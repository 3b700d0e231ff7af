// mcmc_dyn.cu -- the MH ensemble kernel over the dynamic plugins (any
// registered log-density / proposal kind), state padded to MG_DMAX
// coordinates.  Compiled once per MG_DMAX, see csrc/Makefile.
#include "mcmc_kernel.cuh"

#ifndef MG_DMAX
#error "compile with -DMG_DMAX=<max dimension>"
#endif
#define MG_CAT2(a, b) a##b
#define MG_CAT(a, b) MG_CAT2(a, b)

namespace mg {
int MG_CAT(mh_dyn_, MG_DMAX)(mg_ctx *ctx, const DynFnParams &like, const DynFnParams &prior, const DynPropParams &prop,
                             const MhLaunch &L, bool *mom_done) {
  MhArgs<DynFn, DynFn, DynProp, MG_DMAX> a;
  a.like = like; a.prior = prior; a.prop = prop;
  fill_common(a, L);
  return launch_mh(ctx, a, L.mom, mom_done);
}
}  // namespace mg
