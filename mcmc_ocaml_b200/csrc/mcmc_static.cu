// mcmc_static.cu -- one instantiation of the MH ensemble kernel with
// compile-time dimension MG_SD: GAUSS_CORR likelihood, flat prior, box
// proposal, all parameters in the kernel argument block (constant bank).
// Compiled once per dimension (-DMG_SD=<D>), see csrc/Makefile.
#include "mcmc_kernel.cuh"

#include <cstdlib>

#ifndef MG_SD
#error "compile with -DMG_SD=<dimension>"
#endif
#define MG_CAT2(a, b) a##b
#define MG_CAT(a, b) MG_CAT2(a, b)

namespace mg {
int MG_CAT(mh_static_gauss_, MG_SD)(mg_ctx *ctx, const mg_logfn *like, const mg_proposal *prop, const MhLaunch &L,
                                    bool *mom_done) {
  constexpr int D = MG_SD;
  MhArgs<GaussCorr<D>, ZeroFn, BoxProp<D>, D> a;
  GaussCorr<D>::pack(like->params, like->params + D, like->params[D + D * (D + 1) / 2], a.like);
  BoxProp<D>::pack(prop->params, a.prop);
  fill_common(a, L);
  return launch_mh(ctx, a, L.mom, mom_done);
}
}  // namespace mg
