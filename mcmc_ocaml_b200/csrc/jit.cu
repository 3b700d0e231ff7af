// jit.cu -- mg_plugin_register_source: user log-densities compiled at run time.
//
// The reference passes OCaml closures for log_likelihood / log_prior
// (mcmc.mli:58-60).  A closure cannot run on the GPU and an indirect device
// call in the step loop would block inlining, so a user function is given as
// CUDA source, and the sampler kernel is RE-COMPILED with it inlined:
// NVRTC compiles a translation unit made of the user functions, a dispatcher
// on their kind ids (MG_USER_EVAL) and this library's own device headers
// (embedded in the .so at build time), producing an sm_100a cubin that is
// loaded with the driver API and launched on the context's stream.
// libnvrtc and libcuda are opened lazily with dlopen, so the library still
// loads (and the CPU-side tests still run) on a machine without a driver.
#include <dlfcn.h>

#include <map>
#include <mutex>
#include <sstream>

#include "common.cuh"
#include "host_plugins.hpp"
#include "mcmc_kernel.cuh"
#include "nested_kernel_dev.cuh"
#include "rj_kernel_dev.cuh"
#include "tempered_kernel_dev.cuh"

#include "build/embedded_headers.inc"

namespace mg {

struct UserFn { std::string name, body; };
static std::mutex g_mu;
static std::vector<UserFn> g_user;  // kind = MG_FN_USER + index, process wide

bool user_kind_registered(int kind) {
  std::lock_guard<std::mutex> lk(g_mu);
  return kind >= MG_FN_USER && kind < MG_FN_USER + (int)g_user.size();
}

// ---- lazily bound NVRTC / driver entry points --------------------------------
typedef int nvrtcResult_t;
typedef struct _nvrtcProgram *nvrtcProgram_t;
typedef int CUresult_t;
typedef struct CUmod_st *CUmodule_t;
typedef struct CUfunc_st *CUfunction_t;
struct Api {
  bool ok = false;
  std::string why;
  nvrtcResult_t (*nvrtcCreateProgram)(nvrtcProgram_t *, const char *, const char *, int, const char *const *, const char *const *);
  nvrtcResult_t (*nvrtcCompileProgram)(nvrtcProgram_t, int, const char *const *);
  nvrtcResult_t (*nvrtcGetProgramLogSize)(nvrtcProgram_t, size_t *);
  nvrtcResult_t (*nvrtcGetProgramLog)(nvrtcProgram_t, char *);
  nvrtcResult_t (*nvrtcGetCUBINSize)(nvrtcProgram_t, size_t *);
  nvrtcResult_t (*nvrtcGetCUBIN)(nvrtcProgram_t, char *);
  nvrtcResult_t (*nvrtcDestroyProgram)(nvrtcProgram_t *);
  CUresult_t (*cuModuleLoadData)(CUmodule_t *, const void *);
  CUresult_t (*cuModuleGetFunction)(CUfunction_t *, CUmodule_t, const char *);
  CUresult_t (*cuLaunchKernel)(CUfunction_t, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void *, void **, void **);
  CUresult_t (*cuFuncSetAttribute)(CUfunction_t, int, int);
};
static Api &api() {
  static Api a;
  static std::once_flag once;
  std::call_once(once, [] {
    void *hn = nullptr;
    for (const char *n : {"libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so"})
      if ((hn = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
    void *hc = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!hn) { a.why = "libnvrtc.so.12 not found"; return; }
    if (!hc) { a.why = "libcuda.so.1 not found"; return; }
#define MG_BIND(h, f) do { *(void **)(&a.f) = dlsym(h, #f); if (!a.f) { a.why = "missing symbol " #f; return; } } while (0)
    MG_BIND(hn, nvrtcCreateProgram); MG_BIND(hn, nvrtcCompileProgram); MG_BIND(hn, nvrtcGetProgramLogSize);
    MG_BIND(hn, nvrtcGetProgramLog); MG_BIND(hn, nvrtcGetCUBINSize); MG_BIND(hn, nvrtcGetCUBIN);
    MG_BIND(hn, nvrtcDestroyProgram);
    MG_BIND(hc, cuModuleLoadData); MG_BIND(hc, cuModuleGetFunction); MG_BIND(hc, cuLaunchKernel);
    MG_BIND(hc, cuFuncSetAttribute);
#undef MG_BIND
    a.ok = true;
  });
  return a;
}

struct JitKey { int device, dmax; size_t version; bool operator<(const JitKey &o) const {
  return device != o.device ? device < o.device : dmax != o.dmax ? dmax < o.dmax : version < o.version; } };
struct JitMod { CUmodule_t mod = nullptr; CUfunction_t mh = nullptr, eval = nullptr, rj = nullptr, nest_init = nullptr, nest_replace = nullptr, tempered = nullptr; };
static std::map<JitKey, JitMod> g_mods;

static const char *kPrelude =
    "typedef signed char int8_t; typedef unsigned char uint8_t; typedef short int16_t; typedef unsigned short uint16_t;\n"
    "typedef int int32_t; typedef unsigned int uint32_t; typedef long long int64_t; typedef unsigned long long uint64_t;\n";

static std::string make_source(const std::vector<UserFn> &fns, int dmax) {
  std::ostringstream s;
  s << kPrelude << "namespace mg_user {\n";
  for (size_t i = 0; i < fns.size(); ++i)
    s << "// " << fns[i].name << "\n__device__ __forceinline__ double fn_" << i
      << "(const double *x, int dim, const double *p, long long np) {\n" << fns[i].body << "\n}\n";
  s << "__device__ __forceinline__ double eval(int kind, const double *x, int dim, const double *p, long long np) {\n"
       "  switch (kind) {\n";
  for (size_t i = 0; i < fns.size(); ++i) s << "    case " << (MG_FN_USER + (int)i) << ": return fn_" << i << "(x, dim, p, np);\n";
  s << "  }\n  return -__longlong_as_double(0x7FF0000000000000ll);\n}\n}  // namespace mg_user\n"
       "#define MG_USER_EVAL(kind, x, d, p, np) mg_user::eval(kind, x, d, p, (long long)(np))\n"
       "#include \"mcmc_kernel_dev.cuh\"\n"
       "extern \"C\" __global__ void __maxnreg__(255) mg_user_mh(const __grid_constant__ mg::MhArgs<mg::DynFn, mg::DynFn, mg::DynProp, "
    << dmax << "> a) {\n  mg::mh_ensemble_body<mg::DynFn, mg::DynFn, mg::DynProp, " << dmax << ">(a);\n}\n"
       "extern \"C\" __global__ void mg_user_eval(mg::DynFnParams f, const double *x, long long M, double *out) {\n"
       "  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;\n  if (i >= M) return;\n"
       "  double v[" << dmax << "];\n  for (int d = 0; d < " << dmax << "; ++d) v[d] = (d < f.dim) ? x[i * f.dim + d] : 0.0;\n"
       "  out[i] = mg::DynFn::eval<" << dmax << ">(f, nullptr, v, f.dim);\n}\n"
       // Mcmc.rjmcmc_array and Nested.nested_evidence with the user functions as log_likelihood / log_prior
       "#include \"rj_kernel_dev.cuh\"\n#include \"nested_kernel_dev.cuh\"\n"
       "extern \"C\" __global__ void __maxnreg__(255) mg_user_rj(const __grid_constant__ mg::RjArgs a) {\n  mg::rj_ensemble_body<" << dmax << ">(a);\n}\n"
       "extern \"C\" __global__ void mg_user_nest_init(mg::NestArgs a, double *x, double *ll, double *lp) {\n"
       "  mg::nest_init_body<" << dmax << ">(a, x, ll, lp);\n}\n"
       "extern \"C\" __global__ void mg_user_nest_replace(mg::NestArgs a, mg::NestProp p, int s0, int s1, int first, int last, double *cx, double *ccl) {\n"
       "  mg::nest_replace_simple_body<" << dmax << ">(a, p, s0, s1, first, last, cx, ccl);\n}\n"
       // the parallel-tempering evidence kernel (tempered.cu) with the user functions as log_likelihood / log_prior
       "#include \"tempered_kernel_dev.cuh\"\n"
       "extern \"C\" __global__ void __maxnreg__(255) mg_user_tempered(const __grid_constant__ mg::TpArgs a) {\n"
       "  mg::tempered_body<" << dmax << ">(a);\n}\n";
  return s.str();
}

static int get_module(mg_ctx *ctx, int dmax, JitMod *out) {
  Api &a = api();
  if (!a.ok) return set_err(ctx, MG_EFAIL, "run-time plugins unavailable: %s", a.why.c_str());
  std::lock_guard<std::mutex> lk(g_mu);
  const JitKey key{ctx->device, dmax, g_user.size()};
  auto it = g_mods.find(key);
  if (it != g_mods.end()) { *out = it->second; return MG_OK; }
  const std::string src = make_source(g_user, dmax);
  nvrtcProgram_t prog = nullptr;
  if (a.nvrtcCreateProgram(&prog, src.c_str(), "mg_user_plugins.cu", kEmbeddedCount, kEmbeddedSources, kEmbeddedNames))
    return set_err(ctx, MG_EFAIL, "nvrtcCreateProgram failed");
  // -default-device: the C declarations of mcmc_gpu.h carry no execution-space annotation
  const char *opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "--fmad=false", "-lineinfo", "-default-device"};
  const nvrtcResult_t rc = a.nvrtcCompileProgram(prog, 5, opts);
  if (rc != 0) {
    size_t n = 0; a.nvrtcGetProgramLogSize(prog, &n);
    std::string log(n + 1, '\0'); a.nvrtcGetProgramLog(prog, &log[0]);
    a.nvrtcDestroyProgram(&prog);
    if (log.size() > 1500) log.resize(1500);
    return set_err(ctx, MG_EINVAL, "plugin source does not compile: %s", log.c_str());
  }
  size_t nb = 0; a.nvrtcGetCUBINSize(prog, &nb);
  std::vector<char> cubin(nb);
  a.nvrtcGetCUBIN(prog, cubin.data());
  a.nvrtcDestroyProgram(&prog);
  JitMod m;
  MG_CUDA(ctx, cudaSetDevice(ctx->device));
  MG_CUDA(ctx, cudaFree(0));  // make sure the primary context is current
  if (a.cuModuleLoadData(&m.mod, cubin.data())) return set_err(ctx, MG_ECUDA, "cuda: cuModuleLoadData failed for the plugin module");
  if (a.cuModuleGetFunction(&m.mh, m.mod, "mg_user_mh") || a.cuModuleGetFunction(&m.eval, m.mod, "mg_user_eval") ||
      a.cuModuleGetFunction(&m.rj, m.mod, "mg_user_rj") || a.cuModuleGetFunction(&m.nest_init, m.mod, "mg_user_nest_init") ||
      a.cuModuleGetFunction(&m.nest_replace, m.mod, "mg_user_nest_replace") ||
      a.cuModuleGetFunction(&m.tempered, m.mod, "mg_user_tempered"))
    return set_err(ctx, MG_ECUDA, "cuda: plugin module lacks its entry points");
  g_mods[key] = m;
  *out = m;
  return MG_OK;
}

static int dmax_for(int D) { return D <= 2 ? 2 : D <= 4 ? 4 : D <= 8 ? 8 : D <= 16 ? 16 : D <= 32 ? 32 : 64; }

// MH ensemble with user-registered log-densities (called from mg_mcmc_array_dev); it keeps no running moments
int jit_launch_mh(mg_ctx *ctx, const DynFnParams &like, const DynFnParams &prior, const DynPropParams &prop, const MhLaunch &L) {
  const int dmax = dmax_for(L.cfg->dim);
  JitMod m;
  int rc = get_module(ctx, dmax, &m);
  if (rc) return rc;
  // MhArgs has the same layout for every DMAX (the template parameter only sizes registers)
  MhArgs<DynFn, DynFn, DynProp, 2> a;
  a.like = like; a.prior = prior; a.prop = prop;
  fill_common(a, L);
  void *params[] = {&a};
  const unsigned grid = (unsigned)((a.C + MH_BLOCK - 1) / MH_BLOCK);
  time_begin(ctx);
  if (api().cuLaunchKernel(m.mh, grid, 1, 1, MH_BLOCK, 1, 1, 0, ctx->stream, params, nullptr))
    return set_err(ctx, MG_ECUDA, "cuda: launch of the plugin sampler kernel failed");
  ctx->launches++;
  time_end(ctx);
  return MG_OK;
}

int jit_logfn_eval(mg_ctx *ctx, const DynFnParams &f, const double *d_x, int64_t M, double *d_out) {
  JitMod m;
  int rc = get_module(ctx, dmax_for(f.dim), &m);
  if (rc) return rc;
  DynFnParams ff = f; long long MM = M;
  void *params[] = {&ff, &d_x, &MM, &d_out};
  if (api().cuLaunchKernel(m.eval, (unsigned)((M + 127) / 128), 1, 1, 128, 1, 1, 0, ctx->stream, params, nullptr))
    return set_err(ctx, MG_ECUDA, "cuda: launch of the plugin evaluation kernel failed");
  ctx->launches++;
  return MG_OK;
}

// Mcmc.rjmcmc_array with user-registered log-densities (called from mg_rjmcmc_array)
int jit_launch_rj(mg_ctx *ctx, const RjArgs &a, int Dm, unsigned grid, unsigned block, size_t smem) {
  JitMod m;
  int rc = get_module(ctx, dmax_for(Dm), &m);
  if (rc) return rc;
  if (smem > 48 * 1024 && api().cuFuncSetAttribute(m.rj, 8 /* MAX_DYNAMIC_SHARED_SIZE_BYTES */, (int)smem))
    return set_err(ctx, MG_ECUDA, "cuda: cannot size the shared memory of the plugin reversible-jump kernel");
  RjArgs aa = a;
  void *params[] = {&aa};
  if (api().cuLaunchKernel(m.rj, grid, 1, 1, block, 1, 1, (unsigned)smem, ctx->stream, params, nullptr))
    return set_err(ctx, MG_ECUDA, "cuda: launch of the plugin reversible-jump kernel failed");
  return MG_OK;
}

// Nested.nested_evidence with user-registered log-densities (called from mg_nested_evidence)
int jit_launch_nest_init(mg_ctx *ctx, int D, const NestArgs &a, double *x_out, double *ll_out, double *lp_out) {
  JitMod m;
  int rc = get_module(ctx, dmax_for(D), &m);
  if (rc) return rc;
  NestArgs aa = a;
  void *params[] = {&aa, &x_out, &ll_out, &lp_out};
  if (api().cuLaunchKernel(m.nest_init, (unsigned)((a.nlive + 127) / 128), 1, 1, 128, 1, 1, 0, ctx->stream, params, nullptr))
    return set_err(ctx, MG_ECUDA, "cuda: launch of the plugin nested-initialisation kernel failed");
  return MG_OK;
}
int jit_launch_nest_replace(mg_ctx *ctx, int D, const NestArgs &a, const NestProp &p, int s0, int s1, int first, int last,
                            double *chain_x, double *chain_cl) {
  JitMod m;
  int rc = get_module(ctx, dmax_for(D), &m);
  if (rc) return rc;
  NestArgs aa = a; NestProp pp = p;
  void *params[] = {&aa, &pp, &s0, &s1, &first, &last, &chain_x, &chain_cl};
  if (api().cuLaunchKernel(m.nest_replace, (unsigned)((a.K + 63) / 64), 1, 1, 64, 1, 1, 0, ctx->stream, params, nullptr))
    return set_err(ctx, MG_ECUDA, "cuda: launch of the plugin nested-replacement kernel failed");
  return MG_OK;
}

// mg_evidence_tempered with user-registered log-densities (called from tempered.cu)
int jit_launch_tempered(mg_ctx *ctx, const TpArgs &a, int D, unsigned grid, unsigned block) {
  JitMod m;
  int rc = get_module(ctx, dmax_for(D), &m);
  if (rc) return rc;
  TpArgs aa = a;
  void *params[] = {&aa};
  if (api().cuLaunchKernel(m.tempered, grid, 1, 1, block, 1, 1, 0, ctx->stream, params, nullptr))
    return set_err(ctx, MG_ECUDA, "cuda: launch of the plugin parallel-tempering kernel failed");
  return MG_OK;
}

}  // namespace mg

using namespace mg;

extern "C" int mg_plugin_register_source(mg_ctx *ctx, const char *name, const char *body, int32_t *kind) {
  if (!ctx) return MG_EINVAL;
  MG_REQUIRE(ctx, name && body && kind, "plugin_register_source: null argument");
  MG_REQUIRE(ctx, strlen(body) > 0 && strlen(body) < (1u << 20), "plugin_register_source: empty or oversized body");
  *kind = -1;
  int k;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    g_user.push_back(UserFn{name, body});
    k = MG_FN_USER + (int)g_user.size() - 1;
  }
  // compile now so that a syntax error is reported at registration, like a type error at the OCaml call site
  JitMod m;
  int rc = get_module(ctx, 2, &m);
  if (rc) {
    std::lock_guard<std::mutex> lk(g_mu);
    g_user.pop_back();
    return rc;
  }
  *kind = k;
  return MG_OK;
}
