// rng.cuh -- counter-based Philox4x32-10 stream for the device (and the host
// side of the library, which needs the call-key derivation).
//
// The reference draws from OCaml's global Random (mcmc.ml:47,
// interpolate_pdf.ml:115, ...).  A global sequential generator cannot feed
// 65,536 chains; the GPU path keys one Philox stream by (seed, epoch) and
// addresses every draw by (purpose, global chain id, step, draw index), so a
// chain's randomness does not depend on how chains are spread over threads,
// blocks or GPUs.  The stream layout is specified in oracle/og_rng.hpp.
#pragma once
#ifndef __CUDACC_RTC__
#include <cstdint>
#endif

namespace mg {

enum Purpose : uint32_t {
  P_MH = 1, P_RJ = 2, P_RJ_INIT = 3, P_DRAW = 4, P_NEST_INIT = 5,
  P_NEST_MCMC = 6, P_NEST_START = 7, P_POST = 8, P_BOOT = 9, P_PT_SWAP = 10
};

#define MG_PHILOX_M0 0xD2511F53u
#define MG_PHILOX_M1 0xCD9E8D57u
#define MG_PHILOX_W0 0x9E3779B9u
#define MG_PHILOX_W1 0xBB67AE85u

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2,
                                                       uint32_t c3, uint32_t k0, uint32_t k1,
                                                       uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    // one IMAD.WIDE per product: hi and lo halves of 32x32 -> 64
    const uint64_t p0 = (uint64_t)MG_PHILOX_M0 * c0;
    const uint64_t p1 = (uint64_t)MG_PHILOX_M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
    k0 += MG_PHILOX_W0; k1 += MG_PHILOX_W1;  // key is warp-uniform: folded by the compiler
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

struct CallKey { uint32_t k0, k1; };

// The ten round keys of a call key (k + r * W): formed once on the host and passed in the kernel argument
// block, so that the step loop does not re-derive them (2 x 9 uniform-datapath adds per Philox batch).
struct RoundKeys { uint32_t k[20]; };
inline RoundKeys make_round_keys(CallKey ck) {
  RoundKeys rk;
  for (int r = 0; r < 10; ++r) { rk.k[2 * r] = ck.k0 + (uint32_t)r * MG_PHILOX_W0; rk.k[2 * r + 1] = ck.k1 + (uint32_t)r * MG_PHILOX_W1; }
  return rk;
}
__device__ __forceinline__ void philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 const RoundKeys &rk, uint32_t (&out)[4]) {
#ifdef MG_EXP_ROUNDS   /* timing experiment only (tools/mh_ablation.sh): fewer rounds, NOT the shipped generator */
  constexpr int kRounds = MG_EXP_ROUNDS;
#else
  constexpr int kRounds = 10;
#endif
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    const uint64_t p0 = (uint64_t)MG_PHILOX_M0 * c0;
    const uint64_t p1 = (uint64_t)MG_PHILOX_M1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ rk.k[2 * r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ rk.k[2 * r + 1];
    c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

inline CallKey derive_key(uint64_t seed, uint64_t epoch) {
  uint32_t w[4];
  philox4x32_10((uint32_t)epoch, (uint32_t)(epoch >> 32), 0x6d636d63u, 0u, (uint32_t)seed,
                (uint32_t)(seed >> 32), w);
  return CallKey{w[0], w[1]};
}

// Sequential cursor over the draws of one (purpose, g, step).  Draws come in groups of 11 from 5 Philox blocks
// (oracle/og_rng.hpp has the specification): draws 0..9 of a group are the two 64-bit lanes of blocks 0..4 (low 20
// bits of the first word : second word), draw 10 is assembled from the 12 top bits of the first words of blocks
// 0..2, which the lane draws leave unused.  A 10-D proposal plus its accept test is one group: 5 blocks per step.
// In unrolled code the cursor is a compile-time constant and the group arithmetic folds away.
struct Rng {
  uint32_t k0, k1, c1, c2, c3;
  uint32_t w[4];
  uint32_t j;
  uint32_t spA, spB, spC;   // spare bits of the group's blocks 0, 1, 2: (s0 << 12 | s1), (s2 << 12 | s3), s4
  const RoundKeys *rk;   // optional precomputed round keys (kernel argument block)
  __device__ __forceinline__ Rng(CallKey ck, uint32_t purpose, uint64_t g, uint64_t step, const RoundKeys *rk_ = nullptr)
      : k0(ck.k0), k1(ck.k1), c1((uint32_t)step), c2((uint32_t)g),
        c3((uint32_t)((g >> 32) & 0xFFFFu) | ((purpose & 0xFFu) << 16) |
           (uint32_t)(((step >> 32) & 0xFFu) << 24)),
        j(0), spA(0), spB(0), spC(0), rk(rk_) {}
  __device__ __forceinline__ void gen(uint32_t blk) {
    if (rk) philox4x32_10_rk(blk, c1, c2, c3, *rk, w); else philox4x32_10(blk, c1, c2, c3, k0, k1, w);
  }
  // (high 20 bits, low 32 bits) of the next draw's 52 private bits
  __device__ __forceinline__ void next52(uint32_t &hi20, uint32_t &lo32) {
    const uint32_t m = j / 11u, i = j - 11u * m;
    if (i < 10u) {
      if ((i & 1u) == 0u) {
        const uint32_t gi = i >> 1;
        gen(5u * m + gi);
        if (gi == 0u) spA = ((w[0] >> 20) << 12) | (w[2] >> 20);
        else if (gi == 1u) spB = ((w[0] >> 20) << 12) | (w[2] >> 20);
        else if (gi == 2u) spC = w[0] >> 20;
      }
      hi20 = ((i & 1u) ? w[2] : w[0]) & 0xFFFFFu;
      lo32 = (i & 1u) ? w[3] : w[1];
    } else {
      hi20 = spA >> 4;
      lo32 = (spA << 28) | (spB << 4) | (spC >> 8);
    }
    ++j;
  }
  // the draw as a 64-bit word with its 52 bits on top (what Random.int multiplies)
  __device__ __forceinline__ uint64_t lane() {
    uint32_t h, l; next52(h, l);
    return (((uint64_t)h << 32) | l) << 12;
  }
  // Random.float 1.0: 52 random mantissa bits, [0, 1)
  __device__ __forceinline__ double uniform12() {  // 1 + Random.float 1.0, in [1, 2)
    uint32_t h, l; next52(h, l);
    return __hiloint2double((int)(h | 0x3FF00000u), (int)l);
  }
  __device__ __forceinline__ double uniform() { return uniform12() - 1.0; }
  // Random.int n
  __device__ __forceinline__ uint64_t below(uint64_t n) { return __umul64hi(lane(), n); }
};

// Acceptance test  log u < delta  (mcmc.ml:47, strict), decided exactly as the
// float64 comparison would decide it, but without the float64 logarithm in all
// but ~1e-5 of the calls: a single-precision estimate of log u (F2F + MUFU.LG2)
// settles the comparison whenever it is further from delta than a rigorous
// error bound; the rest take the float64 path.
//   |(float)u - u| <= 2^-24 u for u > 1e-30 -> log error <= 6e-8;  __logf: <= 2^-21.41
//   absolute on [0.5, 2], 3 ulp elsewhere -> <= 3.6e-7 (1 + |log u|);  (float)delta and the float subtraction add
//   <= 1.2e-7 (|log u| + |delta|).  Total < 1e-6 (1 + |lf| + |df|); the tolerance used is ten times that.
// u = 0, u < 1e-30, NaN or infinite-minus-infinite cases fail both comparisons and take the exact path.
#ifndef MG_ACCEPT_PREFILTER
#define MG_ACCEPT_PREFILTER 1
#endif
__device__ __forceinline__ bool log_u_less_than(double u, double delta) {
#if MG_ACCEPT_PREFILTER
  const float uf = __double2float_rn(u);
  const float lf = __logf(uf);
  const float df = __double2float_rn(delta);
  const float d = lf - df;
  const float tol = 1e-5f * (1.0f + fabsf(lf) + fabsf(df));
  if (uf > 1e-30f && fabsf(d) > tol) return d < 0.0f;
#endif
  return log(u) < delta;
}

// N draws of one (purpose, g, step) generated up front: lets the sampler issue
// the Philox rounds of step t+1 among the float64 work of step t.
template <int N>
struct RngBuf {
  double u[N];
  int j;
  __device__ __forceinline__ RngBuf() : j(0) {}
  __device__ __forceinline__ void fill(CallKey ck, uint32_t purpose, uint64_t g, uint64_t step) {
    Rng r(ck, purpose, g, step);
#pragma unroll
    for (int k = 0; k < N; ++k) u[k] = r.uniform();
    j = 0;
  }
  __device__ __forceinline__ double uniform() { return u[j++]; }
  __device__ __forceinline__ double uniform12() { return u[j++] + 1.0; }
};

}  // namespace mg
