// mcmc_balanced.cuh -- the Metropolis-Hastings ensemble kernel with the chain
// groups handed out dynamically, so that every warp scheduler of the GPU
// carries the same load.
//
// Why: the step is issue-bound, and one scheduler saturates at three resident
// warps (measured, tools/occupancy_sweep.sh: 56,832 chains = 3 warps on each
// of the 592 schedulers run at 4.27e10 chain-steps/s, 75,776 = 4 warps at
// 4.31e10).  An ensemble whose warps do not divide evenly over the schedulers
// -- config 2: 65,536 chains = 2,048 warps = 3.46 per scheduler -- then runs at
// the pace of the schedulers that hold four (17.5 ms/pass where 15.2 ms would
// do).  Chains cannot be split, but their runs can be cut in time: a task is
// (group of 32 chains, segment of ~128 steps).  A persistent grid of one-warp
// CTAs fills every warp slot of the machine; each warp takes a ticket, waits
// for that ticket's entry in a ring of ready groups, runs the segment with the
// state in registers, writes the state back and pushes the group for its next
// segment.  Tickets are served first-in first-out, so idleness rotates over
// all warps and every scheduler sees the same mean number of busy warps.
// The chains themselves do not change: the random stream of a step depends on
// (chain, step) only, so results are bit-identical to the static kernel.
//
// Progress: ticket k waits for the k-th push; pushes come from segments of
// lower tickets, which are held by running warps and never wait once started,
// so the scheme cannot deadlock even if part of the grid is not resident.
// Every wait is bounded (clock64 budget).  Running out of it does NOT trap (a trap poisons the CUDA context of the
// whole process): the warp writes MG_DEVERR_MH_QUEUE into the context's device error word and leaves; every other
// waiter polls that word and leaves too, and the host reports MG_ECUDA for the call (common.cuh poll_device_error).
#pragma once
#include <cuda.h>   // CUtensorMap (the encoder itself is fetched from the driver at run time, mcmc_kernel.cuh)

#include "mcmc_kernel_dev.cuh"

namespace mg {

// ---- recorded samples through the TMA ------------------------------------------------------------------------------
// Recording a sample with plain stores costs ~45 instructions (12 STG.64 and their 64-bit address arithmetic) on a
// kernel that is bound by instruction issue.  With kTma the warp instead parks its D + 2 fields in shared memory
// (one STS.64 with an immediate offset per field) and, every kTmaSteps recorded samples, ONE elected lane hands the
// [kTmaSteps][D + 2][32 chains] tile to the TMA as a 3-D bulk tensor store (cp.async.bulk.tensor.3d, UTMASTG in SASS)
// into the [n][D + 2][C] block; the box is clipped by the hardware at the ragged last group.  The tile is written
// again only ~kTmaSteps steps later, so the wait for the TMA to have READ it (wait_group.read) never stalls.
constexpr int kTmaSteps = 4;
__device__ __forceinline__ void tma_store_3d(const CUtensorMap *tm, uint32_t smem_addr, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
               :: "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_addr) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Register cap of the balanced kernel: its grid holds exactly three one-warp CTAs per scheduler, which leaves room for
// 170 registers; tools/mh_maxnreg_sweep.sh (D = 10, ms per pass on one box): 128: 15.49, 136: 15.33, 144: 15.21,
// 152: 15.26-15.40, 160: 15.03-15.19, 168: 15.24-15.33.
#ifndef MG_MHB_MAXNREG
#define MG_MHB_MAXNREG(D) ((D) <= 10 ? 160 : MG_MH_MAXNREG(D))
#endif
#ifndef MG_MHB_MOM_MAXNREG
#define MG_MHB_MOM_MAXNREG(D) ((D) <= 10 ? 168 : 255)
#endif

struct MhQueue {
  unsigned long long *ring;  // [cap]: (ticket + 1) << 32 | group; 0 = empty
  unsigned int *ctr;         // [0] next pop ticket, [1] next push ticket
  int32_t *seg_next;         // [ngroups] next segment of each group
  uint32_t cap;              // power of two >= 2 * ngroups
  uint32_t ngroups;
  uint32_t total;            // ngroups * nseg tickets
  int32_t nseg;              // nseg_burn + nseg_rec
  int32_t nseg_burn;         // segments of seg_steps burn-in steps (the last one records slot 0)
  int64_t seg_steps;         // steps per burn-in segment
  int64_t seg_slots;         // recorded samples per sampling segment (nskip steps each)
  long long wait_cycles;     // budget of one wait (kQueueWaitCycles; MCMC_GPU_WAIT_CYCLES overrides it for the tests)
  int *err;                  // mg_ctx::d_devflag
};

constexpr int kDevErrMhQueue = 1;   // = MG_DEVERR_MH_QUEUE (common.cuh; checked where both are visible, mcmc_kernel.cuh)
constexpr long long kQueueWaitCycles = 1ll << 38;  // ~2 min at 2 GHz: far beyond any segment (a heavy data likelihood can take seconds), still finite

static __global__ void mh_queue_init_kernel(MhQueue q) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < q.cap) q.ring[i] = (i < q.ngroups) ? (((unsigned long long)(i + 1u) << 32) | i) : 0ull;
  if (i < q.ngroups) q.seg_next[i] = 0;
  if (i == 0) { q.ctr[0] = 0u; q.ctr[1] = q.ngroups; }
}

// kMom: also accumulate, per chain, sum (v - pivot) and sum (v - pivot)^2 of every recorded field value, pivot =
// the chain's own slot-0 sample -- Stats.multi_mean / multi_std of the block without reading the block back
// (the finishing kernel pools the chains with the parallel-variance formula, stats.cu).  The accumulators live in
// registers (three warps per scheduler leave room for 168), the pivots in shared memory.
template <class Like, class Prior, class Prop, int D, bool kMom, bool kTma = false>
__global__ void __maxnreg__(kMom ? MG_MHB_MOM_MAXNREG(D) : MG_MHB_MAXNREG(D))
mh_balanced_kernel(const __grid_constant__ MhArgs<Like, Prior, Prop, D> a, const __grid_constant__ MhQueue q,
                   const __grid_constant__ CUtensorMap tmap) {
  static_assert(MH_BLOCK == 32, "one warp per CTA");
  __shared__ __align__(128) double s_tile[kTma ? kTmaSteps * (D + 2) * MH_BLOCK : 1];   // [step][field][lane]
  const int dd = Prop::kStaticDim ? D : a.d;
  const int F = dd + 2;
  const int64_t C = a.C;
  __shared__ __align__(16) double smem_params[Like::kSmem + Prior::kSmem + Prop::kSmem + 2];
  double *sl = smem_params, *sp = sl + Like::kSmem, *sj = sp + Prior::kSmem;
  if (Like::kSmem + Prior::kSmem + Prop::kSmem > 0) {
    const double *gl = reinterpret_cast<const double *>(&a.like);
    const double *gp = reinterpret_cast<const double *>(&a.prior);
    const double *gj = reinterpret_cast<const double *>(&a.prop);
    for (int k = threadIdx.x; k < Like::kSmem; k += MH_BLOCK) sl[k] = gl[k];
    for (int k = threadIdx.x; k < Prior::kSmem; k += MH_BLOCK) sp[k] = gp[k];
    for (int k = threadIdx.x; k < Prop::kSmem; k += MH_BLOCK) sj[k] = gj[k];
    __syncwarp();
  }
  const unsigned lane = threadIdx.x;
  const int64_t sample_stride = (int64_t)F * C;
  const uint32_t pitch32 = sample_pitch32(C, F);
  __shared__ double s_piv[kMom ? (D + 2) * MH_BLOCK : 1];   // [field][lane]
  for (;;) {
    // ---- take a ticket and wait for its group
    unsigned long long e = 0ull;
    if (lane == 0) {
      const unsigned ticket = atomicAdd(&q.ctr[0], 1u);
      if (ticket >= q.total) {
        e = ~0ull;
      } else {
        volatile unsigned long long *slot = q.ring + (ticket & (q.cap - 1u));
        const unsigned long long want = (unsigned long long)ticket + 1ull;
        const long long t_begin = clock64();
        unsigned ns = 64;
        for (;;) {
          e = *slot;
          if ((e >> 32) == want) break;
          __nanosleep(ns);
          if (ns < 2048) ns *= 2;
          if (clock64() - t_begin > q.wait_cycles) atomicExch(q.err, kDevErrMhQueue);
          if (*reinterpret_cast<volatile int *>(q.err) != 0) { e = ~0ull; break; }   // someone timed out: everybody leaves
        }
        if (e != ~0ull) *slot = 0ull;
        __threadfence();
      }
    }
    e = __shfl_sync(0xffffffffu, e, 0);
    if (e == ~0ull) break;
    const uint32_t grp = (uint32_t)e;
    int64_t c = (int64_t)grp * MH_BLOCK + lane;
    const bool live = c < C;
    if (!live) c = C - 1;
    const uint64_t g = a.chain_offset + (uint64_t)c;
    const int32_t k = __ldcg(q.seg_next + grp);

    // ---- state into registers
    double x[D];
#pragma unroll
    for (int i = 0; i < D; ++i) x[i] = (i < dd) ? __ldcg(a.state + (int64_t)i * C + c) : 0.0;
    double ll, lp;
    if (k == 0) {  // mcmc.ml:59-61: the start point is evaluated, not trusted
      ll = Like::template eval<D>(a.like, sl, x, dd);
      lp = Prior::template eval<D>(a.prior, sp, x, dd);
    } else {
      ll = __ldcg(a.state + (int64_t)dd * C + c);
      lp = __ldcg(a.state + (int64_t)(dd + 1) * C + c);
    }
    // slot j of the output holds the state after nbin + j * nskip steps (mcmc.ml:63-71); a continuation launch
    // (record_first == 0) owns slots 1.. only and its block starts at slot 1
    double *out = (a.samples && live) ? a.samples + c - (a.record_first ? 0 : sample_stride) : nullptr;
    double m1[kMom ? D + 2 : 1], m2[kMom ? D + 2 : 1];
    if (kMom) {
#pragma unroll
      for (int i = 0; i < D + 2; ++i) {
        const bool on = i < dd + 2;
        s_piv[i * MH_BLOCK + lane] = on ? __ldcg(a.mom + (int64_t)i * C + c) : 0.0;
        m1[i] = on ? __ldcg(a.mom + (int64_t)(F + i) * C + c) : 0.0;
        m2[i] = on ? __ldcg(a.mom + (int64_t)(2 * F + i) * C + c) : 0.0;
      }
    }
    auto accumulate = [&](int i, double v, bool first) {
      if (first) s_piv[i * MH_BLOCK + lane] = v;            // slot 0 is the pivot (deviation 0)
      const double dv = v - s_piv[i * MH_BLOCK + lane];
      m1[i] = m1[i] + dv;
      m2[i] = fma(dv, dv, m2[i]);
    };
    int pend = 0;                       // samples parked in the tile
    bool tile_in_flight = false;        // the TMA may still be reading the tile
    int64_t tile_slot = 0;              // output slot of the tile's first sample
    auto flush_tile = [&]() {           // kTmaSteps samples of 32 chains: one bulk tensor store by one lane
      fence_proxy_async_smem();         // the generic-proxy writes of every lane, before the async proxy reads them
      __syncwarp();
      if (lane == 0) tma_store_3d(&tmap, (uint32_t)__cvta_generic_to_shared(s_tile), (int)(grp * MH_BLOCK), 0, (int)tile_slot);
      tile_slot += kTmaSteps; pend = 0; tile_in_flight = true;
    };
    auto record = [&](bool first) {
      if (kTma && !first) {              // (the launcher selects kTma only with a sample block)
        if (pend == 0 && tile_in_flight) { if (lane == 0) tma_wait_read(); __syncwarp(); tile_in_flight = false; }
        double *tp = s_tile + (size_t)pend * F * MH_BLOCK + lane;
#pragma unroll
        for (int i = 0; i < D; ++i)
          if (i < dd) tp[i * MH_BLOCK] = x[i];
        tp[dd * MH_BLOCK] = ll; tp[(dd + 1) * MH_BLOCK] = lp;
        if (++pend == kTmaSteps) flush_tile();
      } else if (out) {
        store_sample<D>(out, pitch32, C, dd, x, ll, lp);
        out += sample_stride;
      }
      if (kMom) {
#pragma unroll
        for (int i = 0; i < D; ++i)
          if (i < dd) accumulate(i, x[i], first);
        accumulate(dd, ll, first);
        accumulate(dd + 1, lp, first);
      }
    };
    int nacc = 0;
    uint64_t t;
    if (k < q.nseg_burn) {  // :63-65 burn-in, nothing recorded until its last step
      const int64_t s0 = (int64_t)k * q.seg_steps;
      const int64_t s1 = (s0 + q.seg_steps < a.nbin) ? s0 + q.seg_steps : a.nbin;
      t = a.t0 + (uint64_t)s0;
      for (int64_t s = s0; s < s1; ++s, ++t) {
        Rng r(a.key, P_MH, g, t, &a.rk);
        nacc += mh_step<Like, Prior, Prop, D>(a, sl, sp, sj, r, x, ll, lp);
      }
      if (s1 == a.nbin && a.n > 0 && a.record_first) record(true);  // :66 slot 0
    } else {                // :67-71 nskip steps, then a sample
      const int64_t j = k - q.nseg_burn;
      const int64_t slot0 = 1 + j * q.seg_slots;
      const int64_t slot1 = (slot0 + q.seg_slots < a.n) ? slot0 + q.seg_slots : a.n;
      if (a.nbin == 0 && j == 0 && a.n > 0 && a.record_first) record(true);  // no burn-in: slot 0 is the start point
      if (out) out = a.samples + c + (slot0 - (a.record_first ? 0 : 1)) * sample_stride;
      tile_slot = slot0 - (a.record_first ? 0 : 1);
      t = a.t0 + (uint64_t)(a.nbin + (slot0 - 1) * a.nskip);
      for (int64_t slot = slot0; slot < slot1; ++slot) {
        for (int64_t kk = 0; kk < a.nskip; ++kk, ++t) {
          Rng r(a.key, P_MH, g, t, &a.rk);
          nacc += mh_step<Like, Prior, Prop, D>(a, sl, sp, sj, r, x, ll, lp);
        }
        record(false);
      }
      if (kTma) {
        if (pend > 0) {                 // a ragged tail (fewer than kTmaSteps samples left in the segment): plain stores
          __syncwarp();
          if (live) {
            double *o = a.samples + c + tile_slot * sample_stride;
            for (int sft = 0; sft < pend; ++sft, o += sample_stride)
              for (int i = 0; i < F; ++i) __stcs(o + (int64_t)i * C, s_tile[((size_t)sft * F + i) * MH_BLOCK + lane]);
          }
          __syncwarp();
          pend = 0;
        }
        if (lane == 0) tma_wait_all();  // the group's next segment may run anywhere: its stores must follow these
        __syncwarp();
        tile_in_flight = false;
      }
    }

    // ---- state back, group released for its next segment
    if (live) {
#pragma unroll
      for (int i = 0; i < D; ++i)
        if (i < dd) a.state[(int64_t)i * C + c] = x[i];
      a.state[(int64_t)dd * C + c] = ll;
      a.state[(int64_t)(dd + 1) * C + c] = lp;
      if (a.accept && nacc) atomicAdd(a.accept + c, nacc);
      if (kMom) {
#pragma unroll
        for (int i = 0; i < D + 2; ++i)
          if (i < dd + 2) {
            a.mom[(int64_t)i * C + c] = s_piv[i * MH_BLOCK + lane];
            a.mom[(int64_t)(F + i) * C + c] = m1[i];
            a.mom[(int64_t)(2 * F + i) * C + c] = m2[i];
          }
      }
    }
    __threadfence();
    __syncwarp();
    if (lane == 0 && k + 1 < q.nseg) {
      q.seg_next[grp] = k + 1;
      __threadfence();
      const unsigned t2 = atomicAdd(&q.ctr[1], 1u);
      volatile unsigned long long *slot2 = q.ring + (t2 & (q.cap - 1u));
      const long long t_begin = clock64();
      bool ok = true;
      while (*slot2 != 0ull) {
        __nanosleep(64);
        if (clock64() - t_begin > q.wait_cycles) atomicExch(q.err, kDevErrMhQueue);
        if (*reinterpret_cast<volatile int *>(q.err) != 0) { ok = false; break; }
      }
      if (ok) *slot2 = (((unsigned long long)t2 + 1ull) << 32) | grp;
    }
    __syncwarp();
  }
}

}  // namespace mg
