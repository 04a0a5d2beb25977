// gram_fused.cuh -- fused regressor -> normal equations, one persistent warp-specialised kernel per GPU.
//
//   G (+)= sum_s Phi_s^T Phi_s ,  b (+)= sum_s Phi_s^T tau_s ,  tau_sq (+)= sum_s tau_s^T tau_s
//
// Phi never touches HBM.  The kernel runs on the FOLDED chain (fold.cpp: joints that never move are merged into the constant
// transform of the next moving joint, so every joint of the chain the kernel sees is an input and owns a row of Phi).  Per CTA (1 per SM):
//   * generator warps (one per shared-memory slot): one thread walks the chain of one sample (same link-frame recursion as dyn_kernel,
//     kernels.cu) and writes the augmented regressor rows [Phi_row | tau_row] of its 32 samples into its slot (only the structurally
//     non-zero columns, XOR-swizzled, conflict free).  The inputs of the next group are requested BEFORE waiting for the slot, so the DRAM
//     latency hides behind the consumers; sin/cos of all joints are evaluated up front (branch free), so the walk is one basic block.
//   * MMA warps: consume a slot as soon as it is full.  The contraction index k = (sample, joint row); a k-step is 4 samples of one joint
//     row, so the zero pattern of Phi (row of chain joint j is zero in the blocks of the links before j) is known at compile time and whole
//     8x8 tiles are skipped; inside the kernel the columns run tau, last link ... first link, so that every row is a PREFIX of tiles.  The upper-triangular tiles of the (P+1)x(P+1) augmented Gram matrix stay in registers for the whole kernel; the four SM
//     sub-partitions split the k-steps of a slot, GF_TSPLIT warps per sub-partition split the tile rows by parity.  The k-steps of a slot
//     are fully unrolled and software pipelined: the fragments of step n+1 are loaded while the DMMAs of step n issue.
//     tcgen05 has no f64 kind: the FP64 tensor path of sm_100a is mma.sync.m8n8k4.f64 (SASS DMMA).
//   * slots cycle through shared-memory mbarriers (full / empty per slot); as many slots as fit the 227 KB (3 for 7 joints, 4 below).  Chains
//     with only 3 slots still run 4 generator warps, one per SM sub-partition, over them (monotone counters instead of the one-bit mbarrier
//     phase: the writer of a slot changes from use to use).
//   * all-revolute chains drop the columns their walk makes exact zeros (GramGeom Z = 2): m and m c_z of a link on its own joint, and all
//     but I_zz, m c_x, m c_y of the first moving link; tau is no tile column but is accumulated by DFMA on the fragments the MMA warps load
//     anyway (b = Phi^T tau for the tile rows a warp owns, tau^T tau in one warp per k-split): 81 instead of 104 DMMA per 4 samples for 6
//     joints (125 / 149 for 7), plus 32 (42) DFMA.  The extended model keeps Z = 1 (only the own-joint mass dropped, tau in the tiles).
//   * all-revolute chains whose folded axes are all e_z (fold.cpp puts every revolute link in such a canonical frame) run the REV generator,
//     which holds the axis as a compile-time constant: 2 019 instead of 2 412 FP64 instructions per sample for 6 joints (2 658 / 3 119 for 7).
//   * on such chains the launchers run the same kernel compiled at run time against the chain's own constants (gram_jit.cpp, model type M):
//     the products with exact zeros and ones are not issued, 1 347 FP64 instructions per sample for C6 (1 851 for C7), same results.
// Per-CTA partials (tiles, then b and tau^T tau) are summed in a fixed order by gram_fused_reduce_kernel (bit-reproducible for a given n).
// gram_ext_kernel: the extended model [Phi | Phi_c] (friction / spring columns) in ONE pass -- the same slots, the component columns of
// every joint in a small side buffer next to each slot, the MMA warps keep the rigid-body tiles and the cross tiles in registers.
//
// What bounds it (round 2: profiles/r02_micro_datapath_sharing.txt, tools/micro/dfma_halfwarp.cu): DMMA and DFMA share ONE FP64 datapath per
// sub-partition; a DMMA holds it for 16 cycles, a DFMA for 2.  With the two MMA warps of a sub-partition active the generator warp there gets
// NOTHING (measured: DMMA 99 %, DFMA 0.1 % of the datapath; with one DMMA warp the DFMA warp gets 15 %), so generation happens in the gaps
// where the MMA warps wait, and a lone generator warp keeps the datapath ~45 % busy (a third of its instructions are not FP64).  Generation
// alone takes 4.9 ms per 16 M samples, the MMAs alone 6.3 ms, together 9.2 ms (C6).  More generator warps need more samples in flight than
// the shared memory holds; decoupling them through an L2-resident ring was built and measured slower (tools/experiments/README.md).
// Measured slower / no gain and removed: one MMA warp per sub-partition with 254 registers (1.72 vs 1.75 G samples/s), fragments two k-steps
// ahead (no change), row groups split over several generator warps (instruction-cache misses), two lanes per sample, per-row slot release, an
// uneven k-split between the sub-partitions, the ragged row tails by DFMA instead of padded tiles (78 instead of 98 DMMA per 4 samples buy
// 0.5 %: the kernel follows the generator warp, not the tensor work), a register re-partition between the roles (setmaxnreg), paced MMA
// warps, generator warps with the lowest warp ids, an L2 prefetch of the generator's next group.
// The kernel templates live in this header so that gram_jit.cpp can instantiate them at run time, with NVRTC, against the constants of one
// chain (gram_common.cuh: compile-time models); gram_fused.cu holds the precompiled instantiations and the launchers.
#pragma once
#include "gram_common.cuh"

namespace rdb
{

// ---------------------------------------------------------------------------------------------- MMA side
// B fragments of one k-step (4 samples of joint row J, k-step kk of the slot): lane (g, t) holds column 8 I + g of sample 4 kk + t in b[I],
// and (GramGeom::TC == 0) the tau of joint J for that sample in b[T]
template <int NJ, int J, int X = 0, int Z = 0>
__device__ __forceinline__ void gram_load_frags(const double* __restrict__ slot, int kk, int lane, double (&b)[GramGeom<NJ, 0, Z>::NF])
{
  using G = GramGeom<NJ, X, Z>;
  constexpr int T = G::T, L = G::rowlen(J), TJ = G::tj(J);
  const int g = lane >> 2, t = lane & 3;
  const double* rowp = slot + G::rowbase(J) + ((4 * kk + t) ^ (4 * (g & 3)));
#pragma unroll
  for (int I = 0; I < T; I++)
  {
    if (I >= TJ) continue;
    const int col = 8 * I + g;
    if (8 * I + 7 < L || col < L) b[I] = rowp[col * 32];  // only the last tile of the row can be ragged
    else b[I] = 0.0;
  }
  if constexpr (!G::TC) b[T] = slot[G::taubase(J) + 4 * kk + t];
}
template <int NJ, int PAR, int J, int Z>
__device__ __forceinline__ void gram_mma_step(const double (&b)[GramGeom<NJ, 0, Z>::NF], double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2])
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int T = G::T, TJ = G::tj(J);
#pragma unroll
  for (int I = 0; I < T; I++)
  {
    if (I >= TJ || !G::owns(I, GF_TS, PAR)) continue;
#pragma unroll
    for (int K = I; K < T; K++)
      if (K < TJ) dmma884f(acc[G::local(I, K, GF_TS, PAR)][0], acc[G::local(I, K, GF_TS, PAR)][1], b[I], b[K]);
  }
}
// TC == 0: Phi^T tau on the tile rows this warp owns and (par 0) tau^T tau, by DFMA on the fragments of the step's DMMAs
template <int NJ, int PAR, int J, int Z>
__device__ __forceinline__ void gram_tau_step(const double (&b)[GramGeom<NJ, 0, Z>::NF], double (&bacc)[GramGeom<NJ, 0, Z>::nbacc(GF_TS, PAR)])
{
  using G = GramGeom<NJ, 0, Z>;
  if constexpr (!G::TC)
  {
    static_for<0, G::tj(J)>([&](auto Ic) {
      constexpr int I = decltype(Ic)::value;
      if constexpr (G::owns(I, GF_TS, PAR)) bacc[G::bown(I, GF_TS, PAR)] = fma(b[I], b[G::T], bacc[G::bown(I, GF_TS, PAR)]);
    });
    if constexpr (PAR == 0) bacc[G::nbacc(GF_TS, PAR) - 1] = fma(b[G::T], b[G::T], bacc[G::nbacc(GF_TS, PAR) - 1]);
  }
}
// k-steps STEP.. of this warp in one slot; step = (joint row, k-step of the warp); the fragments of the next step are in flight while the
// DMMAs of the current one issue
template <int NJ, int PAR, int STEP, int Z>
__device__ __forceinline__ void gram_consume_steps(const double* __restrict__ slot, int ks, int lane, const double (&bcur)[GramGeom<NJ, 0, Z>::NF],
                                                   double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2],
                                                   double (&bacc)[GramGeom<NJ, 0, Z>::nbacc(GF_TS, PAR)])
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int J = STEP / G::KPW;
  if constexpr (STEP + 1 < G::NSTEPS)
  {
    double bnext[G::NF];
    gram_load_frags<NJ, (STEP + 1) / G::KPW, 0, Z>(slot, ks * G::KPW + (STEP + 1) % G::KPW, lane, bnext);
    gram_mma_step<NJ, PAR, J, Z>(bcur, acc);
    gram_tau_step<NJ, PAR, J, Z>(bcur, bacc);
    gram_consume_steps<NJ, PAR, STEP + 1, Z>(slot, ks, lane, bnext, acc, bacc);
  }
  else
  {
    gram_mma_step<NJ, PAR, J, Z>(bcur, acc);
    gram_tau_step<NJ, PAR, J, Z>(bcur, bacc);
  }
}
// the k-steps of one slot for this warp
template <int NJ, int PAR, int Z>
__device__ __forceinline__ void gram_consume_slot(const double* __restrict__ slot, int ks, int lane,
                                                  double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2],
                                                  double (&bacc)[GramGeom<NJ, 0, Z>::nbacc(GF_TS, PAR)])
{
  using G = GramGeom<NJ, 0, Z>;
  double b0[G::NF];
  gram_load_frags<NJ, 0, 0, Z>(slot, ks * G::KPW, lane, b0);
  gram_consume_steps<NJ, PAR, 0, Z>(slot, ks, lane, b0, acc, bacc);
}

#ifndef GF_SPIN_NS
#define GF_SPIN_NS 32  // back-off of the counter polls
#endif
struct GramBars
{
  uint64_t full[GF_MAX_SLOTS], empty[GF_MAX_SLOTS];
  // GENS != SLOTS (more generator warps than slots, e.g. 4 over the 3 slots of a 7-joint chain): the writer of a slot changes from use to use,
  // so a waiter can be more than one phase behind and the one-bit phase parity of an mbarrier is ambiguous; monotone counters instead
  uint32_t filled[GF_MAX_SLOTS];   // uses of the slot written so far (generator, release)
  uint32_t drained[GF_MAX_SLOTS];  // MMA-warp completions on the slot so far (GF_MMA_WARPS per use, release)
};
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p)
{
  uint32_t v;
  asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v)
{
  asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void red_release_inc(uint32_t* p)
{
  asm volatile("red.release.cta.shared.add.u32 [%0], 1;" ::"r"(smem_u32(p)) : "memory");
}
__device__ __forceinline__ void wait_counter_ge(const uint32_t* p, uint32_t v)
{
  while (ld_acquire_u32(p) < v) __nanosleep(GF_SPIN_NS);
}

// fixed-order reduction over the k-split warps that own the same tiles, into shared memory (the slots are dead by now)
template <int NJ, int PAR, int Z>
__device__ __forceinline__ void gram_mma_reduce(double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2], double* smem, int ks, int lane)
{
  using G = GramGeom<NJ, 0, Z>;
  bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  const int g = lane >> 2, t = lane & 3;
  for (int w = 0; w < GF_KSPLIT; w++)
  {
    if (ks == w)
    {
#pragma unroll
      for (int I = 0; I < G::T; I++)
      {
        if (!G::owns(I, GF_TS, PAR)) continue;
#pragma unroll
        for (int J = I; J < G::T; J++)
        {
          double* o = smem + G::tile(I, J) * 64 + g * 8 + 2 * t;
          const int k = G::local(I, J, GF_TS, PAR);
          if (w == 0)
          {
            o[0] = acc[k][0];
            o[1] = acc[k][1];
          }
          else
          {
            o[0] += acc[k][0];
            o[1] += acc[k][1];
          }
        }
      }
    }
    bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  }
}
// TC == 0: b (8 T doubles by position) and tau^T tau behind the tiles in shared memory, in a fixed order: the four lanes t of a position
// first, then the k-split warps
template <int NJ, int PAR, int Z>
__device__ __forceinline__ void gram_tau_reduce(double (&bacc)[GramGeom<NJ, 0, Z>::nbacc(GF_TS, PAR)], double* smem, int ks, int lane)
{
  using G = GramGeom<NJ, 0, Z>;
  if constexpr (!G::TC)
  {
    constexpr int NB = G::nbacc(GF_TS, PAR);
#pragma unroll
    for (int k = 0; k < NB; k++)
    {
      bacc[k] += __shfl_xor_sync(0xffffffffu, bacc[k], 1);
      bacc[k] += __shfl_xor_sync(0xffffffffu, bacc[k], 2);
    }
    const int g = lane >> 2, t = lane & 3;
    double* ob = smem + G::NT * 64;
    for (int w = 0; w < GF_KSPLIT; w++)
    {
      if (ks == w && t == 0)
      {
#pragma unroll
        for (int I = 0; I < G::T; I++)
        {
          if (!G::owns(I, GF_TS, PAR)) continue;
          double& o = ob[8 * I + g];
          o = w == 0 ? bacc[G::bown(I, GF_TS, PAR)] : o + bacc[G::bown(I, GF_TS, PAR)];
        }
        if (PAR == 0 && g == 0) ob[8 * G::T] = w == 0 ? bacc[NB - 1] : ob[8 * G::T] + bacc[NB - 1];
      }
      bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
    }
  }
}

template <int NJ, int SLOTS, int PAR, int Z>
__device__ __forceinline__ void gram_mma_role(const SamplesDev& in, double* smem, GramBars* bars, int ks, int lane, int dbg)
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int NTP = G::ntiles(GF_TS, PAR);
  double acc[NTP][2], bacc[G::nbacc(GF_TS, PAR)];
#pragma unroll
  for (int k = 0; k < NTP; k++) acc[k][0] = acc[k][1] = 0.0;
#pragma unroll
  for (int k = 0; k < G::nbacc(GF_TS, PAR); k++) bacc[k] = 0.0;
  const int64_t ngroups = (in.n + 31) / 32;
  const int64_t stride = (int64_t)gridDim.x * SLOTS;
  uint32_t parity = 0;
  for (int64_t base = (int64_t)blockIdx.x * SLOTS; base < ngroups; base += stride, parity ^= 1)
  {
#pragma unroll 1
    for (int s = 0; s < SLOTS; s++)
    {
      if (base + s >= ngroups) break;
      const double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
      mbar_wait(&bars->full[s], parity);
      if (!(dbg & 2))
      {
        gram_consume_slot<NJ, PAR, Z>(slot, ks, lane, acc, bacc);
      }
      if (base + s + stride < ngroups)  // the generator will come back for this slot
      {
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->empty[s]);
      }
    }
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);
  gram_tau_reduce<NJ, PAR, Z>(bacc, smem, ks, lane);
}

// ---------------------------------------------------------------------------------------------- MMA side, cross mode
// Extended model [Phi | Phi_c]: the component columns of joint j are non-zero in the row of joint j only, so
//   Phi^T Phi_c [:, comps of j] = sum_s Phi_row_j(s)^T phi_c,j(s)      (one extra 8-wide tile per joint row),
// Phi_c^T Phi_c is block diagonal per joint and Phi_c^T tau rides in the tau column of the last regular tile.  The rigid-body block comes
// from the X = 0 kernel; this mode accumulates only the cross tiles (NXT of them) with the same slots, k-split and software pipelining.
template <int NJ, int J>
__device__ __forceinline__ double gram_load_xfrag(const double* __restrict__ slot, int kk, int lane)
{
  using G = GramGeom<NJ, 1>;
  const int g = lane >> 2, t = lane & 3;
  return slot[G::rowbase(J) + (G::rowlen(J) + g) * 32 + ((4 * kk + t) ^ (4 * (g & 3)))];
}
template <int NJ, int PAR, int J, int Z = 0>
__device__ __forceinline__ void gram_cross_step(const double (&b)[GramGeom<NJ, 0, Z>::NF], double bx,
                                                double (&acc)[GramGeom<NJ, 1, Z>::nxtiles(GF_TS, PAR)][2])
{
  using G = GramGeom<NJ, 1, Z>;
  static_for<0, G::tj(J) + 1>([&](auto Ic) {
    constexpr int I = decltype(Ic)::value;
    if constexpr (G::xowns(J, I, GF_TS, PAR))
    {
      constexpr int k = G::xlocal(J, I, GF_TS, PAR);
      if constexpr (I < G::tj(J)) dmma884f(acc[k][0], acc[k][1], b[I], bx);
      else dmma884f(acc[k][0], acc[k][1], bx, bx);  // (component, component) tile of joint J
    }
  });
}
// fixed-order reduction of the cross tiles over the k-split warps into shared memory at `smem` (NXT tiles of 64 doubles)
template <int NJ, int PAR, int Z = 0>
__device__ __forceinline__ void gram_cross_reduce_smem(double (&acc)[GramGeom<NJ, 1, Z>::nxtiles(GF_TS, PAR)][2], double* smem, int ks, int lane)
{
  using G = GramGeom<NJ, 1, Z>;
  bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  const int g = lane >> 2, t = lane & 3;
  for (int w = 0; w < GF_KSPLIT; w++)
  {
    if (ks == w)
    {
      static_for<0, NJ>([&](auto jc) {
        constexpr int j = decltype(jc)::value;
        static_for<0, G::tj(j) + 1>([&](auto Ic) {
          constexpr int I = decltype(Ic)::value;
          if constexpr (G::xowns(j, I, GF_TS, PAR))
          {
            double* o = smem + G::xtile(j, I) * 64 + g * 8 + 2 * t;
            constexpr int k = G::xlocal(j, I, GF_TS, PAR);
            if (w == 0)
            {
              o[0] = acc[k][0];
              o[1] = acc[k][1];
            }
            else
            {
              o[0] += acc[k][0];
              o[1] += acc[k][1];
            }
          }
        });
      });
    }
    bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  }
}

template <int NJ, int SLOTS, bool REV, int X, int Z, class M>
__device__ __forceinline__ void gram_gen_role(const ChainDev<NJ>& C, const GramComps& comps, const SamplesDev& in,
                                              const double* __restrict__ tau_meas, double* smem, GramBars* bars, int s, int lane, int dbg)
{
  using G = GramGeom<NJ, X, Z>;
  double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
  const int64_t ngroups = (in.n + 31) / 32;
  const int64_t stride = (int64_t)gridDim.x * SLOTS;
  uint32_t parity = 1;  // first wait on an un-arrived barrier with parity 1 returns at once ("previous phase complete")
  for (int64_t grp = (int64_t)blockIdx.x * SLOTS + s; grp < ngroups; grp += stride, parity ^= 1)
  {
    // the inputs are requested BEFORE waiting for the slot: the DRAM latency hides behind the consumers' work on the previous group
    const int64_t i = grp * 32 + lane;
    GenIn<NJ> cur;
    gen_load<NJ>(C, in, min(i, in.n - 1), cur);
    trig_all<NJ>(cur.q, cur.sv, cur.cv);
    mbar_wait(&bars->empty[s], parity);  // consumers released the slot
    if (!(dbg & 1))
    {
      gram_generate<NJ, REV, X, Z, false, false, M>(C, &comps, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
      if (i >= in.n) gram_zero_lane<NJ, X, Z>(slot, lane);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars->full[s]);
  }
}

// ---------------------------------------------------------------------------------------------- GENS generator warps over SLOTS slots
// The k-th group of a CTA (global group blockIdx.x + k gridDim.x) is produced by generator warp k % GENS into slot k % SLOTS (its use k / SLOTS)
// and consumed in order by the MMA warps.  With more generator warps than slots every SM sub-partition hosts a generator (7-joint chains have
// 3 slots: with one generator per slot the fourth sub-partition's FP64 datapath idled whenever the MMA warps waited) and a generator starts
// the walk of its next group while the previous ones are still being consumed.
template <int NJ, int SLOTS, int GENS, bool REV, int Z, class M>
__device__ __forceinline__ void gram_gen_role_c(const ChainDev<NJ>& C, const SamplesDev& in, const double* __restrict__ tau_meas, double* smem,
                                                GramBars* bars, int w, int lane, int dbg)
{
  using G = GramGeom<NJ, 0, Z>;
  const int64_t ngroups = (in.n + 31) / 32;
  const int64_t nk = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  for (int64_t k = w; k < nk; k += GENS)
  {
    const int s = (int)(k % SLOTS);
    const uint32_t u = (uint32_t)(k / SLOTS);
    const int64_t i = ((int64_t)blockIdx.x + k * gridDim.x) * 32 + lane;
    GenIn<NJ> cur;
    gen_load<NJ>(C, in, min(i, in.n - 1), cur);
    trig_all<NJ>(cur.q, cur.sv, cur.cv);
    wait_counter_ge(&bars->drained[s], GF_MMA_WARPS * u);  // every MMA warp is done with the previous use of the slot
    double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
    if (!(dbg & 1))
    {
      gram_generate<NJ, REV, 0, Z, false, false, M>(C, nullptr, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
      if (i >= in.n) gram_zero_lane<NJ, 0, Z>(slot, lane);
    }
    __syncwarp();
    if (lane == 0) st_release_u32(&bars->filled[s], u + 1);
  }
}

template <int NJ, int SLOTS, int PAR, int Z>
__device__ __forceinline__ void gram_mma_role_c(const SamplesDev& in, double* smem, GramBars* bars, int ks, int lane, int dbg)
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int NTP = G::ntiles(GF_TS, PAR);
  double acc[NTP][2], bacc[G::nbacc(GF_TS, PAR)];
#pragma unroll
  for (int k = 0; k < NTP; k++) acc[k][0] = acc[k][1] = 0.0;
#pragma unroll
  for (int k = 0; k < G::nbacc(GF_TS, PAR); k++) bacc[k] = 0.0;
  const int64_t ngroups = (in.n + 31) / 32;
  const int64_t nk = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
#pragma unroll 1
  for (int64_t k = 0; k < nk; k++)
  {
    const int s = (int)(k % SLOTS);
    const uint32_t u = (uint32_t)(k / SLOTS);
    const double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
    wait_counter_ge(&bars->filled[s], u + 1);
    if (!(dbg & 2))
    {
      gram_consume_slot<NJ, PAR, Z>(slot, ks, lane, acc, bacc);
    }
    __syncwarp();
    if (lane == 0) red_release_inc(&bars->drained[s]);
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);
  gram_tau_reduce<NJ, PAR, Z>(bacc, smem, ks, lane);
}

// ---------------------------------------------------------------------------------------------- extended model [Phi | Phi_c] in ONE pass
// The slots carry the rigid-body rows in the geometry of the rigid-body kernel (Z: zero mass column dropped on all-revolute chains).  The
// component columns of a joint -- element-wise functions of that joint's q, Dq (friction_polynomial1.h:45-52, friction_polynomial2.h:42-58,
// ideal_spring.h:64-70), non-zero in the row of that joint only -- go to a small side buffer next to the slots, XC columns per joint (2, 4
// or 8: the widest component set of the chain rounded up) instead of a zero-padded 8-column tile inside every row: for 6 joints with a
// friction model on each the kernel keeps 4 slots (4 x (52.5 + 3) KB) where the padded rows left room for 3 x 66 KB.  The MMA warps keep BOTH
// tile sets in registers -- the upper triangular rigid-body tiles and, per joint row, the (regular tile, component tile) / (component,
// component) cross tiles -- so Phi is generated once.  Counter handshake, GENS generator warps.
template <int NJ, int XC>
__host__ __device__ constexpr int gram_ext_side_doubles()
{
  return NJ * XC * 32;
}
// component columns of all joints for the lane's sample.  q_j, Dq_j are parked in the buffer itself before the walk (columns 1 and 0 of joint
// j; XC >= 2: nothing of them stays in registers through the walk); AFTER the walk ONE rolled loop over (joint, column) evaluates in place
// (~100 instructions).  The order matters: with the loop between the wait for the slot and the walk the kernel ran at 1.02 G samples/s, with
// the loop behind the walk at 1.21 (C6; ncu with the loop in front: no_instruction 23 % of the generator's stall samples).
template <int NJ, int XC>
__device__ __forceinline__ void gram_component_park(const GenIn<NJ>& x, double* __restrict__ side, int lane)
{
  static_assert(XC >= 2, "q and Dq of a joint are staged in its first two columns");
#pragma unroll
  for (int j = 0; j < NJ; j++)
  {
    side[(j * XC) * 32 + lane] = x.dq[j];
    side[(j * XC + 1) * 32 + lane] = x.q[j];
  }
}
template <int NJ, int XC>
__device__ __forceinline__ void gram_component_side(const GramComps& comps, double* __restrict__ side, int lane)
{
#pragma unroll 1
  for (int j = 0; j < NJ; j++)
  {
    double* o = side + (j * XC) * 32 + lane;
    const double dq = o[0], q = o[32];
    const int nc = comps.ncols[j];
#pragma unroll(XC <= 4 ? XC : 1)  // narrow sets: the columns of a joint evaluate side by side (their table reads and chains overlap)
    for (int c = 0; c < XC; c++)
    {
      double val = 0.0;
      if (c < nc)
      {
        const int kd = comps.kind[j][c];
        const double th = comps.thr[j][c], vm = comps.vmax[j][c];
        const double omega = fmin(fmax(dq, -vm), vm);
        if (kd == GXK_OMEGA) val = omega;
        else if (kd == GXK_Q) val = q;
        else if (kd == GXK_ONE) val = 1.0;
        else
        {
          const double r = omega * comps.ithr[j][c];
          if (kd == GXK_SAT) val = fmin(fmax(r, -1.0), 1.0);
          else
          {
            const double sg = omega == 0.0 ? 0.0 : (omega > th ? 1.0 : (omega < -th ? -1.0 : r));
            val = kd == GXK_SGN ? sg : omega * omega * sg;
          }
        }
      }
      o[c * 32] = val;
    }
  }
}
// component fragment of one k-step: lane (g, t) holds column g of joint J for sample 4 kk + t (zero behind the XC stored columns)
template <int J, int XC>
__device__ __forceinline__ double gram_load_xside(const double* __restrict__ side, int kk, int lane)
{
  const int g = lane >> 2, t = lane & 3;
  return g < XC ? side[(J * XC + g) * 32 + 4 * kk + t] : 0.0;
}
template <int NJ, int PAR, int STEP, int Z, int XC>
__device__ __forceinline__ void gram_ext_steps(const double* __restrict__ slot, const double* __restrict__ side, int ks, int lane,
                                               const double (&bcur)[GramGeom<NJ, 0, Z>::NF], double bxcur,
                                               double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2],
                                               double (&xacc)[GramGeom<NJ, 1, Z>::nxtiles(GF_TS, PAR)][2])
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int J = STEP / G::KPW;
  if constexpr (STEP + 1 < G::NSTEPS)
  {
    double bnext[G::NF];
    constexpr int JN = (STEP + 1) / G::KPW;
    const int kn = ks * G::KPW + (STEP + 1) % G::KPW;
    gram_load_frags<NJ, JN, 0, Z>(slot, kn, lane, bnext);
    const double bxn = gram_load_xside<JN, XC>(side, kn, lane);
    gram_mma_step<NJ, PAR, J, Z>(bcur, acc);
    gram_cross_step<NJ, PAR, J, Z>(bcur, bxcur, xacc);
    gram_ext_steps<NJ, PAR, STEP + 1, Z, XC>(slot, side, ks, lane, bnext, bxn, acc, xacc);
  }
  else
  {
    gram_mma_step<NJ, PAR, J, Z>(bcur, acc);
    gram_cross_step<NJ, PAR, J, Z>(bcur, bxcur, xacc);
  }
}

template <int NJ, int SLOTS, int PAR, int Z, int XC>
__device__ __forceinline__ void gram_ext_mma_role(const SamplesDev& in, double* smem, const double* side0, GramBars* bars, int ks, int lane)
{
  using G0 = GramGeom<NJ, 0, Z>;
  using GX = GramGeom<NJ, 1, Z>;
  double acc[G0::ntiles(GF_TS, PAR)][2], xacc[GX::nxtiles(GF_TS, PAR)][2];
#pragma unroll
  for (int k = 0; k < G0::ntiles(GF_TS, PAR); k++) acc[k][0] = acc[k][1] = 0.0;
#pragma unroll
  for (int k = 0; k < GX::nxtiles(GF_TS, PAR); k++) xacc[k][0] = xacc[k][1] = 0.0;
  const int64_t ngroups = (in.n + 31) / 32;
  const int64_t nk = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
#pragma unroll 1
  for (int64_t k = 0; k < nk; k++)
  {
    const int s = (int)(k % SLOTS);
    const uint32_t u = (uint32_t)(k / SLOTS);
    const double* slot = smem + (size_t)s * G0::SLOT_DOUBLES;
    const double* side = side0 + (size_t)s * gram_ext_side_doubles<NJ, XC>();
    wait_counter_ge(&bars->filled[s], u + 1);
    double b0[G0::NF];
    gram_load_frags<NJ, 0, 0, Z>(slot, ks * G0::KPW, lane, b0);
    const double bx0 = gram_load_xside<0, XC>(side, ks * G0::KPW, lane);
    gram_ext_steps<NJ, PAR, 0, Z, XC>(slot, side, ks, lane, b0, bx0, acc, xacc);
    __syncwarp();
    if (lane == 0) red_release_inc(&bars->drained[s]);
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);                           // rigid-body tiles: smem[0, NT * 64)
  gram_cross_reduce_smem<NJ, PAR, Z>(xacc, smem + G0::NT * 64, ks, lane);    // cross tiles behind them
}

// M: model constants (gram_common.cuh) -- RtModel for the precompiled instantiations, a generated model type in gram_jit.cpp
template <int NJ, int SLOTS, int GENS, bool REV, int XC, class M = RtModel>
__global__ void __launch_bounds__(GramGeom<NJ>::threads(GENS), 1)
    gram_ext_kernel(const __grid_constant__ ChainDev<NJ> C, const __grid_constant__ GramComps comps, const SamplesDev in,
                    const double* __restrict__ tau_meas, double* __restrict__ partial)
{
  constexpr int Z = GF_ZCOL && REV ? 1 : 0;
  using G0 = GramGeom<NJ, 0, Z>;
  using GX = GramGeom<NJ, 1, Z>;
  constexpr int NOUT = (G0::NT + GX::NXT) * 64;
  constexpr int SIDE = gram_ext_side_doubles<NJ, XC>();
  extern __shared__ __align__(16) double smem[];
  __shared__ GramBars bars;
  // the component columns of the groups in the slots live behind max(slots, reduction area)
  double* const side0 = smem + (G0::SLOT_DOUBLES * SLOTS > NOUT ? G0::SLOT_DOUBLES * SLOTS : NOUT);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < SLOTS)
  {
    bars.filled[threadIdx.x] = 0;
    bars.drained[threadIdx.x] = 0;
  }
  __syncthreads();
  if (warp >= GF_MMA_WARPS)
  {
    const int w = warp - GF_MMA_WARPS;
    const int64_t ngroups = (in.n + 31) / 32;
    const int64_t nk = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    for (int64_t k = w; k < nk; k += GENS)
    {
      const int s = (int)(k % SLOTS);
      const uint32_t u = (uint32_t)(k / SLOTS);
      const int64_t i = ((int64_t)blockIdx.x + k * gridDim.x) * 32 + lane;
      GenIn<NJ> cur;
      gen_load<NJ>(C, in, min(i, in.n - 1), cur);
      trig_all<NJ>(cur.q, cur.sv, cur.cv);
      wait_counter_ge(&bars.drained[s], GF_MMA_WARPS * u);
      double* slot = smem + (size_t)s * G0::SLOT_DOUBLES;
      double* side = side0 + (size_t)s * SIDE;
      gram_component_park<NJ, XC>(cur, side, lane);
      gram_generate<NJ, REV, 0, Z, false, false, M>(C, nullptr, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
      gram_component_side<NJ, XC>(comps, side, lane);
      if (i >= in.n)
      {
        gram_zero_lane<NJ, 0, Z>(slot, lane);
        for (int c = 0; c < NJ * XC; c++) side[c * 32 + lane] = 0.0;
      }
      __syncwarp();
      if (lane == 0) st_release_u32(&bars.filled[s], u + 1);
    }
    return;
  }
  const int mma_id = warp, ks = mma_id % GF_KSPLIT;
  if (GF_TS == 1 || mma_id < GF_KSPLIT) gram_ext_mma_role<NJ, SLOTS, 0, Z, XC>(in, smem, side0, &bars, ks, lane);
  else gram_ext_mma_role<NJ, SLOTS, 1, Z, XC>(in, smem, side0, &bars, ks, lane);
  double* out = partial + (size_t)blockIdx.x * NOUT;
  for (int k = mma_id * 32 + lane; k < NOUT; k += 32 * GF_MMA_WARPS) out[k] = smem[k];
}

template <int NJ, int SLOTS, bool REV, int X, int GENS = SLOTS, class M = RtModel>
__global__ void __launch_bounds__(GramGeom<NJ>::threads(GENS), 1)
    gram_fused_kernel(const __grid_constant__ ChainDev<NJ> C, const __grid_constant__ GramComps comps, const SamplesDev in,
                      const double* __restrict__ tau_meas, double* __restrict__ partial, const int dbg)
{
  // Z = 2 (gram_common.cuh): on all-revolute chains the exact-zero columns of the REV walk are neither stored nor multiplied, and (TC == 0)
  // tau is accumulated by DFMA beside the tiles: 81 instead of 104 DMMA per 4 samples for 6 joints, 125 instead of 149 for 7
  constexpr int Z = GF_ZCOL && REV && X == 0 ? 2 : 0;
  using G = GramGeom<NJ, X, Z>;
  extern __shared__ __align__(16) double smem[];
  __shared__ GramBars bars;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0)
  {
    for (int s = 0; s < SLOTS; s++)
    {
      mbar_init(&bars.full[s], 1);              // lane 0 of the generator warp, after __syncwarp
      mbar_init(&bars.empty[s], GF_MMA_WARPS);  // lane 0 of every MMA warp
      bars.filled[s] = 0;
      bars.drained[s] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // group of (iteration it, CTA, slot s): (it*gridDim.x + blockIdx.x)*SLOTS + s ; generator warp s fills slot s
  if (warp >= GF_MMA_WARPS)
  {
    if constexpr (GENS != SLOTS) gram_gen_role_c<NJ, SLOTS, GENS, REV, Z, M>(C, in, tau_meas, smem, &bars, warp - GF_MMA_WARPS, lane, dbg);
    else gram_gen_role<NJ, SLOTS, REV, X, Z, M>(C, comps, in, tau_meas, smem, &bars, warp - GF_MMA_WARPS, lane, dbg);
    return;
  }
  // ------------------------------------------------ MMA warps: k-split index = warp % 4 (its SM sub-partition), tile-row parity = warp / 4
  const int mma_id = warp;
  const int ks = mma_id % GF_KSPLIT;
  constexpr int NOUT = X ? G::NXT * 64 : G::PARTIAL;
  static_assert(X == 0, "the extended model runs through gram_ext_kernel");
  {
    if constexpr (GENS != SLOTS)
    {
      if (GF_TS == 1 || mma_id < GF_KSPLIT) gram_mma_role_c<NJ, SLOTS, 0, Z>(in, smem, &bars, ks, lane, dbg);
      else gram_mma_role_c<NJ, SLOTS, 1, Z>(in, smem, &bars, ks, lane, dbg);
    }
    else
    {
      if (GF_TS == 1 || mma_id < GF_KSPLIT) gram_mma_role<NJ, SLOTS, 0, Z>(in, smem, &bars, ks, lane, dbg);
      else gram_mma_role<NJ, SLOTS, 1, Z>(in, smem, &bars, ks, lane, dbg);
    }
  }
  double* out = partial + (size_t)blockIdx.x * NOUT;
  for (int k = mma_id * 32 + lane; k < NOUT; k += 32 * GF_MMA_WARPS) out[k] = smem[k];
}

}  // namespace rdb
