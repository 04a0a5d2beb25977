// gram_fused.cu -- fused regressor -> normal equations, one persistent warp-specialised kernel per GPU.
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
//   * all-revolute chains drop the exact-zero mass column of a link on its own joint (GramGeom Z): the rows are one position shorter,
//     98 instead of 104 DMMA per 4 samples for 6 joints (143 / 149 for 7).
//   * all-revolute chains whose folded axes are all e_z (fold.cpp puts every revolute link in such a canonical frame) run the REV generator,
//     which holds the axis as a compile-time constant: 2 019 instead of 2 412 FP64 instructions per sample for 6 joints (2 658 / 3 119 for 7).
// Per-CTA partials are summed in a fixed order by gram_fused_reduce_kernel (bit-reproducible for a given n).
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
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "gram_common.cuh"

namespace rdb
{

// ---------------------------------------------------------------------------------------------- MMA side
// B fragments of one k-step (4 samples of joint row J, k-step kk of the slot): lane (g, t) holds column 8 I + g of sample 4 kk + t
template <int NJ, int J, int X = 0, int Z = 0>
__device__ __forceinline__ void gram_load_frags(const double* __restrict__ slot, int kk, int lane, double (&b)[GramGeom<NJ, 0, Z>::T])
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
}
template <int NJ, int PAR, int J, int Z>
__device__ __forceinline__ void gram_mma_step(const double (&b)[GramGeom<NJ, 0, Z>::T], double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2])
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
// k-steps STEP.. of this warp in one slot; step = (joint row, k-step of the warp); the fragments of the next step are in flight while the
// DMMAs of the current one issue
template <int NJ, int PAR, int STEP, int Z>
__device__ __forceinline__ void gram_consume_steps(const double* __restrict__ slot, int ks, int lane, const double (&bcur)[GramGeom<NJ, 0, Z>::T],
                                                   double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2])
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int J = STEP / G::KPW;
  if constexpr (STEP + 1 < G::NSTEPS)
  {
    double bnext[G::T];
    gram_load_frags<NJ, (STEP + 1) / G::KPW, 0, Z>(slot, ks * G::KPW + (STEP + 1) % G::KPW, lane, bnext);
    gram_mma_step<NJ, PAR, J, Z>(bcur, acc);
    gram_consume_steps<NJ, PAR, STEP + 1, Z>(slot, ks, lane, bnext, acc);
  }
  else
    gram_mma_step<NJ, PAR, J, Z>(bcur, acc);
}
// the k-steps of one slot for this warp
template <int NJ, int PAR, int Z>
__device__ __forceinline__ void gram_consume_slot(const double* __restrict__ slot, int ks, int lane,
                                                  double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2])
{
  using G = GramGeom<NJ, 0, Z>;
  double b0[G::T];
  gram_load_frags<NJ, 0, 0, Z>(slot, ks * G::KPW, lane, b0);
  gram_consume_steps<NJ, PAR, 0, Z>(slot, ks, lane, b0, acc);
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

template <int NJ, int SLOTS, int PAR, int Z>
__device__ __forceinline__ void gram_mma_role(const SamplesDev& in, double* smem, GramBars* bars, int ks, int lane, int dbg)
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int NTP = G::ntiles(GF_TS, PAR);
  double acc[NTP][2];
#pragma unroll
  for (int k = 0; k < NTP; k++) acc[k][0] = acc[k][1] = 0.0;
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
        gram_consume_slot<NJ, PAR, Z>(slot, ks, lane, acc);
      }
      if (base + s + stride < ngroups)  // the generator will come back for this slot
      {
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->empty[s]);
      }
    }
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);
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
__device__ __forceinline__ void gram_cross_step(const double (&b)[GramGeom<NJ, 0, Z>::T], double bx,
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

template <int NJ, int SLOTS, bool REV, int X, int Z>
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
      gram_generate<NJ, REV, X, Z>(C, &comps, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
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
template <int NJ, int SLOTS, int GENS, bool REV, int Z>
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
      gram_generate<NJ, REV, 0, Z>(C, nullptr, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
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
  double acc[NTP][2];
#pragma unroll
  for (int k = 0; k < NTP; k++) acc[k][0] = acc[k][1] = 0.0;
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
      gram_consume_slot<NJ, PAR, Z>(slot, ks, lane, acc);
    }
    __syncwarp();
    if (lane == 0) red_release_inc(&bars->drained[s]);
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);
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
                                               const double (&bcur)[GramGeom<NJ, 0, Z>::T], double bxcur,
                                               double (&acc)[GramGeom<NJ, 0, Z>::ntiles(GF_TS, PAR)][2],
                                               double (&xacc)[GramGeom<NJ, 1, Z>::nxtiles(GF_TS, PAR)][2])
{
  using G = GramGeom<NJ, 0, Z>;
  constexpr int J = STEP / G::KPW;
  if constexpr (STEP + 1 < G::NSTEPS)
  {
    double bnext[G::T];
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
    double b0[G0::T];
    gram_load_frags<NJ, 0, 0, Z>(slot, ks * G0::KPW, lane, b0);
    const double bx0 = gram_load_xside<0, XC>(side, ks * G0::KPW, lane);
    gram_ext_steps<NJ, PAR, 0, Z, XC>(slot, side, ks, lane, b0, bx0, acc, xacc);
    __syncwarp();
    if (lane == 0) red_release_inc(&bars->drained[s]);
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);                           // rigid-body tiles: smem[0, NT * 64)
  gram_cross_reduce_smem<NJ, PAR, Z>(xacc, smem + G0::NT * 64, ks, lane);    // cross tiles behind them
}

template <int NJ, int SLOTS, int GENS, bool REV, int XC>
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
      gram_generate<NJ, REV, 0, Z>(C, nullptr, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
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

template <int NJ, int SLOTS, bool REV, int X, int GENS = SLOTS>
__global__ void __launch_bounds__(GramGeom<NJ>::threads(GENS), 1)
    gram_fused_kernel(const __grid_constant__ ChainDev<NJ> C, const __grid_constant__ GramComps comps, const SamplesDev in,
                      const double* __restrict__ tau_meas, double* __restrict__ partial, const int dbg)
{
  // Z (gram_common.cuh): on all-revolute chains the mass column of a link on its own joint is an exact zero; it is put last in its block and
  // neither stored nor multiplied (rigid-body mode only: 98 instead of 104 DMMA per 4 samples for 6 joints, 143 instead of 149 for 7)
  constexpr int Z = GF_ZCOL && REV && X == 0 ? 1 : 0;
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
    if constexpr (GENS != SLOTS) gram_gen_role_c<NJ, SLOTS, GENS, REV, Z>(C, in, tau_meas, smem, &bars, warp - GF_MMA_WARPS, lane, dbg);
    else gram_gen_role<NJ, SLOTS, REV, X, Z>(C, comps, in, tau_meas, smem, &bars, warp - GF_MMA_WARPS, lane, dbg);
    return;
  }
  // ------------------------------------------------ MMA warps: k-split index = warp % 4 (its SM sub-partition), tile-row parity = warp / 4
  const int mma_id = warp;
  const int ks = mma_id % GF_KSPLIT;
  constexpr int NOUT = (X ? G::NXT : G::NT) * 64;
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

// fixed-order sum of the per-CTA partials -> gram (full symmetric, column-major), rhs, tau_sq
// zcol: GramGeom Z = 1 position order (the mass column last in every link block; position P does not exist and the row / column of the first
// moving link's mass, an identically zero column of Phi, is written as exact zeros)
__global__ void gram_fused_reduce_kernel(const double* __restrict__ partial, int nparts, int T, int P, double* __restrict__ gram,
                                         double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate, int zcol, int pstride)
{
  const int NT = T * (T + 1) / 2;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NT * 64) return;
  double s = 0.0;
  for (int p = 0; p < nparts; p++) s += partial[(size_t)p * pstride + e];  // pstride: doubles between the partials of two CTAs
  int k = e >> 6, I = 0;
  while (k >= T - I)
  {
    k -= T - I;
    I++;
  }
  const int J = I + k;
  const int rp = 8 * I + ((e >> 3) & 7), cp = 8 * J + (e & 7);  // positions inside the kernel (GramGeom::pos)
  if (zcol && e <= P && !accumulate)  // the untouched mass column of the first moving link (parameter 0): exact zeros
  {
    if (e == P) rhs[0] = 0.0;
    else
    {
      gram[(size_t)e * P] = 0.0;
      gram[e] = 0.0;
    }
  }
  if (rp > P - zcol || cp > P - zcol) return;
  if (I == J && rp > cp) return;  // diagonal tiles hold both halves; keep the upper one
  // position -> column of the (folded) parameter vector, P = tau
  const int nj = P / 10;
  auto col_of = [&](int pos) {
    if (pos == 0) return P;
    const int q = (pos - 1) % 10;
    return 10 * (nj - 1 - (pos - 1) / 10) + (zcol ? (q == 9 ? 0 : q + 1) : q);
  };
  const int row = col_of(rp), col = col_of(cp);
  if (row < P && col < P)
  {
    const double v = accumulate ? gram[(size_t)col * P + row] + s : s;
    gram[(size_t)col * P + row] = v;
    if (row != col) gram[(size_t)row * P + col] = v;
  }
  else if (row < P || col < P)
  {
    const int a = row < P ? row : col;
    rhs[a] = accumulate ? rhs[a] + s : s;
  }
  else if (tau_sq)
    *tau_sq = accumulate ? *tau_sq + s : s;
}

// G = E^T G' E, b = E^T b' (upper triangle computed, mirrored): one thread per entry of the full matrix, 100 products each
__global__ void gram_fold_expand_kernel(const double* __restrict__ T, const int32_t* __restrict__ kof, const double* __restrict__ Gr,
                                        const double* __restrict__ br, const double* __restrict__ tsr, int nj, int Pr, double* __restrict__ gram,
                                        double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  const int P = 10 * nj;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P * (P + 1)) return;
  const int a = e / (P + 1), b = e % (P + 1);  // b == P: right-hand side
  if (e == P && tau_sq) *tau_sq = accumulate ? *tau_sq + *tsr : *tsr;
  if (b < a) return;
  const int la = a / 10, pa = a % 10, ka = kof[la];
  double s = 0.0;
  if (b == P)
  {
    if (ka >= 0)
      for (int c = 0; c < 10; c++) s = fma(T[(size_t)la * 100 + c * 10 + pa], br[10 * ka + c], s);
    rhs[a] = accumulate ? rhs[a] + s : s;
    return;
  }
  const int lb = b / 10, pb = b % 10, kb = kof[lb];
  if (ka >= 0 && kb >= 0)
    for (int c = 0; c < 10; c++)
    {
      double r = 0.0;
      for (int d = 0; d < 10; d++) r = fma(Gr[(size_t)(10 * kb + d) * Pr + 10 * ka + c], T[(size_t)lb * 100 + d * 10 + pb], r);
      s = fma(T[(size_t)la * 100 + c * 10 + pa], r, s);
    }
  const double v = accumulate ? gram[(size_t)b * P + a] + s : s;
  gram[(size_t)b * P + a] = v;
  if (a != b) gram[(size_t)a * P + b] = v;
}

// Timing experiments (1: skip the generation, 2: skip the MMA) exist in development builds only (-DRDB_DEV_SWITCHES); the shipped library
// always computes.
static int gram_dev_switch()
{
#ifdef RDB_DEV_SWITCHES
  static const int dbg = [] { const char* e = getenv("RDB_GRAM_DEBUG"); return e ? atoi(e) : 0; }();
  return dbg;
#else
  return 0;
#endif
}

// the reduced normal equations G' | b' | tau_sq of the folded chain (ch.gram.fold_dev, written by the reduce kernels) -> the reference's full
// parameter vector
cudaError_t launch_fold_expand(ChainHost& ch, double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st)
{
  const int nj = ch.host.nj, Pr = 10 * ch.gram.fold.nj, P = 10 * nj;
  double* Tm = ch.gram.fold_dev;
  double* Gr = Tm + (size_t)nj * 100;
  double* br = Gr + (size_t)Pr * Pr;
  double* tsr = br + Pr;
  const int32_t* kof = reinterpret_cast<const int32_t*>(Gr + (size_t)(Pr + 1) * (Pr + 1));
  gram_fold_expand_kernel<<<(P * (P + 1) + 127) / 128, 128, 0, st>>>(Tm, kof, Gr, br, tsr, nj, Pr, gram, rhs, tau_sq, accumulate);
  count_launch();
  return cudaGetLastError();
}

template <int NJ>
static ChainDev<NJ> narrow_g(const ChainDev<RDB_MAX_JOINTS>& h)
{
  ChainDev<NJ> c;
  c.nj = h.nj;
  c.n_in = h.n_in;
  for (int k = 0; k < 3; k++) c.g[k] = h.g[k];
  for (int j = 0; j < NJ; j++)
  {
    c.joint[j] = h.joint[j];
    c.link[j] = h.link[j];
  }
  return c;
}

static cudaError_t grow(double*& p, size_t& have, size_t need)
{
  if (have >= need) return cudaSuccess;
  if (p) cudaFree(p);
  p = nullptr;
  have = 0;
  cudaError_t e = cudaMalloc(&p, need);
  if (e == cudaSuccess) have = need;
  return e;
}

// generator warps of the rigid-body kernel: one per SM sub-partition even when fewer slots fit (GF_GENS4 = 0: one per slot, as before)
#ifndef GF_GENS4
#define GF_GENS4 1
#endif
template <int SLOTS>
constexpr int gf_gens()
{
  return (GF_GENS4 && GF_TS == 2 && SLOTS < 4) ? 4 : SLOTS;
}

template <int NJ, int SLOTS, bool REV>
static cudaError_t launch_fused_nj(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                   int accumulate, cudaStream_t st)
{
  constexpr int GENS = gf_gens<SLOTS>();
  constexpr int Z = GF_ZCOL && REV ? 1 : 0;  // as in the kernel
  using G = GramGeom<NJ, 0, Z>;
  const size_t smem = sizeof(double) * (size_t)std::max(G::SLOT_DOUBLES * SLOTS, G::NT * 64);
  {
    cudaError_t e = cudaFuncSetAttribute(gram_fused_kernel<NJ, SLOTS, REV, 0, GENS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const int dbg = gram_dev_switch();
  const int64_t ngroups = (in.n + 31) / 32;
  const int grid = (int)std::min<int64_t>(ch.sm_count, GENS != SLOTS ? ngroups : (ngroups + SLOTS - 1) / SLOTS);
  {
    cudaError_t e = grow(ch.gram.fused_partials, ch.gram.fused_bytes, sizeof(double) * (size_t)ch.sm_count * G::NT * 64);
    if (e != cudaSuccess) return e;
  }
  gram_fused_kernel<NJ, SLOTS, REV, 0, GENS><<<grid, G::threads(GENS), smem, st>>>(narrow_g<NJ>(ch.gram.fold), GramComps{}, in, tau_meas,
                                                                                   ch.gram.fused_partials, dbg);
  count_launch();
  if (ch.gram.fold_identity)
  {
    gram_fused_reduce_kernel<<<(G::NT * 64 + 255) / 256, 256, 0, st>>>(ch.gram.fused_partials, grid, G::T, G::P, gram, rhs, tau_sq, accumulate, Z, G::NT * 64);
    count_launch();
    return cudaGetLastError();
  }
  // folded chain: reduce into G', b', then expand to the reference's full parameter vector
  const int nj = ch.host.nj, Pr = G::P;
  double* Tm = ch.gram.fold_dev;
  double* Gr = Tm + (size_t)nj * 100;
  double* br = Gr + (size_t)Pr * Pr;
  double* tsr = br + Pr;
  gram_fused_reduce_kernel<<<(G::NT * 64 + 255) / 256, 256, 0, st>>>(ch.gram.fused_partials, grid, G::T, G::P, Gr, br, tsr, 0, Z, G::NT * 64);
  count_launch();
  return launch_fold_expand(ch, gram, rhs, tau_sq, accumulate, st);
}

// slots that fit the shared memory of an SM (227 KB minus 1 KB of barriers / static data)
template <int NJ, int X = 0>
constexpr int gf_slots()
{
  return std::min<int>(GF_MAX_SLOTS, (int)((227 * 1024 - 1024) / (sizeof(double) * GramGeom<NJ, X>::SLOT_DOUBLES)));
}

// returns cudaErrorNotSupported when the chain does not fit the fused kernel (caller falls back to the general pipeline)
cudaError_t launch_gram_fused(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                              int accumulate, cudaStream_t st)
{
  if (in.n <= 0 || ch.gram.fold_version != ch.model_version) return cudaErrorNotSupported;
  const bool rev = fold_rev_canonical(ch.gram.fold);  // all moving joints revolute about e_z: the specialised generator
  switch (ch.gram.fold.nj)  // moving joints; every joint of the folded chain is an input
  {
#define X(N)                                                                                                    \
  case N:                                                                                                       \
    return rev ? launch_fused_nj<N, gf_slots<N>(), true>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st)  \
               : launch_fused_nj<N, gf_slots<N>(), false>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st);
    X(1) X(2) X(3) X(4) X(5) X(6) X(7)
#undef X
  }
  return cudaErrorNotSupported;
}

// ---------------------------------------------------------------------------------------------- extended model [Phi | Phi_c]
// sum of the per-CTA cross partials in a fixed order
__global__ void gram_cross_reduce_kernel(const double* __restrict__ partial, int nparts, int n, int pstride, double* __restrict__ sum)
{
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  double s = 0.0;
  for (int p = 0; p < nparts; p++) s += partial[(size_t)p * pstride + e];
  sum[e] = s;
}

// the rigid-body block (P x P, rhs, tau_sq) into the extended normal equations (Pt x Pt)
__global__ void gram_ext_scatter_kernel(const double* __restrict__ G, const double* __restrict__ b, const double* __restrict__ ts, int P, int Pt,
                                        double* __restrict__ gram, double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= P * (P + 1)) return;
  const int a = e / (P + 1), c = e % (P + 1);
  if (e == P && tau_sq) *tau_sq = accumulate ? *tau_sq + *ts : *ts;
  if (c == P)
  {
    rhs[a] = accumulate ? rhs[a] + b[a] : b[a];
    return;
  }
  const double v = G[(size_t)c * P + a];
  gram[(size_t)c * Pt + a] = accumulate ? gram[(size_t)c * Pt + a] + v : v;
}

// cross blocks of the extended normal equations from the reduced cross tiles:
//   gram[a][P + cc] (and its mirror) = sum_c T[la][c][pa] X(10 ka + c ; joint, slot of cc)     a < P   (fold expansion of the rigid column)
//   rhs[P + cc] = X(P' ; joint, slot)                                                          (tau column of the last regular tile)
//   gram[P + c2][P + cc] = XX(joint)[slot2][slot] when both components act on the same joint, else 0
// xj / xs: reduced joint and slot of every component column.  One thread per (a in 0 .. P + Pc, cc).
__global__ void gram_cross_finish_kernel(const double* __restrict__ X, const double* __restrict__ Tm, const int32_t* __restrict__ kof,
                                         const int32_t* __restrict__ xj, const int32_t* __restrict__ xs, int nj, int njr, int Pc,
                                         double* __restrict__ gram, double* __restrict__ rhs, int accumulate, int zcol)
{
  const int P = 10 * nj, Pr = 10 * njr, Pt = P + Pc;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (P + 1 + Pc) * Pc) return;
  const int a = e / Pc, cc = e % Pc;
  const int j = xj[cc], g = xs[cc];
  auto tjf = [&](int k) { return (1 + 10 * (njr - k) - zcol + 7) / 8; };  // GramGeom::tj
  int tb = 0;  // first cross tile of joint j
  for (int k = 0; k < j; k++) tb += tjf(k) + 1;
  const int tjj = tjf(j);
  auto xval = [&](int col) -> double {  // reduced regular column `col` (Pr = tau) against (j, g)
    const int p = col % 10;
    const int pos = col == Pr ? 0 : 1 + 10 * (njr - 1 - col / 10) + (zcol ? (p == 0 ? 9 : p - 1) : p);  // GramGeom::pos
    const int I = pos >> 3;
    return (pos >= 1 + 10 * (njr - j) - zcol) ? 0.0 : X[(size_t)(tb + I) * 64 + (pos & 7) * 8 + g];  // behind rowlen(j): an exact zero of Phi
  };
  if (a < P)
  {
    double s = 0.0;
    if (kof)
    {
      const int la = a / 10, pa = a % 10, ka = kof[la];
      if (ka >= 0)
        for (int c = 0; c < 10; c++) s = fma(Tm[(size_t)la * 100 + c * 10 + pa], xval(10 * ka + c), s);
    }
    else
      s = xval(a);
    double* o = gram + (size_t)(P + cc) * Pt + a;
    const double v = accumulate ? *o + s : s;
    *o = v;
    gram[(size_t)a * Pt + P + cc] = v;
  }
  else if (a == P)
  {
    const double s = xval(Pr);
    rhs[P + cc] = accumulate ? rhs[P + cc] + s : s;
  }
  else
  {
    const int c2 = a - P - 1;
    const double s = (xj[c2] == j) ? X[(size_t)(tb + tjj) * 64 + xs[c2] * 8 + g] : 0.0;
    double* o = gram + (size_t)(P + cc) * Pt + P + c2;
    *o = accumulate ? *o + s : s;
  }
}

// slots of the extended-model kernel: rigid-body rows + XC component columns per joint
template <int NJ, int Z, int XC>
constexpr int gf_slots_ext()
{
  return std::min<int>(GF_MAX_SLOTS, (int)((227 * 1024 - 256) / (sizeof(double) * (GramGeom<NJ, 0, Z>::SLOT_DOUBLES + gram_ext_side_doubles<NJ, XC>()))));
}
// single pass (gram_ext_kernel): rigid-body tiles -> Gt | bt | tst (full parameter vector), cross tiles -> xsum
template <int NJ, bool REV, int XC>
static cudaError_t launch_ext_nj(ChainHost& ch, const GramComps& gc, const SamplesDev& in, const double* tau_meas, double* Gt, double* bt, double* tst,
                                 double* xpart, double* xsum, cudaStream_t st)
{
  constexpr int Z = GF_ZCOL && REV ? 1 : 0;  // as in the kernel
  using G0 = GramGeom<NJ, 0, Z>;
  using GX = GramGeom<NJ, 1, Z>;
  constexpr int SLOTS = gf_slots_ext<NJ, Z, XC>();
  static_assert(SLOTS >= 2, "the extended-model kernel needs two slots");
  constexpr int GENS = GF_TS == 2 ? 4 : SLOTS;  // 8 MMA + 4 generator warps (one per SM sub-partition) whatever the number of slots
  constexpr int PSTRIDE = (G0::NT + GX::NXT) * 64;
  const size_t smem = sizeof(double) * ((size_t)std::max(G0::SLOT_DOUBLES * SLOTS, PSTRIDE) + (size_t)SLOTS * gram_ext_side_doubles<NJ, XC>());
  cudaError_t e = cudaFuncSetAttribute(gram_ext_kernel<NJ, SLOTS, GENS, REV, XC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t ngroups = (in.n + 31) / 32;
  const int grid = (int)std::min<int64_t>(ch.sm_count, ngroups);
  gram_ext_kernel<NJ, SLOTS, GENS, REV, XC><<<grid, G0::threads(GENS), smem, st>>>(narrow_g<NJ>(ch.gram.fold), gc, in, tau_meas, xpart);
  count_launch();
  const int nred = (G0::NT * 64 + 255) / 256;
  if (ch.gram.fold_identity)
  {
    gram_fused_reduce_kernel<<<nred, 256, 0, st>>>(xpart, grid, G0::T, G0::P, Gt, bt, tst, 0, Z, PSTRIDE);
    count_launch();
  }
  else
  {
    const int nj = ch.host.nj, Pr = G0::P;
    double* Gr = ch.gram.fold_dev + (size_t)nj * 100;
    double* br = Gr + (size_t)Pr * Pr;
    gram_fused_reduce_kernel<<<nred, 256, 0, st>>>(xpart, grid, G0::T, G0::P, Gr, br, br + Pr, 0, Z, PSTRIDE);
    count_launch();
    e = launch_fold_expand(ch, Gt, bt, tst, 0, st);
    if (e != cudaSuccess) return e;
  }
  gram_cross_reduce_kernel<<<(GX::NXT * 64 + 255) / 256, 256, 0, st>>>(xpart + G0::NT * 64, grid, GX::NXT * 64, PSTRIDE, xsum);
  count_launch();
  return cudaGetLastError();
}

// Normal equations of the extended model in one pass over the samples (gram_ext_kernel); the two-pass scheme (rigid-body kernel, then the cross
// mode of gram_fused_kernel) is kept for development builds (RDB_GRAM_EXT=2).
// cudaErrorNotSupported: more than 7 moving joints, a component on an input no chain joint feeds, or more than GX_COLS component columns
// on one joint (caller falls back to the general pipeline).
cudaError_t launch_gram_fused_ext(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                  int accumulate, cudaStream_t st)
{
  if (in.n <= 0 || ch.gram.fold_version != ch.model_version) return cudaErrorNotSupported;
  const ChainDev<RDB_MAX_JOINTS>& F = ch.gram.fold;
  const int K = F.nj, nj = ch.host.nj, P = 10 * nj, Pc = ch.comps.cols, Pt = P + Pc;
  if (K < 1 || K > 7 || Pc <= 0) return cudaErrorNotSupported;
  GramComps gc{};
  std::vector<int32_t> xmap(2 * (size_t)Pc, 0);
  for (int k = 0; k < ch.comps.n; k++)
  {
    const ComponentDev& c = ch.comps.c[k];
    int j = -1;
    for (int r = 0; r < K; r++)
      if (F.joint[r].in == c.in) j = r;
    if (j < 0 || gc.ncols[j] + c.ncols > GX_COLS) return cudaErrorNotSupported;
    const int kinds[3][3] = {{GXK_SAT, GXK_OMEGA, 0}, {GXK_SGN, GXK_OMEGA, GXK_SQ}, {GXK_Q, GXK_ONE, 0}};
    const int row = c.type == RDB_COMPONENT_FRICTION_POLY1 ? 0 : (c.type == RDB_COMPONENT_FRICTION_POLY2 ? 1 : 2);
    for (int p = 0; p < c.ncols; p++)
    {
      const int g = gc.ncols[j]++;
      gc.kind[j][g] = kinds[row][p];
      gc.thr[j][g] = c.thr;
      gc.ithr[j][g] = 1.0 / c.thr;
      gc.vmax[j][g] = c.vmax;
      xmap[c.col + p] = j;
      xmap[Pc + c.col + p] = g;
    }
  }
  const bool rev = fold_rev_canonical(F);
  const int zc = GF_ZCOL && rev ? 1 : 0;  // GramGeom Z of the kernel that will run
  int xcmax = 0;
  for (int j = 0; j < K; j++) xcmax = std::max(xcmax, (int)gc.ncols[j]);
  int nxt = 0;
  for (int j = 0; j < K; j++) nxt += (1 + 10 * (K - j) - zc + 7) / 8 + 1;  // GramGeom::nxt
  const int Tt = (10 * K + 1 - zc + 7) / 8, ntt = Tt * (Tt + 1) / 2;      // GramGeom::T, NT
  // workspace: rigid block (P*P + P + 1) | cross sums (nxt*64) | per-CTA partials (sm_count*(ntt+nxt)*64) | component map (2 Pc ints)
  const size_t n_rigid = (size_t)P * P + P + 1, n_sum = (size_t)nxt * 64, n_part = (size_t)ch.sm_count * (ntt + nxt) * 64;
  cudaError_t e = grow(ch.gram.ext_dev, ch.gram.ext_bytes, sizeof(double) * (n_rigid + n_sum + n_part) + sizeof(int32_t) * 2 * (size_t)Pc);
  if (e != cudaSuccess) return e;
  double* Gt = ch.gram.ext_dev;
  double* bt = Gt + (size_t)P * P;
  double* tst = bt + P;
  double* xsum = tst + 1;
  double* xpart = xsum + n_sum;
  int32_t* dmap = reinterpret_cast<int32_t*>(xpart + n_part);
  e = cudaMemcpyAsync(dmap, xmap.data(), sizeof(int32_t) * xmap.size(), cudaMemcpyHostToDevice, st);  // pageable source: staged before return
  if (e != cudaSuccess) return e;
  switch (K)
  {
#define XL(N, R)                                                                                                  \
  (xcmax <= 2 ? launch_ext_nj<N, R, 2>(ch, gc, in, tau_meas, Gt, bt, tst, xpart, xsum, st)                         \
              : (xcmax <= 4 ? launch_ext_nj<N, R, 4>(ch, gc, in, tau_meas, Gt, bt, tst, xpart, xsum, st)           \
                            : launch_ext_nj<N, R, 8>(ch, gc, in, tau_meas, Gt, bt, tst, xpart, xsum, st)))
#define X(N)                                \
  case N:                                   \
  e = rev ? XL(N, true) : XL(N, false);     \
  break;
    X(1) X(2) X(3) X(4) X(5) X(6) X(7)
#undef X
#undef XL
  }
  if (e != cudaSuccess) return e;
  gram_ext_scatter_kernel<<<(P * (P + 1) + 255) / 256, 256, 0, st>>>(Gt, bt, tst, P, Pt, gram, rhs, tau_sq, accumulate);
  count_launch();
  const double* Tm1 = ch.gram.fold_identity ? nullptr : ch.gram.fold_dev;
  const int32_t* kof1 = ch.gram.fold_identity
                            ? nullptr
                            : reinterpret_cast<const int32_t*>(ch.gram.fold_dev + (size_t)nj * 100 + (size_t)(10 * K + 1) * (10 * K + 1));
  gram_cross_finish_kernel<<<((P + 1 + Pc) * Pc + 127) / 128, 128, 0, st>>>(xsum, Tm1, kof1, dmap, dmap + Pc, nj, K, Pc, gram, rhs, accumulate, zc);
  count_launch();
  return cudaGetLastError();
}

}  // namespace rdb
