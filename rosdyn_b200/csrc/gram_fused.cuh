// gram_fused.cuh -- fused regressor -> normal equations, one persistent warp-specialised kernel per GPU.
//
//   G (+)= sum_s Phi_s^T Phi_s ,  b (+)= sum_s Phi_s^T tau_s ,  tau_sq (+)= sum_s tau_s^T tau_s
//
// Phi never touches HBM.  The kernel runs on the FOLDED chain (fold.cpp: joints that never move are merged into the constant
// transform of the next moving joint, so every joint of the chain the kernel sees is an input and owns a row of Phi).  Per CTA (1 per SM):
//   * generator warps (one per SM sub-partition): one thread walks the chain of one sample (same link-frame recursion as dyn_kernel,
//     kernels.cu) and writes the augmented regressor rows [Phi_row | tau_row] of its 32 samples into a slot (only the structurally
//     non-zero columns, XOR-swizzled, conflict free).  The inputs of the next group are requested BEFORE waiting for the slot, so the DRAM
//     latency hides behind the consumers; sin/cos of all joints are evaluated up front (branch free), so the walk is one basic block.
//   * MMA warps: consume a slot as soon as it is full.  The contraction index k = (sample, joint row); a k-step is 4 samples of one joint
//     row, so the zero pattern of Phi (row of chain joint j is zero in the blocks of the links before j) is known at compile time and whole
//     8x8 tiles are skipped; inside the kernel the columns run tau, last link ... first link, so that every row is a PREFIX of tiles.  The
//     upper-triangular tiles of the (P+1)x(P+1) augmented Gram matrix stay in registers for the whole kernel; the four SM sub-partitions
//     split the k-steps of a slot, two warps per sub-partition split the tile rows by parity.  The k-steps of a slot
//     are fully unrolled and software pipelined: the fragments of step n+1 are loaded while the DMMAs of step n issue.
//     tcgen05 has no f64 kind: the FP64 tensor path of sm_100a is mma.sync.m8n8k4.f64 (SASS DMMA).
//   * as many slots as fit the 227 KB (3 for 7 joints, 4 below); with 4 each generator warp owns one and the slots cycle through mbarriers,
//     otherwise the 4 generator warps take turns over them and hand over through monotone counters (see the slot hand-off below).
//   * all-revolute chains drop the columns their walk makes exact zeros (GramGeom Z = 2): m and m c_z of a link on its own joint, and all
//     but I_zz, m c_x, m c_y of the first moving link; tau is no tile column but is accumulated by DFMA on the fragments the MMA warps load
//     anyway (b = Phi^T tau for the tile rows a warp owns, tau^T tau in one warp per k-split): 81 instead of 104 DMMA per 4 samples for 6
//     joints (125 / 149 for 7), plus 32 (42) DFMA.  The extended model keeps Z = 1 (only the own-joint mass dropped, tau in the tiles).
//   * all-revolute chains whose folded axes are all e_z (fold.cpp puts every revolute link in such a canonical frame) run the REV generator,
//     which holds the axis as a compile-time constant: 2 019 instead of 2 412 FP64 instructions per sample for 6 joints (2 658 / 3 119 for 7).
//   * on such chains the launchers run the same kernel compiled at run time against the chain's own constants (gram_jit.cpp, model type M):
//     the products with the exact zeros and ones of the model, and of the walk's state that inherits them (the base at rest, gravity, the
//     carried unit twists), are not issued: 1 082 FP64 instructions per sample for C6 (1 522 for C7), same results.
// Per-CTA partials (tiles, then b and tau^T tau) are summed in a fixed order by gram_fused_reduce_kernel (bit-reproducible for a given n).
// XC > 0: the extended model [Phi | Phi_c] (friction / spring columns) in ONE pass -- the same slots, the component columns of every joint
// in a small side buffer next to each slot, the MMA warps keep the rigid-body tiles and the cross tiles in registers.
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

// ---------------------------------------------------------------------------------------------- slot hand-off
// Where every generator warp owns one slot (B == SLOTS below), the slots cycle through mbarriers: one full / one empty per slot, arrive =
// release.cta, wait = acquire.cta, and a waiting warp is suspended by the hardware.  Otherwise (4 generator warps over 3 slots for 7 joints,
// and the extended model) the writer of a slot changes from use to use, a waiter can be more than one phase behind and the one-bit phase
// parity of an mbarrier would be ambiguous: monotone counters per slot instead, polled with a back-off.  Measured on the 4-slot C6 kernel,
// the counters cost 0.8 % (B200, 2.272 against 2.291 G samples/s).
constexpr int GF_POLL_NS = 32;  // back-off of the counter polls
struct GramBars
{
  uint64_t full[GF_MAX_SLOTS], empty[GF_MAX_SLOTS];  // mbarriers
  uint32_t filled[GF_MAX_SLOTS];                     // counters: uses of the slot written so far (generator, release)
  uint32_t drained[GF_MAX_SLOTS];                    // MMA-warp completions on the slot so far (GF_MMA_WARPS per use, release)
};
__device__ __forceinline__ void mbarrier_init(uint64_t* b, int count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarrier_arrive(uint64_t* b)
{
  asm volatile("{\n .reg .b64 st;\n mbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbarrier_wait(uint64_t* b, uint32_t parity)
{
  asm volatile(
      "{\n .reg .pred p;\n"
      "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      " @p bra D;\n bra W;\n"
      "D:\n}" ::"r"(smem_u32(b)),
      "r"(parity)
      : "memory");
}
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
  while (ld_acquire_u32(p) < v) __nanosleep(GF_POLL_NS);
}

// The k-th group of a CTA is produced by generator warp k % GF_GENS into slot k % SLOTS (its use k / SLOTS) and consumed in order by the MMA
// warps.  Global group of the k-th: ((k / B) gridDim.x + blockIdx.x) B + k % B, increasing in k, for a grid of min(SMs, ceil(groups / B))
// CTAs.  B = SLOTS: each CTA takes SLOTS consecutive groups at a time (the rigid-body kernel with 4 slots); B = 1: one group at a time.
// The order fixes which samples every per-CTA partial sums, so it fixes the rounding of the result.
template <int SLOTS, int XC>
__host__ __device__ constexpr int gram_group_block()
{
  return XC == 0 && SLOTS == GF_GENS ? SLOTS : 1;
}
template <int B>
__device__ __forceinline__ int64_t gram_group(int64_t k)
{
  return ((k / B) * gridDim.x + blockIdx.x) * B + k % B;
}
// the groups of this CTA: the number of k with gram_group<B>(k) < ngroups
template <int B>
__device__ __forceinline__ int64_t gram_cta_groups(int64_t ngroups)
{
  if constexpr (B == 1) return ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t nb = (ngroups + B - 1) / B;  // blocks of B groups, the last one possibly short
  if (nb <= blockIdx.x) return 0;
  const int64_t q = (nb - 1 - blockIdx.x) / gridDim.x;  // the last block of this CTA
  return q * B + min((int64_t)B, ngroups - (q * gridDim.x + blockIdx.x) * B);
}
// Which groups a CTA takes, chosen at compile time by the kernel: WIN = false, the CTA-strided walk above over the whole batch
// (gram_fused_kernel); WIN = true, every group of `in` in order (gram_fused_segmented_kernel hands each CTA its own window as `in`)
template <int B, bool WIN>
__device__ __forceinline__ int64_t gram_role_groups(int64_t ngroups)
{
  if constexpr (WIN) return ngroups;
  else return gram_cta_groups<B>(ngroups);
}
template <int B, bool WIN>
__device__ __forceinline__ int64_t gram_role_group(int64_t k)
{
  if constexpr (WIN) return k;
  else return gram_group<B>(k);
}

// ---------------------------------------------------------------------------------------------- extended model [Phi | Phi_c]
// The component columns of a joint -- element-wise functions of that joint's q, Dq (friction_polynomial1.h:45-52, friction_polynomial2.h:42-58,
// ideal_spring.h:64-70), non-zero in the row of that joint only -- go to a small side buffer next to the slots, XC columns per joint (2, 4
// or 8: the widest component set of the chain rounded up) instead of a zero-padded 8-column tile inside every row: for 6 joints with a
// friction model on each the kernel keeps 4 slots (4 x (52.5 + 3) KB) where the padded rows left room for 3 x 66 KB.  Then
//   Phi^T Phi_c [:, comps of j] = sum_s Phi_row_j(s)^T phi_c,j(s)      (one extra 8-wide tile per joint row),
// Phi_c^T Phi_c is block diagonal per joint and Phi_c^T tau rides in the tau column of the last regular tile.  The MMA warps keep BOTH tile
// sets in registers -- the upper triangular rigid-body tiles and, per joint row, the (regular tile, component tile) / (component, component)
// cross tiles -- so Phi is generated once.
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

// per-CTA partial: the rigid-body tiles (then, TC == 0, b and tau^T tau), then (XC) the cross tiles
template <int NJ, int Z, int XC>
__host__ __device__ constexpr int gram_partial_doubles()
{
  return GramGeom<NJ, Z>::PARTIAL + (XC ? GramGeom<NJ, Z>::NXT * 64 : 0);
}
// dynamic shared memory in doubles: the slots (or the partial where that is larger), then (XC) the component side buffer of each slot
template <int NJ, int Z, int SLOTS, int XC>
__host__ __device__ constexpr int gram_side_offset()
{
  return GramGeom<NJ, Z>::SLOT_DOUBLES * SLOTS > gram_partial_doubles<NJ, Z, XC>() ? GramGeom<NJ, Z>::SLOT_DOUBLES * SLOTS
                                                                                   : gram_partial_doubles<NJ, Z, XC>();
}
template <int NJ, int Z, int SLOTS, int XC>
__host__ __device__ constexpr int gram_smem_doubles()
{
  return gram_side_offset<NJ, Z, SLOTS, XC>() + SLOTS * gram_ext_side_doubles<NJ, XC>();
}
// weighted kernels: behind the side buffers, the weight of every (joint row, sample) of each slot, [joint][sample]
template <int NJ, int Z, int SLOTS, int XC, bool W>
__host__ __device__ constexpr int gram_smem_doubles_w()
{
  return gram_smem_doubles<NJ, Z, SLOTS, XC>() + (W ? SLOTS * 32 * NJ : 0);
}

// ---------------------------------------------------------------------------------------------- generator side
// W: weighted normal equations; the generator also stores the weight of each row of its sample (*wt, input order) behind the side buffers,
// [slot][joint][sample] (gram_smem_doubles_w)
template <int NJ, int SLOTS, bool REV, int Z, int XC, class M, bool WIN = false, bool W = false>
__device__ __forceinline__ void gram_gen_role(const ChainDev<NJ>& C, const GramComps& comps, const SamplesDev& in, const double* __restrict__ tau_meas,
                                              double* smem, double* side0, GramBars* bars, int w, int lane, int dbg,
                                              const rdb_gram_weights* wt = nullptr)
{
  using G = GramGeom<NJ, Z>;
  constexpr int B = gram_group_block<SLOTS, XC>();
  const int64_t nk = gram_role_groups<B, WIN>((in.n + 31) / 32);
  for (int64_t k = w; k < nk; k += GF_GENS)
  {
    const int s = (int)(k % SLOTS);
    const uint32_t u = (uint32_t)(k / SLOTS);
    // the inputs are requested BEFORE waiting for the slot: the DRAM latency hides behind the consumers' work on the previous group
    const int64_t i = gram_role_group<B, WIN>(k) * 32 + lane;
    GenIn<NJ> cur;
    gen_load<NJ>(C, in, min(i, in.n - 1), cur);
    double wv[W ? NJ : 1];
    if constexpr (W)
    {
      const int64_t iw = min(i, in.n - 1);
#pragma unroll
      for (int j = 0; j < NJ; j++) wv[j] = __ldg(wt->w + C.joint[j].in * wt->joint_stride + iw * wt->sample_stride);
    }
    trig_all<NJ>(cur.q, cur.sv, cur.cv);
    // every MMA warp is done with the previous use of the slot (mbarrier: the first wait, on parity 1, returns at once)
    if constexpr (B == SLOTS) mbarrier_wait(&bars->empty[s], (u & 1) ^ 1);
    else wait_counter_ge(&bars->drained[s], GF_MMA_WARPS * u);
    double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
    double* side = side0 + (size_t)s * gram_ext_side_doubles<NJ, XC>();
    if constexpr (W)
    {
      double* wrow = side0 + (size_t)SLOTS * gram_ext_side_doubles<NJ, XC>() + (size_t)s * 32 * NJ;
#pragma unroll
      for (int j = 0; j < NJ; j++) wrow[32 * j + lane] = wv[j];
    }
    if (XC > 0 || !(dbg & 1))
    {
      if constexpr (XC > 0) gram_component_park<NJ, XC>(cur, side, lane);
      gram_generate<NJ, REV, Z, M>(C, cur, in, tau_meas, slot, min(i, in.n - 1), lane);
      if constexpr (XC > 0) gram_component_side<NJ, XC>(comps, side, lane);
      if (i >= in.n)
      {
        gram_zero_lane<NJ, Z>(slot, lane);
        for (int c = 0; c < NJ * XC; c++) side[c * 32 + lane] = 0.0;
      }
    }
    __syncwarp();
    if (lane == 0)
    {
      if constexpr (B == SLOTS) mbarrier_arrive(&bars->full[s]);
      else st_release_u32(&bars->filled[s], u + 1);
    }
  }
}

// ---------------------------------------------------------------------------------------------- MMA side
// B fragments of one k-step (4 samples of joint row J, k-step kk of the slot): lane (g, t) holds column 8 I + g of sample 4 kk + t in b[I],
// and (GramGeom::TC == 0) the tau of joint J for that sample in b[T]
template <int NJ, int J, int Z>
__device__ __forceinline__ void gram_load_frags(const double* __restrict__ slot, int kk, int lane, double (&b)[GramGeom<NJ, Z>::NF])
{
  using G = GramGeom<NJ, Z>;
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
// XC: component fragment of one k-step: lane (g, t) holds column g of joint J for sample 4 kk + t (zero behind the XC stored columns)
template <int J, int XC>
__device__ __forceinline__ double gram_load_xside(const double* __restrict__ side, int kk, int lane)
{
  const int g = lane >> 2, t = lane & 3;
  return g < XC ? side[(J * XC + g) * 32 + 4 * kk + t] : 0.0;
}
// a: the A operands of the step -- the fragments b themselves, or in the weighted kernels b scaled by the weight of the lane's sample, so that
// every product of the step carries the weight once: G += A^T B = sum_s w_s Phi_s^T Phi_s (diagonal tiles keep their upper half)
template <int NJ, int PAR, int J, int Z>
__device__ __forceinline__ void gram_mma_step(const double (&a)[GramGeom<NJ, Z>::NF], const double (&b)[GramGeom<NJ, Z>::NF],
                                              double (&acc)[GramGeom<NJ, Z>::ntiles(PAR)][2])
{
  using G = GramGeom<NJ, Z>;
  constexpr int T = G::T, TJ = G::tj(J);
#pragma unroll
  for (int I = 0; I < T; I++)
  {
    if (I >= TJ || !G::owns(I, PAR)) continue;
#pragma unroll
    for (int K = I; K < T; K++)
      if (K < TJ) dmma884f(acc[G::local(I, K, PAR)][0], acc[G::local(I, K, PAR)][1], a[I], b[K]);
  }
}
// TC == 0: Phi^T tau on the tile rows this warp owns and (par 0) tau^T tau, by DFMA on the fragments of the step's DMMAs
template <int NJ, int PAR, int J, int Z>
__device__ __forceinline__ void gram_tau_step(const double (&a)[GramGeom<NJ, Z>::NF], const double (&b)[GramGeom<NJ, Z>::NF],
                                              double (&bacc)[GramGeom<NJ, Z>::nbacc(PAR)])
{
  using G = GramGeom<NJ, Z>;
  static_for<0, G::tj(J)>([&](auto Ic) {
    constexpr int I = decltype(Ic)::value;
    if constexpr (G::owns(I, PAR)) bacc[G::bown(I, PAR)] = fma(a[I], b[G::T], bacc[G::bown(I, PAR)]);
  });
  if constexpr (PAR == 0) bacc[G::nbacc(PAR) - 1] = fma(a[G::T], b[G::T], bacc[G::nbacc(PAR) - 1]);
}
// XC: the cross tiles of joint row J, (regular tile I, component tile) and (component, component); ax: the component fragment as A operand
template <int NJ, int PAR, int J, int Z, int NX>
__device__ __forceinline__ void gram_cross_step(const double (&a)[GramGeom<NJ, Z>::NF], double ax, double bx, double (&xacc)[NX][2])
{
  using G = GramGeom<NJ, Z>;
  static_for<0, G::tj(J) + 1>([&](auto Ic) {
    constexpr int I = decltype(Ic)::value;
    if constexpr (G::xowns(J, I, PAR))
    {
      constexpr int k = G::xlocal(J, I, PAR);
      if constexpr (I < G::tj(J)) dmma884f(xacc[k][0], xacc[k][1], a[I], bx);
      else dmma884f(xacc[k][0], xacc[k][1], ax, bx);  // (component, component) tile of joint J
    }
  });
}
// k-steps STEP.. of this warp in one slot; step = (joint row, k-step of the warp); the fragments of the next step are in flight while the
// DMMAs of the current one issue.  W: wrow holds the weights of the slot [joint][sample], wcur the weight of the lane's sample in this step
template <int NJ, int PAR, int STEP, int Z, int XC, int NX, bool W = false>
__device__ __forceinline__ void gram_consume_steps(const double* __restrict__ slot, const double* __restrict__ side, int ks, int lane,
                                                   const double (&bcur)[GramGeom<NJ, Z>::NF], double bxcur,
                                                   double (&acc)[GramGeom<NJ, Z>::ntiles(PAR)][2], double (&bacc)[GramGeom<NJ, Z>::nbacc(PAR)],
                                                   double (&xacc)[NX][2], const double* __restrict__ wrow = nullptr, double wcur = 1.0)
{
  using G = GramGeom<NJ, Z>;
  constexpr int J = STEP / G::KPW;
  double bnext[G::NF], bxnext = 0.0, wnext = 1.0;
  if constexpr (STEP + 1 < G::NSTEPS)
  {
    constexpr int JN = (STEP + 1) / G::KPW;
    const int kn = ks * G::KPW + (STEP + 1) % G::KPW;
    gram_load_frags<NJ, JN, Z>(slot, kn, lane, bnext);
    if constexpr (XC > 0) bxnext = gram_load_xside<JN, XC>(side, kn, lane);
    if constexpr (W) wnext = wrow[32 * JN + 4 * kn + (lane & 3)];
  }
  if constexpr (W)
  {
    // the A operands carry the weight: one DMUL per fragment this warp uses as A (the others are dead and not issued)
    double a[G::NF];
#pragma unroll
    for (int I = 0; I < G::NF; I++) a[I] = __dmul_rn(bcur[I], wcur);
    gram_mma_step<NJ, PAR, J, Z>(a, bcur, acc);
    if constexpr (!G::TC) gram_tau_step<NJ, PAR, J, Z>(a, bcur, bacc);
    if constexpr (XC > 0) gram_cross_step<NJ, PAR, J, Z>(a, __dmul_rn(bxcur, wcur), bxcur, xacc);
  }
  else
  {
    gram_mma_step<NJ, PAR, J, Z>(bcur, bcur, acc);
    if constexpr (!G::TC) gram_tau_step<NJ, PAR, J, Z>(bcur, bcur, bacc);
    if constexpr (XC > 0) gram_cross_step<NJ, PAR, J, Z>(bcur, bxcur, bxcur, xacc);
  }
  if constexpr (STEP + 1 < G::NSTEPS)
    gram_consume_steps<NJ, PAR, STEP + 1, Z, XC, NX, W>(slot, side, ks, lane, bnext, bxnext, acc, bacc, xacc, wrow, wnext);
}

// fixed-order reduction over the k-split warps that own the same tiles, into shared memory (the slots are dead by now)
template <int NJ, int PAR, int Z>
__device__ __forceinline__ void gram_mma_reduce(double (&acc)[GramGeom<NJ, Z>::ntiles(PAR)][2], double* smem, int ks, int lane)
{
  using G = GramGeom<NJ, Z>;
  bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  const int g = lane >> 2, t = lane & 3;
  for (int w = 0; w < GF_KSPLIT; w++)
  {
    if (ks == w)
    {
#pragma unroll
      for (int I = 0; I < G::T; I++)
      {
        if (!G::owns(I, PAR)) continue;
#pragma unroll
        for (int J = I; J < G::T; J++)
        {
          double* o = smem + G::tile(I, J) * 64 + g * 8 + 2 * t;
          const int k = G::local(I, J, PAR);
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
__device__ __forceinline__ void gram_tau_reduce(double (&bacc)[GramGeom<NJ, Z>::nbacc(PAR)], double* smem, int ks, int lane)
{
  using G = GramGeom<NJ, Z>;
  constexpr int NB = G::nbacc(PAR);
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
        if (!G::owns(I, PAR)) continue;
        double& o = ob[8 * I + g];
        o = w == 0 ? bacc[G::bown(I, PAR)] : o + bacc[G::bown(I, PAR)];
      }
      if (PAR == 0 && g == 0) ob[8 * G::T] = w == 0 ? bacc[NB - 1] : ob[8 * G::T] + bacc[NB - 1];
    }
    bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  }
}
// XC: fixed-order reduction of the cross tiles over the k-split warps into shared memory at `smem` (NXT tiles of 64 doubles)
template <int NJ, int PAR, int Z, int NX>
__device__ __forceinline__ void gram_cross_reduce_smem(double (&xacc)[NX][2], double* smem, int ks, int lane)
{
  using G = GramGeom<NJ, Z>;
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
          if constexpr (G::xowns(j, I, PAR))
          {
            double* o = smem + G::xtile(j, I) * 64 + g * 8 + 2 * t;
            constexpr int k = G::xlocal(j, I, PAR);
            if (w == 0)
            {
              o[0] = xacc[k][0];
              o[1] = xacc[k][1];
            }
            else
            {
              o[0] += xacc[k][0];
              o[1] += xacc[k][1];
            }
          }
        });
      });
    }
    bar_sync(GF_BAR_REDUCE, 32 * GF_MMA_WARPS);
  }
}

template <int NJ, int SLOTS, int PAR, int Z, int XC, bool WIN = false, bool W = false>
__device__ __forceinline__ void gram_mma_role(const SamplesDev& in, double* smem, const double* side0, GramBars* bars, int ks, int lane, int dbg,
                                              const double* wrow0 = nullptr)
{
  using G = GramGeom<NJ, Z>;
  constexpr int B = gram_group_block<SLOTS, XC>();
  constexpr int NTP = G::ntiles(PAR), NB = G::nbacc(PAR), NX = XC ? G::nxtiles(PAR) : 1;
  double acc[NTP][2], bacc[NB], xacc[NX][2];
#pragma unroll
  for (int k = 0; k < NTP; k++) acc[k][0] = acc[k][1] = 0.0;
#pragma unroll
  for (int k = 0; k < NB; k++) bacc[k] = 0.0;
#pragma unroll
  for (int k = 0; k < NX; k++) xacc[k][0] = xacc[k][1] = 0.0;
  const int64_t nk = gram_role_groups<B, WIN>((in.n + 31) / 32);
#pragma unroll 1
  for (int64_t k = 0; k < nk; k++)
  {
    const int s = (int)(k % SLOTS);
    const uint32_t u = (uint32_t)(k / SLOTS);
    const double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
    const double* side = side0 + (size_t)s * gram_ext_side_doubles<NJ, XC>();
    if constexpr (B == SLOTS) mbarrier_wait(&bars->full[s], u & 1);
    else wait_counter_ge(&bars->filled[s], u + 1);
    if (XC > 0 || !(dbg & 2))
    {
      double b0[G::NF], bx0 = 0.0;
      gram_load_frags<NJ, 0, Z>(slot, ks * G::KPW, lane, b0);
      if constexpr (XC > 0) bx0 = gram_load_xside<0, XC>(side, ks * G::KPW, lane);
      if constexpr (W)
      {
        const double* wrow = wrow0 + (size_t)s * 32 * NJ;
        gram_consume_steps<NJ, PAR, 0, Z, XC, NX, true>(slot, side, ks, lane, b0, bx0, acc, bacc, xacc, wrow,
                                                        wrow[4 * ks * G::KPW + (lane & 3)]);
      }
      else gram_consume_steps<NJ, PAR, 0, Z, XC>(slot, side, ks, lane, b0, bx0, acc, bacc, xacc);
    }
    __syncwarp();
    if (lane == 0)
    {
      if constexpr (B == SLOTS) mbarrier_arrive(&bars->empty[s]);
      else red_release_inc(&bars->drained[s]);
    }
  }
  gram_mma_reduce<NJ, PAR, Z>(acc, smem, ks, lane);  // rigid-body tiles: smem[0, NT * 64)
  if constexpr (!G::TC) gram_tau_reduce<NJ, PAR, Z>(bacc, smem, ks, lane);
  if constexpr (XC > 0) gram_cross_reduce_smem<NJ, PAR, Z>(xacc, smem + G::NT * 64, ks, lane);  // cross tiles behind them
}

// XC = 0: the rigid-body model.  XC = 2, 4, 8: the extended model [Phi | Phi_c] in ONE pass, XC component columns per joint.
// M: model constants (gram_common.cuh) -- RtModel for the precompiled instantiations, a generated model type in gram_jit.cpp.
// dbg (development builds only, RDB_GRAM_DEBUG): 1 skips the generation, 2 the MMAs; rigid-body model only (XC = 0): the two tests cost the
// extended kernels spill (C6, XC = 2, not REV: 232 -> 296 bytes).
template <int NJ, int SLOTS, bool REV, int XC, class M = RtModel>
__global__ void __launch_bounds__(GF_THREADS, 1)
    gram_fused_kernel(const __grid_constant__ ChainDev<NJ> C, const __grid_constant__ GramComps comps, const SamplesDev in,
                      const double* __restrict__ tau_meas, double* __restrict__ partial, const int dbg)
{
  // Z (gram_common.cuh): on all-revolute chains the exact-zero columns of the REV walk are neither stored nor multiplied; the extended model
  // drops only the own-joint mass column and keeps tau in the tiles (its Phi_c^T tau rides in the tau column)
  constexpr int Z = REV ? (XC ? 1 : 2) : 0;
  using G = GramGeom<NJ, Z>;
  constexpr int NOUT = gram_partial_doubles<NJ, Z, XC>();
  extern __shared__ __align__(16) double smem[];
  __shared__ GramBars bars;
  double* const side0 = smem + gram_side_offset<NJ, Z, SLOTS, XC>();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if constexpr (gram_group_block<SLOTS, XC>() == SLOTS)
  {
    if (threadIdx.x == 0)
    {
      for (int s = 0; s < SLOTS; s++)
      {
        mbarrier_init(&bars.full[s], 1);              // lane 0 of the generator warp, after __syncwarp
        mbarrier_init(&bars.empty[s], GF_MMA_WARPS);  // lane 0 of every MMA warp
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  else if (threadIdx.x < SLOTS)
  {
    bars.filled[threadIdx.x] = 0;
    bars.drained[threadIdx.x] = 0;
  }
  __syncthreads();
  if (warp >= GF_MMA_WARPS)
  {
    gram_gen_role<NJ, SLOTS, REV, Z, XC, M>(C, comps, in, tau_meas, smem, side0, &bars, warp - GF_MMA_WARPS, lane, dbg);
    return;
  }
  // ------------------------------------------------ MMA warps: k-split index = warp % 4 (its SM sub-partition), tile-row parity = warp / 4
  const int mma_id = warp, ks = mma_id % GF_KSPLIT;
  if (mma_id < GF_KSPLIT) gram_mma_role<NJ, SLOTS, 0, Z, XC>(in, smem, side0, &bars, ks, lane, dbg);
  else gram_mma_role<NJ, SLOTS, 1, Z, XC>(in, smem, side0, &bars, ks, lane, dbg);
  double* out = partial + (size_t)blockIdx.x * NOUT;
  for (int k = mma_id * 32 + lane; k < NOUT; k += 32 * GF_MMA_WARPS) out[k] = smem[k];
}

// Weighted normal equations (rdb_regressor_gram_weighted_batch, rdb_regressor_gram_ext_weighted_batch):
//   G (+)= sum_s Phi_s^T W_s Phi_s ,  b (+)= sum_s Phi_s^T W_s tau_s ,  tau_sq (+)= sum_s tau_s^T W_s tau_s ,  W_s = diag(w of the rows of s)
// The weight of the row of folded joint j in sample i is wt.w[C.joint[j].in * wt.joint_stride + i * wt.sample_stride].  The generator loads
// it with the sample's inputs and stores it beside the slot; the MMA warps scale the A operands of every k-step by it (gram_consume_steps):
// per k-step and warp one shared load and one DMUL per tile row it owns, and nothing more in the generator warp, which bounds the kernel.
// Grid, groups, slots of the rigid-body kernel and every summation order are those of gram_fused_kernel, so w == 1 gives its results bit
// for bit, and a power-of-two weight scales them exactly.  The extended model may keep fewer slots than gram_fused_kernel (the weights take
// shared memory); its CTAs take one group at a time either way, so the order of the sums does not depend on the slots.
// Otherwise this is gram_fused_kernel line for line (kept apart for the reason given at gram_fused_segmented_kernel).
template <int NJ, int SLOTS, bool REV, int XC, class M = RtModel>
__global__ void __launch_bounds__(GF_THREADS, 1)
    gram_fused_weighted_kernel(const __grid_constant__ ChainDev<NJ> C, const __grid_constant__ GramComps comps, const SamplesDev in,
                               const double* __restrict__ tau_meas, const __grid_constant__ rdb_gram_weights wt, double* __restrict__ partial,
                               const int dbg)
{
  constexpr int Z = REV ? (XC ? 1 : 2) : 0;
  constexpr int NOUT = gram_partial_doubles<NJ, Z, XC>();
  extern __shared__ __align__(16) double smem[];
  __shared__ GramBars bars;
  double* const side0 = smem + gram_side_offset<NJ, Z, SLOTS, XC>();
  double* const wrow0 = smem + gram_smem_doubles<NJ, Z, SLOTS, XC>();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if constexpr (gram_group_block<SLOTS, XC>() == SLOTS)
  {
    if (threadIdx.x == 0)
    {
      for (int s = 0; s < SLOTS; s++)
      {
        mbarrier_init(&bars.full[s], 1);
        mbarrier_init(&bars.empty[s], GF_MMA_WARPS);
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  else if (threadIdx.x < SLOTS)
  {
    bars.filled[threadIdx.x] = 0;
    bars.drained[threadIdx.x] = 0;
  }
  __syncthreads();
  if (warp >= GF_MMA_WARPS)
  {
    gram_gen_role<NJ, SLOTS, REV, Z, XC, M, false, true>(C, comps, in, tau_meas, smem, side0, &bars, warp - GF_MMA_WARPS, lane, dbg, &wt);
    return;
  }
  const int mma_id = warp, ks = mma_id % GF_KSPLIT;
  if (mma_id < GF_KSPLIT) gram_mma_role<NJ, SLOTS, 0, Z, XC, false, true>(in, smem, side0, &bars, ks, lane, dbg, wrow0);
  else gram_mma_role<NJ, SLOTS, 1, Z, XC, false, true>(in, smem, side0, &bars, ks, lane, dbg, wrow0);
  double* out = partial + (size_t)blockIdx.x * NOUT;
  for (int k = mma_id * 32 + lane; k < NOUT; k += 32 * GF_MMA_WARPS) out[k] = smem[k];
}

// Segmented normal equations (rdb_regressor_gram_segmented_batch): CTA b owns work item b, the window [items[2 b], + items[2 b + 1]) of the
// batch, which lies inside one segment.  The roles see that window as their batch (plane pointers and tau_meas offset to its start, n = its
// length: ld_in loads by plane stride, so nothing else moves), take its groups in order (WIN), and clamp and zero lanes at its end.  The
// partial of item b goes to partial + b NOUT, in the layout of gram_fused_kernel; gram_fused.cu sums the items of a segment in item order.
// Otherwise this is gram_fused_kernel line for line.  The two do not share a device function for the body: with one more inline level
// ptxas derived other known bits of the lane index and the extended instantiations of gram_fused_kernel compiled to different instructions.
template <int NJ, int SLOTS, bool REV, int XC = 0, class M = RtModel>
__global__ void __launch_bounds__(GF_THREADS, 1)
    gram_fused_segmented_kernel(const __grid_constant__ ChainDev<NJ> C, const __grid_constant__ GramComps comps, const SamplesDev in,
                                const double* __restrict__ tau_meas, const int64_t* __restrict__ items, double* __restrict__ partial,
                                const int dbg)
{
  constexpr int Z = REV ? (XC ? 1 : 2) : 0;
  constexpr int NOUT = gram_partial_doubles<NJ, Z, XC>();
  extern __shared__ __align__(16) double smem[];
  __shared__ GramBars bars;
  // the window lives in shared memory, not in registers: the roles reread it where the unsegmented kernel rereads its parameters
  __shared__ SamplesDev win;
  __shared__ const double* tm;
  double* const side0 = smem + gram_side_offset<NJ, Z, SLOTS, XC>();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 32)
  {
    const int64_t s0 = items[2 * (int64_t)blockIdx.x];
    win = SamplesDev{items[2 * (int64_t)blockIdx.x + 1], in.ld, in.q + s0, in.dq + s0, in.ddq + s0, nullptr};
    tm = tau_meas ? tau_meas + s0 : nullptr;
  }
  if constexpr (gram_group_block<SLOTS, XC>() == SLOTS)
  {
    if (threadIdx.x == 0)
    {
      for (int s = 0; s < SLOTS; s++)
      {
        mbarrier_init(&bars.full[s], 1);
        mbarrier_init(&bars.empty[s], GF_MMA_WARPS);
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  else if (threadIdx.x < SLOTS)
  {
    bars.filled[threadIdx.x] = 0;
    bars.drained[threadIdx.x] = 0;
  }
  __syncthreads();
  if (warp >= GF_MMA_WARPS)
  {
    gram_gen_role<NJ, SLOTS, REV, Z, XC, M, true>(C, comps, win, tm, smem, side0, &bars, warp - GF_MMA_WARPS, lane, dbg);
    return;
  }
  const int mma_id = warp, ks = mma_id % GF_KSPLIT;
  if (mma_id < GF_KSPLIT) gram_mma_role<NJ, SLOTS, 0, Z, XC, true>(win, smem, side0, &bars, ks, lane, dbg);
  else gram_mma_role<NJ, SLOTS, 1, Z, XC, true>(win, smem, side0, &bars, ks, lane, dbg);
  double* out = partial + (size_t)blockIdx.x * NOUT;
  for (int k = mma_id * 32 + lane; k < NOUT; k += 32 * GF_MMA_WARPS) out[k] = smem[k];
}

}  // namespace rdb
