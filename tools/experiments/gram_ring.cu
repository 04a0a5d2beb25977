// gram_ring.cu -- fused regressor -> normal equations, generator warps decoupled from the shared-memory slots through an L2-resident ring.
//
//   G (+)= sum_s Phi_s^T Phi_s ,  b (+)= sum_s Phi_s^T tau_s ,  tau_sq (+)= sum_s tau_s^T tau_s        (Phi never touches HBM)
//
// Why: in gram_fused.cu a generator warp writes its 32 samples straight into a shared-memory slot, so the samples in flight per SM (4 slots =
// 128 samples in 221 KB) cap the generators at ONE warp per SM sub-partition.  One warp cannot keep the FP64 datapath busy on its own (a third of
// its instructions are not FP64, plus instruction-cache and scoreboard stalls: ~50 % utilisation when it runs alone), and while the MMA warps
// hold the datapath the scheduler grants it one DFMA per two DMMAs -- so the phases alternate and 18 % (7-joint chain: 29 %) of the datapath
// cycles stay idle (profiles/r01_gram_fused_v5_ncu.txt, VERDICT round 1).
//
// Here, per CTA (1 per SM, 12 warps):
//   * 8 generator warps (two per sub-partition) walk 32 samples each and write the augmented rows [Phi_row | tau_row] with st.global.cg into
//     their own entry of a ring in GLOBAL memory (8 entries of one slot each per CTA; 65 MB for 148 CTAs of a 6-joint chain: it lives in the
//     126 MB L2 and is overwritten every few microseconds, so it never reaches HBM).  The slot image is the swizzled shared-memory layout.
//   * one elected lane of MMA warp 0 moves finished entries into the shared-memory slots, in group order, with ONE TMA bulk copy each
//     (cp.async.bulk.shared.global with mbarrier complete_tx), as soon as the slot has been released by the four MMA warps.
//   * 4 MMA warps (one per sub-partition, k-split; each owns all upper-triangular tiles) consume the slots exactly as in gram_fused.cu
//     (DMMA m8n8k4, fragments of the next k-step in flight while the current one issues).
// Generation is no longer bounded by the slots: two generator warps per sub-partition overlap each other's stalls and together receive two
// datapath grants per DMMA instead of one per two.
// On all-revolute chains the rows are also one position shorter (GramGeom Z = 1: the mass column of a link on its own joint is an exact zero,
// put last in its block and neither stored nor multiplied): 98 instead of 104 DMMA per 4 samples for the folded 6-joint chain, 143 / 149 for 7.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "gram_common.cuh"
#include "launch.h"

namespace rdb
{

constexpr int GR_GENS = 8;       // generator warps per CTA = ring entries per CTA
constexpr int GR_MMA_WARPS = 4;  // one per SM sub-partition (k-split), each owns all tiles
constexpr int GR_BAR_REDUCE = 1;
constexpr int GR_BAR_PAIR0 = 2;    // named barriers 2..5: the two generator warps of a sub-partition

struct RingBars
{
  uint64_t full[GF_MAX_SLOTS];   // slot filled by the TMA copy (1 arrival + transaction bytes)
  uint64_t empty[GF_MAX_SLOTS];  // slot released by the GR_MMA_WARPS consumers
  uint64_t ring_full[GR_GENS];   // ring entry written by its generator warp
  uint64_t ring_free[GR_GENS];   // ring entry copied out (its TMA completed)
};

__device__ __forceinline__ bool mbar_try(uint64_t* b, uint32_t parity)
{
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      " selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(smem_u32(b)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes)
{
  asm volatile("{\n .reg .b64 st;\n mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
// one TMA bulk copy global -> shared memory of this CTA, completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_bulk(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)), "l"(gsrc),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---------------------------------------------------------------------------------------------- MMA side (geometry G, every warp owns all tiles)
template <class G, int J>
__device__ __forceinline__ void ring_load_frags(const double* __restrict__ slot, int kk, int lane, double (&b)[G::T])
{
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
template <class G, int J>
__device__ __forceinline__ void ring_mma_step(const double (&b)[G::T], double (&acc)[G::NT][2])
{
  constexpr int T = G::T, TJ = G::tj(J);
#pragma unroll
  for (int I = 0; I < T; I++)
  {
    if (I >= TJ) continue;
#pragma unroll
    for (int K = I; K < T; K++)
      if (K < TJ) dmma884f(acc[G::tile(I, K)][0], acc[G::tile(I, K)][1], b[I], b[K]);
  }
}
// k-steps of this warp in one slot, software pipelined: the fragments of step n + 1 are in flight while the DMMAs of step n issue
template <class G, int STEP>
__device__ __forceinline__ void ring_consume_steps(const double* __restrict__ slot, int ks, int lane, const double (&bcur)[G::T], double (&acc)[G::NT][2])
{
  constexpr int J = STEP / G::KPW;
  if constexpr (STEP + 1 < G::NSTEPS)
  {
    double bnext[G::T];
    ring_load_frags<G, (STEP + 1) / G::KPW>(slot, ks * G::KPW + (STEP + 1) % G::KPW, lane, bnext);
    ring_mma_step<G, J>(bcur, acc);
    ring_consume_steps<G, STEP + 1>(slot, ks, lane, bnext, acc);
  }
  else
    ring_mma_step<G, J>(bcur, acc);
}

template <int NJ, int SLOTS, bool REV>
__global__ void __launch_bounds__(32 * (GR_MMA_WARPS + GR_GENS), 1)
    gram_ring_kernel(const __grid_constant__ ChainDev<NJ> C, const SamplesDev in, const double* __restrict__ tau_meas, double* __restrict__ ring,
                     double* __restrict__ partial)
{
  constexpr int Z = REV ? 1 : 0;
  using G = GramGeom<NJ, 0, Z>;
  constexpr uint32_t SLOT_BYTES = (uint32_t)(G::SLOT_DOUBLES * sizeof(double));
  static_assert(SLOT_BYTES % 16 == 0, "TMA bulk copies move multiples of 16 bytes");
  extern __shared__ __align__(128) double smem[];
  __shared__ RingBars bars;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0)
  {
    for (int s = 0; s < SLOTS; s++)
    {
      mbar_init(&bars.full[s], 1);              // the issuing lane's arrive.expect_tx; the copy itself completes the transaction bytes
      mbar_init(&bars.empty[s], GR_MMA_WARPS);  // lane 0 of every MMA warp
    }
    for (int e = 0; e < GR_GENS; e++)
    {
      mbar_init(&bars.ring_full[e], 1);  // lane 0 of the generator warp
      mbar_init(&bars.ring_free[e], 1);  // the issuing lane, once the copy of the entry has landed
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // groups of 32 samples, interleaved over the CTAs: the k-th group of this CTA is group blockIdx.x + k gridDim.x; generator warp k % GR_GENS
  // produces it into its ring entry, slot k % SLOTS receives it
  const int64_t ngroups = (in.n + 31) / 32;
  const int64_t nk = ngroups > blockIdx.x ? (ngroups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  double* const my_ring = ring + (size_t)blockIdx.x * GR_GENS * G::SLOT_DOUBLES;

  if (warp >= GR_MMA_WARPS)
  {
    // ------------------------------------------------ generator warp e: groups e, e + GR_GENS, ...
    // The two generator warps of sub-partition s (warps 4 + s and 8 + s) produce adjacent groups (ring entries 2 s and 2 s + 1) and enter the
    // walk of every group together (named barrier 2 + s): they then go through the ~65 KB of unrolled generator code side by side and share its
    // instruction-cache lines.  Eight warps at eight unrelated places of that code miss the instruction cache on 40 % of their issue slots
    // (profiles/r02_gram_ring_v1_ncu.txt: no_instruction 6.1 stalls per issue).
    const int sp = (warp - GR_MMA_WARPS) & 3, half = (warp - GR_MMA_WARPS) >> 2;
    const int e = 2 * sp + half;
    double* const entry = my_ring + (size_t)e * G::SLOT_DOUBLES;
    const int64_t pair_iters = nk > 2 * sp ? (nk - 2 * sp + GR_GENS - 1) / GR_GENS : 0;  // iterations of the pair's first warp (>= the second's)
    for (int64_t m64 = 0; m64 < pair_iters; m64++)
    {
      const uint32_t m = (uint32_t)m64;  // uses of the entry so far
      const int64_t k = e + m64 * GR_GENS;
      const bool work = k < nk;
      const int64_t i = ((int64_t)blockIdx.x + k * gridDim.x) * 32 + lane;
      GenIn<NJ> cur;
#ifdef RING_EAGER_LOADS
      gen_load<NJ>(C, in, min(i, in.n - 1), cur);
#else
#pragma unroll
      for (int l = 0; l < NJ; l++) cur.q[l] = ld_in(in.q, C.joint[l].in, in.ld, min(i, in.n - 1));
#endif
      trig_all<NJ>(cur.q, cur.sv, cur.cv);
      if (work && m > 0) mbar_wait(&bars.ring_free[e], (m - 1) & 1);  // the previous contents have been copied out
#ifndef RING_UNPAIRED
      bar_sync(GR_BAR_PAIR0 + sp, 64);
#endif
      if (!work) continue;
#ifdef RING_EAGER_LOADS
      gram_generate<NJ, REV, 0, Z, true, false>(C, nullptr, cur, in, tau_meas, entry, min(i, in.n - 1), lane);
#else
      gram_generate<NJ, REV, 0, Z, true, true>(C, nullptr, cur, in, tau_meas, entry, min(i, in.n - 1), lane);
#endif
      if (i >= in.n) gram_zero_lane<NJ, 0, Z, true>(entry, lane);
      // the rows were written through the generic proxy; the TMA engine reads them through the async proxy
#ifndef RING_NO_THREADFENCE
      __threadfence();
#endif
      asm volatile("fence.proxy.async;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.ring_full[e]);
    }
    return;
  }

  // ------------------------------------------------ MMA warps: k-split index = warp (its SM sub-partition)
  const int ks = warp;
  double acc[G::NT][2];
#pragma unroll
  for (int t = 0; t < G::NT; t++) acc[t][0] = acc[t][1] = 0.0;
  int64_t next_issue = 0;  // (warp 0, lane 0) next group whose ring entry -> slot copy has not been issued yet
  for (int64_t k = 0; k < nk; k++)
  {
    const int s = (int)(k % SLOTS);
    if (ks == 0 && lane == 0)
    {
      // issue, in group order, every copy whose ring entry is written and whose slot has been released; group k itself is waited for
      while (next_issue < nk && next_issue < k + SLOTS)
      {
        const int en = (int)(next_issue % GR_GENS), sn = (int)(next_issue % SLOTS);
        const uint32_t pr = (uint32_t)((next_issue / GR_GENS) & 1);       // ring_full: phase = use of the entry
        const uint32_t pe = (uint32_t)(((next_issue / SLOTS) & 1) ^ 1);  // empty: phase use - 1 (use 0: a fresh barrier passes parity 1)
        if (next_issue == k)
        {
          mbar_wait(&bars.ring_full[en], pr);
          mbar_wait(&bars.empty[sn], pe);
        }
        else if (!(mbar_try(&bars.ring_full[en], pr) && mbar_try(&bars.empty[sn], pe)))
          break;
        mbar_expect_tx(&bars.full[sn], SLOT_BYTES);
        tma_load_bulk(smem + (size_t)sn * G::SLOT_DOUBLES, my_ring + (size_t)en * G::SLOT_DOUBLES, SLOT_BYTES, &bars.full[sn]);
        next_issue++;
      }
    }
    __syncwarp();
    const double* slot = smem + (size_t)s * G::SLOT_DOUBLES;
    mbar_wait(&bars.full[s], (uint32_t)((k / SLOTS) & 1));
    if (ks == 0 && lane == 0) mbar_arrive(&bars.ring_free[k % GR_GENS]);  // the copy has landed: the generator may overwrite its entry
    {
      double b0[G::T];
      ring_load_frags<G, 0>(slot, ks * G::KPW, lane, b0);
      ring_consume_steps<G, 0>(slot, ks, lane, b0, acc);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&bars.empty[s]);
  }
  // fixed-order reduction over the k-split warps into shared memory (the slots are dead by now)
  bar_sync(GR_BAR_REDUCE, 32 * GR_MMA_WARPS);
  const int g = lane >> 2, t = lane & 3;
  for (int w = 0; w < GR_MMA_WARPS; w++)
  {
    if (ks == w)
    {
#pragma unroll
      for (int I = 0; I < G::T; I++)
#pragma unroll
        for (int J = I; J < G::T; J++)
        {
          double* o = smem + G::tile(I, J) * 64 + g * 8 + 2 * t;
          const int kt = G::tile(I, J);
          if (w == 0)
          {
            o[0] = acc[kt][0];
            o[1] = acc[kt][1];
          }
          else
          {
            o[0] += acc[kt][0];
            o[1] += acc[kt][1];
          }
        }
    }
    bar_sync(GR_BAR_REDUCE, 32 * GR_MMA_WARPS);
  }
  constexpr int NOUT = G::NT * 64;
  double* out = partial + (size_t)blockIdx.x * NOUT;
  for (int k2 = warp * 32 + lane; k2 < NOUT; k2 += 32 * GR_MMA_WARPS) out[k2] = smem[k2];
}

// fixed-order sum of the per-CTA partials -> gram (full symmetric, column-major), rhs, tau_sq.  zcol: GramGeom Z = 1 position order.
__global__ void gram_ring_reduce_kernel(const double* __restrict__ partial, int nparts, int T, int P, int zcol, double* __restrict__ gram,
                                        double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  const int NT = T * (T + 1) / 2;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NT * 64) return;
  int k = e >> 6, I = 0;
  while (k >= T - I)
  {
    k -= T - I;
    I++;
  }
  const int J = I + k;
  const int rp = 8 * I + ((e >> 3) & 7), cp = 8 * J + (e & 7);  // positions inside the kernel (GramGeom::pos)
  const int npos = P + 1 - zcol;                                // positions that exist
  if (rp >= npos || cp >= npos) return;
  if (I == J && rp > cp) return;  // diagonal tiles hold both halves; keep the upper one
  double s = 0.0;
  for (int p = 0; p < nparts; p++) s += partial[(size_t)p * NT * 64 + e];
  // position -> column of the (folded) parameter vector, P = tau
  const int nj = P / 10;
  auto col_of = [&](int pos) {
    if (pos == 0) return P;
    const int l = nj - 1 - (pos - 1) / 10, q = (pos - 1) % 10;
    return 10 * l + (zcol ? (q == 9 ? 0 : q + 1) : q);
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
// Z = 1 never touches the mass column of the first moving link (position 10 NJ): its row / column of the normal equations is exactly zero
__global__ void gram_ring_zero_first_mass_kernel(int P, double* __restrict__ gram, double* __restrict__ rhs, int accumulate)
{
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (accumulate || e > P) return;
  if (e == P)
  {
    rhs[0] = 0.0;
    return;
  }
  gram[(size_t)e * P] = 0.0;  // column e, row 0
  gram[e] = 0.0;              // column 0, row e
}

template <int NJ>
static ChainDev<NJ> narrow_r(const ChainDev<RDB_MAX_JOINTS>& h)
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

static cudaError_t grow_r(double*& p, size_t& have, size_t need)
{
  if (have >= need) return cudaSuccess;
  if (p) cudaFree(p);
  p = nullptr;
  have = 0;
  cudaError_t e = cudaMalloc(&p, need);
  if (e == cudaSuccess) have = need;
  return e;
}

template <int NJ, int Z>
constexpr int gr_slots()
{
  return std::min<int>(GF_MAX_SLOTS, (int)((227 * 1024 - 1024) / (sizeof(double) * GramGeom<NJ, 0, Z>::SLOT_DOUBLES)));
}

template <int NJ, bool REV>
static cudaError_t launch_ring_nj(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                  int accumulate, cudaStream_t st)
{
  constexpr int Z = REV ? 1 : 0;
  using G = GramGeom<NJ, 0, Z>;
  constexpr int SLOTS = gr_slots<NJ, Z>();
  const size_t smem = sizeof(double) * (size_t)std::max(G::SLOT_DOUBLES * SLOTS, G::NT * 64);
  cudaError_t e = cudaFuncSetAttribute(gram_ring_kernel<NJ, SLOTS, REV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t ngroups = (in.n + 31) / 32;
  const int grid = (int)std::min<int64_t>(ch.sm_count, ngroups);
  e = grow_r(ch.gram.fused_partials, ch.gram.fused_bytes, sizeof(double) * (size_t)ch.sm_count * (GramGeom<NJ>::NT + 1) * 64);
  if (e != cudaSuccess) return e;
  e = grow_r(ch.gram.ring, ch.gram.ring_bytes, sizeof(double) * (size_t)ch.sm_count * GR_GENS * G::SLOT_DOUBLES);
  if (e != cudaSuccess) return e;
  gram_ring_kernel<NJ, SLOTS, REV><<<grid, 32 * (GR_MMA_WARPS + GR_GENS), smem, st>>>(narrow_r<NJ>(ch.gram.fold), in, tau_meas, ch.gram.ring,
                                                                                     ch.gram.fused_partials);
  count_launch();
  const int nred = (G::NT * 64 + 255) / 256;
  if (ch.gram.fold_identity)
  {
    if (Z)
    {
      gram_ring_zero_first_mass_kernel<<<(G::P + 1 + 127) / 128, 128, 0, st>>>(G::P, gram, rhs, accumulate);
      count_launch();
    }
    gram_ring_reduce_kernel<<<nred, 256, 0, st>>>(ch.gram.fused_partials, grid, G::T, G::P, Z, gram, rhs, tau_sq, accumulate);
    count_launch();
    return cudaGetLastError();
  }
  // folded chain: reduce into G', b', then expand to the reference's full parameter vector (gram_fold_expand_kernel, gram_fused.cu)
  const int nj = ch.host.nj, Pr = G::P;
  double* Tm = ch.gram.fold_dev;
  double* Gr = Tm + (size_t)nj * 100;
  double* br = Gr + (size_t)Pr * Pr;
  double* tsr = br + Pr;
  if (Z)
  {
    gram_ring_zero_first_mass_kernel<<<(Pr + 1 + 127) / 128, 128, 0, st>>>(Pr, Gr, br, 0);
    count_launch();
  }
  gram_ring_reduce_kernel<<<nred, 256, 0, st>>>(ch.gram.fused_partials, grid, G::T, G::P, Z, Gr, br, tsr, 0);
  count_launch();
  return launch_fold_expand(ch, gram, rhs, tau_sq, accumulate, st);
}

// cudaErrorNotSupported when the chain does not fit (the caller tries the slot kernel of gram_fused.cu, then the general pipeline)
cudaError_t launch_gram_ring(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                             int accumulate, cudaStream_t st)
{
  if (in.n <= 0 || ch.gram.fold_version != ch.model_version) return cudaErrorNotSupported;
  const bool rev = fold_rev_canonical(ch.gram.fold);  // all moving joints revolute about e_z: the specialised generator and the shorter rows
  switch (ch.gram.fold.nj)
  {
#define X(N)                                                                                              \
  case N:                                                                                                 \
    return rev ? launch_ring_nj<N, true>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st)            \
               : launch_ring_nj<N, false>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st);
    X(1) X(2) X(3) X(4) X(5) X(6) X(7)
#undef X
  }
  return cudaErrorNotSupported;
}

}  // namespace rdb
