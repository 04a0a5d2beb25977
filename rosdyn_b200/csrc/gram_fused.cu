// gram_fused.cu -- launchers of the fused regressor -> normal-equation kernels (gram_fused.cuh), the reductions behind them and the
// fold expansion.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "gram_fused.cuh"
#include "launch.h"

namespace rdb
{

// fixed-order sum of the per-CTA partials (GramGeom<NJ, Z>::PARTIAL doubles each, pstride apart) -> gram (full symmetric,
// column-major), rhs, tau_sq.  One thread per partial entry, and per entry of the P x (P + 1) output: the parameter columns without a position
// (identically zero columns of Phi, GramGeom::has_pos) get exact zeros in their row, column and rhs.
template <int NJ, int Z>
__device__ __forceinline__ void gram_fused_reduce_entry(int e, const double* __restrict__ partial, int nparts, int pstride, double* __restrict__ gram,
                                                        double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  using G = GramGeom<NJ, Z>;
  constexpr int P = G::P;
  if (!accumulate && e < P * (P + 1))
  {
    const int c = e / (P + 1), r = e % (P + 1);  // r == P: rhs
    if (!G::has_pos(c))
    {
      if (r == P) rhs[c] = 0.0;
      else
      {
        gram[(size_t)c * P + r] = 0.0;
        gram[(size_t)r * P + c] = 0.0;
      }
    }
  }
  if (e >= G::PARTIAL) return;
  double s = 0.0;
  for (int p = 0; p < nparts; p++) s += partial[(size_t)p * pstride + e];
  if (e >= G::NT * 64)  // TC == 0: b by position, then tau^T tau
  {
    const int q = e - G::NT * 64;
    if (q == 8 * G::T)
    {
      if (tau_sq) *tau_sq = accumulate ? *tau_sq + s : s;
    }
    else if (q < G::NPOS)
    {
      const int a = G::col_of(q);
      rhs[a] = accumulate ? rhs[a] + s : s;
    }
    return;
  }
  int k = e >> 6, I = 0;
  while (k >= G::T - I)
  {
    k -= G::T - I;
    I++;
  }
  const int J = I + k;
  const int rp = 8 * I + ((e >> 3) & 7), cp = 8 * J + (e & 7);  // positions inside the kernel (GramGeom::pos)
  if (rp >= G::NPOS || cp >= G::NPOS) return;
  if (I == J && rp > cp) return;  // diagonal tiles hold both halves; keep the upper one
  const int row = G::col_of(rp), col = G::col_of(cp);  // P: tau
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
template <int NJ, int Z>
__global__ void gram_fused_reduce_kernel(const double* __restrict__ partial, int nparts, int pstride, double* __restrict__ gram,
                                         double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  gram_fused_reduce_entry<NJ, Z>(blockIdx.x * blockDim.x + threadIdx.x, partial, nparts, pstride, gram, rhs, tau_sq, accumulate);
}
// segmented: blockIdx.y is row y of the wave's segment table (rows[3 y ..]: first item of the wave, item count, segment), which sums its
// items' partials in item order.  Output o = the segment (by_segment) or y, at gram + o gstride, rhs + o rstride, tau_sq + o tstride.  A row
// without items writes zeros (the host lists empty segments only when the call does not accumulate).
template <int NJ, int Z>
__global__ void gram_fused_reduce_segmented_kernel(const double* __restrict__ partial, const int64_t* __restrict__ rows, int pstride,
                                                   double* __restrict__ gram, double* __restrict__ rhs, double* __restrict__ tau_sq,
                                                   int64_t gstride, int64_t rstride, int64_t tstride, int by_segment, int accumulate)
{
  const int64_t* r = rows + 3 * (int64_t)blockIdx.y;
  const int64_t o = by_segment ? r[2] : (int64_t)blockIdx.y;
  gram_fused_reduce_entry<NJ, Z>(blockIdx.x * blockDim.x + threadIdx.x, partial + r[0] * pstride, (int)r[1], pstride, gram + o * gstride,
                                 rhs + o * rstride, tau_sq ? tau_sq + o * tstride : nullptr, accumulate);
}
template <int NJ, int Z>
static void launch_fused_reduce(const double* partial, int nparts, int pstride, double* gram, double* rhs, double* tau_sq, int accumulate,
                                cudaStream_t st)
{
  using G = GramGeom<NJ, Z>;
  const int n = std::max(G::PARTIAL, G::P * (G::P + 1));
  gram_fused_reduce_kernel<NJ, Z><<<(n + 255) / 256, 256, 0, st>>>(partial, nparts, pstride, gram, rhs, tau_sq, accumulate);
  count_launch();
}

// G = E^T G' E, b = E^T b' (upper triangle computed, mirrored): one thread per entry of the full matrix, 100 products each
__device__ __forceinline__ void gram_fold_expand_entry(int e, const double* __restrict__ T, const int32_t* __restrict__ kof,
                                                       const double* __restrict__ Gr, const double* __restrict__ br, const double* __restrict__ tsr,
                                                       int nj, int Pr, double* __restrict__ gram, double* __restrict__ rhs,
                                                       double* __restrict__ tau_sq, int accumulate)
{
  const int P = 10 * nj;
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
__global__ void gram_fold_expand_kernel(const double* __restrict__ T, const int32_t* __restrict__ kof, const double* __restrict__ Gr,
                                        const double* __restrict__ br, const double* __restrict__ tsr, int nj, int Pr, double* __restrict__ gram,
                                        double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  gram_fold_expand_entry(blockIdx.x * blockDim.x + threadIdx.x, T, kof, Gr, br, tsr, nj, Pr, gram, rhs, tau_sq, accumulate);
}
// segmented: blockIdx.y is row y of the wave's segment table; its reduced equations sit at red + y rstride (G' | b' | tau_sq), its output
// is segment rows[3 y + 2] of gram / rhs / tau_sq
__global__ void gram_fold_expand_segmented_kernel(const double* __restrict__ T, const int32_t* __restrict__ kof, const double* __restrict__ red,
                                                  int64_t rstride, const int64_t* __restrict__ rows, int nj, int Pr, double* __restrict__ gram,
                                                  double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  const int64_t P = 10 * nj, k = rows[3 * (int64_t)blockIdx.y + 2];
  const double* Gr = red + (int64_t)blockIdx.y * rstride;
  gram_fold_expand_entry(blockIdx.x * blockDim.x + threadIdx.x, T, kof, Gr, Gr + (size_t)Pr * Pr, Gr + (size_t)Pr * Pr + Pr, nj, Pr,
                         gram + k * P * P, rhs + k * P, tau_sq ? tau_sq + k : nullptr, accumulate);
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

// the reduced normal equations G' | b' | tau_sq of the folded chain (reduced_row(ch, 0), written by the reduce kernels) -> the reference's
// full parameter vector
cudaError_t launch_fold_expand(ChainHost& ch, double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st)
{
  const int nj = ch.host.nj, Pr = 10 * ch.gram.fold.nj, P = 10 * nj;
  const FoldMaps fm = fold_maps(ch);
  const ReducedRow r = reduced_row(ch, 0);
  gram_fold_expand_kernel<<<(P * (P + 1) + 127) / 128, 128, 0, st>>>(fm.T, fm.kof, r.G, r.b, r.tau_sq, nj, Pr, gram, rhs, tau_sq, accumulate);
  count_launch();
  return cudaGetLastError();
}

// the reduced normal equations of `rows` systems of the folded chain (ch.gram.reduced)
static cudaError_t grow_reduced(ChainHost& ch, int64_t rows)
{
  return ch.gram.reduced.grow(sizeof(double) * rows * ReducedRow::doubles(10 * ch.gram.fold.nj), ch.gram.done);
}

// slots that fit the shared memory of an SM (227 KB minus 1 KB of barriers / static data): the rows, XC component columns per joint and (WT)
// the weight of every row
template <int NJ, int Z, int XC, bool WT = false>
constexpr int gf_slots()
{
  return std::min<int>(GF_MAX_SLOTS, (int)((227 * 1024 - 1024) / (sizeof(double) * (GramGeom<NJ, Z>::SLOT_DOUBLES + gram_ext_side_doubles<NJ, XC>() +
                                                                                     (WT ? 32 * NJ : 0)))));
}

// gram_fused_kernel on the folded chain, one per-CTA partial (gram_partial_doubles) each into `partials`: *grid CTAs.  On REV chains the
// kernel is the one specialised at run time to the chain's constants when it can be built (gram_jit.cpp), else the precompiled
// instantiation; other chains always run the precompiled generic kernel.
// SEG: gram_fused_segmented_kernel instead, one CTA per work item of items[0 .. 2 *grid) (device table of start, length).
// WT: gram_fused_weighted_kernel instead, with the weights wt (same grid).
template <int NJ, bool REV, int XC, bool SEG = false, bool WT = false>
static cudaError_t launch_fused_kernel(ChainHost& ch, const GramComps& gc, const SamplesDev& in, const double* tau_meas, double* partials,
                                       int* grid, cudaStream_t st, const int64_t* items = nullptr, const rdb_gram_weights& wt = {})
{
  static_assert(!(SEG && WT), "no weighted segmented kernel");
  constexpr int Z = REV ? (XC ? 1 : 2) : 0;  // as in the kernel
  constexpr int SLOTS = gf_slots<NJ, Z, XC, WT>();
  static_assert(SLOTS >= 2, "the fused kernel needs two slots");
  static_assert(!WT || XC > 0 || SLOTS == gf_slots<NJ, Z, XC>(), "the weighted rigid-body kernel keeps the slots, hence the groups, of gram_fused_kernel");
  const char* name = SEG ? "gram_fused_segmented_kernel" : (WT ? "gram_fused_weighted_kernel" : "gram_fused_kernel");
  const void* kfn = nullptr;
  if constexpr (SEG) kfn = reinterpret_cast<const void*>(gram_fused_segmented_kernel<NJ, SLOTS, REV, XC>);
  else if constexpr (WT) kfn = reinterpret_cast<const void*>(gram_fused_weighted_kernel<NJ, SLOTS, REV, XC>);
  else kfn = reinterpret_cast<const void*>(gram_fused_kernel<NJ, SLOTS, REV, XC>);
  if (REV)
  {
    char args[64];
    snprintf(args, sizeof args, "%s<%d, %d, true, %d", name, NJ, SLOTS, XC);
    if (const void* jk = gram_jit_kernel(ch, args)) kfn = jk;
  }
  else
  {
    ch.gram.kernel_specialised = 0;
    ch.gram.kernel_why = "precompiled kernel: not every folded joint is revolute about e_z (generic generator)";
  }
  // rdb_chain_gram_kernel_info names the segmented and the weighted kernel
  if (SEG || WT) ch.gram.kernel_why = std::string(name) + ", " + ch.gram.kernel_why;
  const size_t smem = sizeof(double) * (size_t)gram_smem_doubles_w<NJ, Z, SLOTS, XC, WT>();
  cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (!SEG)
  {
    const int64_t ngroups = (in.n + 31) / 32;
    constexpr int B = gram_group_block<SLOTS, XC>();
    *grid = (int)std::min<int64_t>(ch.sm_count, (ngroups + B - 1) / B);
  }
  ChainDev<NJ> C = narrow<NJ>(ch.gram.fold);
  GramComps comps = gc;
  SamplesDev ins = in;
  const double* tm = tau_meas;
  const int64_t* it = items;
  rdb_gram_weights w = wt;
  double* part = partials;
  int dbg = gram_dev_switch();
  void* args_whole[] = {&C, &comps, &ins, &tm, &part, &dbg};
  void* args_seg[] = {&C, &comps, &ins, &tm, &it, &part, &dbg};
  void* args_w[] = {&C, &comps, &ins, &tm, &w, &part, &dbg};
  e = cudaLaunchKernel(kfn, dim3(*grid), dim3(GF_THREADS), SEG ? args_seg : (WT ? args_w : args_whole), smem, st);
  if (e != cudaSuccess) return e;
  count_launch();
  return cudaSuccess;
}
// the same, weighted when wt is given
template <int NJ, bool REV, int XC>
static cudaError_t launch_fused_kernel(ChainHost& ch, const GramComps& gc, const SamplesDev& in, const double* tau_meas, double* partials,
                                       int* grid, cudaStream_t st, const rdb_gram_weights* wt)
{
  return wt ? launch_fused_kernel<NJ, REV, XC, false, true>(ch, gc, in, tau_meas, partials, grid, st, nullptr, *wt)
            : launch_fused_kernel<NJ, REV, XC>(ch, gc, in, tau_meas, partials, grid, st);
}

template <int NJ, bool REV>
static cudaError_t launch_fused_nj(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                   int accumulate, cudaStream_t st, const rdb_gram_weights* wt)
{
  constexpr int Z = REV ? 2 : 0;  // as in the kernel
  using G = GramGeom<NJ, Z>;
  cudaError_t e = ch.gram.fused_partials.grow(sizeof(double) * (size_t)ch.sm_count * G::PARTIAL, ch.gram.done);
  if (e == cudaSuccess && !ch.gram.fold_identity) e = grow_reduced(ch, 1);
  if (e != cudaSuccess) return e;
  double* part = ch.gram.fused_partials.get();
  int grid = 0;
  e = launch_fused_kernel<NJ, REV, 0>(ch, GramComps{}, in, tau_meas, part, &grid, st, wt);
  if (e != cudaSuccess) return e;
  if (ch.gram.fold_identity)
  {
    launch_fused_reduce<NJ, Z>(part, grid, G::PARTIAL, gram, rhs, tau_sq, accumulate, st);
    return cudaGetLastError();
  }
  // folded chain: reduce into G', b', then expand to the reference's full parameter vector
  const ReducedRow r = reduced_row(ch, 0);
  launch_fused_reduce<NJ, Z>(part, grid, G::PARTIAL, r.G, r.b, r.tau_sq, 0, st);
  return launch_fold_expand(ch, gram, rhs, tau_sq, accumulate, st);
}

// returns cudaErrorNotSupported when the chain does not fit the fused kernel (caller falls back to the general pipeline)
cudaError_t launch_gram_fused(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                              int accumulate, cudaStream_t st, const rdb_gram_weights* wt)
{
  if (in.n <= 0 || ch.gram.fold_version != ch.model_version) return cudaErrorNotSupported;
  const bool rev = fold_rev_canonical(ch.gram.fold);  // all moving joints revolute about e_z: the specialised generator
  switch (ch.gram.fold.nj)  // moving joints; every joint of the folded chain is an input
  {
#define X(N)                                                                                  \
  case N:                                                                                     \
    return rev ? launch_fused_nj<N, true>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st, wt) \
               : launch_fused_nj<N, false>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st, wt);
    X(1) X(2) X(3) X(4) X(5) X(6) X(7)
#undef X
  }
  return cudaErrorNotSupported;
}

// ---------------------------------------------------------------------------------------------- segmented normal equations
// Work items: every segment is cut, from its start, into items of `item` samples (the last one short); each item is one CTA of
// gram_fused_segmented_kernel.  The items run in waves of at most `wave` items and `wave` segment rows, so the workspace of partials is
// bounded by the wave, not by the number of segments.  A wave holds whole segments; a segment of more than `wave` items runs alone over
// ceil(items / wave) waves, each one after the first added into its output.  Both cuts depend on the segment's length alone, and every sum runs
// in item order, so a segment's result depends on its own samples only, bit for bit, wherever it sits in the call.
// Chosen by measurement on a B200 (tools/bench_gram_segmented.py, profiles/gram_segmented_bench*.json, DESIGN.md 3.3.1): 128 groups (4 096
// samples) per item, 8 items per SM per wave.  The environment variables RDB_GRAM_SEG_ITEM_GROUPS and RDB_GRAM_SEG_WAVE_PER_SM override
// them for such measurements; results are reproducible for a given setting.
constexpr int GF_SEG_ITEM_GROUPS = 128;
constexpr int GF_SEG_WAVE_PER_SM = 8;

static int64_t seg_knob(const char* env, int64_t dflt, int64_t hi)
{
  const char* e = getenv(env);
  const long long v = e && *e ? atoll(e) : 0;
  return v >= 1 && v <= hi ? (int64_t)v : dflt;
}

struct SegPlan
{
  struct Wave
  {
    int64_t item0, nitems, row0, nrows;
    int accumulate;
  };
  std::vector<Wave> waves;
  std::vector<int64_t> tab;  // offsets [K + 1] | items (start, length) | rows (first item in the wave, items, segment)
  int64_t nitems = 0, max_rows = 0, wave = 0;
};

static SegPlan plan_segments(int64_t nseg, const int64_t* offsets, int64_t item, int64_t wave, int accumulate)
{
  SegPlan p;
  p.wave = wave;
  std::vector<int64_t> items, rows;
  SegPlan::Wave cur{0, 0, 0, 0, accumulate};
  auto flush = [&] {
    if (cur.nitems || cur.nrows) p.waves.push_back(cur);
    p.max_rows = std::max(p.max_rows, cur.nrows);
    cur = SegPlan::Wave{(int64_t)items.size() / 2, 0, (int64_t)rows.size() / 3, 0, accumulate};
  };
  auto add_items = [&](int64_t lo, int64_t hi, int64_t i0, int64_t ni) {
    for (int64_t i = i0; i < i0 + ni; i++)
    {
      items.push_back(lo + i * item);
      items.push_back(std::min(item, hi - lo - i * item));
    }
  };
  for (int64_t k = 0; k < nseg; k++)
  {
    const int64_t lo = offsets[k], hi = offsets[k + 1], ni = (hi - lo + item - 1) / item;
    if (ni > wave)  // alone, over several waves
    {
      flush();
      for (int64_t w0 = 0; w0 < ni; w0 += wave)
      {
        const int64_t nw = std::min(wave, ni - w0);
        rows.insert(rows.end(), {0, nw, k});
        add_items(lo, hi, w0, nw);
        cur.nitems = nw;
        cur.nrows = 1;
        cur.accumulate = w0 ? 1 : accumulate;
        flush();
      }
      continue;
    }
    if (ni == 0 && accumulate) continue;  // an empty segment is left as it is
    if (cur.nitems + ni > wave || cur.nrows == wave) flush();
    rows.insert(rows.end(), {cur.nitems, ni, k});  // an empty segment: a row without items, which writes zeros
    add_items(lo, hi, 0, ni);
    cur.nitems += ni;
    cur.nrows++;
  }
  flush();
  p.nitems = (int64_t)items.size() / 2;
  p.tab.assign(offsets, offsets + nseg + 1);
  p.tab.insert(p.tab.end(), items.begin(), items.end());
  p.tab.insert(p.tab.end(), rows.begin(), rows.end());
  return p;
}

template <int NJ, bool REV>
static cudaError_t launch_fused_segmented_nj(ChainHost& ch, const SamplesDev& in, const double* tau_meas, int64_t nseg, const SegPlan& plan,
                                             double* gram, double* rhs, double* tau_sq, int accumulate, bool unfed, cudaStream_t st)
{
  constexpr int Z = REV ? 2 : 0;  // as in the kernel
  using G = GramGeom<NJ, Z>;
  const int nj = ch.host.nj, Pr = G::P, P = 10 * nj;
  const bool fold = !ch.gram.fold_identity;
  // workspace: per-item partials of one wave | (unfed) the fused tau^T tau of every segment | the plan's table; (folded chain) the reduced
  // equations of each row of a wave
  const size_t n_part = (size_t)plan.wave * G::PARTIAL, n_ts = unfed ? (size_t)nseg : 0;
  cudaError_t e = ch.gram.seg_dev.grow(sizeof(double) * (n_part + n_ts) + sizeof(int64_t) * plan.tab.size(), ch.gram.done);
  if (e == cudaSuccess && fold) e = grow_reduced(ch, plan.max_rows);
  if (e != cudaSuccess) return e;
  double* part = ch.gram.seg_dev.get();
  double* ts = part + n_part;
  int64_t* tab = reinterpret_cast<int64_t*>(ts + n_ts);
  e = cudaMemcpyAsync(tab, plan.tab.data(), sizeof(int64_t) * plan.tab.size(), cudaMemcpyHostToDevice, st);  // pageable: staged before return
  if (e != cudaSuccess) return e;
  const int64_t* items = tab + nseg + 1;
  const int64_t* rows = items + 2 * plan.nitems;
  if (unfed) cudaMemsetAsync(ts, 0, sizeof(double) * nseg, st);
  double* tso = unfed ? ts : tau_sq;
  const int nred = std::max(G::PARTIAL, Pr * (Pr + 1));
  for (const SegPlan::Wave& w : plan.waves)
  {
    if (w.nitems)
    {
      int grid = (int)w.nitems;
      e = launch_fused_kernel<NJ, REV, 0, true>(ch, GramComps{}, in, tau_meas, part, &grid, st, items + 2 * w.item0);
      if (e != cudaSuccess) return e;
    }
    const int64_t* wr = rows + 3 * w.row0;
    const dim3 rg((nred + 255) / 256, (unsigned)w.nrows);
    if (!fold)
      gram_fused_reduce_segmented_kernel<NJ, Z><<<rg, 256, 0, st>>>(part, wr, G::PARTIAL, gram, rhs, tso, (int64_t)P * P, P, 1, 1, w.accumulate);
    else
    {
      const FoldMaps fm = fold_maps(ch);
      const ReducedRow r = reduced_row(ch, 0);
      const int64_t RS = ReducedRow::doubles(Pr);
      gram_fused_reduce_segmented_kernel<NJ, Z><<<rg, 256, 0, st>>>(part, wr, G::PARTIAL, r.G, r.b, r.tau_sq, RS, RS, RS, 0, 0);
      count_launch();
      gram_fold_expand_segmented_kernel<<<dim3((P * (P + 1) + 127) / 128, (unsigned)w.nrows), 128, 0, st>>>(fm.T, fm.kof, r.G, RS, wr, nj, Pr, gram,
                                                                                                             rhs, tso, w.accumulate);
    }
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if (unfed) return launch_unfed_tau_sq(ch, tau_meas, in.ld, in.n, tab, nseg, ts, tau_sq, accumulate, st);
  return cudaSuccess;
}

// returns cudaErrorNotSupported when the chain does not fit the fused kernel (caller runs the general pipeline per segment).  unfed: measured
// torques also sit on inputs no chain joint feeds (their squares join tau_sq per segment, launch_unfed_tau_sq_segmented)
cudaError_t launch_gram_fused_segmented(ChainHost& ch, const SamplesDev& in, const double* tau_meas, int64_t nseg, const int64_t* offsets,
                                        double* gram, double* rhs, double* tau_sq, int accumulate, bool unfed, cudaStream_t st)
{
  if (ch.gram.fold_version != ch.model_version || ch.gram.fold.nj < 1 || ch.gram.fold.nj > 7) return cudaErrorNotSupported;
  const int64_t item = 32 * seg_knob("RDB_GRAM_SEG_ITEM_GROUPS", GF_SEG_ITEM_GROUPS, 1 << 20);
  const int64_t wave = ch.sm_count * seg_knob("RDB_GRAM_SEG_WAVE_PER_SM", GF_SEG_WAVE_PER_SM, 65535 / std::max(ch.sm_count, 1));
  const SegPlan plan = plan_segments(nseg, offsets, item, wave, accumulate);
  const bool rev = fold_rev_canonical(ch.gram.fold);
  switch (ch.gram.fold.nj)
  {
#define X(N)                                                                                                            \
  case N:                                                                                                               \
    return rev ? launch_fused_segmented_nj<N, true>(ch, in, tau_meas, nseg, plan, gram, rhs, tau_sq, accumulate, unfed, st) \
               : launch_fused_segmented_nj<N, false>(ch, in, tau_meas, nseg, plan, gram, rhs, tau_sq, accumulate, unfed, st);
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

// cross blocks of the extended normal equations from the reduced cross tiles X of the folded chain (NJ joints, layout GramGeom<NJ, Z>):
//   gram[a][P + cc] (and its mirror) = sum_c T[la][c][pa] X(10 ka + c ; joint, slot of cc)     a < P   (fold expansion of the rigid column)
//   rhs[P + cc] = X(P' ; joint, slot)                                                          (tau column of the last regular tile)
//   gram[P + c2][P + cc] = XX(joint)[slot2][slot] when both components act on the same joint, else 0
// xj / xs: reduced joint and slot of every component column.  One thread per (a in 0 .. P + Pc, cc).
template <int NJ, int Z>
__global__ void gram_cross_finish_kernel(const double* __restrict__ X, const double* __restrict__ Tm, const int32_t* __restrict__ kof,
                                         const int32_t* __restrict__ xj, const int32_t* __restrict__ xs, int nj, int Pc, double* __restrict__ gram,
                                         double* __restrict__ rhs, int accumulate)
{
  using G = GramGeom<NJ, Z>;
  static_assert(G::TC == 1, "tau is the tile column at position 0");
  const int P = 10 * nj, Pt = P + Pc;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (P + 1 + Pc) * Pc) return;
  const int a = e / Pc, cc = e % Pc;
  const int j = xj[cc], g = xs[cc];
  const int tb = G::xtile(j, 0);  // first cross tile of joint j
  auto xval = [&](int col) -> double {  // reduced regular column `col` (G::P = tau) against (j, g)
    const int pos = col == G::P ? 0 : G::pos(col / 10, col % 10);
    return pos >= G::rowlen(j) ? 0.0 : X[(size_t)(tb + (pos >> 3)) * 64 + (pos & 7) * 8 + g];  // behind rowlen(j): an exact zero of Phi
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
    const double s = xval(G::P);
    rhs[P + cc] = accumulate ? rhs[P + cc] + s : s;
  }
  else
  {
    const int c2 = a - P - 1;
    const double s = (xj[c2] == j) ? X[(size_t)(tb + G::tj(j)) * 64 + xs[c2] * 8 + g] : 0.0;
    double* o = gram + (size_t)(P + cc) * Pt + P + c2;
    *o = accumulate ? *o + s : s;
  }
}

// weighted extended model: the (component, component) tiles are sums of (w x_m) x_n, whose two halves round differently; gram_cross_finish_kernel
// writes both.  Keep the upper one (row < column), as the reduction does for the diagonal tiles of the rigid-body block: one thread per pair
// (c2 > cc) of component columns on the same joint.  With w == 1 both halves are equal and nothing changes.
__global__ void gram_ext_mirror_kernel(const int32_t* __restrict__ xj, int P, int Pc, double* __restrict__ gram)
{
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Pc * Pc) return;
  const int c2 = e / Pc, cc = e % Pc;
  if (c2 <= cc || xj[c2] != xj[cc]) return;
  const int64_t Pt = P + Pc;
  gram[(int64_t)(P + cc) * Pt + P + c2] = gram[(int64_t)(P + c2) * Pt + P + cc];
}

// one pass of gram_fused_kernel<.., XC> over the samples: rigid-body tiles -> Gt | bt | tst (full parameter vector) -> the rigid block of the
// extended normal equations; cross tiles -> xsum -> the cross blocks.  xmap: reduced joint, then slot, of every component column.
template <int NJ, bool REV, int XC>
static cudaError_t launch_ext_nj(ChainHost& ch, const GramComps& gc, const std::vector<int32_t>& xmap, const SamplesDev& in, const double* tau_meas,
                                 double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st, const rdb_gram_weights* wt)
{
  constexpr int Z = REV ? 1 : 0;  // as in the kernel
  using G = GramGeom<NJ, Z>;
  constexpr int PSTRIDE = gram_partial_doubles<NJ, Z, XC>();
  const int nj = ch.host.nj, P = 10 * nj, Pc = ch.comps.cols, Pt = P + Pc;
  // workspace: rigid block (P*P + P + 1) | cross sums (NXT*64) | per-CTA partials (sm_count*PSTRIDE) | component map (2 Pc ints)
  const size_t n_rigid = (size_t)P * P + P + 1, n_sum = (size_t)G::NXT * 64, n_part = (size_t)ch.sm_count * PSTRIDE;
  cudaError_t e = ch.gram.ext_dev.grow(sizeof(double) * (n_rigid + n_sum + n_part) + sizeof(int32_t) * 2 * (size_t)Pc, ch.gram.done);
  if (e == cudaSuccess && !ch.gram.fold_identity) e = grow_reduced(ch, 1);
  if (e != cudaSuccess) return e;
  double* Gt = ch.gram.ext_dev.get();
  double* bt = Gt + (size_t)P * P;
  double* tst = bt + P;
  double* xsum = tst + 1;
  double* xpart = xsum + n_sum;
  int32_t* dmap = reinterpret_cast<int32_t*>(xpart + n_part);
  e = cudaMemcpyAsync(dmap, xmap.data(), sizeof(int32_t) * xmap.size(), cudaMemcpyHostToDevice, st);  // pageable source: staged before return
  if (e != cudaSuccess) return e;
  int grid = 0;
  e = launch_fused_kernel<NJ, REV, XC>(ch, gc, in, tau_meas, xpart, &grid, st, wt);
  if (e != cudaSuccess) return e;
  if (ch.gram.fold_identity) launch_fused_reduce<NJ, Z>(xpart, grid, PSTRIDE, Gt, bt, tst, 0, st);
  else
  {
    const ReducedRow r = reduced_row(ch, 0);
    launch_fused_reduce<NJ, Z>(xpart, grid, PSTRIDE, r.G, r.b, r.tau_sq, 0, st);
    e = launch_fold_expand(ch, Gt, bt, tst, 0, st);
    if (e != cudaSuccess) return e;
  }
  gram_cross_reduce_kernel<<<(G::NXT * 64 + 255) / 256, 256, 0, st>>>(xpart + G::NT * 64, grid, G::NXT * 64, PSTRIDE, xsum);
  count_launch();
  gram_ext_scatter_kernel<<<(P * (P + 1) + 255) / 256, 256, 0, st>>>(Gt, bt, tst, P, Pt, gram, rhs, tau_sq, accumulate);
  count_launch();
  const FoldMaps fm = ch.gram.fold_identity ? FoldMaps{nullptr, nullptr} : fold_maps(ch);
  gram_cross_finish_kernel<NJ, Z><<<((P + 1 + Pc) * Pc + 127) / 128, 128, 0, st>>>(xsum, fm.T, fm.kof, dmap, dmap + Pc, nj, Pc, gram, rhs, accumulate);
  count_launch();
  if (wt)
  {
    gram_ext_mirror_kernel<<<(Pc * Pc + 127) / 128, 128, 0, st>>>(dmap, P, Pc, gram);
    count_launch();
  }
  return cudaGetLastError();
}

// Normal equations of the extended model in one pass over the samples.
// cudaErrorNotSupported: more than 7 moving joints, a component on an input no chain joint feeds, or more than GX_COLS component columns
// on one joint (caller falls back to the general pipeline).
cudaError_t launch_gram_fused_ext(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                  int accumulate, cudaStream_t st, const rdb_gram_weights* wt)
{
  if (in.n <= 0 || ch.gram.fold_version != ch.model_version) return cudaErrorNotSupported;
  const ChainDev<RDB_MAX_JOINTS>& F = ch.gram.fold;
  const int K = F.nj, Pc = ch.comps.cols;
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
  int xcmax = 0;
  for (int j = 0; j < K; j++) xcmax = std::max(xcmax, (int)gc.ncols[j]);
  switch (K)
  {
#define XL(N, R)                                                                                                  \
  (xcmax <= 2 ? launch_ext_nj<N, R, 2>(ch, gc, xmap, in, tau_meas, gram, rhs, tau_sq, accumulate, st, wt)               \
              : (xcmax <= 4 ? launch_ext_nj<N, R, 4>(ch, gc, xmap, in, tau_meas, gram, rhs, tau_sq, accumulate, st, wt) \
                            : launch_ext_nj<N, R, 8>(ch, gc, xmap, in, tau_meas, gram, rhs, tau_sq, accumulate, st, wt)))
#define X(N) \
  case N:    \
    return rev ? XL(N, true) : XL(N, false);
    X(1) X(2) X(3) X(4) X(5) X(6) X(7)
#undef X
#undef XL
  }
  return cudaErrorNotSupported;
}

// the row layout of gram_fused_kernel on all-revolute chains (host entry for tests, rdb_gram_row_layout)
template <int NJ>
static void gram_row_layout_nj(int32_t* pos, int32_t* rowlen, int32_t* tau_col)
{
  using G = GramGeom<NJ, 2>;
  for (int j = 0; j < NJ; j++)
  {
    rowlen[j] = G::rowlen(j);
    for (int c = 0; c < G::P; c++) pos[j * G::P + c] = c / 10 >= j && G::stored(j, c / 10, c % 10) ? G::pos(c / 10, c % 10) : -1;
  }
  *tau_col = G::TC;
}

}  // namespace rdb

extern "C" rdb_status rdb_gram_row_layout(int32_t nj, int32_t* pos, int32_t* rowlen, int32_t* tau_col)
{
  if (!pos || !rowlen || !tau_col) return RDB_ERR_INVALID_ARG;
  switch (nj)
  {
#define X(N)                                                \
  case N:                                                   \
    rdb::gram_row_layout_nj<N>(pos, rowlen, tau_col);       \
    return RDB_OK;
    X(1) X(2) X(3) X(4) X(5) X(6) X(7)
#undef X
  }
  return RDB_ERR_INVALID_ARG;
}
