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
__global__ void gram_fused_reduce_kernel(const double* __restrict__ partial, int nparts, int pstride, double* __restrict__ gram,
                                         double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  using G = GramGeom<NJ, Z>;
  constexpr int P = G::P;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
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
static void launch_fused_reduce(const double* partial, int nparts, int pstride, double* gram, double* rhs, double* tau_sq, int accumulate,
                                cudaStream_t st)
{
  using G = GramGeom<NJ, Z>;
  const int n = std::max(G::PARTIAL, G::P * (G::P + 1));
  gram_fused_reduce_kernel<NJ, Z><<<(n + 255) / 256, 256, 0, st>>>(partial, nparts, pstride, gram, rhs, tau_sq, accumulate);
  count_launch();
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

// done: the handle's Gram event (launch_gram); the previous Gram call, possibly on another stream, may still use the old buffer
static cudaError_t grow(double*& p, size_t& have, size_t need, cudaEvent_t done)
{
  if (have >= need) return cudaSuccess;
  if (p)
  {
    const cudaError_t e = cudaEventSynchronize(done);
    if (e != cudaSuccess) return e;
    cudaFree(p);
  }
  p = nullptr;
  have = 0;
  cudaError_t e = cudaMalloc(&p, need);
  if (e == cudaSuccess) have = need;
  return e;
}

// slots that fit the shared memory of an SM (227 KB minus 1 KB of barriers / static data): the rows, and XC component columns per joint
template <int NJ, int Z, int XC>
constexpr int gf_slots()
{
  return std::min<int>(GF_MAX_SLOTS,
                       (int)((227 * 1024 - 1024) / (sizeof(double) * (GramGeom<NJ, Z>::SLOT_DOUBLES + gram_ext_side_doubles<NJ, XC>()))));
}

// gram_fused_kernel on the folded chain, one per-CTA partial (gram_partial_doubles) each into `partials`: *grid CTAs.  On REV chains the
// kernel is the one specialised at run time to the chain's constants when it can be built (gram_jit.cpp), else the precompiled
// instantiation; other chains always run the precompiled generic kernel.
template <int NJ, bool REV, int XC>
static cudaError_t launch_fused_kernel(ChainHost& ch, const GramComps& gc, const SamplesDev& in, const double* tau_meas, double* partials,
                                       int* grid, cudaStream_t st)
{
  constexpr int Z = REV ? (XC ? 1 : 2) : 0;  // as in the kernel
  constexpr int SLOTS = gf_slots<NJ, Z, XC>();
  static_assert(SLOTS >= 2, "the fused kernel needs two slots");
  const void* kfn = reinterpret_cast<const void*>(gram_fused_kernel<NJ, SLOTS, REV, XC>);
  if (REV)
  {
    char args[64];
    snprintf(args, sizeof args, "gram_fused_kernel<%d, %d, true, %d", NJ, SLOTS, XC);
    if (const void* jk = gram_jit_kernel(ch, args)) kfn = jk;
  }
  else
  {
    ch.gram.kernel_specialised = 0;
    ch.gram.kernel_why = "precompiled kernel: not every folded joint is revolute about e_z (generic generator)";
  }
  const size_t smem = sizeof(double) * (size_t)gram_smem_doubles<NJ, Z, SLOTS, XC>();
  cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int64_t ngroups = (in.n + 31) / 32;
  constexpr int B = gram_group_block<SLOTS, XC>();
  *grid = (int)std::min<int64_t>(ch.sm_count, (ngroups + B - 1) / B);
  ChainDev<NJ> C = narrow_g<NJ>(ch.gram.fold);
  GramComps comps = gc;
  SamplesDev ins = in;
  const double* tm = tau_meas;
  double* part = partials;
  int dbg = gram_dev_switch();
  void* args[] = {&C, &comps, &ins, &tm, &part, &dbg};
  e = cudaLaunchKernel(kfn, dim3(*grid), dim3(GF_THREADS), args, smem, st);
  if (e != cudaSuccess) return e;
  count_launch();
  return cudaSuccess;
}

template <int NJ, bool REV>
static cudaError_t launch_fused_nj(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                   int accumulate, cudaStream_t st)
{
  constexpr int Z = REV ? 2 : 0;  // as in the kernel
  using G = GramGeom<NJ, Z>;
  cudaError_t e = grow(ch.gram.fused_partials, ch.gram.fused_bytes, sizeof(double) * (size_t)ch.sm_count * G::PARTIAL, ch.gram.done);
  if (e != cudaSuccess) return e;
  int grid = 0;
  e = launch_fused_kernel<NJ, REV, 0>(ch, GramComps{}, in, tau_meas, ch.gram.fused_partials, &grid, st);
  if (e != cudaSuccess) return e;
  if (ch.gram.fold_identity)
  {
    launch_fused_reduce<NJ, Z>(ch.gram.fused_partials, grid, G::PARTIAL, gram, rhs, tau_sq, accumulate, st);
    return cudaGetLastError();
  }
  // folded chain: reduce into G', b', then expand to the reference's full parameter vector
  const int nj = ch.host.nj, Pr = G::P;
  double* Tm = ch.gram.fold_dev;
  double* Gr = Tm + (size_t)nj * 100;
  double* br = Gr + (size_t)Pr * Pr;
  double* tsr = br + Pr;
  launch_fused_reduce<NJ, Z>(ch.gram.fused_partials, grid, G::PARTIAL, Gr, br, tsr, 0, st);
  return launch_fold_expand(ch, gram, rhs, tau_sq, accumulate, st);
}

// returns cudaErrorNotSupported when the chain does not fit the fused kernel (caller falls back to the general pipeline)
cudaError_t launch_gram_fused(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                              int accumulate, cudaStream_t st)
{
  if (in.n <= 0 || ch.gram.fold_version != ch.model_version) return cudaErrorNotSupported;
  const bool rev = fold_rev_canonical(ch.gram.fold);  // all moving joints revolute about e_z: the specialised generator
  switch (ch.gram.fold.nj)  // moving joints; every joint of the folded chain is an input
  {
#define X(N)                                                                                  \
  case N:                                                                                     \
    return rev ? launch_fused_nj<N, true>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st) \
               : launch_fused_nj<N, false>(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st);
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

// one pass of gram_fused_kernel<.., XC> over the samples: rigid-body tiles -> Gt | bt | tst (full parameter vector) -> the rigid block of the
// extended normal equations; cross tiles -> xsum -> the cross blocks.  xmap: reduced joint, then slot, of every component column.
template <int NJ, bool REV, int XC>
static cudaError_t launch_ext_nj(ChainHost& ch, const GramComps& gc, const std::vector<int32_t>& xmap, const SamplesDev& in, const double* tau_meas,
                                 double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st)
{
  constexpr int Z = REV ? 1 : 0;  // as in the kernel
  using G = GramGeom<NJ, Z>;
  constexpr int PSTRIDE = gram_partial_doubles<NJ, Z, XC>();
  const int nj = ch.host.nj, P = 10 * nj, Pc = ch.comps.cols, Pt = P + Pc;
  // workspace: rigid block (P*P + P + 1) | cross sums (NXT*64) | per-CTA partials (sm_count*PSTRIDE) | component map (2 Pc ints)
  const size_t n_rigid = (size_t)P * P + P + 1, n_sum = (size_t)G::NXT * 64, n_part = (size_t)ch.sm_count * PSTRIDE;
  cudaError_t e = grow(ch.gram.ext_dev, ch.gram.ext_bytes, sizeof(double) * (n_rigid + n_sum + n_part) + sizeof(int32_t) * 2 * (size_t)Pc,
                       ch.gram.done);
  if (e != cudaSuccess) return e;
  double* Gt = ch.gram.ext_dev;
  double* bt = Gt + (size_t)P * P;
  double* tst = bt + P;
  double* xsum = tst + 1;
  double* xpart = xsum + n_sum;
  int32_t* dmap = reinterpret_cast<int32_t*>(xpart + n_part);
  e = cudaMemcpyAsync(dmap, xmap.data(), sizeof(int32_t) * xmap.size(), cudaMemcpyHostToDevice, st);  // pageable source: staged before return
  if (e != cudaSuccess) return e;
  int grid = 0;
  e = launch_fused_kernel<NJ, REV, XC>(ch, gc, in, tau_meas, xpart, &grid, st);
  if (e != cudaSuccess) return e;
  if (ch.gram.fold_identity) launch_fused_reduce<NJ, Z>(xpart, grid, PSTRIDE, Gt, bt, tst, 0, st);
  else
  {
    double* Gr = ch.gram.fold_dev + (size_t)nj * 100;
    double* br = Gr + (size_t)G::P * G::P;
    launch_fused_reduce<NJ, Z>(xpart, grid, PSTRIDE, Gr, br, br + G::P, 0, st);
    e = launch_fold_expand(ch, Gt, bt, tst, 0, st);
    if (e != cudaSuccess) return e;
  }
  gram_cross_reduce_kernel<<<(G::NXT * 64 + 255) / 256, 256, 0, st>>>(xpart + G::NT * 64, grid, G::NXT * 64, PSTRIDE, xsum);
  count_launch();
  gram_ext_scatter_kernel<<<(P * (P + 1) + 255) / 256, 256, 0, st>>>(Gt, bt, tst, P, Pt, gram, rhs, tau_sq, accumulate);
  count_launch();
  const double* Tm1 = ch.gram.fold_identity ? nullptr : ch.gram.fold_dev;
  const int32_t* kof1 =
      ch.gram.fold_identity ? nullptr : reinterpret_cast<const int32_t*>(ch.gram.fold_dev + (size_t)nj * 100 + (size_t)(G::P + 1) * (G::P + 1));
  gram_cross_finish_kernel<NJ, Z><<<((P + 1 + Pc) * Pc + 127) / 128, 128, 0, st>>>(xsum, Tm1, kof1, dmap, dmap + Pc, nj, Pc, gram, rhs, accumulate);
  count_launch();
  return cudaGetLastError();
}

// Normal equations of the extended model in one pass over the samples.
// cudaErrorNotSupported: more than 7 moving joints, a component on an input no chain joint feeds, or more than GX_COLS component columns
// on one joint (caller falls back to the general pipeline).
cudaError_t launch_gram_fused_ext(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                  int accumulate, cudaStream_t st)
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
  (xcmax <= 2 ? launch_ext_nj<N, R, 2>(ch, gc, xmap, in, tau_meas, gram, rhs, tau_sq, accumulate, st)               \
              : (xcmax <= 4 ? launch_ext_nj<N, R, 4>(ch, gc, xmap, in, tau_meas, gram, rhs, tau_sq, accumulate, st) \
                            : launch_ext_nj<N, R, 8>(ch, gc, xmap, in, tau_meas, gram, rhs, tau_sq, accumulate, st)))
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
