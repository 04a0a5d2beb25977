// gram.cu -- regressor -> normal equations (Phi^T Phi, Phi^T tau, tau^T tau) on the FP64 tensor path.
//
// tcgen05 has no f64 kind, so the Blackwell FP64 tensor path is mma.sync.m8n8k4.f64 (SASS: DMMA).
// The contraction index k runs over (sample, input-row) pairs; the augmented row [Phi_row | tau_row] gives
// G, b and tau^T tau from one symmetric rank-k update of a (P+1)x(P+1) matrix.
//
// General pipeline (any chain; the fused kernels of gram_fused.cu take over whenever the folded chain has at most 7 moving joints):
// materialise Phi for a chunk of samples into an L2-sized workspace (dyn_kernel) -> syrk_dmma_kernel streams it back (L2 hits) into
// per-CTA partials -> fixed-order reduction (bit-reproducible for a given launch geometry).  Correct for every chain and component
// set, but slow: it multiplies all structural zeros and feeds 9 DMMAs from 6 dependent L2 loads (0.076 G samples/s for the extended C6
// model, against 0.73 on the fused path).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "launch.h"

namespace rdb
{

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b)
{
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

constexpr int TB = 3;               // tiles per block side: a CTA owns a (TB*8) x (TB*8) block of the Gram matrix
constexpr int BLK = TB * 8;         // 24 columns
constexpr int SY_THREADS = 128;     // 4 warps, each takes a quarter of the CTA's samples
constexpr int TILE_ELEMS = TB * TB * 64;

// column c of the augmented row of (sample s, input row r): Phi plane c*n_in+r, or tau for c == P, 0 beyond
__device__ __forceinline__ double aug_load(const double* __restrict__ phi, const double* __restrict__ tau, int64_t ld, int n_in, int P, int c,
                                           int r, int64_t s, int64_t n)
{
  if (s >= n || c > P) return 0.0;
  const double* p = (c < P) ? phi + ((int64_t)c * n_in + r) * ld + s : tau + (int64_t)r * ld + s;
  return __ldg(p);
}

// partial[blockIdx.x][pair][TB*TB tiles][64]  (tile element (m,n) at m*8+n)
__global__ void __launch_bounds__(SY_THREADS) syrk_dmma_kernel(const double* __restrict__ phi, const double* __restrict__ tau, int64_t ld,
                                                               int64_t n, int n_in, int P, int nblk, double* __restrict__ partial)
{
  __shared__ double red[TILE_ELEMS];
  // decode the block pair (bi <= bj) from blockIdx.y
  int bi = 0, bj = 0;
  {
    int idx = blockIdx.y;
    for (bi = 0; bi < nblk; bi++)
    {
      const int cnt = nblk - bi;
      if (idx < cnt)
      {
        bj = bi + idx;
        break;
      }
      idx -= cnt;
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  double acc[TB][TB][2];
#pragma unroll
  for (int a = 0; a < TB; a++)
#pragma unroll
    for (int b = 0; b < TB; b++) acc[a][b][0] = acc[a][b][1] = 0.0;

  // samples are dealt to (CTA, warp) in groups of 4 (one k-step per input row)
  const int64_t groups = (n + 3) / 4;
  const int64_t nwarps = (int64_t)gridDim.x * 4;
  for (int64_t grp = (int64_t)blockIdx.x * 4 + warp; grp < groups; grp += nwarps)
  {
    const int64_t s = grp * 4 + t;
    for (int r = 0; r < n_in; r++)
    {
      double fa[TB], fb[TB];
#pragma unroll
      for (int a = 0; a < TB; a++) fa[a] = aug_load(phi, tau, ld, n_in, P, bi * BLK + a * 8 + g, r, s, n);
#pragma unroll
      for (int b = 0; b < TB; b++) fb[b] = (bi == bj) ? fa[b] : aug_load(phi, tau, ld, n_in, P, bj * BLK + b * 8 + g, r, s, n);
#pragma unroll
      for (int a = 0; a < TB; a++)
#pragma unroll
        for (int b = 0; b < TB; b++) dmma884(acc[a][b][0], acc[a][b][1], fa[a], fb[b]);
    }
  }

  // fixed-order reduction over the 4 warps, then one partial per CTA
  for (int w = 0; w < 4; w++)
  {
    if (warp == w)
    {
#pragma unroll
      for (int a = 0; a < TB; a++)
#pragma unroll
        for (int b = 0; b < TB; b++)
        {
          double* o = red + (a * TB + b) * 64 + g * 8 + 2 * t;
          if (w == 0)
          {
            o[0] = acc[a][b][0];
            o[1] = acc[a][b][1];
          }
          else
          {
            o[0] += acc[a][b][0];
            o[1] += acc[a][b][1];
          }
        }
    }
    __syncthreads();
  }
  double* out = partial + ((int64_t)blockIdx.x * gridDim.y + blockIdx.y) * TILE_ELEMS;
  for (int k = threadIdx.x; k < TILE_ELEMS; k += SY_THREADS) out[k] = red[k];
}

// G_aug = sum over CTAs (fixed order) of the partials; scatter to gram (full symmetric, column-major), rhs, tau_sq
__global__ void gram_reduce_kernel(const double* __restrict__ partial, int nparts, int npairs, int nblk, int P, double* __restrict__ gram,
                                   double* __restrict__ rhs, double* __restrict__ tau_sq, int accumulate)
{
  const int pair = blockIdx.x;
  int bi = 0, bj = 0;
  {
    int idx = pair;
    for (bi = 0; bi < nblk; bi++)
    {
      const int cnt = nblk - bi;
      if (idx < cnt)
      {
        bj = bi + idx;
        break;
      }
      idx -= cnt;
    }
  }
  for (int e = threadIdx.x; e < TILE_ELEMS; e += blockDim.x)
  {
    double s = 0.0;
    for (int p = 0; p < nparts; p++) s += partial[((int64_t)p * npairs + pair) * TILE_ELEMS + e];
    const int tile = e >> 6, m = (e >> 3) & 7, nn = e & 7;
    const int row = bi * BLK + (tile / TB) * 8 + m;
    const int col = bj * BLK + (tile % TB) * 8 + nn;
    if (row > P || col > P) continue;
    if (bi == bj && row > col) continue;  // diagonal blocks hold both halves; keep the upper one
    if (col < P)
    {
      // row <= col < P : G(row,col) and its mirror
      double* a = gram + (int64_t)col * P + row;
      double* b = gram + (int64_t)row * P + col;
      const double v = accumulate ? *a + s : s;
      *a = v;
      if (row != col) *b = v;
    }
    else if (row < P)
      rhs[row] = accumulate ? rhs[row] + s : s;
    else if (tau_sq)
      *tau_sq = accumulate ? *tau_sq + s : s;
  }
}

// tau_sq[k] = (accumulate ? tau_sq[k] : 0) + (part[k] + the measured torques of the inputs no chain joint feeds over segment k, squared and
// summed).  The fused kernels walk the folded chain, whose rows are the fed inputs only; such an input has a zero regressor row (nothing to
// add to G or b) but its torque is part of the residual |tau - Phi pi|^2.  part: the fused kernels' tau^T tau of this call.  One block per
// segment [offsets[k], offsets[k + 1]) (device offsets; nullptr: the one segment [0, n)), fixed order: reproducible.
struct UnfedRows
{
  int32_t n, row[RDB_MAX_JOINTS];
};
// W: the weighted sum of squares w t t (gram_unfed_tau_sq_weighted_kernel), in the same order
template <bool W>
__device__ __forceinline__ void gram_unfed_tau_sq_body(const double* __restrict__ tau, int64_t ld, int64_t n, const int64_t* __restrict__ offsets,
                                                       int64_t nseg, const UnfedRows& u, const double* __restrict__ part, double* __restrict__ tau_sq,
                                                       int accumulate, const rdb_gram_weights& wt)
{
  __shared__ double red[256];
  for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x)
  {
    const int64_t lo = offsets ? offsets[k] : 0, hi = offsets ? offsets[k + 1] : n;
    if (accumulate && lo == hi) continue;
    double s = 0.0;
    for (int r = 0; r < u.n; r++)
      for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x)
      {
        const double t = tau[(int64_t)u.row[r] * ld + i];
        if constexpr (W) s = fma(__dmul_rn(wt.w[u.row[r] * wt.joint_stride + i * wt.sample_stride], t), t, s);
        else s = fma(t, t, s);
      }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1)
    {
      if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
      __syncthreads();
    }
    if (threadIdx.x == 0)
    {
      const double v = part[k] + red[0];
      tau_sq[k] = accumulate ? tau_sq[k] + v : v;
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(256) gram_unfed_tau_sq_segmented_kernel(const double* __restrict__ tau, int64_t ld, int64_t n,
                                                                          const int64_t* __restrict__ offsets, int64_t nseg, UnfedRows u,
                                                                          const double* __restrict__ part, double* __restrict__ tau_sq,
                                                                          int accumulate)
{
  gram_unfed_tau_sq_body<false>(tau, ld, n, offsets, nseg, u, part, tau_sq, accumulate, rdb_gram_weights{});
}
__global__ void __launch_bounds__(256) gram_unfed_tau_sq_weighted_kernel(const double* __restrict__ tau, int64_t ld, int64_t n,
                                                                         const int64_t* __restrict__ offsets, int64_t nseg, UnfedRows u,
                                                                         const double* __restrict__ part, double* __restrict__ tau_sq,
                                                                         int accumulate, const rdb_gram_weights wt)
{
  gram_unfed_tau_sq_body<true>(tau, ld, n, offsets, nseg, u, part, tau_sq, accumulate, wt);
}

// the inputs no chain joint feeds
static UnfedRows unfed_rows(const ChainHost& ch)
{
  UnfedRows u{};
  std::vector<char> fed(ch.host.n_in, 0);
  for (int j = 0; j < ch.host.nj; j++)
    if (ch.host.joint[j].in >= 0) fed[ch.host.joint[j].in] = 1;
  for (int i = 0; i < ch.host.n_in; i++)
    if (!fed[i]) u.row[u.n++] = i;
  return u;
}

cudaError_t launch_unfed_tau_sq(const ChainHost& ch, const double* tau, int64_t ld, int64_t n, const int64_t* offsets, int64_t nseg,
                                const double* part, double* tau_sq, int accumulate, cudaStream_t st, const rdb_gram_weights* wt)
{
  if (nseg <= 0) return cudaSuccess;
  const unsigned grid = (unsigned)std::min<int64_t>(nseg, 65535);
  if (wt) gram_unfed_tau_sq_weighted_kernel<<<grid, 256, 0, st>>>(tau, ld, n, offsets, nseg, unfed_rows(ch), part, tau_sq, accumulate, *wt);
  else gram_unfed_tau_sq_segmented_kernel<<<grid, 256, 0, st>>>(tau, ld, n, offsets, nseg, unfed_rows(ch), part, tau_sq, accumulate);
  count_launch();
  return cudaGetLastError();
}

// General pipeline, weighted: row r of every Phi plane of a chunk (plane c n_in + r, c < P) and of the staged tau, times sqrt(w) of that row
// and sample, so that the SYRK's sums of products carry w once.  Sample s of the chunk is sample off + s of the call.
__global__ void gram_weight_rows_kernel(double* __restrict__ phi, double* __restrict__ tau, int64_t ld, int64_t len, int n_in, int P,
                                        const rdb_gram_weights wt, int64_t off)
{
  const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (s >= len) return;
  const double sw = sqrt(wt.w[r * wt.joint_stride + (off + s) * wt.sample_stride]);
  for (int c = 0; c < P; c++) phi[((int64_t)c * n_in + r) * ld + s] *= sw;
  tau[(int64_t)r * ld + s] *= sw;
}

// rdb_chain_gram_kernel_info after a call on the general pipeline: why the fused kernels did not take it
static std::string general_pipeline_why(const ChainHost& ch, bool force_v0, bool with_components)
{
  const int K = ch.gram.fold.nj;
  if (force_v0) return "general pipeline: RDB_GRAM_IMPL=v0";
  if (K > 7) return "general pipeline: more than 7 moving joints (" + std::to_string(K) + ")";
  if (K < 1) return "general pipeline: no moving joint";
  if (with_components)
    return "general pipeline: a component set the one-pass kernel refuses (a component on an input no chain joint feeds, "
           "or more than 8 component columns on one joint)";
  return "general pipeline: the fused kernel does not take this chain";
}

// Development builds (-DRDB_DEV_SWITCHES, never the shipped library) can force the general pipeline with RDB_GRAM_IMPL=v0
static bool gram_force_v0()
{
#ifdef RDB_DEV_SWITCHES
  static const bool force_v0 = [] { const char* e = getenv("RDB_GRAM_IMPL"); return e && e[0] == 'v'; }();
  return force_v0;
#else
  return false;
#endif
}

static cudaError_t gram_launches(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                 int accumulate, cudaStream_t st, bool with_components, const rdb_gram_weights* wt = nullptr)
{
  const int n_in = ch.host.n_in, Pr = 10 * ch.host.nj;     // rigid-body columns
  const int P = Pr + (with_components ? ch.comps.cols : 0);  // + component columns (extended model)
  if (in.n <= 0 || n_in == 0 || P == 0)
  {
    if (!accumulate)
    {
      cudaMemsetAsync(gram, 0, sizeof(double) * P * P, st);
      cudaMemsetAsync(rhs, 0, sizeof(double) * P, st);
      if (tau_sq) cudaMemsetAsync(tau_sq, 0, sizeof(double), st);
    }
    return cudaGetLastError();
  }
  {
    // fused warp-specialised kernel (gram_fused.cu) whenever the chain fits it
    const bool force_v0 = gram_force_v0();
    if (!force_v0)
    {
      cudaError_t e = cudaErrorNotSupported;
      // measured torques on inputs no chain joint feeds: the fused kernels' tau^T tau goes to a zeroed scratch word first
      const bool unfed = tau_meas && tau_sq && !ch.inputs_cover_all;
      if (unfed)
      {
        e = ch.gram.tau_sq_part.grow(sizeof(double), ch.gram.done);
        if (e != cudaSuccess) return e;
        cudaMemsetAsync(ch.gram.tau_sq_part.get(), 0, sizeof(double), st);
      }
      double* ts = unfed ? ch.gram.tau_sq_part.get() : tau_sq;
      if (P == Pr)
        e = launch_gram_fused(ch, in, tau_meas, gram, rhs, ts, accumulate, st, wt);
      else
        e = launch_gram_fused_ext(ch, in, tau_meas, gram, rhs, ts, accumulate, st, wt);
      if (e == cudaSuccess && unfed) e = launch_unfed_tau_sq(ch, tau_meas, in.ld, in.n, nullptr, 1, ts, tau_sq, accumulate, st, wt);
      if (e != cudaErrorNotSupported) return e;
    }
    // rdb_chain_gram_kernel_info describes the last Gram call: say that this one ran the general pipeline, and why
    ch.gram.kernel_specialised = 2;
    ch.gram.kernel_why = general_pipeline_why(ch, force_v0, P != Pr);
  }
  const int nblk = (P + 1 + BLK - 1) / BLK;
  const int npairs = nblk * (nblk + 1) / 2;
  // chunk: Phi (+tau) of the chunk should stay L2 resident (~126 MB L2): <= 48 MB
  const int64_t bytes_per_sample = sizeof(double) * ((int64_t)P * n_in + n_in);
  int64_t chunk = std::max<int64_t>(1024, (48ll << 20) / bytes_per_sample);
  chunk = std::min<int64_t>((chunk / 128) * 128, std::max<int64_t>(in.n, 128));
  const int gx = std::max(1, std::min<int>(ch.sm_count * 2 / std::max(1, npairs) + 1, (int)((chunk + 15) / 16)));
  const size_t need = sizeof(double) * ((size_t)chunk * (P * n_in + n_in) + (size_t)gx * npairs * TILE_ELEMS);
  cudaError_t e = ch.gram.partials.grow(need, ch.gram.done);
  if (e != cudaSuccess) return e;
  double* w_phi = ch.gram.partials.get();
  double* w_tau = w_phi + (size_t)chunk * P * n_in;
  double* w_part = w_tau + (size_t)chunk * n_in;
  for (int64_t off = 0; off < in.n; off += chunk)
  {
    const int64_t len = std::min<int64_t>(chunk, in.n - off);
    SamplesDev v{len, in.ld, in.q + off, in.dq + off, in.ddq + off, nullptr};
    const bool own_tau = (tau_meas == nullptr);
    if (!ch.inputs_cover_all) cudaMemsetAsync(w_phi, 0, sizeof(double) * (size_t)chunk * (P * n_in + n_in), st);
    e = launch_dyn(ch, own_tau ? (DYN_REGRESSOR_ | DYN_TORQUE_) : DYN_REGRESSOR_, v, w_phi, own_tau ? w_tau : nullptr, nullptr, chunk, st);
    if (e != cudaSuccess) return e;
    if (P > Pr)  // component planes follow the rigid-body planes (plane index = col * n_in + row)
    {
      e = launch_components_regressor(ch, v, w_phi + (size_t)Pr * n_in * chunk, chunk, st);
      if (e != cudaSuccess) return e;
    }
    const double* tau = own_tau ? w_tau : tau_meas + off;
    const int64_t tau_ld = own_tau ? chunk : in.ld;
    // the SYRK kernel takes one ld for both; when tau comes from the caller with another stride, stage it (weighted: always, it is scaled)
    if (!own_tau && (tau_ld != chunk || wt))
    {
      e = cudaMemcpy2DAsync(w_tau, chunk * sizeof(double), tau, tau_ld * sizeof(double), len * sizeof(double), n_in, cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) return e;
      tau = w_tau;
    }
    if (wt)
    {
      gram_weight_rows_kernel<<<dim3((unsigned)((len + 255) / 256), n_in), 256, 0, st>>>(w_phi, w_tau, chunk, len, n_in, P, *wt, off);
      count_launch();
    }
    syrk_dmma_kernel<<<dim3(gx, npairs), SY_THREADS, 0, st>>>(w_phi, tau, chunk, len, n_in, P, nblk, w_part);
    count_launch();
    gram_reduce_kernel<<<npairs, 256, 0, st>>>(w_part, gx, npairs, nblk, P, gram, rhs, tau_sq, (accumulate || off > 0) ? 1 : 0);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// Every Gram call of a handle (device entries, the host entry's chunks, the group's shards) runs its launches through here.  The workspace
// of ch.gram is shared by all of them, and callers may pass any stream: each call's stream first waits for the device work of the previous
// call (free on the same stream), and the call's own work is recorded for the next one.
template <class F>
static cudaError_t ordered_gram_call(ChainHost& ch, cudaStream_t st, F&& launches)
{
  cudaError_t e = ch.gram.done.ensure();
  if (e != cudaSuccess) return e;
  e = cudaStreamWaitEvent(st, ch.gram.done, 0);
  if (e != cudaSuccess) return e;
  e = launches();
  const cudaError_t r = cudaEventRecord(ch.gram.done, st);  // also after a failed launch: whatever was queued stays ordered
  return e != cudaSuccess ? e : r;
}

cudaError_t launch_gram(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq, int accumulate,
                        cudaStream_t st, bool with_components, const rdb_gram_weights* wt)
{
  return ordered_gram_call(ch, st, [&] { return gram_launches(ch, in, tau_meas, gram, rhs, tau_sq, accumulate, st, with_components, wt); });
}

static cudaError_t gram_segmented_launches(ChainHost& ch, const SamplesDev& in, const double* tau_meas, int64_t nseg, const int64_t* offsets,
                                           double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st)
{
  const int64_t P = 10 * ch.host.nj;
  const bool force_v0 = gram_force_v0();
  if (!force_v0 && ch.host.n_in > 0 && P > 0)
  {
    const bool unfed = tau_meas && tau_sq && !ch.inputs_cover_all;
    const cudaError_t e = launch_gram_fused_segmented(ch, in, tau_meas, nseg, offsets, gram, rhs, tau_sq, accumulate, unfed, st);
    if (e != cudaErrorNotSupported) return e;
  }
  // the general pipeline, one pass per segment: correct for every chain, slow for many short segments.  ch.gram.done is recorded behind
  // every segment, so that a workspace which grows for a longer segment is freed only once the segments before it are done with it
  for (int64_t k = 0; k < nseg; k++)
  {
    const int64_t lo = offsets[k], hi = offsets[k + 1];
    auto at = [&](const double* p) { return p ? p + lo : nullptr; };
    const SamplesDev v{hi - lo, in.ld, at(in.q), at(in.dq), at(in.ddq), nullptr};
    cudaError_t e = gram_launches(ch, v, at(tau_meas), gram + k * P * P, rhs + k * P, tau_sq ? tau_sq + k : nullptr, accumulate, st, false);
    if (e != cudaSuccess) return e;
    e = cudaEventRecord(ch.gram.done, st);
    if (e != cudaSuccess) return e;
  }
  ch.gram.kernel_specialised = 2;
  ch.gram.kernel_why = "general pipeline: one pass per segment (slow for short segments); " +
                       general_pipeline_why(ch, force_v0, false).substr(sizeof("general pipeline: ") - 1);
  return cudaSuccess;
}

cudaError_t launch_gram_segmented(ChainHost& ch, const SamplesDev& in, const double* tau_meas, int64_t nseg, const int64_t* offsets, double* gram,
                                  double* rhs, double* tau_sq, int accumulate, cudaStream_t st)
{
  return ordered_gram_call(ch, st, [&] { return gram_segmented_launches(ch, in, tau_meas, nseg, offsets, gram, rhs, tau_sq, accumulate, st); });
}

// ---------------------------------------------------------------------------------------------------------
// FP64 pipe micro-benchmarks: the repo's own roofline denominator for the Gram path
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double x)
{
  double a[16];
#pragma unroll
  for (int k = 0; k < 16; k++) a[k] = threadIdx.x * 1e-3 + k;
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int k = 0; k < 16; k++) a[k] = fma(a[k], x, 1e-9);
  }
  double s = 0;
#pragma unroll
  for (int k = 0; k < 16; k++) s += a[k];
  if (s == 12345.678) out[0] = s;
}
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double x)
{
  double c[16][2];
#pragma unroll
  for (int k = 0; k < 16; k++) c[k][0] = c[k][1] = threadIdx.x * 1e-3 + k;
  const double a = x, b = 1.0 - x * 1e-12;
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int k = 0; k < 16; k++) dmma884(c[k][0], c[k][1], a, b);
  }
  double s = 0;
#pragma unroll
  for (int k = 0; k < 16; k++) s += c[k][0] + c[k][1];
  if (s == 12345.678) out[0] = s;
}

// both at once, independent accumulators: tells whether DFMA and DMMA share one FP64 datapath (sum ~= single peak) or not
__global__ void __launch_bounds__(256) dmix_peak_kernel(double* out, int iters, double x)
{
  double c[8][2], a[16];
#pragma unroll
  for (int k = 0; k < 8; k++) c[k][0] = c[k][1] = threadIdx.x * 1e-3 + k;
#pragma unroll
  for (int k = 0; k < 16; k++) a[k] = threadIdx.x * 1e-3 + k;
  const double fa = x, fb = 1.0 - x * 1e-12;
  for (int it = 0; it < iters; it++)
  {
#pragma unroll
    for (int k = 0; k < 8; k++)
    {
      dmma884(c[k][0], c[k][1], fa, fb);
      a[2 * k] = fma(a[2 * k], x, 1e-9);
      a[2 * k + 1] = fma(a[2 * k + 1], x, 1e-9);
    }
  }
  double s = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) s += c[k][0] + c[k][1] + a[2 * k] + a[2 * k + 1];
  if (s == 12345.678) out[0] = s;
}

cudaError_t fp64_peak(int kind, int reps, double* tflops)
{
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double* d = nullptr;
  cudaError_t e = cudaMalloc(&d, 64);
  if (e != cudaSuccess) return e;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  const int iters = 4096, blocks = sms * 8, threads = 256;
  double best = 0;
  for (int r = 0; r < std::max(1, reps) + 1; r++)
  {
    cudaEventRecord(e0);
    if (kind == 0) dfma_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999);
    else if (kind == 1) dmma_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999);
    else dmix_peak_kernel<<<blocks, threads>>>(d, iters, 0.999999);
    count_launch();
    cudaEventRecord(e1);
    e = cudaEventSynchronize(e1);
    if (e != cudaSuccess) break;
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    // DFMA: 2 flop per lane-instruction; DMMA m8n8k4: 2*8*8*4 = 512 flop per warp-instruction
    const double flop = kind == 0   ? 2.0 * 16 * iters * (double)blocks * threads
                        : kind == 1 ? 512.0 * 16 * iters * (double)blocks * (threads / 32)
                                    : (512.0 * 8 * (threads / 32) + 2.0 * 16 * threads) * iters * (double)blocks;
    if (r > 0) best = std::max(best, flop / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *tflops = best;
  return e;
}

}  // namespace rdb
