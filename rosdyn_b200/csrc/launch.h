// launch.h -- host-side handle contents and kernel launcher declarations (internal).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "chain_dev.h"

namespace rdb
{

// An owning allocation of device memory (Pinned = false) or of pinned host memory (cudaHostAlloc with the flags given at construction),
// viewed as T.  It only grows.  Move-only; it makes no CUDA call at all while it holds nothing, so that handles built without a device
// (rdb_gram_specialised_cubin) stay free of CUDA calls.
template <class T, bool Pinned>
class Buffer
{
 public:
  explicit Buffer(unsigned flags = cudaHostAllocDefault) : flags_(flags) {}
  Buffer(Buffer&& o) noexcept : p_(o.p_), bytes_(o.bytes_), flags_(o.flags_)
  {
    o.p_ = nullptr;
    o.bytes_ = 0;
  }
  Buffer& operator=(Buffer&& o) noexcept
  {
    std::swap(p_, o.p_);
    std::swap(bytes_, o.bytes_);
    std::swap(flags_, o.flags_);
    return *this;
  }
  ~Buffer() { reset(); }
  // at least `bytes`, contents not kept when it has to grow.  wait_before_free, when given, is synchronised before the old allocation is
  // freed: device work recorded before it may still use that allocation.  On a failed allocation the buffer is empty and the error returned.
  cudaError_t grow(size_t bytes, cudaEvent_t wait_before_free)
  {
    if (bytes_ >= bytes) return cudaSuccess;
    if (p_ && wait_before_free)
    {
      const cudaError_t e = cudaEventSynchronize(wait_before_free);
      if (e != cudaSuccess) return e;
    }
    reset();
    void* p = nullptr;
    const cudaError_t e = Pinned ? cudaHostAlloc(&p, bytes, flags_) : cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return e;
    p_ = static_cast<T*>(p);
    bytes_ = bytes;
    return cudaSuccess;
  }
  void reset()
  {
    if (!p_) return;
    if (Pinned) cudaFreeHost(p_);
    else cudaFree(p_);
    p_ = nullptr;
    bytes_ = 0;
  }
  T* get() const { return p_; }

 private:
  T* p_ = nullptr;
  size_t bytes_ = 0;
  unsigned flags_;
};
template <class T = double>
using DeviceBuffer = Buffer<T, false>;
template <class T = double>
using PinnedBuffer = Buffer<T, true>;

// A stream (non-blocking) or event (no timing) of the handle: created on first use, destroyed with the handle; no CUDA call while it holds
// nothing.
template <class H>
class Owned
{
 public:
  Owned() = default;
  Owned(const Owned&) = delete;
  Owned& operator=(const Owned&) = delete;
  ~Owned()
  {
    if (h_) destroy(h_);
  }
  cudaError_t ensure() { return h_ ? cudaSuccess : create(&h_); }
  operator H() const { return h_; }

 private:
  static cudaError_t create(cudaStream_t* s) { return cudaStreamCreateWithFlags(s, cudaStreamNonBlocking); }
  static cudaError_t create(cudaEvent_t* e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming); }
  static void destroy(cudaStream_t s) { cudaStreamDestroy(s); }
  static void destroy(cudaEvent_t e) { cudaEventDestroy(e); }
  H h_ = nullptr;
};
using OwnedStream = Owned<cudaStream_t>;
using OwnedEvent = Owned<cudaEvent_t>;

// Every buffer below but `fold_dev` is Gram-call scratch: it grows with wait_before_free = `done`.
struct GramWorkspace
{
  DeviceBuffer<> partials;  // general pipeline (gram.cu): Phi and tau of a chunk | per-CTA partial normal equations
  DeviceBuffer<> fused_partials;  // gram_fused.cu: per-CTA partial (P+1)x(P+1) upper-triangular tiles
  // fold.cpp: the chain with its never-moving joints folded away (fold_chain), rebuilt when the model changes
  ChainDev<RDB_MAX_JOINTS> fold;
  uint64_t fold_version = ~0ull;
  bool fold_identity = true;   // nothing was folded: no expansion step
  DeviceBuffer<> fold_dev;     // fold maps (fold_maps): parameter maps T | link -> reduced link; written by fold_chain only
  DeviceBuffer<> reduced;      // reduced normal equations of the folded chain, one row per system (reduced_row)
  DeviceBuffer<> ext_dev;      // extended model: rigid-body block | cross-tile sums | cross partials | component map
  DeviceBuffer<> tau_sq_part;  // gram.cu: the fused kernels' tau^T tau when measured torques also sit on inputs no chain joint feeds
  DeviceBuffer<> seg_dev;      // gram_fused.cu, segmented calls: item partials of a wave | per-segment tau^T tau | item table
  // recorded after the last launch of every Gram call (launch_gram): the next call's stream waits for it before it touches the buffers
  // above, so the Gram calls of one handle run their device work in call order whatever streams they come on; a buffer is freed only
  // once it has completed
  OwnedEvent done;
  // which kernel the last Gram call ran (rdb_chain_gram_kernel_info): 1 run-time specialised (gram_jit.cpp), 0 precompiled, 2 general
  // pipeline (gram.cu), -1 none yet
  int kernel_specialised = -1;
  std::string kernel_why = "no fused Gram call yet";
};

// persistent pipeline of rdb_regressor_gram_batch_host (capi.cu)
struct GramHostPipe
{
  static constexpr int NSLOT = 3;
  OwnedStream copy, comp;
  DeviceBuffer<> stage[NSLOT];  // q | dq | ddq | tau_meas planes of one chunk
  OwnedEvent copied[NSLOT], freed[NSLOT];
  DeviceBuffer<> d_out;  // gram | rhs | tau_sq
  // pageable callers (std::vector, numpy): pinned bounce buffers filled by host threads, so that the copies to the device stay asynchronous
  // and run at the link's rate instead of the driver's single-threaded staging (11 GB/s measured)
  PinnedBuffer<> pin[NSLOT];
  bool pin_failed = false;
};

// additive joint components (friction_polynomial1.h / friction_polynomial2.h / ideal_spring.h), device image
struct ComponentDev
{
  int32_t type, in, col, ncols;
  double thr, vmax;
};
struct ComponentsDev
{
  int32_t n, cols;
  ComponentDev c[RDB_MAX_COMPONENTS];
};
struct ComponentParams
{
  double p[3 * RDB_MAX_COMPONENTS];
};

// staging arena of the *_host entry points (kinematics / torque / regressor / inertia): device buffers and streams kept in the handle, so that
// a host call does not pay cudaMalloc / cudaFree of its (up to GB-sized) double buffers every time
struct HostArena
{
  DeviceBuffer<> base;
  OwnedStream st[2];
  // small calls (a handful of samples, the per-sample getters of the C++ facade): one mapped pinned buffer that the kernels read and write
  // in place over PCIe -- one launch and one synchronisation instead of a copy call per array
  PinnedBuffer<> map_h{cudaHostAllocMapped};
  double* map_d = nullptr;  // device alias of map_h
  bool map_failed = false;
  // pageable callers: pinned mirror of the device arena; host threads gather inputs into it / scatter outputs out of it, so that every copy
  // to or from the device is asynchronous and contiguous (the driver stages copies on pageable memory synchronously on one thread)
  PinnedBuffer<> pin;
  bool pin_failed = false;
};
constexpr size_t RDB_HOST_MAPPED_BYTES = 256 << 10;

struct ChainHost
{
  ComponentsDev comps{};
  ChainDev<RDB_MAX_JOINTS> host;           // model constants, host copy
  DeviceBuffer<ChainDev<RDB_MAX_JOINTS>> dev;  // same, in device memory (generic kernels)
  int device = 0;
  bool inputs_cover_all = true;  // every input index is fed by a chain joint (else outputs are pre-zeroed)
  double nominal[10 * RDB_MAX_JOINTS];
  GramWorkspace gram;
  GramHostPipe gram_host;
  HostArena host_arena;
  int sm_count = 148;
  uint64_t model_version = 0;  // bumped by every upload of the model (creation, rdb_chain_set_input_joints)
  // serialises the entries that touch the handle's mutable state (model upload, Gram workspaces, the staging pipelines of the *_host entries):
  // two host threads may share one handle -- their calls run one after the other instead of racing
  std::recursive_mutex mu;
};

// the fold maps of the handle (ch.gram.fold_dev, folded chains only): T, 10 x 10 per link of the model, then link -> reduced link (-1: none)
struct FoldMaps
{
  double* T;
  int32_t* kof;
};
inline FoldMaps fold_maps(const ChainHost& ch)
{
  double* T = ch.gram.fold_dev.get();
  return {T, reinterpret_cast<int32_t*>(T + (size_t)ch.host.nj * 100)};
}
// reduced normal equations r of the folded chain (ch.gram.reduced): row r of a segmented wave, row 0 for the unsegmented calls
struct ReducedRow
{
  double *G, *b, *tau_sq;  // G' (Pr x Pr, Pr = 10 moving joints) | b' (Pr) | tau^T tau
  static int64_t doubles(int Pr) { return (int64_t)Pr * Pr + Pr + 1; }  // row stride
};
inline ReducedRow reduced_row(const ChainHost& ch, int64_t r)
{
  const int Pr = 10 * ch.gram.fold.nj;
  double* G = ch.gram.reduced.get() + r * ReducedRow::doubles(Pr);
  return {G, G + (size_t)Pr * Pr, G + (size_t)Pr * Pr + Pr};
}

// the model's first NJ joints and links, by value for the kernels instantiated per joint count
template <int NJ>
inline ChainDev<NJ> narrow(const ChainDev<RDB_MAX_JOINTS>& h)
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

// RAII: make the handle's device current for the duration of an entry point and restore the caller's device afterwards
struct DeviceScope
{
  int prev = -1;
  bool switched = false;
  cudaError_t err = cudaSuccess;
  explicit DeviceScope(int device)
  {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device)
    {
      err = cudaSetDevice(device);
      switched = err == cudaSuccess;
    }
  }
  ~DeviceScope()
  {
    if (switched) cudaSetDevice(prev);
  }
  DeviceScope(const DeviceScope&) = delete;
  DeviceScope& operator=(const DeviceScope&) = delete;
};

extern std::atomic<uint64_t> g_launches;
inline void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

cudaError_t launch_dyn(const ChainHost& ch, int mode, const SamplesDev& in, double* phi, double* tau, double* M, int64_t ld_out,
                       cudaStream_t st);
cudaError_t launch_dyn(const ChainHost& ch, int mode, const SamplesDev& in, const DynOutDev& out, cudaStream_t st);
cudaError_t launch_kin(const ChainHost& ch, unsigned want, const SamplesDev& in, const KinOutDev& o, cudaStream_t st);
cudaError_t launch_fill_uniform(double* x, int n_planes, int64_t n, int64_t ld, uint64_t seed, int stream_id, cudaStream_t st);
void fill_uniform_host(double* x, int n_planes, int64_t n, int64_t ld, uint64_t seed, int stream_id);

// gram.cu
// with_components: the extended model [Phi | Phi_c] (general pipeline); else the rigid-body columns only (fused kernel when it fits).
// wt: the weighted normal equations (rdb_regressor_gram_weighted_batch), nullptr: unweighted.
// Ordered after the previous Gram call of the handle on any stream (ch.gram.done).
cudaError_t launch_gram(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                        int accumulate, cudaStream_t st, bool with_components = false, const rdb_gram_weights* wt = nullptr);
// aux.cu: getWrench / getJointTorque with external wrenches, getJacobianLink (two-pass kernels, not the throughput path)
cudaError_t launch_aux(const ChainHost& ch, const SamplesDev& in, const double* ext, int64_t ld_ext, double* torque, double* wrenches,
                       double* jac_link, int link, int64_t ld_out, cudaStream_t st);
// ik.cu: batched local IK (Chain::computeLocalIk, primitives_impl.h:1398-1468)
cudaError_t launch_ik(const ChainHost& ch, int64_t n, int64_t ld, const double* target, const double* seed, const double* q_min,
                      const double* q_max, const double* weight, double tol, int max_iter, double* sol, int32_t* status, int32_t* iters,
                      double* err, cudaStream_t st);
// components.cu
cudaError_t launch_components_regressor(const ChainHost& ch, const SamplesDev& in, double* phi_c, int64_t ld_out, cudaStream_t st);
cudaError_t launch_components_torque(const ChainHost& ch, const SamplesDev& in, const ComponentParams& prm, double* torque, int64_t ld_out,
                                     int accumulate, cudaStream_t st);
cudaError_t fp64_peak(int kind, int reps, double* tflops);
// fold.cpp: the chain with its never-moving joints folded away and its revolute axes on +z (ch.gram.fold); rebuilt by every model upload.
// upload = true rewrites the fold maps (ch.gram.fold_dev): no work that reads them may be queued or running (upload_model synchronises the
// device first)
cudaError_t fold_chain(ChainHost& ch, bool upload = true);  // upload = false: the host image ch.gram.fold only
// every joint of the folded chain is revolute about exactly e_z of its link frame: the fused kernels' REV generators (gram_common.cuh) hold
// the axis as a compile-time constant; any other chain takes the generic generator
inline bool fold_rev_canonical(const ChainDev<RDB_MAX_JOINTS>& F)
{
  bool rev = true;
  for (int j = 0; j < F.nj; j++)
    rev = rev && F.joint[j].type == RDB_JOINT_REVOLUTE && F.joint[j].ax[0] == REV_AXIS[0] && F.joint[j].ax[1] == REV_AXIS[1] &&
          F.joint[j].ax[2] == REV_AXIS[2];
  return rev;
}
// gram_jit.cpp: the fused kernel `kernel_args` ("gram_fused_kernel<6, 4, true, 0": template arguments without the model) compiled at run
// time against the constants of ch.gram.fold, or nullptr when the precompiled instantiation has to run; records which one and why in ch.gram.
const void* gram_jit_kernel(ChainHost& ch, const char* kernel_args);
// gram_jit.cpp: the same kernel's cubin for `arch` (e.g. "sm_100a") without a device (rdb_gram_specialised_cubin)
bool gram_jit_cubin(const ChainDev<RDB_MAX_JOINTS>& F, const char* kernel_args, const char* arch, std::vector<char>& cubin, std::string& why);
// gram_fused.cu: cudaErrorNotSupported when the chain does not fit the fused kernel; wt: weighted (gram_fused_weighted_kernel)
cudaError_t launch_gram_fused(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                              int accumulate, cudaStream_t st, const rdb_gram_weights* wt = nullptr);
// gram.cu: the normal equations of every segment [offsets[k], offsets[k + 1]) of the batch (host offsets, k < nseg), segment k at gram + k P P,
// rhs + k P, tau_sq + k; fused segmented kernel when the chain fits it, else the general pipeline once per segment.  Ordered like launch_gram.
cudaError_t launch_gram_segmented(ChainHost& ch, const SamplesDev& in, const double* tau_meas, int64_t nseg, const int64_t* offsets, double* gram,
                                  double* rhs, double* tau_sq, int accumulate, cudaStream_t st);
// gram_fused.cu: the fused part of the above; cudaErrorNotSupported when the chain does not fit the fused kernel.  unfed: tau_sq gets the
// measured torques of the inputs no chain joint feeds too (launch_unfed_tau_sq)
cudaError_t launch_gram_fused_segmented(ChainHost& ch, const SamplesDev& in, const double* tau_meas, int64_t nseg, const int64_t* offsets,
                                        double* gram, double* rhs, double* tau_sq, int accumulate, bool unfed, cudaStream_t st);
// gram.cu: tau_sq[k] = (accumulate ? tau_sq[k] : 0) + part[k] + the squares of the measured torques of the inputs no chain joint feeds over
// segment k (device offsets [nseg + 1]; nullptr: the one segment [0, n)); an empty segment is left as it is when accumulating.
// wt: each square times its weight (one segment only)
cudaError_t launch_unfed_tau_sq(const ChainHost& ch, const double* tau, int64_t ld, int64_t n, const int64_t* offsets, int64_t nseg,
                                const double* part, double* tau_sq, int accumulate, cudaStream_t st, const rdb_gram_weights* wt = nullptr);
// gram_fused.cu: G = E^T G' E, b = E^T b' from the reduced (folded-chain) normal equations of reduced_row(ch, 0)
cudaError_t launch_fold_expand(ChainHost& ch, double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st);
// same for the extended model [Phi | Phi_c] (gram is Pt x Pt, Pt = 10 nJ + component columns)
cudaError_t launch_gram_fused_ext(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                  int accumulate, cudaStream_t st, const rdb_gram_weights* wt = nullptr);

enum : int
{
  DYN_REGRESSOR_ = 1,
  DYN_TORQUE_ = 2,
  DYN_INERTIA_ = 4,
  DYN_FD_ = 8
};

}  // namespace rdb
