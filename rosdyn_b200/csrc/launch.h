// launch.h -- host-side handle contents and kernel launcher declarations (internal).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "chain_dev.h"

namespace rdb
{

struct GramWorkspace
{
  double* partials = nullptr;  // per-CTA partial normal equations
  size_t bytes = 0;
  int ctas = 0;
  double* fused_partials = nullptr;  // gram_fused.cu: per-CTA partial (P+1)x(P+1) upper-triangular tiles
  size_t fused_bytes = 0;
  // fold.cpp: the chain with its never-moving joints folded away (fold_chain), rebuilt when the model changes
  ChainDev<RDB_MAX_JOINTS> fold;
  uint64_t fold_version = ~0ull;
  bool fold_identity = true;   // nothing was folded: no expansion step
  double* fold_dev = nullptr;  // parameter maps T | reduced normal equations | link -> reduced link
  size_t fold_bytes = 0;
  double* ext_dev = nullptr;   // extended model: rigid-body block | cross-tile sums | cross partials | component map
  size_t ext_bytes = 0;
  double* tau_sq_part = nullptr;  // gram.cu: the fused kernels' tau^T tau when measured torques also sit on inputs no chain joint feeds
  // which kernel the last Gram call ran (rdb_chain_gram_kernel_info): 1 run-time specialised (gram_jit.cpp), 0 precompiled, 2 general
  // pipeline (gram.cu), -1 none yet
  int kernel_specialised = -1;
  std::string kernel_why = "no fused Gram call yet";
};

// persistent pipeline of rdb_regressor_gram_batch_host (capi.cu)
struct GramHostPipe
{
  static constexpr int NSLOT = 3;
  cudaStream_t copy = nullptr, comp = nullptr;
  double* stage[NSLOT] = {nullptr, nullptr, nullptr};  // q | dq | ddq | tau_meas planes of one chunk
  cudaEvent_t copied[NSLOT] = {nullptr, nullptr, nullptr}, freed[NSLOT] = {nullptr, nullptr, nullptr};
  double* d_out = nullptr;  // gram | rhs | tau_sq
  size_t n_out = 0;
  int planes = -1;
  // pageable callers (std::vector, numpy): pinned bounce buffers filled by host threads, so that the copies to the device stay asynchronous
  // and run at the link's rate instead of the driver's single-threaded staging (11 GB/s measured)
  double* pin[NSLOT] = {nullptr, nullptr, nullptr};
  size_t pin_doubles = 0;
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
  double* base = nullptr;
  size_t bytes = 0;
  cudaStream_t st[2] = {nullptr, nullptr};
  // small calls (a handful of samples, the per-sample getters of the C++ facade): one mapped pinned buffer that the kernels read and write
  // in place over PCIe -- one launch and one synchronisation instead of a copy call per array
  double* map_h = nullptr;
  double* map_d = nullptr;
  bool map_failed = false;
  // pageable callers: pinned mirror of the device arena; host threads gather inputs into it / scatter outputs out of it, so that every copy
  // to or from the device is asynchronous and contiguous (the driver stages copies on pageable memory synchronously on one thread)
  double* pin = nullptr;
  size_t pin_bytes = 0;
  bool pin_failed = false;
};
constexpr size_t RDB_HOST_MAPPED_BYTES = 256 << 10;

struct ChainHost
{
  ComponentsDev comps{};
  ChainDev<RDB_MAX_JOINTS> host;           // model constants, host copy
  ChainDev<RDB_MAX_JOINTS>* dev = nullptr;  // same, in device memory (generic kernels)
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
// with_components: the extended model [Phi | Phi_c] (general pipeline); else the rigid-body columns only (fused kernel when it fits)
cudaError_t launch_gram(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                        int accumulate, cudaStream_t st, bool with_components = false);
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
// fold.cpp: the chain with its never-moving joints folded away and its revolute axes on +z (ch.gram.fold); rebuilt by every model upload
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
// gram_fused.cu: cudaErrorNotSupported when the chain does not fit the fused kernel
cudaError_t launch_gram_fused(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                              int accumulate, cudaStream_t st);
// gram_fused.cu: G = E^T G' E, b = E^T b' from the reduced (folded-chain) normal equations kept in ch.gram.fold_dev
cudaError_t launch_fold_expand(ChainHost& ch, double* gram, double* rhs, double* tau_sq, int accumulate, cudaStream_t st);
// same for the extended model [Phi | Phi_c] (gram is Pt x Pt, Pt = 10 nJ + component columns)
cudaError_t launch_gram_fused_ext(ChainHost& ch, const SamplesDev& in, const double* tau_meas, double* gram, double* rhs, double* tau_sq,
                                  int accumulate, cudaStream_t st);

enum : int
{
  DYN_REGRESSOR_ = 1,
  DYN_TORQUE_ = 2,
  DYN_INERTIA_ = 4,
  DYN_FD_ = 8
};

}  // namespace rdb
