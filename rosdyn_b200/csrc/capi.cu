// capi.cu -- implementation of the C-ABI declared in include/rosdyn_b200.h.
// Host-side model build (the cold path of Joint::fromUrdf / Link::fromUrdf / Chain::init, reference
// primitives_impl.h:50-83, 288-319, 399-417, 580-742) + argument checking + launches.  No CPU fallback.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "launch.h"

namespace rdb
{
std::atomic<uint64_t> g_launches{0};
static thread_local std::string t_err;

static rdb_status fail(rdb_status s, const std::string& what)
{
  t_err = what;
  return s;
}
rdb_status set_error(rdb_status s, const std::string& what) { return fail(s, what); }  // for urdf.cpp
static rdb_status cuda_fail(cudaError_t e, const char* where)
{
  return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? RDB_ERR_NO_DEVICE : RDB_ERR_CUDA,
              std::string(where) + ": " + cudaGetErrorString(e));
}
#define RDB_CUDA(call)                                   \
  do                                                     \
  {                                                      \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

// entry-point prologue: the handle's device becomes current (restored on return); RDB_LOCK serialises the entries that touch the handle's
// mutable state (model, workspaces, staging pipelines)
#define RDB_ENTER(chain)                                                          \
  DeviceScope dev__((chain)->device);                                             \
  if (dev__.err != cudaSuccess) return cuda_fail(dev__.err, "cudaSetDevice(device of the handle)")
#define RDB_LOCK(chain) std::lock_guard<std::recursive_mutex> lock__((chain)->mu)

static void mat3_mul(const double* a, const double* b, double* c)
{
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++)
    {
      double s = 0;
      for (int k = 0; k < 3; k++) s += a[3 * i + k] * b[3 * k + j];
      c[3 * i + j] = s;
    }
}
static void skew(const double* v, double* m)
{
  m[0] = 0; m[1] = -v[2]; m[2] = v[1];
  m[3] = v[2]; m[4] = 0; m[5] = -v[0];
  m[6] = -v[1]; m[7] = v[0]; m[8] = 0;
}

// Joint::fromUrdf (primitives_impl.h:54-83) + Link::fromUrdf (288-319) + getNominalParameters (399-417)
static rdb_status build_model(const rdb_chain_desc* d, ChainHost* ch)
{
  ChainDev<RDB_MAX_JOINTS>& H = ch->host;
  std::memset(&H, 0, sizeof(H));
  H.nj = d->n_joints;
  H.n_in = d->n_inputs;
  for (int k = 0; k < 3; k++) H.g[k] = d->gravity[k];
  for (int j = 0; j < d->n_joints; j++)
  {
    const rdb_joint_desc& s = d->joints[j];
    JointDev& o = H.joint[j];
    if (s.type != RDB_JOINT_FIXED && s.type != RDB_JOINT_REVOLUTE && s.type != RDB_JOINT_PRISMATIC)
      return fail(RDB_ERR_INVALID_ARG, "joint type must be RDB_JOINT_FIXED/REVOLUTE/PRISMATIC");
    if (s.input_index < -1 || s.input_index >= d->n_inputs) return fail(RDB_ERR_INVALID_ARG, "joint input_index out of range");
    o.type = s.type;
    o.in = s.input_index;
    const double n = std::sqrt(s.axis[0] * s.axis[0] + s.axis[1] * s.axis[1] + s.axis[2] * s.axis[2]);
    for (int k = 0; k < 3; k++) o.ax[k] = n > 0 ? s.axis[k] / n : s.axis[k];
    double K[9], K2[9];
    skew(o.ax, K);
    mat3_mul(K, K, K2);
    std::memcpy(o.A, s.rot, sizeof(o.A));
    mat3_mul(s.rot, K, o.B);
    mat3_mul(s.rot, K2, o.C);
    for (int r = 0; r < 3; r++)
    {
      o.t[r] = s.xyz[r];
      o.axp[r] = s.rot[3 * r] * o.ax[0] + s.rot[3 * r + 1] * o.ax[1] + s.rot[3 * r + 2] * o.ax[2];
    }
  }
  for (int l = 0; l < d->n_joints; l++)
  {
    const rdb_link_desc& s = d->links[l + 1];
    double I[9] = {s.inertia[0], s.inertia[1], s.inertia[2], s.inertia[1], s.inertia[3], s.inertia[4], s.inertia[2], s.inertia[4], s.inertia[5]};
    double Rt[9], t[9], Ir[9], cs[9], cst[9], cc[9];
    for (int i = 0; i < 3; i++)
      for (int k = 0; k < 3; k++) Rt[3 * i + k] = s.inertial_rot[3 * k + i];
    mat3_mul(s.inertial_rot, I, t);
    mat3_mul(t, Rt, Ir);
    skew(s.cog, cs);
    for (int i = 0; i < 3; i++)
      for (int k = 0; k < 3; k++) cst[3 * i + k] = cs[3 * k + i];
    mat3_mul(cs, cst, cc);
    double I0[9];
    for (int k = 0; k < 9; k++) I0[k] = Ir[k] + s.mass * cc[k];  // spacevect_algebra.h:238
    double* P = H.link[l].pi;
    P[0] = s.mass;
    for (int k = 0; k < 3; k++) P[1 + k] = s.cog[k] * s.mass;
    P[4] = I0[0]; P[5] = I0[1]; P[6] = I0[2];
    P[7] = I0[4]; P[8] = I0[5]; P[9] = I0[8];
    std::memcpy(ch->nominal + 10 * l, P, 10 * sizeof(double));
  }
  std::vector<int> fed(std::max(d->n_inputs, 1), 0);
  for (int j = 0; j < d->n_joints; j++)
    if (H.joint[j].in >= 0)
    {
      if (fed[H.joint[j].in]) return fail(RDB_ERR_INVALID_ARG, "two chain joints share one input index");
      fed[H.joint[j].in] = 1;
    }
  ch->inputs_cover_all = true;
  for (int i = 0; i < d->n_inputs; i++) ch->inputs_cover_all = ch->inputs_cover_all && fed[i];
  return RDB_OK;
}

// the handle's device (fixed at creation) must be current: every caller holds a DeviceScope
static rdb_status upload_model(ChainHost* ch)
{
  if (!ch->dev) RDB_CUDA(cudaMalloc(&ch->dev, sizeof(ch->host)));
  RDB_CUDA(cudaMemcpy(ch->dev, &ch->host, sizeof(ch->host), cudaMemcpyHostToDevice));
  cudaDeviceGetAttribute(&ch->sm_count, cudaDevAttrMultiProcessorCount, ch->device);
  ch->model_version++;
  RDB_CUDA(fold_chain(*ch));
  return RDB_OK;
}

static rdb_status check_samples(const ChainHost* ch, const rdb_samples* in, bool need_q)
{
  if (!ch || !in) return fail(RDB_ERR_INVALID_ARG, "null chain or samples");
  if (in->n < 0 || in->ld < in->n) return fail(RDB_ERR_INVALID_ARG, "samples: need 0 <= n <= ld");
  if (need_q && !in->q && ch->host.n_in > 0 && in->n > 0) return fail(RDB_ERR_DIM_MISMATCH, "q is required");
  return RDB_OK;
}

static SamplesDev to_dev(const rdb_samples* in) { return SamplesDev{in->n, in->ld, in->q, in->dq, in->ddq, in->dddq}; }

static unsigned kin_mask(const rdb_kinematics_out* o)
{
  unsigned m = 0;
  if (o->T_tool) m |= K_TTOOL;
  if (o->T_links) m |= K_TLINKS;
  if (o->jacobian) m |= K_JAC;
  if (o->twist) m |= K_TWIST;
  if (o->dtwist) m |= K_DTWIST;
  if (o->dtwist_lin) m |= K_DTWIST_LIN;
  if (o->dtwist_nonlin) m |= K_DTWIST_NONLIN;
  if (o->ddtwist) m |= K_DDTWIST;
  if (o->ddtwist_lin) m |= K_DDTWIST_LIN;
  if (o->ddtwist_nonlin) m |= K_DDTWIST_NONLIN;
  if (o->torque) m |= K_TORQUE;
  return m;
}

// rows/columns of inputs that no chain joint feeds stay zero in the reference (S has a zero column there)
static rdb_status prezero(const ChainHost* ch, double* p, int64_t planes, int64_t ld, int64_t n, cudaStream_t st, bool eigen = false)
{
  if (ch->inputs_cover_all || !p || n <= 0 || planes <= 0) return RDB_OK;
  if (eigen) RDB_CUDA(cudaMemsetAsync(p, 0, sizeof(double) * (size_t)n * planes, st));  // dense per-sample records
  else RDB_CUDA(cudaMemset2DAsync(p, ld * sizeof(double), 0, n * sizeof(double), planes, st));
  return RDB_OK;
}
static bool bad_layout(int32_t l) { return l != RDB_LAYOUT_SOA && l != RDB_LAYOUT_EIGEN; }

}  // namespace rdb

using namespace rdb;

struct rdb_chain : public rdb::ChainHost
{
};

extern "C" {

int32_t rdb_abi_version(void) { return RDB_ABI_VERSION; }
const char* rdb_last_error(void) { return t_err.c_str(); }
const char* rdb_status_string(rdb_status s)
{
  switch (s)
  {
    case RDB_OK: return "ok";
    case RDB_ERR_INVALID_ARG: return "invalid argument";
    case RDB_ERR_DIM_MISMATCH: return "Input data dimensions mismatch";
    case RDB_ERR_CUDA: return "CUDA error";
    case RDB_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    case RDB_ERR_NOT_FOUND: return "not found";
    case RDB_ERR_ALLOC: return "allocation failed";
  }
  return "unknown status";
}
int32_t rdb_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess)
  {
    cudaGetLastError();
    return 0;
  }
  return n;
}
uint64_t rdb_kernel_launch_count(void) { return g_launches.load(); }

rdb_status rdb_chain_create(const rdb_chain_desc* desc, rdb_chain** out)
{
  if (!desc || !out) return fail(RDB_ERR_INVALID_ARG, "null descriptor or output");
  *out = nullptr;
  if (desc->n_joints < 0 || desc->n_joints > RDB_MAX_JOINTS) return fail(RDB_ERR_INVALID_ARG, "n_joints out of range");
  if (desc->n_inputs < 0 || desc->n_inputs > RDB_MAX_JOINTS) return fail(RDB_ERR_INVALID_ARG, "n_inputs out of range");
  if (desc->n_joints > 0 && !desc->joints) return fail(RDB_ERR_INVALID_ARG, "null joints");
  if (!desc->links) return fail(RDB_ERR_INVALID_ARG, "null links");
  rdb_chain* ch = new (std::nothrow) rdb_chain();
  if (!ch) return fail(RDB_ERR_ALLOC, "out of host memory");
  rdb_status s = build_model(desc, ch);
  if (s == RDB_OK)
  {
    if (rdb_device_count() <= 0) s = fail(RDB_ERR_NO_DEVICE, "no CUDA device: rosdyn_b200 has no CPU fallback");
    else if (cudaGetDevice(&ch->device) != cudaSuccess) s = fail(RDB_ERR_CUDA, "cudaGetDevice failed");  // the handle lives on the CURRENT device
    else s = upload_model(ch);
  }
  if (s != RDB_OK)
  {
    if (ch->dev) cudaFree(ch->dev);
    delete ch;
    return s;
  }
  *out = ch;
  return RDB_OK;
}

void rdb_chain_destroy(rdb_chain* chain)
{
  if (!chain) return;
  DeviceScope dev__(chain->device);
  if (chain->dev) cudaFree(chain->dev);
  if (chain->gram.partials) cudaFree(chain->gram.partials);
  if (chain->gram.fused_partials) cudaFree(chain->gram.fused_partials);
  if (chain->gram.fold_dev) cudaFree(chain->gram.fold_dev);
  if (chain->gram.ext_dev) cudaFree(chain->gram.ext_dev);
  if (chain->gram.tau_sq_part) cudaFree(chain->gram.tau_sq_part);
  if (chain->host_arena.base) cudaFree(chain->host_arena.base);
  if (chain->host_arena.map_h) cudaFreeHost(chain->host_arena.map_h);
  if (chain->host_arena.pin) cudaFreeHost(chain->host_arena.pin);
  for (int k = 0; k < GramHostPipe::NSLOT; k++)
    if (chain->gram_host.pin[k]) cudaFreeHost(chain->gram_host.pin[k]);
  for (int k = 0; k < 2; k++)
    if (chain->host_arena.st[k]) cudaStreamDestroy(chain->host_arena.st[k]);
  GramHostPipe& hp = chain->gram_host;
  for (int k = 0; k < GramHostPipe::NSLOT; k++)
  {
    if (hp.stage[k]) cudaFree(hp.stage[k]);
    if (hp.copied[k]) cudaEventDestroy(hp.copied[k]);
    if (hp.freed[k]) cudaEventDestroy(hp.freed[k]);
  }
  if (hp.d_out) cudaFree(hp.d_out);
  if (hp.copy) cudaStreamDestroy(hp.copy);
  if (hp.comp) cudaStreamDestroy(hp.comp);
  delete chain;
}

rdb_status rdb_chain_set_input_joints(rdb_chain* chain, int32_t n_inputs, const int32_t* chain_joint_of_input)
{
  if (!chain || n_inputs < 0 || n_inputs > RDB_MAX_JOINTS || (n_inputs > 0 && !chain_joint_of_input))
    return fail(RDB_ERR_INVALID_ARG, "bad input-joint selection");
  RDB_ENTER(chain);
  RDB_LOCK(chain);
  std::vector<int> in(chain->host.nj, -1);
  bool all = true;
  for (int i = 0; i < n_inputs; i++)
  {
    const int j = chain_joint_of_input[i];
    if (j < 0 || j >= chain->host.nj)
    {
      all = false;  // "Joint named '%s' not found" (primitives_impl.h:734): the input keeps a zero column of S
      continue;
    }
    if (in[j] >= 0) return fail(RDB_ERR_INVALID_ARG, "chain joint selected twice");
    in[j] = i;
  }
  for (int j = 0; j < chain->host.nj; j++) chain->host.joint[j].in = in[j];
  chain->host.n_in = n_inputs;
  chain->inputs_cover_all = all;
  // the components were registered against the OLD input vector (their input_index may be out of range now, or name another joint):
  // they are dropped and must be set again after the inputs change (the reference builds its components from the joint-name list, base_component.h:95-108)
  chain->comps = ComponentsDev{};
  return upload_model(chain);
}

int32_t rdb_chain_joints_number(const rdb_chain* chain) { return chain ? chain->host.nj : -1; }
int32_t rdb_chain_links_number(const rdb_chain* chain) { return chain ? chain->host.nj + 1 : -1; }
int32_t rdb_chain_active_joints_number(const rdb_chain* chain) { return chain ? chain->host.n_in : -1; }
rdb_status rdb_chain_gravity(const rdb_chain* chain, double out[3])
{
  if (!chain || !out) return fail(RDB_ERR_INVALID_ARG, "null argument");
  for (int k = 0; k < 3; k++) out[k] = chain->host.g[k];
  return RDB_OK;
}
rdb_status rdb_chain_nominal_parameters(const rdb_chain* chain, double* out)
{
  if (!chain || !out) return fail(RDB_ERR_INVALID_ARG, "null argument");
  std::memcpy(out, chain->nominal, sizeof(double) * 10 * chain->host.nj);
  return RDB_OK;
}

// ------------------------------------------------------------------------------------------- device entries
rdb_status rdb_kinematics_batch(const rdb_chain* chain, const rdb_samples* in, const rdb_kinematics_out* out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (!out || bad_layout(out->layout)) return fail(RDB_ERR_INVALID_ARG, "kinematics_out: null or unknown layout");
  const bool eig = out->layout == RDB_LAYOUT_EIGEN;
  if (!eig && out->ld < in->n) return fail(RDB_ERR_INVALID_ARG, "kinematics_out: need ld >= n");
  const unsigned mask = kin_mask(out);
  if (!mask || in->n == 0) return RDB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int n_in = chain->host.n_in;
  if ((s = prezero(chain, out->jacobian, 6 * n_in, out->ld, in->n, st, eig)) != RDB_OK) return s;
  if ((s = prezero(chain, out->torque, n_in, out->ld, in->n, st, eig)) != RDB_OK) return s;
  KinOutDev o{out->ld,         out->T_tool,        out->T_links, out->jacobian,    out->twist,          out->dtwist,
              out->dtwist_lin, out->dtwist_nonlin, out->ddtwist, out->ddtwist_lin, out->ddtwist_nonlin, out->torque, eig ? 1 : 0};
  RDB_CUDA(launch_kin(*chain, mask, to_dev(in), o, st));
  return RDB_OK;
}

rdb_status rdb_torque_batch(const rdb_chain* chain, const rdb_samples* in, double* torque, int64_t ld_out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (in->n == 0) return RDB_OK;
  if (!torque || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "torque: null or ld_out < n");
  cudaStream_t st = (cudaStream_t)stream;
  if ((s = prezero(chain, torque, chain->host.n_in, ld_out, in->n, st)) != RDB_OK) return s;
  RDB_CUDA(launch_dyn(*chain, DYN_TORQUE_, to_dev(in), nullptr, torque, nullptr, ld_out, st));
  return RDB_OK;
}

rdb_status rdb_regressor_batch(const rdb_chain* chain, const rdb_samples* in, double* phi, double* torque, int64_t ld_out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  // Chain::getRegressor throws std::invalid_argument("Input data dimensions mismatch") (primitives_impl.h:1299-1309)
  if (in->n > 0 && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  if (in->n == 0) return RDB_OK;
  if (!phi || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "phi: null or ld_out < n");
  cudaStream_t st = (cudaStream_t)stream;
  const int n_in = chain->host.n_in;
  if ((s = prezero(chain, phi, (int64_t)10 * chain->host.nj * n_in, ld_out, in->n, st)) != RDB_OK) return s;
  if ((s = prezero(chain, torque, n_in, ld_out, in->n, st)) != RDB_OK) return s;
  RDB_CUDA(launch_dyn(*chain, torque ? (DYN_REGRESSOR_ | DYN_TORQUE_) : DYN_REGRESSOR_, to_dev(in), phi, torque, nullptr, ld_out, st));
  return RDB_OK;
}

rdb_status rdb_inertia_batch(const rdb_chain* chain, const rdb_samples* in, double* inertia, int64_t ld_out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (in->n == 0) return RDB_OK;
  if (!inertia || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "inertia: null or ld_out < n");
  cudaStream_t st = (cudaStream_t)stream;
  const int n_in = chain->host.n_in;
  if ((s = prezero(chain, inertia, (int64_t)n_in * n_in, ld_out, in->n, st)) != RDB_OK) return s;
  RDB_CUDA(launch_dyn(*chain, DYN_INERTIA_, to_dev(in), nullptr, nullptr, inertia, ld_out, st));
  return RDB_OK;
}

rdb_status rdb_forward_dynamics_batch(const rdb_chain* chain, const rdb_samples* in, const double* tau, double* ddq, int64_t ld_out,
                                      int32_t* info, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (in->n == 0) return RDB_OK;
  if (!ddq || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "ddq: null or ld_out < n");
  cudaStream_t st = (cudaStream_t)stream;
  if ((s = prezero(chain, ddq, chain->host.n_in, ld_out, in->n, st)) != RDB_OK) return s;
  SamplesDev sd = to_dev(in);
  sd.ddq = sd.dddq = nullptr;  // the walk runs with DDq = 0
  DynOutDev o = dyn_out_soa(nullptr, ddq, nullptr, ld_out);
  o.tau_in = tau;
  o.info = info;
  RDB_CUDA(launch_dyn(*chain, DYN_FD_, sd, o, st));
  return RDB_OK;
}

rdb_status rdb_dynamics_batch(const rdb_chain* chain, const rdb_samples* in, const rdb_dynamics_out* out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (!out || bad_layout(out->layout)) return fail(RDB_ERR_INVALID_ARG, "dynamics_out: null or unknown layout");
  const bool eig = out->layout == RDB_LAYOUT_EIGEN;
  if (!eig && out->ld < in->n) return fail(RDB_ERR_INVALID_ARG, "dynamics_out: need ld >= n");
  // Chain::getRegressor throws std::invalid_argument("Input data dimensions mismatch") (primitives_impl.h:1299-1309)
  if (out->regressor && in->n > 0 && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  if (in->n == 0 || (!out->regressor && !out->torque && !out->inertia)) return RDB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_in = chain->host.n_in, P = (int64_t)10 * chain->host.nj;
  if ((s = prezero(chain, out->regressor, P * n_in, out->ld, in->n, st, eig)) != RDB_OK) return s;
  if ((s = prezero(chain, out->torque, n_in, out->ld, in->n, st, eig)) != RDB_OK) return s;
  if ((s = prezero(chain, out->inertia, n_in * n_in, out->ld, in->n, st, eig)) != RDB_OK) return s;
  DynOutDev o{out->regressor, out->torque, out->inertia, eig ? 1 : out->ld, eig ? P * n_in : 1, eig ? n_in : 1, eig ? n_in * n_in : 1};
  if (out->regressor) RDB_CUDA(launch_dyn(*chain, out->torque ? (DYN_REGRESSOR_ | DYN_TORQUE_) : DYN_REGRESSOR_, to_dev(in), o, st));
  else if (out->torque) RDB_CUDA(launch_dyn(*chain, DYN_TORQUE_, to_dev(in), o, st));
  if (out->inertia) RDB_CUDA(launch_dyn(*chain, DYN_INERTIA_, to_dev(in), o, st));
  return RDB_OK;
}

rdb_status rdb_regressor_gram_batch(rdb_chain* chain, const rdb_samples* in, const double* tau_meas, double* gram, double* rhs,
                                    double* tau_sq, int32_t accumulate, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  RDB_LOCK(chain);  // the per-CTA partials live in the handle
  if (in->n > 0 && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  if (!gram || !rhs) return fail(RDB_ERR_INVALID_ARG, "gram / rhs must not be null");
  RDB_CUDA(launch_gram(*chain, to_dev(in), tau_meas, gram, rhs, tau_sq, accumulate, (cudaStream_t)stream));
  return RDB_OK;
}

rdb_status rdb_wrench_batch(const rdb_chain* chain, const rdb_samples* in, const double* ext_wrenches, int64_t ld_ext, double* torque,
                            double* wrenches, int64_t ld_out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (in->n == 0 || (!torque && !wrenches)) return RDB_OK;
  if (ld_out < in->n || (ext_wrenches && ld_ext < in->n)) return fail(RDB_ERR_INVALID_ARG, "wrench_batch: ld < n");
  cudaStream_t st = (cudaStream_t)stream;
  if ((s = prezero(chain, torque, chain->host.n_in, ld_out, in->n, st)) != RDB_OK) return s;
  RDB_CUDA(launch_aux(*chain, to_dev(in), ext_wrenches, ld_ext, torque, wrenches, nullptr, 0, ld_out, st));
  return RDB_OK;
}

rdb_status rdb_jacobian_link_batch(const rdb_chain* chain, const rdb_samples* in, int32_t link_index, double* jacobian, int64_t ld_out,
                                   void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (link_index < 0 || link_index > chain->host.nj) return fail(RDB_ERR_NOT_FOUND, "link is not member of the chain");
  if (in->n == 0) return RDB_OK;
  if (!jacobian || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "jacobian: null or ld_out < n");
  cudaStream_t st = (cudaStream_t)stream;
  if ((s = prezero(chain, jacobian, 6 * chain->host.n_in, ld_out, in->n, st)) != RDB_OK) return s;
  RDB_CUDA(launch_aux(*chain, to_dev(in), nullptr, 0, nullptr, nullptr, jacobian, link_index, ld_out, st));
  return RDB_OK;
}

rdb_status rdb_local_ik_batch(const rdb_chain* chain, int64_t n, int64_t ld, const double* target, const double* seed, const double* q_min,
                              const double* q_max, const double* weight, double toll, int32_t max_iter, double* sol, int32_t* status,
                              int32_t* iterations, double* error_norm, void* stream)
{
  if (!chain) return fail(RDB_ERR_INVALID_ARG, "null chain");
  if (n < 0 || ld < n) return fail(RDB_ERR_INVALID_ARG, "need 0 <= n <= ld");
  if (chain->host.n_in > RDB_IK_MAX_INPUTS) return fail(RDB_ERR_INVALID_ARG, "local IK supports at most RDB_IK_MAX_INPUTS input joints");
  if (n == 0) return RDB_OK;
  if (!target || !sol || (!seed && chain->host.n_in > 0)) return fail(RDB_ERR_INVALID_ARG, "target, seed and sol are required");
  if (max_iter < 0 || !(toll >= 0.0)) return fail(RDB_ERR_INVALID_ARG, "max_iter and toll must be non-negative");
  RDB_ENTER(chain);
  RDB_CUDA(launch_ik(*chain, n, ld, target, seed, q_min, q_max, weight, toll, max_iter, sol, status, iterations, error_norm,
                     (cudaStream_t)stream));
  return RDB_OK;
}

// ------------------------------------------------------------------------------------------- components (N2)
int32_t rdb_component_columns(int32_t type)
{
  switch (type)
  {
    case RDB_COMPONENT_FRICTION_POLY1: return 2;
    case RDB_COMPONENT_FRICTION_POLY2: return 3;
    case RDB_COMPONENT_IDEAL_SPRING: return 2;
  }
  return -1;
}

rdb_status rdb_chain_set_components(rdb_chain* chain, int32_t n, const rdb_component_desc* components)
{
  if (!chain || n < 0 || n > RDB_MAX_COMPONENTS || (n > 0 && !components)) return fail(RDB_ERR_INVALID_ARG, "bad component list");
  RDB_LOCK(chain);
  ComponentsDev C{};
  for (int k = 0; k < n; k++)
  {
    const rdb_component_desc& d = components[k];
    const int nc = rdb_component_columns(d.type);
    if (nc < 0) return fail(RDB_ERR_INVALID_ARG, "unknown component type");
    // "Component Joint name ... is not a elemente of joint_names" (base_component.h:103-104)
    if (d.input_index < 0 || d.input_index >= chain->host.n_in) return fail(RDB_ERR_NOT_FOUND, "component joint is not an input joint");
    ComponentDev& c = C.c[k];
    c.type = d.type;
    c.in = d.input_index;
    c.col = C.cols;
    c.ncols = nc;
    c.thr = d.min_velocity;
    c.vmax = d.max_velocity;
    if (d.type != RDB_COMPONENT_IDEAL_SPRING)
    {
      if (c.thr < 1e-6) c.thr = 1.0e-6;                                             // friction_polynomial1.h:75-80, friction_polynomial2.h:84-89
      if (d.type == RDB_COMPONENT_FRICTION_POLY1 && c.vmax <= 0) c.vmax = 1.0e6;    // friction_polynomial1.h:82-87
      if (d.type == RDB_COMPONENT_FRICTION_POLY2 && c.vmax < 0) c.thr = 1.0e6;      // friction_polynomial2.h:91-96 (sic: the threshold)
    }
    C.cols += nc;
  }
  C.n = n;
  chain->comps = C;
  return RDB_OK;
}

int32_t rdb_chain_component_columns(const rdb_chain* chain) { return chain ? chain->comps.cols : -1; }

rdb_status rdb_components_regressor_batch(const rdb_chain* chain, const rdb_samples* in, double* phi_c, int64_t ld_out, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (in->n == 0 || chain->comps.cols == 0) return RDB_OK;
  if (!phi_c || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "phi_c: null or ld_out < n");
  RDB_CUDA(launch_components_regressor(*chain, to_dev(in), phi_c, ld_out, (cudaStream_t)stream));
  return RDB_OK;
}

rdb_status rdb_components_torque_batch(const rdb_chain* chain, const rdb_samples* in, const double* parameters, double* torque, int64_t ld_out,
                                       int32_t accumulate, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  if (in->n == 0) return RDB_OK;
  if (!torque || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "torque: null or ld_out < n");
  if (chain->comps.cols > 0 && !parameters) return fail(RDB_ERR_INVALID_ARG, "parameters is null");
  ComponentParams prm{};
  for (int k = 0; k < chain->comps.cols; k++) prm.p[k] = parameters[k];
  RDB_CUDA(launch_components_torque(*chain, to_dev(in), prm, torque, ld_out, accumulate, (cudaStream_t)stream));
  return RDB_OK;
}

rdb_status rdb_regressor_gram_ext_batch(rdb_chain* chain, const rdb_samples* in, const double* tau_meas, double* gram, double* rhs,
                                        double* tau_sq, int32_t accumulate, void* stream)
{
  rdb_status s = check_samples(chain, in, true);
  if (s != RDB_OK) return s;
  RDB_ENTER(chain);
  RDB_LOCK(chain);
  if (in->n > 0 && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  if (!gram || !rhs) return fail(RDB_ERR_INVALID_ARG, "gram / rhs must not be null");
  RDB_CUDA(launch_gram(*chain, to_dev(in), tau_meas, gram, rhs, tau_sq, accumulate, (cudaStream_t)stream, true));
  return RDB_OK;
}

rdb_status rdb_fill_uniform(double* x, int32_t n_planes, int64_t n, int64_t ld, uint64_t seed, int32_t stream_id, void* stream)
{
  if (!x || n_planes < 0 || n_planes > 64 || n < 0 || ld < n || stream_id < 0 || stream_id > 3)
    return fail(RDB_ERR_INVALID_ARG, "fill_uniform: bad argument");
  if (rdb_device_count() <= 0) return fail(RDB_ERR_NO_DEVICE, "no CUDA device");
  RDB_CUDA(launch_fill_uniform(x, n_planes, n, ld, seed, stream_id, (cudaStream_t)stream));
  return RDB_OK;
}
void rdb_fill_uniform_host(double* x, int32_t n_planes, int64_t n, int64_t ld, uint64_t seed, int32_t stream_id)
{
  fill_uniform_host(x, n_planes, n, ld, seed, stream_id);
}

rdb_status rdb_fp64_peak(int32_t kind, int32_t reps, double* tflops)
{
  if (!tflops || kind < 0 || kind > 2) return fail(RDB_ERR_INVALID_ARG, "fp64_peak: bad argument");
  if (rdb_device_count() <= 0) return fail(RDB_ERR_NO_DEVICE, "no CUDA device");
  RDB_CUDA(fp64_peak(kind, reps, tflops));
  return RDB_OK;
}

rdb_status rdb_chain_create_on(const rdb_chain_desc* desc, int32_t device, rdb_chain** out)
{
  int cur = 0;
  if (rdb_device_count() <= 0) return fail(RDB_ERR_NO_DEVICE, "no CUDA device: rosdyn_b200 has no CPU fallback");
  RDB_CUDA(cudaGetDevice(&cur));
  RDB_CUDA(cudaSetDevice(device));
  const rdb_status s = rdb_chain_create(desc, out);
  cudaSetDevice(cur);
  return s;
}

int32_t rdb_chain_device(const rdb_chain* chain) { return chain ? chain->device : -1; }

rdb_status rdb_gram_specialised_cubin(const rdb_chain_desc* desc, const char* kernel_args, const char* arch, const char* path, char* reason,
                                      int32_t reason_len)
{
  if (!desc || !kernel_args || !arch || !path) return fail(RDB_ERR_INVALID_ARG, "null argument");
  if (desc->n_joints < 0 || desc->n_joints > RDB_MAX_JOINTS) return fail(RDB_ERR_INVALID_ARG, "n_joints out of range");
  if (desc->n_inputs < 0 || desc->n_inputs > RDB_MAX_JOINTS) return fail(RDB_ERR_INVALID_ARG, "n_inputs out of range");
  if (desc->n_joints > 0 && !desc->joints) return fail(RDB_ERR_INVALID_ARG, "null joints");
  if (!desc->links) return fail(RDB_ERR_INVALID_ARG, "null links");
  std::unique_ptr<ChainHost> ch(new (std::nothrow) ChainHost());
  if (!ch) return fail(RDB_ERR_ALLOC, "out of host memory");
  rdb_status s = build_model(desc, ch.get());
  if (s != RDB_OK) return s;
  if (fold_chain(*ch, false) != cudaSuccess) return fail(RDB_ERR_INVALID_ARG, "fold_chain failed");
  if (!fold_rev_canonical(ch->gram.fold)) return fail(RDB_ERR_INVALID_ARG, "the folded chain is not all-revolute about e_z: no specialised kernel");
  std::vector<char> cubin;
  std::string why;
  const bool ok = gram_jit_cubin(ch->gram.fold, kernel_args, arch, cubin, why);
  if (reason && reason_len > 0) snprintf(reason, (size_t)reason_len, "%s", why.c_str());
  if (!ok) return fail(RDB_ERR_CUDA, "NVRTC: " + why);
  FILE* f = fopen(path, "wb");
  if (!f) return fail(RDB_ERR_INVALID_ARG, std::string("cannot write ") + path);
  const bool wrote = fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size();
  if (fclose(f) != 0 || !wrote) return fail(RDB_ERR_INVALID_ARG, std::string("writing ") + path + " failed");
  return RDB_OK;
}

rdb_status rdb_chain_gram_kernel_info(const rdb_chain* chain, int32_t* specialised, char* reason, int32_t reason_len)
{
  if (!chain) return fail(RDB_ERR_INVALID_ARG, "null chain");
  rdb_chain* ch = const_cast<rdb_chain*>(chain);
  RDB_LOCK(ch);
  if (specialised) *specialised = ch->gram.kernel_specialised;
  if (reason && reason_len > 0) snprintf(reason, (size_t)reason_len, "%s", ch->gram.kernel_why.c_str());
  return RDB_OK;
}

rdb_status rdb_regressor_gram_sharded_host(rdb_chain* const* chains, int32_t n_chains, const rdb_samples* in, const double* tau_meas,
                                           double* gram, double* rhs, double* tau_sq, int32_t accumulate)
{
  if (!chains || n_chains <= 0 || !in) return fail(RDB_ERR_INVALID_ARG, "null chains or samples");
  for (int r = 0; r < n_chains; r++)
    if (!chains[r] || chains[r]->host.nj != chains[0]->host.nj || chains[r]->host.n_in != chains[0]->host.n_in)
      return fail(RDB_ERR_INVALID_ARG, "the handles must describe the same chain");
  {
    const rdb_status cs = check_samples(chains[0], in, true);
    if (cs != RDB_OK) return cs;
  }
  if (!gram || !rhs) return fail(RDB_ERR_INVALID_ARG, "gram / rhs must not be null");
  const int R = n_chains, P = 10 * chains[0]->host.nj;
  const size_t n_out = (size_t)P * P + P + 1;
  std::vector<double> part((size_t)R * n_out, 0.0);
  std::vector<rdb_status> st((size_t)R, RDB_OK);
  std::vector<std::string> msg((size_t)R);
  std::vector<std::thread> th;
  for (int r = 0; r < R; r++)
    th.emplace_back([&, r] {
      cudaSetDevice(chains[r]->device);
      const int64_t lo = (int64_t)r * in->n / R, hi = (int64_t)(r + 1) * in->n / R;
      rdb_samples v{hi - lo, in->ld, in->q ? in->q + lo : nullptr, in->dq ? in->dq + lo : nullptr, in->ddq ? in->ddq + lo : nullptr, nullptr};
      double* o = part.data() + (size_t)r * n_out;
      st[r] = rdb_regressor_gram_batch_host(chains[r], &v, tau_meas ? tau_meas + lo : nullptr, o, o + (size_t)P * P, o + (size_t)P * P + P, 0);
      if (st[r] != RDB_OK) msg[r] = rdb_last_error();  // thread-local text of this worker
    });
  for (auto& t : th) t.join();
  for (int r = 0; r < R; r++)
    if (st[r] != RDB_OK) return fail(st[r], "shard " + std::to_string(r) + ": " + msg[r]);
  for (size_t e = 0; e < n_out; e++)
  {
    double* dst = e < (size_t)P * P ? gram + e : (e < (size_t)P * P + P ? rhs + (e - (size_t)P * P) : tau_sq);
    if (!dst) continue;
    double s = accumulate ? *dst : 0.0;
    for (int r = 0; r < R; r++) s += part[(size_t)r * n_out + e];  // rank order: reproducible for a given R
    *dst = s;
  }
  return RDB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------- host wrappers
// Chunked, double-buffered: H2D of chunk k+1 and D2H of chunk k-1 overlap the kernel of chunk k when the
// caller's buffers are pinned (cudaMemcpy2DAsync gathers each plane's slice).
namespace rdb
{
struct Plane
{
  const double* h_in = nullptr;  // host source (inputs)
  double* h_out = nullptr;       // host destination (outputs)
  int64_t planes = 0;
  int64_t ld = 0;  // host plane stride
  bool records = false;  // RDB_LAYOUT_EIGEN output: [sample][planes] dense records on both sides (one contiguous copy per chunk)
  int64_t es = sizeof(double);  // bytes per element of an output plane (int32 status planes: 4; the device side keeps a double-sized slot)
  double* d[2] = {nullptr, nullptr};
  double* hm = nullptr;  // mapped mode: host alias of d[0]
  double* hp[2] = {nullptr, nullptr};  // bounce mode: pinned mirror of d[slot]
  void* out_at(int64_t r, int64_t off) const { return reinterpret_cast<char*>(h_out) + (r * ld + off) * es; }  // caller's element (plane r, sample off)
};

// host threads of the gather / scatter loops: the hardware threads shared out over the visible GPUs (one rank or one handle per GPU is the
// usual deployment), 2 .. 16; measured on a 16-thread B200 host, pageable fused Gram: 2 / 4 / 8 / 12 / 16 threads -> 110 / 183 / 225 / 266 /
// 295 M samples/s.  RDB_HOST_THREADS (1 .. 64) is a tuning knob only -- it never changes results.
static int host_threads()
{
  static const int n = [] {
    const char* e = getenv("RDB_HOST_THREADS");
    if (e) return (int)std::min<long>(std::max<long>(atol(e), 1), 64);
    int ndev = 1;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
    {
      cudaGetLastError();
      ndev = 1;
    }
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    return (int)std::min(16u, std::max(2u, hw / (unsigned)ndev));
  }();
  return n;
}
// n_tasks independent pieces of host work on a few threads (gather / scatter of plane slices between caller memory and pinned buffers)
template <class F>
static void host_parallel(int64_t n_tasks, F&& task)
{
  const int n_workers = (int)std::min<int64_t>(n_tasks, host_threads());
  std::atomic<int64_t> next{0};
  auto work = [&] {
    for (int64_t t = next.fetch_add(1); t < n_tasks; t = next.fetch_add(1)) task(t);
  };
  std::vector<std::thread> pool;
  for (int w = 1; w < n_workers; w++) pool.emplace_back(work);
  work();
  for (std::thread& th : pool) th.join();
}
static bool is_pageable(const void* p)
{
  if (!p) return false;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess)
  {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

struct HostPipe
{
  cudaStream_t st[2] = {nullptr, nullptr};
  std::vector<Plane*> all;
  int64_t chunk = 0;
  bool mapped = false;  // the whole call fits the handle's mapped pinned buffer: no copy calls, the kernels work on host memory
  struct Pending
  {
    Plane* p;
    int64_t off, len;
  };
  std::vector<Pending> pending;  // mapped mode: outputs to hand to the caller after the synchronisation
  bool bounce = false;           // pageable caller memory: every transfer goes through the pinned mirror of the arena
  std::vector<Pending> waiting[2];  // bounce mode: outputs of the last chunk of a slot, still to be scattered to the caller
  // device buffers and streams come from the handle's arena (grown on demand, freed with the handle); one host call at a time per handle
  rdb_status init(HostArena& ar, int64_t n, int64_t chunk_max, std::vector<Plane*> planes)
  {
    all = planes;
    chunk = std::min<int64_t>(std::max<int64_t>(n, 1), chunk_max);
    if (!ar.pin_failed && n >= (1 << 12))
      for (Plane* p : all)
        if (p->planes > 0 && (is_pageable(p->h_in) || is_pageable(p->h_out)))
        {
          bounce = true;
          break;
        }
    if (bounce)
    {
      // at most 64 MB of pinned memory per slot
      int64_t total = 0;
      for (Plane* p : all)
        if ((p->h_in || p->h_out) && p->planes > 0) total += p->planes;
      const int64_t cap = std::max<int64_t>(1024, ((int64_t)(64 << 20) / (8 * std::max<int64_t>(total, 1))) & ~(int64_t)1023);
      chunk = std::min(chunk, cap);
    }
    const int slots = n > chunk ? 2 : 1;
    for (int k = 0; k < 2; k++)
    {
      if (!ar.st[k]) RDB_CUDA(cudaStreamCreateWithFlags(&ar.st[k], cudaStreamNonBlocking));
      st[k] = ar.st[k];
    }
    size_t need = 0;
    for (Plane* p : all)
      if ((p->h_in || p->h_out) && p->planes > 0) need += sizeof(double) * (size_t)p->planes * chunk * slots;
    if (slots == 1 && need <= RDB_HOST_MAPPED_BYTES)
    {
      if (!ar.map_h && !ar.map_failed)
      {
        // no mapped pinned memory on this host (locked-memory limit, ...): remembered, the copy path below serves small calls as well
        if (cudaHostAlloc(&ar.map_h, RDB_HOST_MAPPED_BYTES, cudaHostAllocMapped) != cudaSuccess ||
            cudaHostGetDevicePointer(&ar.map_d, ar.map_h, 0) != cudaSuccess)
        {
          cudaGetLastError();
          if (ar.map_h) cudaFreeHost(ar.map_h);
          ar.map_h = ar.map_d = nullptr;
          ar.map_failed = true;
        }
      }
      if (ar.map_h)
      {
        mapped = true;
        size_t o = 0;
        for (Plane* p : all)
          if ((p->h_in || p->h_out) && p->planes > 0)
          {
            p->d[0] = ar.map_d + o;
            p->hm = ar.map_h + o;
            o += (size_t)p->planes * chunk;
          }
        return RDB_OK;
      }
    }
    if (ar.bytes < need)
    {
      if (ar.base) cudaFree(ar.base);
      ar.base = nullptr;
      ar.bytes = 0;
      RDB_CUDA(cudaMalloc(&ar.base, need));
      ar.bytes = need;
    }
    if (bounce && ar.pin_bytes < need)
    {
      if (ar.pin) cudaFreeHost(ar.pin);
      ar.pin = nullptr;
      ar.pin_bytes = 0;
      if (cudaHostAlloc(&ar.pin, need, cudaHostAllocDefault) == cudaSuccess) ar.pin_bytes = need;
      else
      {
        cudaGetLastError();
        ar.pin = nullptr;
        ar.pin_failed = true;  // no pinned memory to spare: the driver's staging serves
        bounce = false;
      }
    }
    double* cur = ar.base;
    double* hcur = ar.pin;
    for (Plane* p : all)
      if ((p->h_in || p->h_out) && p->planes > 0)
        for (int k = 0; k < slots; k++)
        {
          p->d[k] = cur;
          cur += (size_t)p->planes * chunk;
          if (bounce)
          {
            p->hp[k] = hcur;
            hcur += (size_t)p->planes * chunk;
          }
        }
    return RDB_OK;
  }
  // bounce mode: hand the outputs of the previous chunk of this slot to the caller (its copies into the pinned mirror are awaited here, while
  // the other slot's chunk keeps the device busy)
  rdb_status begin(int slot)
  {
    if (!bounce) return RDB_OK;
    RDB_CUDA(cudaStreamSynchronize(st[slot]));  // also covers the previous copy OUT of this slot's pinned input regions
    scatter(slot);
    return RDB_OK;
  }
  void scatter(int slot)
  {
    for (const Pending& q : waiting[slot])
    {
      const Plane& p = *q.p;
      const double* src = p.hp[slot];
      if (p.records)
      {
        const int64_t total = q.len * p.planes, piece = (total + 15) / 16;
        host_parallel(16, [&](int64_t t) {
          const int64_t a = t * piece, b = std::min(total, a + piece);
          if (a < b) memcpy(p.h_out + q.off * p.planes + a, src + a, sizeof(double) * (size_t)(b - a));
        });
      }
      else
        host_parallel(p.planes, [&](int64_t r) { memcpy(p.out_at(r, q.off), src + r * chunk, p.es * (size_t)q.len); });
    }
    waiting[slot].clear();
  }
  rdb_status h2d(Plane& p, int slot, int64_t off, int64_t len)
  {
    if (!p.h_in || p.planes == 0) return RDB_OK;
    if (mapped)
    {
      for (int64_t r = 0; r < p.planes; r++) memcpy(p.hm + r * chunk, p.h_in + r * p.ld + off, sizeof(double) * (size_t)len);
      return RDB_OK;
    }
    if (bounce)
    {
      // the previous copy out of this pinned region belongs to the chunk begin(slot) has waited for, or to one that ran before its kernel
      double* dst = p.hp[slot];
      host_parallel(p.planes, [&](int64_t r) { memcpy(dst + r * chunk, p.h_in + r * p.ld + off, sizeof(double) * (size_t)len); });
      RDB_CUDA(cudaMemcpy2DAsync(p.d[slot], chunk * sizeof(double), dst, chunk * sizeof(double), len * sizeof(double), p.planes,
                                 cudaMemcpyHostToDevice, st[slot]));
      return RDB_OK;
    }
    RDB_CUDA(cudaMemcpy2DAsync(p.d[slot], chunk * sizeof(double), p.h_in + off, p.ld * sizeof(double), len * sizeof(double), p.planes,
                               cudaMemcpyHostToDevice, st[slot]));
    return RDB_OK;
  }
  rdb_status d2h(Plane& p, int slot, int64_t off, int64_t len)
  {
    if (!p.h_out || p.planes == 0) return RDB_OK;
    if (mapped)
    {
      pending.push_back({&p, off, len});
      return RDB_OK;
    }
    if (bounce)
    {
      if (p.records)
        RDB_CUDA(cudaMemcpyAsync(p.hp[slot], p.d[slot], sizeof(double) * (size_t)len * p.planes, cudaMemcpyDeviceToHost, st[slot]));
      else
        RDB_CUDA(cudaMemcpy2DAsync(p.hp[slot], chunk * sizeof(double), p.d[slot], chunk * sizeof(double), len * p.es, p.planes,
                                   cudaMemcpyDeviceToHost, st[slot]));
      waiting[slot].push_back({&p, off, len});
      return RDB_OK;
    }
    if (p.records)
      RDB_CUDA(cudaMemcpyAsync(p.h_out + off * p.planes, p.d[slot], sizeof(double) * (size_t)len * p.planes, cudaMemcpyDeviceToHost, st[slot]));
    else
      RDB_CUDA(cudaMemcpy2DAsync(p.out_at(0, off), p.ld * p.es, p.d[slot], chunk * sizeof(double), len * p.es, p.planes,
                                 cudaMemcpyDeviceToHost, st[slot]));
    return RDB_OK;
  }
  rdb_status finish()
  {
    for (int k = 0; k < 2; k++)
      if (st[k] && (k == 0 || !mapped)) RDB_CUDA(cudaStreamSynchronize(st[k]));
    if (bounce)
      for (int k = 0; k < 2; k++) scatter(k);
    for (const Pending& q : pending)
    {
      const Plane& p = *q.p;
      if (p.records) memcpy(p.h_out + q.off * p.planes, p.hm, sizeof(double) * (size_t)q.len * p.planes);
      else
        for (int64_t r = 0; r < p.planes; r++) memcpy(p.out_at(r, q.off), p.hm + r * chunk, p.es * (size_t)q.len);
    }
    pending.clear();
    return RDB_OK;
  }
};

struct HostIn
{
  Plane q, dq, ddq, dddq;
  void bind(const rdb_samples* in, int n_in)
  {
    const double* src[4] = {in->q, in->dq, in->ddq, in->dddq};
    Plane* dst[4] = {&q, &dq, &ddq, &dddq};
    for (int k = 0; k < 4; k++)
    {
      dst[k]->h_in = src[k];
      dst[k]->planes = src[k] ? n_in : 0;
      dst[k]->ld = in->ld;
    }
  }
  rdb_samples view(int slot, int64_t len, int64_t chunk) const
  {
    return rdb_samples{len, chunk, q.d[slot], dq.d[slot], ddq.d[slot], dddq.d[slot]};
  }
};
}  // namespace rdb

#define RDB_TRY(x)                    \
  do                                  \
  {                                   \
    rdb_status s__ = (x);             \
    if (s__ != RDB_OK) return s__;    \
  } while (0)

extern "C" {

rdb_status rdb_kinematics_batch_host(rdb_chain* chain, const rdb_samples* in, const rdb_kinematics_out* out)
{
  RDB_TRY(check_samples(chain, in, true));
  RDB_ENTER(chain);
  RDB_LOCK(chain);  // the staging arena and its streams live in the handle
  if (!out || bad_layout(out->layout)) return fail(RDB_ERR_INVALID_ARG, "kinematics_out: null or unknown layout");
  const bool eig = out->layout == RDB_LAYOUT_EIGEN;
  if (!eig && out->ld < in->n) return fail(RDB_ERR_INVALID_ARG, "kinematics_out: need ld >= n");
  const int nL = chain->host.nj + 1, n_in = chain->host.n_in;
  const int64_t pose = eig ? 16 : 12;  // doubles per pose: Affine3d image / 3x4 [R|p]
  HostIn hi;
  hi.bind(in, n_in);
  double* const outs[11] = {out->T_tool,        out->T_links, out->jacobian,    out->twist,          out->dtwist, out->dtwist_lin,
                            out->dtwist_nonlin, out->ddtwist, out->ddtwist_lin, out->ddtwist_nonlin, out->torque};
  const int64_t rows[11] = {pose, pose * nL, 6 * n_in, 6 * nL, 6 * nL, 6 * nL, 6 * nL, 6 * nL, 6 * nL, 6 * nL, n_in};
  Plane po[11];
  std::vector<Plane*> all = {&hi.q, &hi.dq, &hi.ddq, &hi.dddq};
  for (int k = 0; k < 11; k++)
  {
    po[k].h_out = outs[k];
    po[k].planes = outs[k] ? rows[k] : 0;
    po[k].ld = out->ld;
    po[k].records = eig;
    all.push_back(&po[k]);
  }
  HostPipe pipe;
  RDB_TRY(pipe.init(chain->host_arena, in->n, 1 << 20, all));
  int slot = 0;
  for (int64_t off = 0; off < in->n; off += pipe.chunk, slot ^= 1)
  {
    const int64_t len = std::min<int64_t>(pipe.chunk, in->n - off);
    RDB_TRY(pipe.begin(slot));
    RDB_TRY(pipe.h2d(hi.q, slot, off, len));
    RDB_TRY(pipe.h2d(hi.dq, slot, off, len));
    RDB_TRY(pipe.h2d(hi.ddq, slot, off, len));
    RDB_TRY(pipe.h2d(hi.dddq, slot, off, len));
    rdb_samples v = hi.view(slot, len, pipe.chunk);
    rdb_kinematics_out o{pipe.chunk,    po[0].d[slot], po[1].d[slot], po[2].d[slot], po[3].d[slot], po[4].d[slot],
                         po[5].d[slot], po[6].d[slot], po[7].d[slot], po[8].d[slot], po[9].d[slot], po[10].d[slot], out->layout};
    RDB_TRY(rdb_kinematics_batch(chain, &v, &o, pipe.st[slot]));
    for (int k = 0; k < 11; k++) RDB_TRY(pipe.d2h(po[k], slot, off, len));
  }
  return pipe.finish();
}

// what: 0 regressor (+ torque), 1 torque, 2 inertia, 3 rdb_dynamics_batch (any subset)
static rdb_status dyn_host(rdb_chain* chain, const rdb_samples* in, double* phi, double* torque, double* inertia, int64_t ld_out, int what,
                           int32_t layout = RDB_LAYOUT_SOA)
{
  RDB_TRY(check_samples(chain, in, true));
  RDB_ENTER(chain);
  RDB_LOCK(chain);
  const bool eig = layout == RDB_LAYOUT_EIGEN;
  if (!eig && ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "ld_out < n");
  const int n_in = chain->host.n_in;
  HostIn hi;
  hi.bind(in, n_in);
  Plane pphi, ptau, pM;
  pphi.h_out = phi; pphi.planes = phi ? (int64_t)10 * chain->host.nj * n_in : 0; pphi.ld = ld_out;
  ptau.h_out = torque; ptau.planes = torque ? n_in : 0; ptau.ld = ld_out;
  pM.h_out = inertia; pM.planes = inertia ? (int64_t)n_in * n_in : 0; pM.ld = ld_out;
  pphi.records = ptau.records = pM.records = eig;
  HostPipe pipe;
  RDB_TRY(pipe.init(chain->host_arena, in->n, phi ? (1 << 18) : (1 << 21), {&hi.q, &hi.dq, &hi.ddq, &hi.dddq, &pphi, &ptau, &pM}));
  int slot = 0;
  for (int64_t off = 0; off < in->n; off += pipe.chunk, slot ^= 1)
  {
    const int64_t len = std::min<int64_t>(pipe.chunk, in->n - off);
    RDB_TRY(pipe.begin(slot));
    RDB_TRY(pipe.h2d(hi.q, slot, off, len));
    RDB_TRY(pipe.h2d(hi.dq, slot, off, len));
    RDB_TRY(pipe.h2d(hi.ddq, slot, off, len));
    rdb_samples v = hi.view(slot, len, pipe.chunk);
    if (what == 0) RDB_TRY(rdb_regressor_batch(chain, &v, pphi.d[slot], ptau.d[slot], pipe.chunk, pipe.st[slot]));
    if (what == 1) RDB_TRY(rdb_torque_batch(chain, &v, ptau.d[slot], pipe.chunk, pipe.st[slot]));
    if (what == 2) RDB_TRY(rdb_inertia_batch(chain, &v, pM.d[slot], pipe.chunk, pipe.st[slot]));
    if (what == 3)
    {
      rdb_dynamics_out o{pipe.chunk, pphi.d[slot], ptau.d[slot], pM.d[slot], layout};
      RDB_TRY(rdb_dynamics_batch(chain, &v, &o, pipe.st[slot]));
    }
    RDB_TRY(pipe.d2h(pphi, slot, off, len));
    RDB_TRY(pipe.d2h(ptau, slot, off, len));
    RDB_TRY(pipe.d2h(pM, slot, off, len));
  }
  return pipe.finish();
}

rdb_status rdb_torque_batch_host(rdb_chain* chain, const rdb_samples* in, double* torque, int64_t ld_out)
{
  if (!torque) return fail(RDB_ERR_INVALID_ARG, "torque is null");
  return dyn_host(chain, in, nullptr, torque, nullptr, ld_out, 1);
}
rdb_status rdb_regressor_batch_host(rdb_chain* chain, const rdb_samples* in, double* phi, double* torque, int64_t ld_out)
{
  if (!phi) return fail(RDB_ERR_INVALID_ARG, "phi is null");
  if (in && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  return dyn_host(chain, in, phi, torque, nullptr, ld_out, 0);
}
rdb_status rdb_inertia_batch_host(rdb_chain* chain, const rdb_samples* in, double* inertia, int64_t ld_out)
{
  if (!inertia) return fail(RDB_ERR_INVALID_ARG, "inertia is null");
  return dyn_host(chain, in, nullptr, nullptr, inertia, ld_out, 2);
}

rdb_status rdb_forward_dynamics_batch_host(rdb_chain* chain, const rdb_samples* in, const double* tau, double* ddq, int64_t ld_out,
                                           int32_t* info)
{
  RDB_TRY(check_samples(chain, in, true));
  RDB_ENTER(chain);
  RDB_LOCK(chain);
  if (in->n == 0) return RDB_OK;
  if (!ddq || ld_out < in->n) return fail(RDB_ERR_INVALID_ARG, "ddq: null or ld_out < n");
  const int n_in = chain->host.n_in;
  HostIn hi;
  hi.bind(in, n_in);
  // forward dynamics ignores DDq / DDDq: tau travels in the DDq slot
  hi.ddq.h_in = tau;
  hi.ddq.planes = tau ? n_in : 0;
  hi.dddq.h_in = nullptr;
  hi.dddq.planes = 0;
  Plane pdd, pinfo;
  pdd.h_out = ddq; pdd.planes = n_in; pdd.ld = ld_out;
  pinfo.h_out = reinterpret_cast<double*>(info); pinfo.planes = info ? 1 : 0; pinfo.ld = in->n; pinfo.es = sizeof(int32_t);
  HostPipe pipe;
  RDB_TRY(pipe.init(chain->host_arena, in->n, 1 << 21, {&hi.q, &hi.dq, &hi.ddq, &pdd, &pinfo}));
  int slot = 0;
  for (int64_t off = 0; off < in->n; off += pipe.chunk, slot ^= 1)
  {
    const int64_t len = std::min<int64_t>(pipe.chunk, in->n - off);
    RDB_TRY(pipe.begin(slot));
    RDB_TRY(pipe.h2d(hi.q, slot, off, len));
    RDB_TRY(pipe.h2d(hi.dq, slot, off, len));
    RDB_TRY(pipe.h2d(hi.ddq, slot, off, len));
    const rdb_samples v{len, pipe.chunk, hi.q.d[slot], hi.dq.d[slot], nullptr, nullptr};
    RDB_TRY(rdb_forward_dynamics_batch(chain, &v, hi.ddq.d[slot], pdd.d[slot], pipe.chunk, info ? reinterpret_cast<int32_t*>(pinfo.d[slot]) : nullptr,
                                       pipe.st[slot]));
    RDB_TRY(pipe.d2h(pdd, slot, off, len));
    RDB_TRY(pipe.d2h(pinfo, slot, off, len));
  }
  return pipe.finish();
}

rdb_status rdb_dynamics_batch_host(rdb_chain* chain, const rdb_samples* in, const rdb_dynamics_out* out)
{
  if (!out || bad_layout(out->layout)) return fail(RDB_ERR_INVALID_ARG, "dynamics_out: null or unknown layout");
  if (out->regressor && in && in->n > 0 && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  if (!out->regressor && !out->torque && !out->inertia) return RDB_OK;
  return dyn_host(chain, in, out->regressor, out->torque, out->inertia, out->ld, 3, out->layout);
}

rdb_status rdb_regressor_gram_batch_host(rdb_chain* chain, const rdb_samples* in, const double* tau_meas, double* gram, double* rhs,
                                         double* tau_sq, int32_t accumulate)
{
  // Streaming pipeline kept in the handle (streams, 3 staging slots, events): H2D of chunk k+1/k+2 on the copy
  // stream overlaps the fused kernel of chunk k on the compute stream; only (P^2+P+1) doubles come back.
  // One host call at a time per handle (the handle's workspace is not shared between threads).
  RDB_TRY(check_samples(chain, in, true));
  if (in->n > 0 && (!in->dq || !in->ddq)) return fail(RDB_ERR_DIM_MISMATCH, "Input data dimensions mismatch");
  if (!gram || !rhs) return fail(RDB_ERR_INVALID_ARG, "gram / rhs must not be null");
  RDB_ENTER(chain);
  RDB_LOCK(chain);  // streams, staging slots and events of the pipeline live in the handle
  rdb_chain* ch = chain;
  GramHostPipe& hp = ch->gram_host;
  const int n_in = ch->host.n_in, P = 10 * ch->host.nj;
  // chunk: measured on B200 (C6, 4 M samples per call, pinned inputs): 2^16 354, 2^17 330, 2^18 375, 2^19 372 M samples/s end to end
  // RDB_HOST_CHUNK (samples per staged chunk) is a tuning knob only -- it never changes results; clamped to [2^10, 2^24]
  static const int64_t chunk = [] {
    const char* e = getenv("RDB_HOST_CHUNK");
    const int64_t v = e ? (int64_t)atoll(e) : (int64_t)(1 << 18);
    return std::min<int64_t>(std::max<int64_t>(v, 1 << 10), 1 << 24);
  }();
  const size_t n_out = (size_t)P * P + P + 1;
  if (!hp.copy)
  {
    RDB_CUDA(cudaStreamCreateWithFlags(&hp.copy, cudaStreamNonBlocking));
    RDB_CUDA(cudaStreamCreateWithFlags(&hp.comp, cudaStreamNonBlocking));
    for (int k = 0; k < GramHostPipe::NSLOT; k++)
    {
      RDB_CUDA(cudaEventCreateWithFlags(&hp.copied[k], cudaEventDisableTiming));
      RDB_CUDA(cudaEventCreateWithFlags(&hp.freed[k], cudaEventDisableTiming));
    }
  }
  if (hp.planes != n_in || !hp.stage[0])
  {
    for (int k = 0; k < GramHostPipe::NSLOT; k++)
    {
      if (hp.stage[k]) cudaFree(hp.stage[k]);
      hp.stage[k] = nullptr;
      RDB_CUDA(cudaMalloc(&hp.stage[k], sizeof(double) * 4 * (size_t)std::max(n_in, 1) * chunk));
    }
    if (hp.d_out) cudaFree(hp.d_out);
    hp.d_out = nullptr;
    RDB_CUDA(cudaMalloc(&hp.d_out, sizeof(double) * n_out));
    hp.planes = n_in;
    hp.n_out = n_out;
  }
  else if (hp.n_out < n_out)
  {
    cudaFree(hp.d_out);
    hp.d_out = nullptr;
    RDB_CUDA(cudaMalloc(&hp.d_out, sizeof(double) * n_out));
    hp.n_out = n_out;
  }
  double* dG = hp.d_out;
  double* db = dG + (size_t)P * P;
  double* dt = db + P;
  if (accumulate)
  {
    RDB_CUDA(cudaMemcpyAsync(dG, gram, sizeof(double) * P * P, cudaMemcpyHostToDevice, hp.comp));
    RDB_CUDA(cudaMemcpyAsync(db, rhs, sizeof(double) * P, cudaMemcpyHostToDevice, hp.comp));
    if (tau_sq) RDB_CUDA(cudaMemcpyAsync(dt, tau_sq, sizeof(double), cudaMemcpyHostToDevice, hp.comp));
    else RDB_CUDA(cudaMemsetAsync(dt, 0, sizeof(double), hp.comp));
  }
  else if (in->n == 0)
    RDB_CUDA(cudaMemsetAsync(dG, 0, sizeof(double) * n_out, hp.comp));
  // Pageable inputs: gather each chunk into a pinned bounce buffer with a few host threads (one plane slice per task), then ONE contiguous
  // asynchronous copy -- the driver would otherwise stage every cudaMemcpy2DAsync synchronously through its own buffer on one thread.
  bool bounce = false;
  if (in->n >= (1 << 14) && n_in > 0 && !hp.pin_failed)
  {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, in->q) == cudaSuccess && at.type == cudaMemoryTypeUnregistered) bounce = true;
    else cudaGetLastError();
  }
  const size_t slot_doubles = 4 * (size_t)std::max(n_in, 1) * chunk;
  if (bounce && hp.pin_doubles < slot_doubles)
  {
    for (int s = 0; s < GramHostPipe::NSLOT; s++)
    {
      if (hp.pin[s]) cudaFreeHost(hp.pin[s]);
      hp.pin[s] = nullptr;
    }
    hp.pin_doubles = 0;
    bool ok = true;
    for (int s = 0; s < GramHostPipe::NSLOT && ok; s++) ok = cudaHostAlloc(&hp.pin[s], sizeof(double) * slot_doubles, cudaHostAllocDefault) == cudaSuccess;
    if (ok) hp.pin_doubles = slot_doubles;
    else
    {
      cudaGetLastError();
      for (int s = 0; s < GramHostPipe::NSLOT; s++)
      {
        if (hp.pin[s]) cudaFreeHost(hp.pin[s]);
        hp.pin[s] = nullptr;
      }
      hp.pin_failed = true;  // no pinned memory to spare: the driver's staging serves
      bounce = false;
    }
  }
  const int n_workers = bounce ? rdb::host_threads() : 0;
  int64_t k = 0;
  for (int64_t off = 0; off < in->n; off += chunk, k++)
  {
    const int slot = (int)(k % GramHostPipe::NSLOT);
    const int64_t len = std::min<int64_t>(chunk, in->n - off);
    if (k >= GramHostPipe::NSLOT) RDB_CUDA(cudaStreamWaitEvent(hp.copy, hp.freed[slot], 0));
    double* base = hp.stage[slot];
    const double* src[4] = {in->q, in->dq, in->ddq, tau_meas};
    if (bounce)
    {
      if (k >= GramHostPipe::NSLOT) RDB_CUDA(cudaEventSynchronize(hp.copied[slot]));  // the previous copy out of this bounce buffer is done
      double* pb = hp.pin[slot];
      const int n_arr = tau_meas ? 4 : 3, n_tasks = n_arr * n_in;
      std::atomic<int> next{0};
      auto work = [&] {
        for (int t = next.fetch_add(1); t < n_tasks; t = next.fetch_add(1))
        {
          const int a = t / n_in, r = t % n_in;
          memcpy(pb + ((size_t)a * n_in + r) * chunk, src[a] + (size_t)r * in->ld + off, sizeof(double) * (size_t)len);
        }
      };
      std::vector<std::thread> pool;
      for (int w = 1; w < n_workers; w++) pool.emplace_back(work);
      work();
      for (std::thread& th : pool) th.join();
      RDB_CUDA(cudaMemcpyAsync(base, pb, sizeof(double) * (size_t)n_arr * n_in * chunk, cudaMemcpyHostToDevice, hp.copy));
    }
    else
      for (int a = 0; a < 4; a++)
        if (src[a] && n_in > 0)
          RDB_CUDA(cudaMemcpy2DAsync(base + (size_t)a * n_in * chunk, chunk * sizeof(double), src[a] + off, in->ld * sizeof(double),
                                     len * sizeof(double), n_in, cudaMemcpyHostToDevice, hp.copy));
    RDB_CUDA(cudaEventRecord(hp.copied[slot], hp.copy));
    RDB_CUDA(cudaStreamWaitEvent(hp.comp, hp.copied[slot], 0));
    rdb_samples v{len, chunk, base, base + (size_t)n_in * chunk, base + (size_t)2 * n_in * chunk, nullptr};
    RDB_TRY(rdb_regressor_gram_batch(chain, &v, tau_meas ? base + (size_t)3 * n_in * chunk : nullptr, dG, db, dt, (accumulate || k > 0) ? 1 : 0,
                                     hp.comp));
    RDB_CUDA(cudaEventRecord(hp.freed[slot], hp.comp));
  }
  RDB_CUDA(cudaMemcpyAsync(gram, dG, sizeof(double) * P * P, cudaMemcpyDeviceToHost, hp.comp));
  RDB_CUDA(cudaMemcpyAsync(rhs, db, sizeof(double) * P, cudaMemcpyDeviceToHost, hp.comp));
  if (tau_sq) RDB_CUDA(cudaMemcpyAsync(tau_sq, dt, sizeof(double), cudaMemcpyDeviceToHost, hp.comp));
  RDB_CUDA(cudaStreamSynchronize(hp.comp));
  return RDB_OK;
}

}  // extern "C"
