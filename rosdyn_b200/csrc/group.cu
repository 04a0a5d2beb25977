// group.cu -- the sample-sharded fused Gram over several B200s with ONE NCCL all-reduce of the small normal-equation partials over
// NVLink / NVSwitch, reachable from the C-ABI (SURVEY.md section 8b/8e: rdb_group_create / rdb_regressor_gram_sharded).
//
// Samples are independent, so every device runs gram_fused_kernel on its own shard with no data-path collective; the only exchange is the sum of
// the packed partials [G | b | tau_sq] (P^2 + P + 1 doubles, 39.8 KB for 7 joints).  The fused kernel's epilogue writes straight into the group's
// packed device buffer, ncclAllReduce(ncclDouble, ncclSum) runs in place on the same stream, and one small kernel adds / stores the result into
// the caller's arrays -- no host round trip, no pack copies.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): the library has no link-time dependency on it, a process that already loaded an NCCL
// (e.g. through torch) shares that copy, and everything else in the C-ABI keeps working on a box without NCCL.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "launch.h"

namespace rdb
{
rdb_status set_error(rdb_status s, const std::string& what);  // capi.cu

// the few NCCL declarations used here (stable across NCCL 2.x: nccl.h:37-38, 260, 286)
typedef struct ncclComm* ncclComm_t;
struct NcclUniqueId
{
  char internal[128];
};
enum : int
{
  kNcclSuccess = 0,
  kNcclSum = 0,
  kNcclDouble = 8
};
struct NcclApi
{
  void* lib = nullptr;
  int (*GetUniqueId)(NcclUniqueId*) = nullptr;
  int (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, NcclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::string why;
};

static NcclApi& nccl()
{
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    for (const char* name : {"libnccl.so.2", "libnccl.so"})
    {
      api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (api.lib) break;
    }
    if (!api.lib)
    {
      const char* e = dlerror();
      api.why = std::string("NCCL not found (dlopen libnccl.so.2): ") + (e ? e : "");
      return;
    }
    auto sym = [&](const char* n) {
      void* p = dlsym(api.lib, n);
      if (!p && api.why.empty()) api.why = std::string("NCCL symbol missing: ") + n;
      return p;
    };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  return api;
}

// out (+)= packed, split into the caller's three arrays (any of them may be null)
__global__ void group_unpack_kernel(const double* __restrict__ packed, int P, double* __restrict__ gram, double* __restrict__ rhs,
                                    double* __restrict__ tau_sq, int accumulate)
{
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int nG = P * P;
  if (e >= nG + P + 1) return;
  double* dst = e < nG ? (gram ? gram + e : nullptr) : (e < nG + P ? (rhs ? rhs + (e - nG) : nullptr) : tau_sq);
  if (!dst) return;
  *dst = accumulate ? *dst + packed[e] : packed[e];
}

}  // namespace rdb

using namespace rdb;

struct rdb_group
{
  std::vector<rdb_chain*> chains;    // one handle per local device (owned)
  std::vector<ncclComm_t> comms;     // one communicator per local device
  std::vector<double*> packed;       // [G | b | tau_sq] on each local device
  std::vector<cudaStream_t> streams; // default streams of the group (used when the caller passes none)
  std::vector<cudaEvent_t> done;     // recorded after the last use of packed[k] by a call; the next call on device k waits for it
  int nranks = 0;                    // ranks in the communicator (local devices for rdb_group_create, all processes for rdb_group_create_rank)
  int P = 0;
  std::mutex mu;
};

static rdb_status nccl_fail(int r, const char* where)
{
  NcclApi& a = nccl();
  return set_error(RDB_ERR_CUDA, std::string(where) + ": NCCL: " + (a.GetErrorString ? a.GetErrorString(r) : "error"));
}
static rdb_status cuda_fail_g(cudaError_t e, const char* where) { return set_error(RDB_ERR_CUDA, std::string(where) + ": " + cudaGetErrorString(e)); }

static rdb_status group_alloc(rdb_group* g, const rdb_chain_desc* desc, int ndev, const int32_t* dev_ids)
{
  g->P = 10 * desc->n_joints;
  const size_t n_out = (size_t)g->P * g->P + g->P + 1;
  for (int k = 0; k < ndev; k++)
  {
    rdb_chain* ch = nullptr;
    const rdb_status s = rdb_chain_create_on(desc, dev_ids[k], &ch);
    if (s != RDB_OK) return s;
    g->chains.push_back(ch);
    DeviceScope dev(dev_ids[k]);
    if (dev.err != cudaSuccess) return cuda_fail_g(dev.err, "cudaSetDevice");
    double* p = nullptr;
    cudaError_t e = cudaMalloc(&p, sizeof(double) * n_out);
    if (e != cudaSuccess) return cuda_fail_g(e, "cudaMalloc(group partials)");
    g->packed.push_back(p);
    cudaStream_t st = nullptr;
    e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    if (e != cudaSuccess) return cuda_fail_g(e, "cudaStreamCreate");
    g->streams.push_back(st);
    cudaEvent_t ev = nullptr;
    e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return cuda_fail_g(e, "cudaEventCreate");
    g->done.push_back(ev);
  }
  return RDB_OK;
}

extern "C" {

void rdb_group_destroy(rdb_group* g)
{
  if (!g) return;
  NcclApi& a = nccl();
  for (size_t k = 0; k < g->chains.size(); k++)
  {
    DeviceScope dev(rdb_chain_device(g->chains[k]));
    if (k < g->comms.size() && g->comms[k] && a.CommDestroy) a.CommDestroy(g->comms[k]);
    if (k < g->packed.size() && g->packed[k]) cudaFree(g->packed[k]);
    if (k < g->streams.size() && g->streams[k]) cudaStreamDestroy(g->streams[k]);
    if (k < g->done.size() && g->done[k]) cudaEventDestroy(g->done[k]);
  }
  for (rdb_chain* ch : g->chains) rdb_chain_destroy(ch);
  delete g;
}

rdb_status rdb_group_create(const rdb_chain_desc* desc, int32_t ndev, const int32_t* dev_ids, rdb_group** out)
{
  if (!desc || !out || ndev <= 0 || ndev > 64) return set_error(RDB_ERR_INVALID_ARG, "group_create: null argument or bad device count");
  *out = nullptr;
  const int have = rdb_device_count();
  if (have <= 0) return set_error(RDB_ERR_NO_DEVICE, "no CUDA device: rosdyn_b200 has no CPU fallback");
  std::vector<int32_t> ids((size_t)ndev);
  for (int k = 0; k < ndev; k++)
  {
    ids[k] = dev_ids ? dev_ids[k] : k;  // NULL: devices 0 .. ndev-1
    if (ids[k] < 0 || ids[k] >= have) return set_error(RDB_ERR_INVALID_ARG, "group_create: device id out of range");
    for (int j = 0; j < k; j++)
      if (ids[j] == ids[k]) return set_error(RDB_ERR_INVALID_ARG, "group_create: device listed twice");
  }
  rdb_group* g = new (std::nothrow) rdb_group();
  if (!g) return set_error(RDB_ERR_ALLOC, "out of host memory");
  rdb_status s = group_alloc(g, desc, ndev, ids.data());
  if (s == RDB_OK && ndev > 1)
  {
    NcclApi& a = nccl();
    if (!a.CommInitAll || !a.why.empty()) s = set_error(RDB_ERR_NOT_FOUND, a.why.empty() ? "NCCL unavailable" : a.why);
    else
    {
      g->comms.assign((size_t)ndev, nullptr);
      std::vector<int> di(ids.begin(), ids.end());
      const int r = a.CommInitAll(g->comms.data(), ndev, di.data());
      if (r != kNcclSuccess) s = nccl_fail(r, "ncclCommInitAll");
    }
  }
  if (s != RDB_OK)
  {
    rdb_group_destroy(g);
    return s;
  }
  g->nranks = ndev;
  *out = g;
  return RDB_OK;
}

rdb_status rdb_group_unique_id(uint8_t id[128])
{
  if (!id) return set_error(RDB_ERR_INVALID_ARG, "group_unique_id: null argument");
  NcclApi& a = nccl();
  if (!a.GetUniqueId || !a.why.empty()) return set_error(RDB_ERR_NOT_FOUND, a.why.empty() ? "NCCL unavailable" : a.why);
  NcclUniqueId u;
  const int r = a.GetUniqueId(&u);
  if (r != kNcclSuccess) return nccl_fail(r, "ncclGetUniqueId");
  std::memcpy(id, u.internal, 128);
  return RDB_OK;
}

rdb_status rdb_group_create_rank(const rdb_chain_desc* desc, int32_t device, int32_t nranks, int32_t rank, const uint8_t id[128], rdb_group** out)
{
  if (!desc || !out || nranks <= 0 || rank < 0 || rank >= nranks || (nranks > 1 && !id))
    return set_error(RDB_ERR_INVALID_ARG, "group_create_rank: bad argument");
  *out = nullptr;
  const int have = rdb_device_count();
  if (have <= 0) return set_error(RDB_ERR_NO_DEVICE, "no CUDA device: rosdyn_b200 has no CPU fallback");
  if (device < 0 || device >= have) return set_error(RDB_ERR_INVALID_ARG, "group_create_rank: device id out of range");
  rdb_group* g = new (std::nothrow) rdb_group();
  if (!g) return set_error(RDB_ERR_ALLOC, "out of host memory");
  const int32_t ids[1] = {device};
  rdb_status s = group_alloc(g, desc, 1, ids);
  if (s == RDB_OK && nranks > 1)
  {
    NcclApi& a = nccl();
    if (!a.CommInitRank || !a.why.empty()) s = set_error(RDB_ERR_NOT_FOUND, a.why.empty() ? "NCCL unavailable" : a.why);
    else
    {
      DeviceScope dev(device);
      NcclUniqueId u;
      std::memcpy(u.internal, id, 128);
      g->comms.assign(1, nullptr);
      const int r = a.CommInitRank(&g->comms[0], nranks, u, rank);
      if (r != kNcclSuccess) s = nccl_fail(r, "ncclCommInitRank");
    }
  }
  if (s != RDB_OK)
  {
    rdb_group_destroy(g);
    return s;
  }
  g->nranks = nranks;
  *out = g;
  return RDB_OK;
}

int32_t rdb_group_size(const rdb_group* g) { return g ? (int32_t)g->chains.size() : -1; }
int32_t rdb_group_ranks(const rdb_group* g) { return g ? g->nranks : -1; }
rdb_chain* rdb_group_chain(rdb_group* g, int32_t k) { return (g && k >= 0 && k < (int32_t)g->chains.size()) ? g->chains[(size_t)k] : nullptr; }

rdb_status rdb_regressor_gram_sharded(rdb_group* g, const rdb_samples* shards, const double* const* tau_meas, double* const* gram,
                                      double* const* rhs, double* const* tau_sq, int32_t accumulate, void* const* streams)
{
  if (!g || !shards) return set_error(RDB_ERR_INVALID_ARG, "gram_sharded: null group or shards");
  std::lock_guard<std::mutex> lock(g->mu);
  const int nd = (int)g->chains.size(), P = g->P;
  const size_t n_out = (size_t)P * P + P + 1;
  NcclApi& a = nccl();
  // 1. every local device: fused regressor -> normal equations of its shard, written straight into the packed buffer once the previous
  //    call, whatever its stream, has unpacked it
  for (int k = 0; k < nd; k++)
  {
    cudaStream_t st = streams ? (cudaStream_t)streams[k] : g->streams[(size_t)k];  // an entry of `streams` may be 0 = the default stream
    double* pk = g->packed[(size_t)k];
    {
      DeviceScope dev(rdb_chain_device(g->chains[(size_t)k]));
      const cudaError_t e = cudaStreamWaitEvent(st, g->done[(size_t)k], 0);
      if (e != cudaSuccess) return cuda_fail_g(e, "cudaStreamWaitEvent");
    }
    const rdb_status s = rdb_regressor_gram_batch(g->chains[(size_t)k], &shards[k], tau_meas ? tau_meas[k] : nullptr, pk, pk + (size_t)P * P,
                                                  pk + (size_t)P * P + P, 0, st);
    if (s != RDB_OK) return s;
  }
  // 2. ONE all-reduce of the partials over NVLink (in place, on each device's stream)
  if (g->nranks > 1)
  {
    int r = nd > 1 ? a.GroupStart() : kNcclSuccess;
    if (r != kNcclSuccess) return nccl_fail(r, "ncclGroupStart");
    for (int k = 0; k < nd; k++)
    {
      cudaStream_t st = streams ? (cudaStream_t)streams[k] : g->streams[(size_t)k];  // an entry of `streams` may be 0 = the default stream
      DeviceScope dev(rdb_chain_device(g->chains[(size_t)k]));
      r = a.AllReduce(g->packed[(size_t)k], g->packed[(size_t)k], n_out, kNcclDouble, kNcclSum, g->comms[(size_t)k], st);
      if (r != kNcclSuccess) break;
    }
    const int r2 = nd > 1 ? a.GroupEnd() : kNcclSuccess;
    if (r != kNcclSuccess) return nccl_fail(r, "ncclAllReduce");
    if (r2 != kNcclSuccess) return nccl_fail(r2, "ncclGroupEnd");
  }
  // 3. into the caller's arrays; packed[k] is free for the next call after this
  for (int k = 0; k < nd; k++)
  {
    double* G = gram ? gram[k] : nullptr;
    double* b = rhs ? rhs[k] : nullptr;
    double* t = tau_sq ? tau_sq[k] : nullptr;
    cudaStream_t st = streams ? (cudaStream_t)streams[k] : g->streams[(size_t)k];  // an entry of `streams` may be 0 = the default stream
    DeviceScope dev(rdb_chain_device(g->chains[(size_t)k]));
    if (G || b || t)
    {
      group_unpack_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, st>>>(g->packed[(size_t)k], P, G, b, t, accumulate);
      count_launch();
      const cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return cuda_fail_g(e, "group_unpack_kernel");
    }
    const cudaError_t e = cudaEventRecord(g->done[(size_t)k], st);
    if (e != cudaSuccess) return cuda_fail_g(e, "cudaEventRecord");
  }
  return RDB_OK;
}

rdb_status rdb_group_synchronize(rdb_group* g)
{
  if (!g) return set_error(RDB_ERR_INVALID_ARG, "null group");
  for (size_t k = 0; k < g->chains.size(); k++)
  {
    DeviceScope dev(rdb_chain_device(g->chains[k]));
    const cudaError_t e = cudaStreamSynchronize(g->streams[k]);
    if (e != cudaSuccess) return cuda_fail_g(e, "cudaStreamSynchronize");
  }
  return RDB_OK;
}

}  // extern "C"
