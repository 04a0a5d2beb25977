// gram_jit.cpp -- run-time specialisation of the fused Gram kernels to the constants of one chain.
//
// The precompiled kernels read the model (A', t', pi', g of the folded chain) from the constant bank, so ptxas cannot see that most of it is
// exact zeros and ones (signed-permutation rotations, translations along one axis, zero centres of mass and products of inertia) and issues
// every product.  On the first Gram call of an all-revolute (REV) folded chain this file emits a translation unit that defines those
// constants as constexpr data (hexfloat literals: the exact values), instantiates the same kernel template against it (gram_fused.cuh,
// compile-time model of gram_common.cuh), compiles it with NVRTC for the device's architecture and loads the cubin.  The generator then skips
// the products with exact zeros and passes through the ones with +-1; every other operation is the precompiled kernel's, in the same order.
//
// NVRTC is bound at run time (dlopen "libnvrtc.so.12", RDB_NVRTC_LIB overrides the name): the library has no link-time dependency on it.
// When NVRTC is missing, compilation or loading fails, or RDB_GRAM_JIT=0 is set, the precompiled instantiation runs and the handle records
// why (rdb_chain_gram_kernel_info).  Compiled modules are cached for the process, keyed by the generated source (every constant), the
// kernel and the architecture: handles of the same chain share one compilation, and a failure is not retried.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvrtc.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "launch.h"

namespace rdb
{

// the kernel headers as text (generated from csrc/ at build time, rosdyn_b200/build.py)
extern const int gram_jit_nheaders;
extern const char* const gram_jit_header_names[];
extern const char* const gram_jit_header_texts[];

namespace
{

// NVRTC has no system headers; the kernel headers need the fixed-width integer types only
const char* const kStdint =
    "#pragma once\n"
    "typedef signed char int8_t; typedef short int16_t; typedef int int32_t; typedef long long int64_t;\n"
    "typedef unsigned char uint8_t; typedef unsigned short uint16_t; typedef unsigned int uint32_t; typedef unsigned long long uint64_t;\n";

struct NvrtcApi
{
  void* lib = nullptr;
  std::string why;
  decltype(&nvrtcCreateProgram) create = nullptr;
  decltype(&nvrtcDestroyProgram) destroy = nullptr;
  decltype(&nvrtcAddNameExpression) add_name = nullptr;
  decltype(&nvrtcCompileProgram) compile = nullptr;
  decltype(&nvrtcGetProgramLogSize) log_size = nullptr;
  decltype(&nvrtcGetProgramLog) log = nullptr;
  decltype(&nvrtcGetCUBINSize) cubin_size = nullptr;
  decltype(&nvrtcGetCUBIN) cubin = nullptr;
  decltype(&nvrtcGetLoweredName) lowered = nullptr;
  decltype(&nvrtcGetErrorString) err = nullptr;
};

const NvrtcApi& nvrtc()
{
  static const NvrtcApi api = [] {
    NvrtcApi a;
    const char* env = getenv("RDB_NVRTC_LIB");
    const char* name = env && *env ? env : "libnvrtc.so.12";
    a.lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
    if (!a.lib)
    {
      const char* e = dlerror();
      a.why = std::string("NVRTC not found (dlopen ") + name + "): " + (e ? e : "");
      return a;
    }
    bool ok = true;
    auto sym = [&](auto& fn, const char* n) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(a.lib, n));
      ok = ok && fn != nullptr;
    };
    sym(a.create, "nvrtcCreateProgram");
    sym(a.destroy, "nvrtcDestroyProgram");
    sym(a.add_name, "nvrtcAddNameExpression");
    sym(a.compile, "nvrtcCompileProgram");
    sym(a.log_size, "nvrtcGetProgramLogSize");
    sym(a.log, "nvrtcGetProgramLog");
    sym(a.cubin_size, "nvrtcGetCUBINSize");
    sym(a.cubin, "nvrtcGetCUBIN");
    sym(a.lowered, "nvrtcGetLoweredName");
    sym(a.err, "nvrtcGetErrorString");
    if (!ok)
    {
      a.why = std::string("NVRTC library ") + name + " lacks an entry point this library needs";
      a.create = nullptr;
    }
    return a;
  }();
  return api;
}

void append_hex(std::string& s, double v)
{
  char b[40];
  snprintf(b, sizeof b, "%a", v);
  s += b;
}
void append_array(std::string& s, const char* decl, const double* v, int n)
{
  s += decl;
  s += " = {";
  for (int k = 0; k < n; k++)
  {
    if (k) s += ", ";
    append_hex(s, v[k]);
  }
  s += "};\n";
}

struct Entry
{
  cudaLibrary_t lib = nullptr;
  cudaKernel_t kernel = nullptr;
  std::string why;  // failure, or how the module was made
};
std::mutex g_mu;
std::map<std::string, Entry> g_cache;

// NVRTC: the cubin of kernel `expr` from `src` and its lowered name; false with the reason in `why`
bool compile_cubin(const std::string& src, const std::string& expr, const std::string& arch, std::vector<char>& cubin, std::string& kname,
                   std::string& why)
{
  const NvrtcApi& api = nvrtc();
  if (!api.create)
  {
    why = api.why;
    return false;
  }
  std::vector<const char*> names{"stdint.h"}, texts{kStdint};
  for (int k = 0; k < gram_jit_nheaders; k++)
  {
    names.push_back(gram_jit_header_names[k]);
    texts.push_back(gram_jit_header_texts[k]);
  }
  nvrtcProgram prog = nullptr;
  nvrtcResult r = api.create(&prog, src.c_str(), "gram_jit_model.cu", (int)names.size(), texts.data(), names.data());
  if (r != NVRTC_SUCCESS)
  {
    why = std::string("nvrtcCreateProgram: ") + api.err(r);
    return false;
  }
  api.add_name(prog, expr.c_str());
  // the flags of the precompiled library (rosdyn_b200/build.py): -O3 is NVRTC's default, FMA contraction stays on (--fmad=true).
  // -default-device: the host entry points the public header declares (chain_dev.h includes it for the joint types) are never called here
  const std::string arch_opt = "--gpu-architecture=" + arch;
  const char* opts[] = {arch_opt.c_str(), "-std=c++17", "--fmad=true", "-default-device"};
  r = api.compile(prog, (int)(sizeof opts / sizeof opts[0]), opts);
  if (r != NVRTC_SUCCESS)
  {
    size_t n = 0;
    api.log_size(prog, &n);
    std::string log(n, '\0');
    if (n) api.log(prog, &log[0]);
    why = std::string("NVRTC compilation failed (") + api.err(r) + "): " + log.substr(0, 2000);
    api.destroy(&prog);
    return false;
  }
  size_t nc = 0;
  api.cubin_size(prog, &nc);
  cubin.assign(nc, 0);
  const char* lowered = nullptr;
  const bool ok = nc > 0 && api.cubin(prog, cubin.data()) == NVRTC_SUCCESS && api.lowered(prog, expr.c_str(), &lowered) == NVRTC_SUCCESS && lowered;
  if (ok) kname = lowered;  // owned by the program
  else why = "NVRTC produced no cubin or kernel name";
  api.destroy(&prog);
  return ok;
}

Entry compile_entry(const std::string& src, const std::string& expr, const std::string& arch)
{
  Entry e;
  std::vector<char> cubin;
  std::string kname;
  const auto t0 = std::chrono::steady_clock::now();
  if (!compile_cubin(src, expr, arch, cubin, kname, e.why)) return e;
  const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  cudaError_t ce = cudaLibraryLoadData(&e.lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
  if (ce == cudaSuccess) ce = cudaLibraryGetKernel(&e.kernel, e.lib, kname.c_str());
  if (ce != cudaSuccess)
  {
    cudaGetLastError();
    if (e.lib) cudaLibraryUnload(e.lib);
    e.lib = nullptr;
    e.kernel = nullptr;
    e.why = std::string("loading the NVRTC cubin failed: ") + cudaGetErrorString(ce);
    return e;
  }
  char b[160];
  snprintf(b, sizeof b, "specialised to the chain's constants, compiled by NVRTC for %s in %.0f ms", arch.c_str(), ms);
  e.why = b;
  return e;
}

// the translation unit of a folded chain: its constants as the compile-time model GramJitModel; "" when a constant is not finite
std::string model_source(const ChainDev<RDB_MAX_JOINTS>& F)
{
  const int K = F.nj;
  std::vector<double> A(9 * K), t(3 * K), pi(10 * K);
  bool finite = true;
  for (int l = 0; l < K; l++)
  {
    for (int k = 0; k < 9; k++) A[9 * l + k] = F.joint[l].A[k];
    for (int k = 0; k < 3; k++) t[3 * l + k] = F.joint[l].t[k];
    for (int k = 0; k < 10; k++) pi[10 * l + k] = F.link[l].pi[k];
  }
  for (double v : A) finite = finite && std::isfinite(v);
  for (double v : t) finite = finite && std::isfinite(v);
  for (double v : pi) finite = finite && std::isfinite(v);
  for (int k = 0; k < 3; k++) finite = finite && std::isfinite(F.g[k]);
  if (!finite) return "";
  std::string src = "#include \"gram_fused.cuh\"\nnamespace rdb\n{\nstruct GramJitModel\n{\n  static constexpr bool RUNTIME = false;\n";
  const std::string nk = std::to_string(K);
  append_array(src, ("  static constexpr double A[" + nk + "][9]").c_str(), A.data(), 9 * K);
  append_array(src, ("  static constexpr double t[" + nk + "][3]").c_str(), t.data(), 3 * K);
  append_array(src, ("  static constexpr double pi[" + nk + "][10]").c_str(), pi.data(), 10 * K);
  append_array(src, "  static constexpr double g[3]", F.g, 3);
  src +=
      "  __host__ __device__ static constexpr double val(int f, int l, int k)\n  {\n"
      "    return f == MK_A ? A[l][k] : (f == MK_T ? t[l][k] : (f == MK_PI ? pi[l][k] : g[k]));\n  }\n};\n}  // namespace rdb\n";
  return src;
}

std::string kernel_expr(const char* kernel_args) { return std::string("&rdb::") + kernel_args + ", rdb::GramJitModel>"; }

}  // namespace

const void* gram_jit_kernel(ChainHost& ch, const char* kernel_args)
{
  std::string& why = ch.gram.kernel_why;
  ch.gram.kernel_specialised = 0;
  const char* env = getenv("RDB_GRAM_JIT");
  if (env && strcmp(env, "0") == 0)
  {
    why = "precompiled kernel: run-time specialisation disabled (RDB_GRAM_JIT=0)";
    return nullptr;
  }
  const std::string src = model_source(ch.gram.fold);
  if (src.empty())
  {
    why = "precompiled kernel: the model has non-finite constants";
    return nullptr;
  }
  const std::string expr = kernel_expr(kernel_args);
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, ch.device);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, ch.device);
  // the architecture-specific target (sm_100a) where there is one, as the precompiled library uses
  const std::string arch = "sm_" + std::to_string(major) + std::to_string(minor) + (major >= 9 ? "a" : "");
  const std::string ckey = src + expr + "|" + arch;  // the generated source holds every constant, exactly
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_cache.find(ckey);
  if (it == g_cache.end()) it = g_cache.emplace(ckey, compile_entry(src, expr, arch)).first;
  if (!it->second.kernel)
  {
    why = "precompiled kernel: " + it->second.why;
    return nullptr;
  }
  ch.gram.kernel_specialised = 1;
  why = it->second.why;
  return reinterpret_cast<const void*>(it->second.kernel);
}

bool gram_jit_cubin(const ChainDev<RDB_MAX_JOINTS>& F, const char* kernel_args, const char* arch, std::vector<char>& cubin, std::string& why)
{
  const std::string model = model_source(F);
  if (model.empty())
  {
    why = "the model has non-finite constants";
    return false;
  }
  std::string kname;
  return compile_cubin(model, kernel_expr(kernel_args), arch, cubin, kname, why);
}

}  // namespace rdb
