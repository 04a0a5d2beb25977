// Weighted normal equations through the C++ facade (include/rosdyn_b200/chain.hpp): the getRegressorGram / getRegressorGramExt overloads
// that take rdb_gram_weights, on device arrays.  tests/test_gram_weighted.py compiles and links this file against the library and the CUDA
// runtime; without a CUDA device it only reports that it linked (the engine has no CPU fallback).  On a device: unit weights give the
// unweighted results bit for bit, weights of 4 exactly four times them (per joint, per sample, as planes), one-hot per-joint weights sum to
// the unweighted normal equations, and a negative stride throws like every other argument error.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <vector>

#include "rosdyn_b200/chain.hpp"

using rosdyn_b200::Chain;

static rdb_joint_desc joint(int type, double x, double y, double z, double r, double p, double yw, double ax, double ay, double az, int in)
{
  rdb_joint_desc j{};
  j.type = type;
  j.input_index = in;
  j.xyz[0] = x; j.xyz[1] = y; j.xyz[2] = z;
  rosdyn_b200::rpyToRot(r, p, yw, j.rot);
  j.axis[0] = ax; j.axis[1] = ay; j.axis[2] = az;
  return j;
}

static std::vector<double> get(const double* d, size_t n)
{
  std::vector<double> h(n);
  cudaMemcpy(h.data(), d, sizeof(double) * n, cudaMemcpyDeviceToHost);
  return h;
}

int main()
{
  if (rdb_device_count() <= 0)
  {
    std::printf("no CUDA device: compiled and linked only\n");
    return 0;
  }
  // revolute, fixed, revolute, prismatic, revolute: the folded chain has 4 moving joints and a fold expansion
  std::vector<rdb_joint_desc> J = {joint(RDB_JOINT_REVOLUTE, 0, 0, 0.1, 0, 0, 0, 0, 0, 1, 0), joint(RDB_JOINT_FIXED, 0, 0.05, 0.1, 0.2, 0, 0, 0, 0, 1, -1),
                                   joint(RDB_JOINT_REVOLUTE, 0, 0.2, 0, 0, 1.57, 0, 0, 1, 0, 1),
                                   joint(RDB_JOINT_PRISMATIC, 0.3, 0, 0, 0.1, 0, 0.2, 1, 0, 0, 2),
                                   joint(RDB_JOINT_REVOLUTE, 0.1, 0, 0.05, 0, 0.3, 0, 0, 0, 1, 3)};
  const int nj = (int)J.size(), n_in = 4, P = 10 * nj;
  std::vector<rdb_link_desc> L(nj + 1);
  for (int l = 1; l <= nj; l++)
  {
    L[l].mass = 1.0 + l;
    L[l].cog[0] = 0.02 * l;
    L[l].cog[2] = 0.1 * l;
    L[l].inertial_rot[0] = L[l].inertial_rot[4] = L[l].inertial_rot[8] = 1.0;
    L[l].inertia[0] = L[l].inertia[3] = 0.02 * l;
    L[l].inertia[5] = 0.01 * l;
  }
  rdb_chain_desc desc{nj, n_in, {0, 0, -9.806}, J.data(), L.data()};
  Chain ch(desc);
  int fail = 0;

  const int64_t n = 7011, ld = 7013, ldw = 7020;
  const size_t NOUT = (size_t)P * P + P + 1;
  double *x = nullptr, *w = nullptr, *o0 = nullptr, *o1 = nullptr;
  if (cudaMalloc(&x, sizeof(double) * 4 * n_in * ld) != cudaSuccess || cudaMalloc(&w, sizeof(double) * n_in * ldw) != cudaSuccess ||
      cudaMalloc(&o0, sizeof(double) * NOUT) != cudaSuccess || cudaMalloc(&o1, sizeof(double) * NOUT) != cudaSuccess)
  {
    std::printf("FAIL cudaMalloc\n");
    return 1;
  }
  for (int a = 0; a < 4; a++) rdb_fill_uniform(x + (size_t)a * n_in * ld, n_in, n, ld, 0x3E1, a, nullptr);
  const rdb_samples in{n, ld, x, x + n_in * ld, x + 2 * n_in * ld, nullptr};
  const double* tau = x + 3 * n_in * ld;
  ch.getRegressorGram(in, tau, o0, o0 + P * P, o0 + P * P + P, false);
  const std::vector<double> base = get(o0, NOUT);

  // unit weights and weights of 4 in the per-joint, per-sample and plane forms
  const rdb_gram_weights forms[3] = {{w, 1, 0}, {w, 0, 1}, {w, ldw, 1}};
  for (double c : {1.0, 4.0})
  {
    std::vector<double> hw((size_t)n_in * ldw, c);
    cudaMemcpy(w, hw.data(), sizeof(double) * hw.size(), cudaMemcpyHostToDevice);
    for (const rdb_gram_weights& f : forms)
    {
      ch.getRegressorGram(in, tau, f, o1, o1 + P * P, o1 + P * P + P, false);
      const std::vector<double> r = get(o1, NOUT);
      for (size_t e = 0; e < NOUT; e++)
        if (r[e] != c * base[e]) fail++;
    }
  }
  // one-hot per-joint weights: the per-joint normal equations add up to the unweighted ones
  double scale = 0.0;
  for (double v : base) scale = std::max(scale, std::fabs(v));
  for (int r = 0; r < n_in; r++)
  {
    std::vector<double> hw(n_in, 0.0);
    hw[r] = 1.0;
    cudaMemcpy(w, hw.data(), sizeof(double) * n_in, cudaMemcpyHostToDevice);
    ch.getRegressorGram(in, tau, rdb_gram_weights{w, 1, 0}, o1, o1 + P * P, o1 + P * P + P, r > 0);
  }
  const std::vector<double> sum = get(o1, NOUT);
  for (size_t e = 0; e < NOUT; e++)
    if (!(std::fabs(sum[e] - base[e]) <= 1e-13 * scale)) fail++;

  // a negative stride throws like every other argument error
  bool threw = false;
  try
  {
    ch.getRegressorGram(in, tau, rdb_gram_weights{w, -1, 0}, o1, o1 + P * P, o1 + P * P + P, false);
  }
  catch (const std::invalid_argument&)
  {
    threw = true;
  }
  if (!threw) fail++;
  if (cudaDeviceSynchronize() != cudaSuccess) fail++;
  cudaFree(x);
  cudaFree(w);
  cudaFree(o0);
  cudaFree(o1);

  std::printf(fail ? "FAIL %d\n" : "weighted gram facade ok\n", fail);
  return fail ? 1 : 0;
}
