// Segmented normal equations through the C++ facade (include/rosdyn_b200/chain.hpp): getRegressorGramSegmented on device arrays.
// tests/test_gram_segmented.py compiles and links this file against the library and the CUDA runtime; without a CUDA device it only reports
// that it linked (the engine has no CPU fallback).  On a device every segment's (G, b, tau^T tau) is compared with getRegressorGram over the
// same samples (pointer-offset inputs), an empty segment must come back as zeros, and accumulate must add exactly.
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

static double maxabs(const std::vector<double>& v, size_t lo, size_t hi)
{
  double m = 0.0;
  for (size_t k = lo; k < hi; k++) m = std::max(m, std::fabs(v[k]));
  return m;
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

  const std::vector<int64_t> offsets = {3, 3, 40, 1040, 7000};  // an empty segment, short ones, one of several work items; 3 samples before
  const int64_t n = 7011, ld = 7013, K = (int64_t)offsets.size() - 1;
  double *x = nullptr, *G = nullptr, *b = nullptr, *t = nullptr, *g1 = nullptr;
  if (cudaMalloc(&x, sizeof(double) * 3 * n_in * ld) != cudaSuccess || cudaMalloc(&G, sizeof(double) * (K * P * P + K * P + K)) != cudaSuccess ||
      cudaMalloc(&g1, sizeof(double) * (P * P + P + 1)) != cudaSuccess)
  {
    std::printf("FAIL cudaMalloc\n");
    return 1;
  }
  b = G + K * P * P;
  t = b + K * P;
  for (int a = 0; a < 3; a++) rdb_fill_uniform(x + (size_t)a * n_in * ld, n_in, n, ld, 0x5E9, a, nullptr);
  const rdb_samples in{n, ld, x, x + n_in * ld, x + 2 * n_in * ld, nullptr};
  ch.getRegressorGramSegmented(in, nullptr, offsets, G, b, t, false);
  std::vector<double> seg((size_t)(K * P * P + K * P + K)), one((size_t)(P * P + P + 1));
  cudaMemcpy(seg.data(), G, sizeof(double) * seg.size(), cudaMemcpyDeviceToHost);
  for (int64_t k = 0; k < K; k++)
  {
    const int64_t lo = offsets[k], len = offsets[k + 1] - lo;
    const rdb_samples s{len, ld, x + lo, x + n_in * ld + lo, x + 2 * n_in * ld + lo, nullptr};
    ch.getRegressorGram(s, nullptr, g1, g1 + P * P, g1 + P * P + P, false);
    cudaMemcpy(one.data(), g1, sizeof(double) * one.size(), cudaMemcpyDeviceToHost);
    const size_t og = (size_t)k * P * P, ob = (size_t)(K * P * P + k * P), ot = (size_t)(K * P * P + K * P + k);
    const double sg = std::max(maxabs(one, 0, P * P), 1.0), sb = std::max(maxabs(one, P * P, P * P + P), 1.0);
    for (int e = 0; e < P * P; e++)
      if (!(std::fabs(seg[og + e] - one[e]) <= 1e-10 * sg)) fail++;
    for (int e = 0; e < P; e++)
      if (!(std::fabs(seg[ob + e] - one[P * P + e]) <= 1e-10 * sb)) fail++;
    if (!(std::fabs(seg[ot] - one[P * P + P]) <= 1e-10 * std::max(one[P * P + P], 1.0))) fail++;
    if (len == 0 && (maxabs(seg, og, og + P * P) != 0.0 || seg[ot] != 0.0)) fail++;
  }
  // accumulate adds the same sums onto the first call's exactly
  ch.getRegressorGramSegmented(in, nullptr, offsets, G, b, t, true);
  std::vector<double> twice(seg.size());
  cudaMemcpy(twice.data(), G, sizeof(double) * twice.size(), cudaMemcpyDeviceToHost);
  for (size_t e = 0; e < seg.size(); e++)
    if (twice[e] != seg[e] + seg[e]) fail++;

  // bad offsets throw like every other argument error
  bool threw = false;
  try
  {
    ch.getRegressorGramSegmented(in, nullptr, {0, 50, 20}, G, b, t, false);
  }
  catch (const std::invalid_argument&)
  {
    threw = true;
  }
  if (!threw) fail++;
  if (cudaDeviceSynchronize() != cudaSuccess) fail++;
  cudaFree(x);
  cudaFree(G);
  cudaFree(g1);

  std::printf(fail ? "FAIL %d\n" : "segmented gram facade ok\n", fail);
  return fail ? 1 : 0;
}
