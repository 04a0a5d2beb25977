// Forward dynamics through the C++ facade (include/rosdyn_b200/chain.hpp): getJointAcceleration in its std, Eigen and batched host forms.
// tests/test_forward_dynamics.py compiles and links this file against the Eigen subset of oracle/shim; without a CUDA device it only reports
// that it linked (the engine has no CPU fallback).  On a device it checks M ddq + h = tau with the facade's own inertia and torque getters.
#include <cmath>
#include <cstdio>
#include <vector>

#include "rosdyn_b200/chain.hpp"

#ifndef ROSDYN_B200_HAVE_EIGEN
#error "compile with -I oracle/shim (or a real Eigen3) so that <Eigen/Core> exists"
#endif

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

static bool near(double a, double b) { return std::fabs(a - b) <= 1e-10 * (1 + std::fabs(b)); }

int main()
{
  if (rdb_device_count() <= 0)
  {
    std::printf("no CUDA device: compiled and linked only\n");
    return 0;
  }
  // revolute, fixed, revolute, prismatic, revolute: the walker folds the fixed joint away
  std::vector<rdb_joint_desc> J = {joint(RDB_JOINT_REVOLUTE, 0, 0, 0.1, 0, 0, 0, 0, 0, 1, 0), joint(RDB_JOINT_FIXED, 0, 0.05, 0.1, 0.2, 0, 0, 0, 0, 1, -1),
                                   joint(RDB_JOINT_REVOLUTE, 0, 0.2, 0, 0, 1.57, 0, 0, 1, 0, 1),
                                   joint(RDB_JOINT_PRISMATIC, 0.3, 0, 0, 0.1, 0, 0.2, 1, 0, 0, 2),
                                   joint(RDB_JOINT_REVOLUTE, 0.1, 0, 0.05, 0, 0.3, 0, 0, 0, 1, 3)};
  const int nj = (int)J.size(), n = 4;
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
  rdb_chain_desc desc{nj, n, {0, 0, -9.806}, J.data(), L.data()};
  Chain ch(desc);
  int fail = 0;

  // std containers
  const rosdyn_b200::VectorXd q = {0.3, -0.7, 0.2, 0.9}, dq = {0.5, 0.1, -0.4, 0.2}, tau = {1.5, -4.0, 7.0, 0.3};
  const rosdyn_b200::VectorXd ddq = ch.getJointAcceleration(q, dq, tau);
  const rosdyn_b200::VectorXd M = ch.getJointInertia(q), h = ch.getJointTorqueNonLinearPart(q, dq), tau2 = ch.getJointTorque(q, dq, ddq);
  for (int r = 0; r < n; r++)
  {
    double s = h[r];
    for (int c = 0; c < n; c++) s += M[(size_t)c * n + r] * ddq[c];
    if (!near(s, tau[r])) fail++;
    if (!near(tau2[r], tau[r])) fail++;
  }

  // Eigen overloads
  Eigen::VectorXd eq(n), edq(n), etau(n);
  for (int k = 0; k < n; k++)
  {
    eq(k) = q[k];
    edq(k) = dq[k];
    etau(k) = tau[k];
  }
  const Eigen::VectorXd eddq = ch.getJointAcceleration(eq, edq, etau);
  const Eigen::MatrixXd eM = ch.getJointInertia(eq);
  const Eigen::VectorXd eh = ch.getJointTorqueNonLinearPart(eq, edq);
  const Eigen::VectorXd res = eM * eddq + eh;
  for (int k = 0; k < n; k++)
  {
    if (!near(res(k), etau(k))) fail++;
    if (eddq(k) != ddq[k]) fail++;  // one engine behind both overloads
  }

  // batched host sibling: sample 0 is the per-sample call, bit for bit
  const int N = 9;
  std::vector<double> Q((size_t)n * N), DQ((size_t)n * N), T((size_t)n * N), DDQ((size_t)n * N);
  for (int i = 0; i < N; i++)
    for (int k = 0; k < n; k++)
    {
      Q[(size_t)k * N + i] = q[k] + 0.1 * i;
      DQ[(size_t)k * N + i] = dq[k];
      T[(size_t)k * N + i] = tau[k];
    }
  std::vector<int32_t> info(N, -1);
  const rdb_samples in{N, N, Q.data(), DQ.data(), nullptr, nullptr};
  ch.getJointAccelerationHost(in, T.data(), DDQ.data(), N, info.data());
  for (int k = 0; k < n; k++)
    if (DDQ[(size_t)k * N] != ddq[k]) fail++;
  for (int i = 0; i < N; i++)
    if (info[i] != 0) fail++;

  // a size mismatch throws like every other getter
  bool threw = false;
  try
  {
    ch.getJointAcceleration(q, dq, rosdyn_b200::VectorXd(n + 1, 0.0));
  }
  catch (const std::invalid_argument&)
  {
    threw = true;
  }
  if (!threw) fail++;

  std::printf(fail ? "FAIL %d\n" : "forward dynamics facade ok\n", fail);
  return fail ? 1 : 0;
}
