// fold.cpp -- the chain with its never-moving joints folded away and every revolute joint's axis on +z of its link frame (host side; used by
// the fused Gram kernel and by the torque / inertia walkers).
#include <cuda_runtime.h>

#include <cmath>
#include <vector>

#include "launch.h"

namespace rdb
{

// ---------------------------------------------------------------------------------------------- folded chain (host)
// A joint that never moves (FIXED, or a joint that is not an input: the reference gives it q = 0) rigidly attaches its child link to the last
// moving link A before it.  tau is linear in the inertial parameters, so the regressor block of such a link B is the block of A times a
// CONSTANT 10x10 matrix:  Phi[:, B] = Phi[:, A] T_AB,  T_AB = d(parameters of the body referred to frame A) / d(parameters referred to
// frame B)  (rotation + parallel-axis shift, linear in m, m c, I).  The fused kernel therefore runs on the chain with those joints folded
// into the constant transform of the next moving joint (nJ' = moving joints, lumped parameters for tau), and the normal equations of the
// reference's full parameter vector follow as  G = E^T G' E,  b = E^T b'  with E = blockdiag-like(I | T_AB) -- exact identities, evaluated
// once per call on 70x70 numbers.  UR10-like C6 (6 revolute + fixed tool): 60 instead of 70 columns, 109 instead of 146 DMMA per 4 samples,
// 21 instead of 28 (joint, link) pairs per sample, and a slot small enough for FOUR slots / generator warps per SM.
// Canonical frames: the frame of every revolute moving link is turned about its origin, x_old = Q x_new with Q e_z = axis (det +1), so that
// the folded chain's revolute axes are all exactly e_z.  Nothing the chain returns depends on the frame a link's parameters are referred to:
// the moving link's own block gets T = T(Q^T, 0) in E like a rigidly attached link, and the generators of the fused kernels (gram_common.cuh,
// REV) take the axis as a compile-time constant instead of paying for a runtime one in every rotation, rate and projection.
struct FoldXf
{
  double R[9], t[3];  // x_parent = R x_child + t
};
static void xf_mul(const FoldXf& a, const double* Rb, const double* tb, FoldXf& c)
{
  for (int i = 0; i < 3; i++)
  {
    for (int j = 0; j < 3; j++) c.R[3 * i + j] = a.R[3 * i] * Rb[j] + a.R[3 * i + 1] * Rb[3 + j] + a.R[3 * i + 2] * Rb[6 + j];
    c.t[i] = a.R[3 * i] * tb[0] + a.R[3 * i + 1] * tb[1] + a.R[3 * i + 2] * tb[2] + a.t[i];
  }
}
static void rot9(const double* R, const double* M, double* out)  // R M
{
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) out[3 * i + j] = R[3 * i] * M[j] + R[3 * i + 1] * M[3 + j] + R[3 * i + 2] * M[6 + j];
}
// T[c * 10 + p]: parameters [m, m c, Ixx, Ixy, Ixz, Iyy, Iyz, Izz] (inertia about the frame origin, frame axes; primitives_impl.h:399-417)
// of a body referred to frame A as a linear function of the same referred to frame B, x_A = R x_B + t
static void fold_param_map(const FoldXf& X, double* T)
{
  const double* R = X.R;
  const double* t = X.t;
  for (int p = 0; p < 10; p++)
  {
    double e[10] = {0};
    e[p] = 1.0;
    const double m = e[0], h[3] = {e[1], e[2], e[3]};
    const double I[9] = {e[4], e[5], e[6], e[5], e[7], e[8], e[6], e[8], e[9]};
    double Rh[3], RI[9], Io[9];
    for (int i = 0; i < 3; i++) Rh[i] = R[3 * i] * h[0] + R[3 * i + 1] * h[1] + R[3 * i + 2] * h[2];
    rot9(R, I, RI);
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) Io[3 * i + j] = RI[3 * i] * R[3 * j] + RI[3 * i + 1] * R[3 * j + 1] + RI[3 * i + 2] * R[3 * j + 2];  // R I R^T
    const double rht = Rh[0] * t[0] + Rh[1] * t[1] + Rh[2] * t[2], tt = t[0] * t[0] + t[1] * t[1] + t[2] * t[2];
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++)
        Io[3 * i + j] += (i == j ? 2.0 * rht + m * tt : 0.0) - (Rh[i] * t[j] + t[i] * Rh[j]) - m * t[i] * t[j];
    const double o[10] = {m, Rh[0] + m * t[0], Rh[1] + m * t[1], Rh[2] + m * t[2], Io[0], Io[1], Io[2], Io[4], Io[5], Io[8]};
    for (int c = 0; c < 10; c++) T[c * 10 + p] = o[c];
  }
}

// Q (row-major, det +1) with Q e_z = ax, ax a unit axis: columns (c0, c1, ax), c0 x c1 = ax.  An axis along a coordinate axis, +-e_i (every
// axis of C6 / C7 and of most URDF arms), gets the exact signed permutation c0 = e_{i+1}, c1 = +-e_{i+2}, so that the folded constants and the
// parameter map are exact (+e_z: Q = I); an oblique axis gets c0 = unit(e_k x ax), k its smallest component, orthonormal to rounding.
// false (Q = I) for an axis that is not a unit vector (a zero axis): that joint keeps its runtime axis.
static bool canonical_frame(const double* ax, double* Q)
{
  for (int k = 0; k < 9; k++) Q[k] = (k % 4 == 0) ? 1.0 : 0.0;
  if (!(std::fabs(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2] - 1.0) <= 1e-12)) return false;
  double c0[3] = {0, 0, 0}, c1[3] = {0, 0, 0};
  int i = -1;
  for (int k = 0; k < 3; k++)
    if ((ax[k] == 1.0 || ax[k] == -1.0) && ax[(k + 1) % 3] == 0.0 && ax[(k + 2) % 3] == 0.0) i = k;
  if (i >= 0)
  {
    c0[(i + 1) % 3] = 1.0;
    c1[(i + 2) % 3] = ax[i];
  }
  else
  {
    int k = 0;
    for (int r = 1; r < 3; r++)
      if (std::fabs(ax[r]) < std::fabs(ax[k])) k = r;
    double e[3] = {0, 0, 0};
    e[k] = 1.0;
    const double x[3] = {e[1] * ax[2] - e[2] * ax[1], e[2] * ax[0] - e[0] * ax[2], e[0] * ax[1] - e[1] * ax[0]};
    const double n = std::sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
    for (int r = 0; r < 3; r++) c0[r] = x[r] / n;
    c1[0] = ax[1] * c0[2] - ax[2] * c0[1];
    c1[1] = ax[2] * c0[0] - ax[0] * c0[2];
    c1[2] = ax[0] * c0[1] - ax[1] * c0[0];
  }
  for (int r = 0; r < 3; r++)
  {
    Q[3 * r] = c0[r];
    Q[3 * r + 1] = c1[r];
    Q[3 * r + 2] = ax[r];
  }
  return true;
}

}  // namespace rdb
// host-only entry for tests: the parameter map of a rigid attachment x_A = R x_B + t (row-major R), T[c * 10 + p]
extern "C" rdb_status rdb_fold_parameter_map(const double* R, const double* t, double* T)
{
  if (!R || !t || !T) return RDB_ERR_INVALID_ARG;
  rdb::FoldXf X;
  for (int k = 0; k < 9; k++) X.R[k] = R[k];
  for (int k = 0; k < 3; k++) X.t[k] = t[k];
  rdb::fold_param_map(X, T);
  return RDB_OK;
}
// host-only entry for tests: the rotation Q (row-major) that turns a link frame so that its revolute axis becomes e_z, Q e_z = axis
extern "C" rdb_status rdb_fold_canonical_frame(const double* axis, double* Q)
{
  if (!axis || !Q) return RDB_ERR_INVALID_ARG;
  return rdb::canonical_frame(axis, Q) ? RDB_OK : RDB_ERR_INVALID_ARG;
}
namespace rdb
{

// (re)builds ch.gram.fold* for the current model (called by every model upload, capi.cu)
cudaError_t fold_chain(ChainHost& ch, bool upload)
{
  GramWorkspace& w = ch.gram;
  if (w.fold_version == ch.model_version) return cudaSuccess;
  const ChainDev<RDB_MAX_JOINTS>& H = ch.host;
  ChainDev<RDB_MAX_JOINTS>& F = w.fold;
  F = ChainDev<RDB_MAX_JOINTS>{};
  F.n_in = H.n_in;
  for (int k = 0; k < 3; k++) F.g[k] = H.g[k];
  std::vector<double> T((size_t)H.nj * 100, 0.0);
  std::vector<int32_t> kof(H.nj, -1);
  FoldXf X{{1, 0, 0, 0, 1, 0, 0, 0, 1}, {0, 0, 0}};
  int K = 0;
  bool rotated = false;  // some Q != I
  for (int l = 0; l < H.nj; l++)
  {
    const JointDev& J = H.joint[l];
    if (J.in < 0)  // never moves: q = 0, T_pc = [A | t]
    {
      FoldXf Y;
      xf_mul(X, J.A, J.t, Y);
      X = Y;
      if (K > 0)
      {
        kof[l] = K - 1;
        fold_param_map(X, &T[(size_t)l * 100]);
        for (int c = 0; c < 10; c++)
          for (int p = 0; p < 10; p++) F.link[K - 1].pi[c] += T[(size_t)l * 100 + c * 10 + p] * H.link[l].pi[p];
      }
      continue;
    }
    JointDev& o = F.joint[K];
    o = J;
    // revolute: the child link in its canonical frame, x_old = Q x_new (prismatic joints keep Q = I)
    double Q[9];
    const bool canon = J.type == RDB_JOINT_REVOLUTE && canonical_frame(J.ax, Q);
    if (!canon) for (int k = 0; k < 9; k++) Q[k] = (k % 4 == 0) ? 1.0 : 0.0;
    double XA[9];
    rot9(X.R, J.A, XA);
    rot9(XA, Q, o.A);  // A' = X.R A Q
    if (canon)
    {
      // ax' = e_z; B' = A' skew(e_z), C' = A' skew(e_z)^2: columns of A' moved, exact (R_pc(q) = A' Rz(q))
      static_assert(REV_AXIS[0] == 0.0 && REV_AXIS[1] == 0.0 && REV_AXIS[2] == 1.0, "Q e_z = axis: the canonical axis is e_z");
      for (int k = 0; k < 3; k++) o.ax[k] = REV_AXIS[k];
      for (int i = 0; i < 3; i++)
      {
        o.B[3 * i] = o.A[3 * i + 1];
        o.B[3 * i + 1] = -o.A[3 * i];
        o.B[3 * i + 2] = 0.0;
        o.C[3 * i] = -o.A[3 * i];
        o.C[3 * i + 1] = -o.A[3 * i + 1];
        o.C[3 * i + 2] = 0.0;
      }
    }
    else
    {
      rot9(X.R, J.B, o.B);
      rot9(X.R, J.C, o.C);
    }
    for (int i = 0; i < 3; i++)
    {
      o.t[i] = X.R[3 * i] * J.t[0] + X.R[3 * i + 1] * J.t[1] + X.R[3 * i + 2] * J.t[2] + X.t[i];
      o.axp[i] = X.R[3 * i] * J.axp[0] + X.R[3 * i + 1] * J.axp[1] + X.R[3 * i + 2] * J.axp[2];
    }
    // the frame change of the link is a rigid attachment {Q^T, 0} of its own body: parameters T pi, and everything attached behind it is
    // referred to the new frame through X
    FoldXf Y{{Q[0], Q[3], Q[6], Q[1], Q[4], Q[7], Q[2], Q[5], Q[8]}, {0, 0, 0}};
    fold_param_map(Y, &T[(size_t)l * 100]);
    for (int c = 0; c < 10; c++)
    {
      F.link[K].pi[c] = 0.0;
      for (int p = 0; p < 10; p++) F.link[K].pi[c] += T[(size_t)l * 100 + c * 10 + p] * H.link[l].pi[p];
    }
    rotated = rotated || (canon && !(Q[0] == 1.0 && Q[4] == 1.0 && Q[8] == 1.0));
    kof[l] = K;
    K++;
    X = Y;
  }
  F.nj = K;
  w.fold_identity = (K == H.nj) && !rotated;
  if (upload && !w.fold_identity && K > 0)
  {
    // the caller (upload_model) has synchronised the device: no kernel still reads the fold maps, so they may be freed and rewritten here
    cudaError_t e = w.fold_dev.grow(sizeof(double) * T.size() + sizeof(int32_t) * kof.size(), nullptr);
    if (e != cudaSuccess) return e;
    const FoldMaps fm = fold_maps(ch);
    e = cudaMemcpy(fm.T, T.data(), sizeof(double) * T.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
    e = cudaMemcpy(fm.kof, kof.data(), sizeof(int32_t) * kof.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return e;
  }
  if (upload) w.fold_version = ch.model_version;
  return cudaSuccess;
}

}  // namespace rdb
