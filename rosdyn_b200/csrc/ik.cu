// ik.cu -- batched local inverse kinematics: Chain::computeLocalIk / computeWeigthedLocalIk (primitives_impl.h:1398-1468).
//
// The reference iterates, per pose,   e = getFrameDistance(T_target, T(sol))            (frame_distance.h:44-49)
//                                     if |w . e| < toll: done
//                                     dq = argmin 1/2 dq^T (J^T W J) dq - (J^T W e)^T dq   s.t.  q_min <= sol + dq <= q_max
//                                     sol += dq
// until a WALL-CLOCK budget (ros::Duration) runs out, the QP being solved by Eigen::solve_quadprog of the un-vendored eigen_matrix_utils
// (Goldfarb-Idnani; its answer is the unique minimiser of a strictly convex QP).  Here: one thread per target pose, an ITERATION budget
// instead of the wall clock, and the box-constrained QP solved exactly by a primal active-set method on the (at most 8) input joints --
// the same statement of the problem, not the same code path; the CPU oracle restates the loop the same way (oracle/rosdyn_oracle.c).
// Not a throughput kernel: runtime loops over the chain, model read from global memory.
#include <cuda_runtime.h>

#include "launch.h"
#include "spatial.cuh"

namespace rdb
{

constexpr int IK_MAXN = RDB_IK_MAX_INPUTS;

// Eigen::AngleAxisd(Eigen::Matrix3d) = AngleAxis(Quaternion(m)): angle * axis of the rotation m (row-major)
__device__ void angle_axis_vec(const double* m, double* out)
{
  double q[4];  // x y z w
  double t = m[0] + m[4] + m[8];
  if (t > 0.0)
  {
    t = sqrt(t + 1.0);
    q[3] = 0.5 * t;
    t = 0.5 / t;
    q[0] = (m[7] - m[5]) * t;
    q[1] = (m[2] - m[6]) * t;
    q[2] = (m[3] - m[1]) * t;
  }
  else
  {
    int i = 0;
    if (m[4] > m[0]) i = 1;
    if (m[8] > m[4 * i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrt(m[4 * i] - m[4 * j] - m[4 * k] + 1.0);
    q[i] = 0.5 * t;
    t = 0.5 / t;
    q[3] = (m[3 * k + j] - m[3 * j + k]) * t;
    q[j] = (m[3 * j + i] + m[3 * i + j]) * t;
    q[k] = (m[3 * k + i] + m[3 * i + k]) * t;
  }
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2]);
  if (n != 0.0)
  {
    const double angle = 2.0 * atan2(n, fabs(q[3]));
    if (q[3] < 0.0) n = -n;
    for (int c = 0; c < 3; c++) out[c] = angle * (q[c] / n);
  }
  else
    out[0] = out[1] = out[2] = 0.0;
}

// min 1/2 x^T H x + f^T x,  lo <= x <= hi  (H symmetric positive semi-definite, n <= IK_MAXN): primal active-set method.
// Free variables move along the Newton direction of the free block until the first bound blocks; at a free-block minimiser the bound
// with the most wrong-signed multiplier is released.  Directions in which H is (numerically) singular are left where they are.
__device__ void box_qp(int n, const double* H, const double* f, const double* lo, const double* hi, double* x)
{
  int state[IK_MAXN];  // 0 free, 1 at lo, 2 at hi, 3 pinned (lo >= hi)
  double hmx = 0.0, fmx = 0.0;
  for (int i = 0; i < n; i++)
  {
    hmx = fmax(hmx, H[i * n + i]);
    fmx = fmax(fmx, fabs(f[i]));
    x[i] = 0.0;  // start from "no move", clamped into the box (a seed outside its limits is pulled back by the bounds)
    state[i] = 0;
    if (lo[i] >= hi[i])
    {
      x[i] = lo[i];
      state[i] = 3;
    }
    else if (x[i] <= lo[i])
    {
      x[i] = lo[i];
      state[i] = 1;
    }
    else if (x[i] >= hi[i])
    {
      x[i] = hi[i];
      state[i] = 2;
    }
  }
  const double ptol = 1e-13 * hmx, gtol = 1e-12 * (fmx + hmx);
  for (int it = 0; it < 6 * IK_MAXN + 8; it++)
  {
    double g[IK_MAXN], d[IK_MAXN], L[IK_MAXN * IK_MAXN];
    int idx[IK_MAXN], m = 0;
    for (int i = 0; i < n; i++)
    {
      double s = f[i];
      for (int k = 0; k < n; k++) s += H[i * n + k] * x[k];
      g[i] = s;
      d[i] = 0.0;
      if (state[i] == 0) idx[m++] = i;
    }
    // Cholesky of the free block (pivot guard: a singular direction keeps d = 0), then L L^T d = -g
    bool ok[IK_MAXN];
    for (int a = 0; a < m; a++)
    {
      for (int b = 0; b <= a; b++)
      {
        double s = H[idx[a] * n + idx[b]];
        for (int k = 0; k < b; k++) s -= L[a * IK_MAXN + k] * L[b * IK_MAXN + k];
        if (a == b)
        {
          ok[a] = s > ptol;
          L[a * IK_MAXN + a] = ok[a] ? sqrt(s) : 1.0;
          if (!ok[a])
            for (int k = 0; k < a; k++) L[a * IK_MAXN + k] = 0.0;
        }
        else
          L[a * IK_MAXN + b] = ok[b] ? s / L[b * IK_MAXN + b] : 0.0;
      }
    }
    double y[IK_MAXN];
    for (int a = 0; a < m; a++)
    {
      double s = ok[a] ? -g[idx[a]] : 0.0;
      for (int k = 0; k < a; k++) s -= L[a * IK_MAXN + k] * y[k];
      y[a] = s / L[a * IK_MAXN + a];
    }
    for (int a = m - 1; a >= 0; a--)
    {
      double s = y[a];
      for (int k = a + 1; k < m; k++) s -= L[k * IK_MAXN + a] * d[idx[k]];
      d[idx[a]] = ok[a] ? s / L[a * IK_MAXN + a] : 0.0;
    }
    // longest feasible step along d
    double alpha = 1.0;
    int blocking = -1, bstate = 0;
    for (int a = 0; a < m; a++)
    {
      const int i = idx[a];
      if (d[i] > 0.0 && x[i] + d[i] > hi[i])
      {
        const double s = (hi[i] - x[i]) / d[i];
        if (s < alpha)
        {
          alpha = s;
          blocking = i;
          bstate = 2;
        }
      }
      else if (d[i] < 0.0 && x[i] + d[i] < lo[i])
      {
        const double s = (lo[i] - x[i]) / d[i];
        if (s < alpha)
        {
          alpha = s;
          blocking = i;
          bstate = 1;
        }
      }
    }
    for (int a = 0; a < m; a++) x[idx[a]] += alpha * d[idx[a]];
    if (blocking >= 0)
    {
      x[blocking] = bstate == 1 ? lo[blocking] : hi[blocking];
      state[blocking] = bstate;
      continue;
    }
    // minimiser of the free block reached: multipliers of the active bounds
    int worst = -1;
    double wv = gtol;
    for (int i = 0; i < n; i++)
    {
      if (state[i] != 1 && state[i] != 2) continue;
      double s = f[i];
      for (int k = 0; k < n; k++) s += H[i * n + k] * x[k];
      const double viol = state[i] == 1 ? -s : s;  // at lo the gradient must be >= 0, at hi <= 0
      if (viol > wv)
      {
        wv = viol;
        worst = i;
      }
    }
    if (worst < 0) break;
    state[worst] = 0;
  }
}

struct IkParams
{
  double q_min[IK_MAXN], q_max[IK_MAXN], weight[6];
  double tol;
  int32_t max_iter, weighted;
};

__global__ void __launch_bounds__(128) ik_kernel(const ChainDev<RDB_MAX_JOINTS>* __restrict__ C, const __grid_constant__ IkParams prm, int64_t n,
                                                 int64_t ld, const double* __restrict__ target, const double* __restrict__ seed,
                                                 double* __restrict__ sol_out, int32_t* __restrict__ status, int32_t* __restrict__ iters,
                                                 double* __restrict__ err_out)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int nj = C->nj, n_in = C->n_in;
  double Ta[12];
  for (int k = 0; k < 12; k++) Ta[k] = target[(int64_t)k * ld + i];
  const double Ra[9] = {Ta[0], Ta[1], Ta[2], Ta[4], Ta[5], Ta[6], Ta[8], Ta[9], Ta[10]};
  const double pa[3] = {Ta[3], Ta[7], Ta[11]};
  double sol[IK_MAXN];
  for (int r = 0; r < n_in; r++) sol[r] = seed[(int64_t)r * ld + i];
  int done = 0, it = 0;
  double en = 0.0;
  for (;; it++)
  {
    // computeFrames + computeScrews + getJacobian at sol (PI.h:863-882, 927-949)
    double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    V3 p = v3(0, 0, 0);
    V3 ab[IK_MAXN], pj[IK_MAXN];
    int ty[IK_MAXN];
    for (int r = 0; r < n_in; r++) ty[r] = RDB_JOINT_FIXED;
    for (int l = 0; l < nj; l++)
    {
      const JointDev& J = C->joint[l];
      const int r = J.in;
      double Rpc[9], Rn[9];
      V3 t;
      joint_transform(J, r >= 0 ? sol[r] : 0.0, Rpc, t);
      const V3 axb = rot(R, v3(J.axp));
      p = p + rot(R, t);
      mul33(R, Rpc, Rn);
      for (int k = 0; k < 9; k++) R[k] = Rn[k];
      if (r >= 0)
      {
        ab[r] = axb;
        pj[r] = p;
        ty[r] = J.type;
      }
    }
    double Jm[6 * IK_MAXN];  // column-major 6 x n_in
    for (int r = 0; r < n_in; r++)
    {
      V3 lin = v3(0, 0, 0), ang = v3(0, 0, 0);
      if (ty[r] == RDB_JOINT_REVOLUTE)
      {
        lin = cross(ab[r], p - pj[r]);
        ang = ab[r];
      }
      else if (ty[r] == RDB_JOINT_PRISMATIC)
        lin = ab[r];
      Jm[6 * r + 0] = lin.x;
      Jm[6 * r + 1] = lin.y;
      Jm[6 * r + 2] = lin.z;
      Jm[6 * r + 3] = ang.x;
      Jm[6 * r + 4] = ang.y;
      Jm[6 * r + 5] = ang.z;
    }
    // getFrameDistance(T_target, T(sol)) (frame_distance.h:44-49): [p_a - p_b ; -R_a (angle axis)(R_a^T R_b)]
    double e[6], Rab[9], aa[3];
    e[0] = pa[0] - p.x;
    e[1] = pa[1] - p.y;
    e[2] = pa[2] - p.z;
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) Rab[3 * a + b] = Ra[a] * R[b] + Ra[3 + a] * R[3 + b] + Ra[6 + a] * R[6 + b];
    angle_axis_vec(Rab, aa);
    for (int a = 0; a < 3; a++) e[3 + a] = -(Ra[3 * a] * aa[0] + Ra[3 * a + 1] * aa[1] + Ra[3 * a + 2] * aa[2]);
    en = 0.0;
    for (int k = 0; k < 6; k++)
    {
      const double we = prm.weighted ? prm.weight[k] * e[k] : e[k];
      en += we * we;
    }
    en = sqrt(en);
    if (en < prm.tol)
    {
      done = 1;
      break;
    }
    if (it >= prm.max_iter) break;
    double H[IK_MAXN * IK_MAXN], f[IK_MAXN], lo[IK_MAXN], hi[IK_MAXN], dq[IK_MAXN];
    for (int a = 0; a < n_in; a++)
    {
      for (int b = 0; b < n_in; b++)
      {
        double s = 0.0;
        for (int k = 0; k < 6; k++) s += Jm[6 * a + k] * (prm.weighted ? prm.weight[k] : 1.0) * Jm[6 * b + k];
        H[a * n_in + b] = s;
      }
      double s = 0.0;
      for (int k = 0; k < 6; k++) s += Jm[6 * a + k] * (prm.weighted ? prm.weight[k] : 1.0) * e[k];
      f[a] = -s;
      lo[a] = prm.q_min[a] - sol[a];
      hi[a] = prm.q_max[a] - sol[a];
    }
    box_qp(n_in, H, f, lo, hi, dq);
    for (int a = 0; a < n_in; a++) sol[a] += dq[a];
  }
  for (int r = 0; r < n_in; r++) sol_out[(int64_t)r * ld + i] = sol[r];
  if (status) status[i] = done;
  if (iters) iters[i] = it;
  if (err_out) err_out[i] = en;
}

cudaError_t launch_ik(const ChainHost& ch, int64_t n, int64_t ld, const double* target, const double* seed, const double* q_min,
                      const double* q_max, const double* weight, double tol, int max_iter, double* sol, int32_t* status, int32_t* iters,
                      double* err, cudaStream_t st)
{
  if (n <= 0) return cudaSuccess;
  IkParams prm{};
  for (int r = 0; r < ch.host.n_in && r < IK_MAXN; r++)
  {
    prm.q_min[r] = q_min ? q_min[r] : -1e10;  // Joint defaults without <limit> (PI.h:92-93)
    prm.q_max[r] = q_max ? q_max[r] : 1e10;
  }
  prm.weighted = weight != nullptr;
  for (int k = 0; k < 6; k++) prm.weight[k] = weight ? weight[k] : 1.0;
  prm.tol = tol;
  prm.max_iter = max_iter;
  ik_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(ch.dev.get(), prm, n, ld, target, seed, sol, status, iters, err);
  count_launch();
  return cudaGetLastError();
}

}  // namespace rdb
