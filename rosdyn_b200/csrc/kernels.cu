// kernels.cu -- hand-written sm_100a fp64 kernels for the rosdyn::Chain hot path.
//
// One thread walks the serial chain of one sample.  q/Dq/DDq/DDDq are read from SoA planes (one coalesced
// 8-byte load per lane per plane, streamed), every result is written to SoA planes (coalesced streaming
// stores), the model lives in the kernel-parameter constant bank (chain_dev.h).  Two families:
//
//   * kin_kernel      -- base-frame walker: everything the reference returns in the base frame
//                        (frames, Jacobian, twist / acceleration / jerk recursions, RNEA torque);
//                        replaces computeFrames/computeScrews/getJacobian/getTwist/getDTwist*/getDDTwist*/
//                        getWrench/getJointTorque  (primitives_impl.h:863-1293).
//   * dyn_kernel      -- link-frame walker for the dynamics that only need scalars per joint:
//                        inertial regressor (getRegressor, primitives_impl.h:1295-1355), RNEA torque, the
//                        joint inertia matrix (getJointInertia, primitives_impl.h:1357-1379) and forward dynamics
//                        (both of the last two in one walk, then an in-register Cholesky solve).
//
// Both are FORWARD-ONLY: instead of the reference's backward wrench pass they carry, for every joint j
// already passed, its unit twist ("Jacobian column") expressed at the current link, and project each
// link's wrench / wrench-regressor on it.  That keeps the live state small enough for registers
// (no per-link frame storage) and lets every output leave the thread the moment it is computed.
#include <cuda_runtime.h>

#include "launch.h"
#include "spatial.cuh"

namespace rdb
{

#define RDB_BLOCK 128
#ifndef RDB_KIN_MINB
#define RDB_KIN_MINB 4  // min CTAs/SM asked of ptxas (register cap 65536/(128*MINB) = 128): measured on B200, config 2 runs
                        // 2.59 -> 3.20 G samples/s and the jerk walker 5.22 -> 5.51 vs. the uncapped 244-register build
#endif
#ifndef RDB_DYN_MINB
#define RDB_DYN_MINB 4  // link-frame walker, torque / inertia modes (FP64-pipe bound): <= 128 registers
#endif
#ifndef RDB_FD_MINB
#define RDB_FD_MINB 3  // forward dynamics (h and M accumulators, then the solve): <= 168 registers, some spills; measured on B200 over 1e8
                       // samples, C6 / C7 4.45 / 3.27 G samples/s vs 3.95 / 3.20 at 2 (255 registers) and 4.05 / 2.00 at 4 (128, power-capped)
                       // (profiles/fd_ptxas.txt)
#endif
#ifndef RDB_REG_MINB
#define RDB_REG_MINB 3  // regressor modes (HBM-write bound): <= 168 registers, measured 0.92 -> 0.96 (C6) / 0.95 -> 0.99 (C7) of HBM peak vs. 4
#endif

template <int NJ_T>
struct Cap
{
  static constexpr int value = NJ_T > 0 ? NJ_T : RDB_MAX_JOINTS;
};

// =============================================================================================================
// link-frame walker
// =============================================================================================================
enum : int
{
  DYN_REGRESSOR = 1,  // write Phi
  DYN_TORQUE = 2,     // write tau
  DYN_INERTIA = 4,    // write M
  DYN_FD = 8          // forward dynamics: walk with DDq = 0 accumulating h and M, solve M ddq = tau_in - h, write ddq (into out.tau) and info
};

// Link-frame state of the walker after joint l: twist (v,w), acceleration (a,al) and gravity g of link l in link-l
// axes at the link-l origin, and the unit twists (U[j],S[j]) of all joints j <= l at the same point/axes.
// REV (unrolled torque / inertia kernels on the folded chain): every joint is revolute, so the joint type is a compile-time fact -- no type
// selects and the linear half of the joint screws (an exact zero) is never multiplied
// REC (regressor modes, RDB_LAYOUT_EIGEN): the 10 n_act values a link contributes to a sample's record (a contiguous piece of the column-major
// n_act x 10 nJ matrix) are staged in a per-warp shared-memory tile [32 samples][10 n_act + 1] and written out row by row, 32 lanes on
// consecutive doubles -- full sectors instead of one 8-byte piece of 32 different lines per store instruction (0.21 -> see DESIGN.md).
// `stage` is the warp's tile, `i_live` the number of samples of this warp that exist (all 32 lanes take part in the cooperative copies).
template <int NJ_T, int MODE, bool REV = false, bool REC = false, class ChainT>
__device__ __forceinline__ void dyn_body(const ChainT& C, const SamplesDev& in, const DynOutDev& out, int64_t i, double* stage = nullptr,
                                         int i_live = 32)
{
  // element (plane p, sample i) of an output array: base + p * ld_out + i * ss (SoA planes: ld_out = ld, ss = 1; Eigen records: ld_out = 1)
  double* __restrict__ const phi = out.phi + i * out.ss_phi;
  double* __restrict__ const tau_out = out.tau;
  double* __restrict__ const M_out = out.M;
  const int64_t ld_out = out.ps, i_tau = i * out.ss_tau, i_M = i * out.ss_M;
  constexpr int CAP = Cap<NJ_T>::value;
  const int nj = NJ_T > 0 ? NJ_T : C.nj;
  const int n_in = C.n_in;
  constexpr bool kReg = (MODE & DYN_REGRESSOR) != 0;
  constexpr bool kFd = (MODE & DYN_FD) != 0;
  constexpr bool kTau = (MODE & (DYN_TORQUE | DYN_FD)) != 0;
  constexpr bool kInr = (MODE & (DYN_INERTIA | DYN_FD)) != 0;
  constexpr bool kDyn = kReg || kTau;  // needs velocities / accelerations
  const int lane_r = threadIdx.x & 31;
  const int W = 10 * n_in, RS = W + 1;                // REC: doubles of one link block of a record, tile row stride (odd: conflict free)
  double* const my_row = REC ? stage + lane_r * RS : nullptr;
  if (REC)
  {
    for (int c = 0; c < W; c++) my_row[c] = 0.0;      // rows of inputs that no chain joint feeds stay zero (never written below)
  }

  V3 U[CAP], S[CAP];
  double tau[kTau ? CAP : 1];
  double M[kInr ? CAP * (CAP + 1) / 2 : 1];
  if (kInr)
  {
#pragma unroll
    for (int k = 0; k < (kInr ? CAP * (CAP + 1) / 2 : 1); k++)
      if (NJ_T > 0 || k < nj * (nj + 1) / 2) M[k] = 0.0;
  }

  V3 v = v3(0, 0, 0), w = v3(0, 0, 0), a = v3(0, 0, 0), al = v3(0, 0, 0);
  V3 g = v3(C.g);

  // unrolled instantiations: every angle is loaded and its sin / cos evaluated up front (branch free), see trig_all
  constexpr int NT = NJ_T > 0 ? NJ_T : 1;
  double qv[NT], sv[NT], cv[NT];
  if (NJ_T > 0)
  {
#pragma unroll
    for (int l = 0; l < NT; l++) qv[l] = ld_in(in.q, C.joint[l].in, in.ld, i);
    trig_all<NT>(qv, sv, cv);
  }

  // regressor modes (HBM bound): the rates are all pulled into L2 up front (no register held), then loaded one link ahead of their use;
  // measured slower for the FP64-bound torque walker (9.0 -> 8.5 G samples/s), which keeps the plain per-link loads
  double dq_nx = 0.0, ddq_nx = 0.0;
  if (NJ_T > 0 && kReg)
  {
#pragma unroll
    for (int l = 1; l < NT; l++)
    {
      prefetch_in(in.dq, C.joint[l].in, in.ld, i);
      prefetch_in(in.ddq, C.joint[l].in, in.ld, i);
    }
    dq_nx = ld_in(in.dq, C.joint[0].in, in.ld, i);
    ddq_nx = ld_in(in.ddq, C.joint[0].in, in.ld, i);
  }

#pragma unroll
  for (int l = 0; l < (NJ_T > 0 ? NJ_T : nj); l++)
  {
    const JointDev& J = C.joint[l];
    double R[9];
    V3 t;
    if (REV)
    {
      t = v3(J.t);
      const double c1 = 1.0 - cv[NJ_T > 0 ? l : 0];
#pragma unroll
      for (int k = 0; k < 9; k++) R[k] = fma(c1, J.C[k], fma(sv[NJ_T > 0 ? l : 0], J.B[k], J.A[k]));
    }
    else if (NJ_T > 0)
      joint_transform_sc(J, qv[NJ_T > 0 ? l : 0], sv[NJ_T > 0 ? l : 0], cv[NJ_T > 0 ? l : 0], R, t);
    else
      joint_transform(J, ld_in(in.q, J.in, in.ld, i), R, t);

    // child-frame screw of joint l: [0;ax] revolute, [ax;0] prismatic, 0 fixed (R_pc^T axis_p == axis_j)
    const V3 axj = v3(J.ax);
    const V3 su = (!REV && J.type == RDB_JOINT_PRISMATIC) ? axj : v3(0, 0, 0);
    const V3 ss = (REV || J.type == RDB_JOINT_REVOLUTE) ? axj : v3(0, 0, 0);

    if (kDyn)
    {
      double dql, ddql;
      if (NJ_T > 0 && kReg)  // requested one link earlier
      {
        dql = dq_nx;
        ddql = ddq_nx;
        if (l + 1 < NJ_T)
        {
          const int inn = C.joint[l + 1 < CAP ? l + 1 : 0].in;
          dq_nx = ld_in(in.dq, inn, in.ld, i);
          ddq_nx = ld_in(in.ddq, inn, in.ld, i);
        }
      }
      else
      {
        dql = ld_in(in.dq, J.in, in.ld, i);
        ddql = kFd ? 0.0 : ld_in(in.ddq, J.in, in.ld, i);
      }
      // getTwist (primitives_impl.h:1007-1008) and getDTwist (1116-1117) moved to the child frame
      v = rotT(R, cross_add(v, w, t));
      w = rotT(R, w);
      a = rotT(R, cross_add(a, al, t));
      al = rotT(R, al);
      g = rotT(R, g);
      // forward dynamics walks with DDq = 0 (the bias torque h): its DDq terms are left out, not multiplied by zero
      if (REV)
      {
        w = axpy(w, ss, dql);
        a = axpy(a, cross(v, ss), dql);
        al = axpy(al, cross(w, ss), dql);
        if (!kFd) al = axpy(al, ss, ddql);
      }
      else
      {
        v = axpy(v, su, dql);
        w = axpy(w, ss, dql);
        // (v x s) Dq + s DDq, spatial cross of spacevect_algebra.h:88-93
        const V3 xl = cross_add(cross(w, su), v, ss);
        const V3 xa = cross(w, ss);
        a = axpy(a, xl, dql);
        al = axpy(al, xa, dql);
        if (!kFd)
        {
          a = axpy(a, su, ddql);
          al = axpy(al, ss, ddql);
        }
      }
    }

    // unit twists of the joints already passed, moved to link l
#pragma unroll
    for (int j = 0; j < l; j++)
    {
      U[j] = rotT(R, cross_add(U[j], S[j], t));
      S[j] = rotT(R, S[j]);
    }
    U[l] = su;
    S[l] = ss;
    if (kTau) tau[l] = 0.0;

    const double* P = C.link[l].pi;

    if (kReg)
    {
      // Closed form of the wrench regressor of link l in link axes (primitives_impl.h:1324-1339):
      //   col m    : [ fm ; 0 ]                         fm = a + w x v - g
      //   col mc_k : [ (al^ + w^ w^) e_k ; e_k x fm ]
      //   col I_p  : [ 0 ; E_p al + w x (E_p w) ]
      // projected on the unit twist (u,s) of joint j (primitives_impl.h:1341-1347):
      //   m   : u.fm
      //   mc  : u x al + w x (w x u) + fm x s          (vector of the three mc columns)
      //   I_p : s.(E_p al) + (s x w).(E_p w)
      const V3 fm = cross_add(a - g, w, v);
      const int64_t colbase = (int64_t)10 * l * n_in;
#pragma unroll
      for (int j = 0; j <= l; j++)
      {
        const int r = C.joint[j].in;
        const V3 u = U[j], s = S[j];
        const double e0 = dot(u, fm);
        const V3 wu = cross(w, u);
        const V3 h = cross_add(cross_add(cross(u, al), w, wu), fm, s);
        const V3 rho = cross(s, w);
        const double e4 = fma(s.x, al.x, rho.x * w.x);
        const double e5 = fma(s.x, al.y, fma(s.y, al.x, fma(rho.x, w.y, rho.y * w.x)));
        const double e6 = fma(s.x, al.z, fma(s.z, al.x, fma(rho.x, w.z, rho.z * w.x)));
        const double e7 = fma(s.y, al.y, rho.y * w.y);
        const double e8 = fma(s.y, al.z, fma(s.z, al.y, fma(rho.y, w.z, rho.z * w.y)));
        const double e9 = fma(s.z, al.z, rho.z * w.z);
        if (kTau)
        {
          double tj = tau[j];
          tj = fma(e0, P[0], tj);
          tj = fma(h.x, P[1], tj);
          tj = fma(h.y, P[2], tj);
          tj = fma(h.z, P[3], tj);
          tj = fma(e4, P[4], tj);
          tj = fma(e5, P[5], tj);
          tj = fma(e6, P[6], tj);
          tj = fma(e7, P[7], tj);
          tj = fma(e8, P[8], tj);
          tj = fma(e9, P[9], tj);
          tau[j] = tj;
        }
        if (r >= 0)
        {
          if (REC)
          {
            double* o = my_row + r;
            o[0] = e0;
            o[n_in] = h.x;
            o[2 * n_in] = h.y;
            o[3 * n_in] = h.z;
            o[4 * n_in] = e4;
            o[5 * n_in] = e5;
            o[6 * n_in] = e6;
            o[7 * n_in] = e7;
            o[8 * n_in] = e8;
            o[9 * n_in] = e9;
          }
          else
          {
            double* o = phi + (colbase + r) * ld_out;
            const int64_t st = (int64_t)n_in * ld_out;
            __stcs(o, e0);
            __stcs(o + st, h.x);
            __stcs(o + 2 * st, h.y);
            __stcs(o + 3 * st, h.z);
            __stcs(o + 4 * st, e4);
            __stcs(o + 5 * st, e5);
            __stcs(o + 6 * st, e6);
            __stcs(o + 7 * st, e7);
            __stcs(o + 8 * st, e8);
            __stcs(o + 9 * st, e9);
          }
        }
      }
      // rows of the joints after link l are structural zeros of this column block (exact 0.0)
#pragma unroll
      for (int j = l + 1; j < (NJ_T > 0 ? NJ_T : nj); j++)
      {
        const int r = C.joint[j].in;
        if (r >= 0)
        {
          if (REC)
          {
#pragma unroll
            for (int p = 0; p < 10; p++) my_row[p * n_in + r] = 0.0;
          }
          else
          {
            double* o = phi + (colbase + r) * ld_out;
            const int64_t st = (int64_t)n_in * ld_out;
#pragma unroll
            for (int p = 0; p < 10; p++) __stcs(o + p * st, 0.0);
          }
        }
      }
      if (REC)
      {
        // the warp's 32 record pieces of this link leave together: sample s -> out.phi + (i - lane + s) * ss_phi + 10 l n_act + [0, W)
        __syncwarp();
        const int64_t i0 = __shfl_sync(0xffffffffu, i, 0);  // lane 0 always holds a live sample: the warp's first
        double* const base = out.phi + i0 * out.ss_phi + colbase;
        for (int srow = 0; srow < i_live; srow++)
        {
          const double* src = stage + srow * RS;
          double* dst = base + (int64_t)srow * out.ss_phi;
          for (int c = lane_r; c < W; c += 32) __stcs(dst + c, src[c]);
        }
        __syncwarp();
      }
    }
    else if (kTau)
    {
      // RNEA wrench of link l about its origin in link axes (primitives_impl.h:1240-1250; gravity folded into a):
      //   h(x,y) = I_cc [x;y] = [ m x + y x mc ; mc x x + I0 y ]
      //   f = h_lin(a-g, al) + w x h_lin(v,w) ;  n = h_ang(a-g, al) + w x h_ang(v,w) + v x h_lin(v,w)
      const V3 mc = v3(P[1], P[2], P[3]);
      const V3 ag = a - g;
      const V3 hl1 = cross_add(ag * P[0], al, mc);
      const V3 hl2 = cross_add(v * P[0], w, mc);
      const V3 Ial = v3(fma(P[4], al.x, fma(P[5], al.y, P[6] * al.z)), fma(P[5], al.x, fma(P[7], al.y, P[8] * al.z)),
                        fma(P[6], al.x, fma(P[8], al.y, P[9] * al.z)));
      const V3 Iw = v3(fma(P[4], w.x, fma(P[5], w.y, P[6] * w.z)), fma(P[5], w.x, fma(P[7], w.y, P[8] * w.z)),
                       fma(P[6], w.x, fma(P[8], w.y, P[9] * w.z)));
      const V3 ha1 = cross_add(Ial, mc, ag);
      const V3 ha2 = cross_add(Iw, mc, v);
      const V3 f = cross_add(hl1, w, hl2);
      const V3 n = cross_add(cross_add(ha1, w, ha2), v, hl2);
#pragma unroll
      for (int j = 0; j <= l; j++) tau[j] += (REV && j == l) ? dot(S[j], n) : dot(U[j], f) + dot(S[j], n);
    }

    if (kInr)
    {
      // M += J_l^T I_cc(l) J_l with J_l = unit twists at link l in link axes (primitives_impl.h:1366-1375)
      const V3 mc = v3(P[1], P[2], P[3]);
#pragma unroll
      for (int j = 0; j <= l; j++)
      {
        const V3 u = U[j], s = S[j];
        const bool own = REV && j == l;  // u == 0 exactly
        const V3 hl = own ? cross(s, mc) : cross_add(u * P[0], s, mc);
        const V3 Is = v3(fma(P[4], s.x, fma(P[5], s.y, P[6] * s.z)), fma(P[5], s.x, fma(P[7], s.y, P[8] * s.z)),
                         fma(P[6], s.x, fma(P[8], s.y, P[9] * s.z)));
        const V3 ha = own ? Is : cross_add(Is, mc, u);
#pragma unroll
        for (int k = 0; k <= j; k++) M[j * (j + 1) / 2 + k] += (own && k == j) ? dot(S[k], ha) : dot(U[k], hl) + dot(S[k], ha);
      }
    }
  }

  if (kTau && !kFd)
  {
#pragma unroll
    for (int j = 0; j < (NJ_T > 0 ? NJ_T : nj); j++)
    {
      const int r = C.joint[j].in;
      if (r >= 0 && (!REC || lane_r < i_live)) st_out(tau_out, r, ld_out, i_tau, tau[j]);
    }
  }
  if (kFd)
  {
    // Forward dynamics: tau[] holds h(q, Dq) (the walk ran with DDq = 0) and M[] the packed lower triangle of the joint inertia matrix.
    // Joints that feed no input, and fixed joints, are locked: their row / column becomes the identity's and their right-hand side zero, so
    // they drop out (ddq = 0 exactly).  M ddq = tau_in - h is solved in place: Cholesky M = L L^T row by row (L_jk over M_jk, the diagonal
    // slot keeps 1 / L_jj), then L y = b and L^T ddq = y over tau[].
    const int n = NJ_T > 0 ? NJ_T : nj;
#pragma unroll
    for (int j = 0; j < n; j++)
    {
      const int rj = C.joint[j].in;
      const bool lock_j = rj < 0 || (!REV && C.joint[j].type == RDB_JOINT_FIXED);
      tau[j] = lock_j ? 0.0 : ld_in(out.tau_in, rj, in.ld, i) - tau[j];
#pragma unroll
      for (int k = 0; k <= j; k++)
        if (lock_j || C.joint[k].in < 0 || (!REV && C.joint[k].type == RDB_JOINT_FIXED)) M[j * (j + 1) / 2 + k] = j == k ? 1.0 : 0.0;
    }
    bool ok = true;
#pragma unroll
    for (int j = 0; j < n; j++)
    {
      const int jj = j * (j + 1) / 2;
#pragma unroll
      for (int k = 0; k < j; k++)
      {
        const int kk = k * (k + 1) / 2;
        double s = M[jj + k];
#pragma unroll
        for (int m = 0; m < k; m++) s = fma(-M[jj + m], M[kk + m], s);
        M[jj + k] = s * M[kk + k];
      }
      double d = M[jj + j];
#pragma unroll
      for (int m = 0; m < j; m++) d = fma(-M[jj + m], M[jj + m], d);
      ok = ok && d > 0.0 && isfinite(d);  // a NaN pivot fails the first test
      M[jj + j] = rsqrt(d);
    }
#pragma unroll
    for (int j = 0; j < n; j++)
    {
      const int jj = j * (j + 1) / 2;
      double y = tau[j];
#pragma unroll
      for (int m = 0; m < j; m++) y = fma(-M[jj + m], tau[m], y);
      tau[j] = y * M[jj + j];
    }
#pragma unroll
    for (int j = n - 1; j >= 0; j--)
    {
      double x = tau[j];
#pragma unroll
      for (int m = j + 1; m < n; m++) x = fma(-M[m * (m + 1) / 2 + j], tau[m], x);
      tau[j] = x * M[j * (j + 1) / 2 + j];
    }
    if (ok)
    {
#pragma unroll
      for (int j = 0; j < n; j++)
      {
        const int r = C.joint[j].in;
        if (r >= 0) st_out(tau_out, r, ld_out, i_tau, tau[j]);
      }
    }
    else
      for (int r = 0; r < n_in; r++) st_out(tau_out, r, ld_out, i_tau, __longlong_as_double(0x7ff8000000000000ll));  // every component NaN
    if (out.info) __stcs(out.info + i, ok ? 0 : 1);
  }
  if (kInr && !kFd)
  {
#pragma unroll
    for (int j = 0; j < (NJ_T > 0 ? NJ_T : nj); j++)
#pragma unroll
      for (int k = 0; k <= j; k++)
      {
        const int rj = C.joint[j].in, rk = C.joint[k].in;
        if (rj >= 0 && rk >= 0)
        {
          const double m = M[j * (j + 1) / 2 + k];
          st_out(M_out, (int64_t)rj * n_in + rk, ld_out, i_M, m);
          if (j != k) st_out(M_out, (int64_t)rk * n_in + rj, ld_out, i_M, m);
        }
      }
  }
}

template <int NJ, int MODE, bool REV = false, bool REC = false>
__global__ void __launch_bounds__(RDB_BLOCK, (MODE & DYN_REGRESSOR) ? RDB_REG_MINB : ((MODE & DYN_FD) ? RDB_FD_MINB : RDB_DYN_MINB))
    dyn_kernel(const __grid_constant__ ChainDev<NJ> C, const SamplesDev in, const DynOutDev out)
{
  const int64_t i = (int64_t)blockIdx.x * RDB_BLOCK + threadIdx.x;
  if (REC)
  {
    // every lane of a warp that holds at least one sample takes part in the staged copies; lanes past the end recompute the last sample
    extern __shared__ double dyn_stage[];
    const int64_t i0 = i - (threadIdx.x & 31);
    if (i0 >= in.n) return;
    const int live = (int)min((int64_t)32, in.n - i0);
    dyn_body<NJ, MODE, REV, true>(C, in, out, min(i, in.n - 1), dyn_stage + (size_t)(threadIdx.x >> 5) * 32 * (10 * C.n_in + 1), live);
    return;
  }
  if (i >= in.n) return;
  dyn_body<NJ, MODE, REV>(C, in, out, i);
}

template <int MODE>
__global__ void __launch_bounds__(RDB_BLOCK) dyn_kernel_generic(const ChainDev<RDB_MAX_JOINTS>* __restrict__ C, const SamplesDev in,
                                                                const DynOutDev out)
{
  const int64_t i = (int64_t)blockIdx.x * RDB_BLOCK + threadIdx.x;
  if (i >= in.n) return;
  dyn_body<0, MODE>(*C, in, out, i);
}

// =============================================================================================================
// base-frame walker
// =============================================================================================================
struct Tw
{
  V3 l, a;  // linear, angular
};
__device__ __forceinline__ Tw tw0() { return Tw{v3(0, 0, 0), v3(0, 0, 0)}; }
// spatialTranslation, spacevect_algebra.h:129-133
__device__ __forceinline__ Tw transl(Tw t, V3 d) { return Tw{cross_add(t.l, t.a, d), t.a}; }
// spatialCrossProduct, spacevect_algebra.h:88-93
__device__ __forceinline__ Tw scross(Tw a, Tw b) { return Tw{cross_add(cross(a.a, b.l), a.l, b.a), cross(a.a, b.a)}; }
__device__ __forceinline__ Tw tw_axpy(Tw y, Tw x, double s) { return Tw{axpy(y.l, x.l, s), axpy(y.a, x.a, s)}; }
// y + x s where the linear half of x is a compile-time zero (ZL)
template <bool ZL>
__device__ __forceinline__ Tw tw_axpy_s(Tw y, Tw x, double s)
{
  return ZL ? Tw{y.l, axpy(y.a, x.a, s)} : Tw{axpy(y.l, x.l, s), axpy(y.a, x.a, s)};
}
__device__ __forceinline__ void st_tw(double* p, int link, int64_t ld, int64_t i, Tw t)
{
  st3(p, (int64_t)6 * link, ld, i, t.l);
  st3(p, (int64_t)6 * link + 3, ld, i, t.a);
}
__device__ __forceinline__ void st_pose(double* p, int64_t plane0, int64_t ld, int64_t i, const double* R, V3 t)
{
#pragma unroll
  for (int r = 0; r < 3; r++)
  {
    __stcs(p + (plane0 + 4 * r + 0) * ld + i, R[3 * r + 0]);
    __stcs(p + (plane0 + 4 * r + 1) * ld + i, R[3 * r + 1]);
    __stcs(p + (plane0 + 4 * r + 2) * ld + i, R[3 * r + 2]);
    __stcs(p + (plane0 + 4 * r + 3) * ld + i, r == 0 ? t.x : (r == 1 ? t.y : t.z));
  }
}

// the same pose as an Eigen::Affine3d image (internal/types.h:137): 4x4 column-major, 16 contiguous doubles with the [0 0 0 1] row; `p` points at
// the sample's record
__device__ __forceinline__ void st_pose_eigen(double* p, const double* R, V3 t)
{
#pragma unroll
  for (int c = 0; c < 3; c++)
  {
    __stcs(p + 4 * c + 0, R[c]);
    __stcs(p + 4 * c + 1, R[3 + c]);
    __stcs(p + 4 * c + 2, R[6 + c]);
    __stcs(p + 4 * c + 3, 0.0);
  }
  __stcs(p + 12, t.x);
  __stcs(p + 13, t.y);
  __stcs(p + 14, t.z);
  __stcs(p + 15, 1.0);
}

// Per-joint state of the base-frame walker that must outlive the walk: the base-frame axis and the origin of every joint (the Jacobian needs
// p_tool, the forward torque projection reads all earlier joints at every link).  In registers it is 6 doubles per joint -- with the torque
// accumulators, more than the 128-register budget of 4 CTAs/SM holds, and the spills go through L1/L2 to DRAM (ncu: +11 % traffic).  The
// unrolled torque kernels keep it in SHARED memory instead ([component][thread], conflict free, never written back): written once per joint,
// read once per (joint, link) pair and once for the Jacobian.
template <int CAP, bool SM>
struct JointStore;
template <int CAP>
struct JointStore<CAP, false>
{
  V3 a[CAP], p[CAP];
  __device__ __forceinline__ explicit JointStore(double*) {}
  __device__ __forceinline__ void set(int j, V3 ab, V3 pj)
  {
    a[j] = ab;
    p[j] = pj;
  }
  __device__ __forceinline__ V3 ab(int j) const { return a[j]; }
  __device__ __forceinline__ V3 pj(int j) const { return p[j]; }
};
template <int CAP>
struct JointStore<CAP, true>
{
  double* b;  // shared memory, already offset by threadIdx.x; component k of joint j at b[(6 j + k) RDB_BLOCK]
  __device__ __forceinline__ explicit JointStore(double* base) : b(base) {}
  __device__ __forceinline__ void set(int j, V3 ab, V3 pj)
  {
    double* q = b + 6 * j * RDB_BLOCK;
    q[0] = ab.x;
    q[RDB_BLOCK] = ab.y;
    q[2 * RDB_BLOCK] = ab.z;
    q[3 * RDB_BLOCK] = pj.x;
    q[4 * RDB_BLOCK] = pj.y;
    q[5 * RDB_BLOCK] = pj.z;
  }
  __device__ __forceinline__ V3 ab(int j) const
  {
    const double* q = b + 6 * j * RDB_BLOCK;
    return v3(q[0], q[RDB_BLOCK], q[2 * RDB_BLOCK]);
  }
  __device__ __forceinline__ V3 pj(int j) const
  {
    const double* q = b + (6 * j + 3) * RDB_BLOCK;
    return v3(q[0], q[RDB_BLOCK], q[2 * RDB_BLOCK]);
  }
};
// shared-memory joint store: unrolled kernels that need the Jacobian or project the torque forward
template <int NJ_T, unsigned MASK>
struct KinSm
{
  static constexpr bool value = NJ_T > 0 && (MASK & (K_JAC | K_TORQUE)) != 0;
  static constexpr size_t bytes = value ? sizeof(double) * 6 * NJ_T * RDB_BLOCK : 0;
};

// NP (unrolled kernels): the chain has no prismatic joint, so the linear half of every base-frame screw is a compile-time zero
template <int NJ_T, unsigned MASK, bool NP = false, class ChainT>
__device__ __forceinline__ void kin_body(const ChainT& C, const SamplesDev& in, const KinOutDev& o, int64_t i, double* smp = nullptr)
{
  constexpr int CAP = Cap<NJ_T>::value;
  const int nj = NJ_T > 0 ? NJ_T : C.nj;
  const int n_in = C.n_in;
  // element (plane p, sample i) of an output array: base + p * ld + i * ss.  SoA planes: ld = o.ld, ss = 1.  Eigen records (o.eigen): ld = 1
  // and ss = planes of the array, i.e. every sample owns a dense record laid out as the reference's Eigen object (6-vectors of all links back to
  // back = VectorOfVector6d, Jacobian 6 x n_act column-major); poses become 16-double Affine3d images (st_pose_eigen)
  const bool eig = o.eigen != 0;
  const int64_t ld = eig ? 1 : o.ld;
  const int64_t i_tw = eig ? i * (6 * (nj + 1)) : i, i_jac = eig ? i * (6 * n_in) : i, i_tau = eig ? i * n_in : i;
  double* const Tl_e = o.T_links + i * (16 * (nj + 1));  // Eigen records of the link poses (used when eig)

  constexpr bool cJer = (MASK & (K_DDTWIST | K_DDTWIST_NONLIN)) != 0;
  constexpr bool cAcc = (MASK & (K_DTWIST | K_TORQUE)) != 0 || cJer;
  constexpr bool cVel = (MASK & (K_TWIST | K_DTWIST_NONLIN)) != 0 || cAcc;
  constexpr bool cJac = (MASK & (K_JAC | K_TORQUE)) != 0;

  const bool wTl = (MASK & K_TLINKS) && o.T_links;
  const bool wV = (MASK & K_TWIST) && o.twist;
  const bool wA = (MASK & K_DTWIST) && o.dtwist;
  const bool wAl = (MASK & K_DTWIST_LIN) && o.dtwist_lin;
  const bool wAn = (MASK & K_DTWIST_NONLIN) && o.dtwist_nonlin;
  const bool wJ = (MASK & K_DDTWIST) && o.ddtwist;
  const bool wJl = (MASK & K_DDTWIST_LIN) && o.ddtwist_lin;
  const bool wJn = (MASK & K_DDTWIST_NONLIN) && o.ddtwist_nonlin;
  const bool wTau = (MASK & K_TORQUE) && o.torque;

  double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};  // base <- current link
  V3 p = v3(0, 0, 0);
  Tw v = tw0(), a = tw0(), al = tw0(), an = tw0(), jf = tw0(), jl = tw0(), jn = tw0();
  // base-frame screw of joint j = [0; ab[j]] (revolute) / [ab[j]; 0] (prismatic) / 0 (fixed): one 3-vector + the joint type
  JointStore<cJac ? CAP : 1, KinSm<NJ_T, MASK>::value> js(smp);
  double tau[(MASK & K_TORQUE) ? CAP : 1];
  constexpr int NT = NJ_T > 0 ? NJ_T : 1;
  double qv[NT], sv[NT], cv[NT];
  if (NJ_T > 0)
  {
#pragma unroll
    for (int l = 0; l < NT; l++) qv[l] = ld_in(in.q, C.joint[l].in, in.ld, i);
    trig_all<NT>(qv, sv, cv);
  }

  double dq_nx = 0.0, ddq_nx = 0.0, dddq_nx = 0.0;  // rates of the next link (unrolled kernels)
  if (NJ_T > 0)
  {
    // every rate the walk will need is pulled into L2 now (no register held), then loaded one link ahead of its use
#pragma unroll
    for (int l = 1; l < NT; l++)
    {
      const int inl = C.joint[l].in;
      if (cVel) prefetch_in(in.dq, inl, in.ld, i);
      if ((MASK & (K_DTWIST | K_DTWIST_LIN | K_TORQUE)) != 0 || cJer) prefetch_in(in.ddq, inl, in.ld, i);
      if ((MASK & (K_DDTWIST | K_DDTWIST_LIN)) != 0) prefetch_in(in.dddq, inl, in.ld, i);
    }
    const int in0 = C.joint[0].in;
    if (cVel) dq_nx = ld_in(in.dq, in0, in.ld, i);
    if ((MASK & (K_DTWIST | K_DTWIST_LIN | K_TORQUE)) != 0 || cJer) ddq_nx = ld_in(in.ddq, in0, in.ld, i);
    if ((MASK & (K_DDTWIST | K_DDTWIST_LIN)) != 0) dddq_nx = ld_in(in.dddq, in0, in.ld, i);
  }
  // link 0 = base: identity pose, zero twists (primitives_impl.h:661-677, 697)
  if (wTl)
  {
    if (eig) st_pose_eigen(Tl_e, R, p);
    else st_pose(o.T_links, 0, ld, i, R, p);
  }
  if (wV) st_tw(o.twist, 0, ld, i_tw, v);
  if (wA) st_tw(o.dtwist, 0, ld, i_tw, v);
  if (wAl) st_tw(o.dtwist_lin, 0, ld, i_tw, v);
  if (wAn) st_tw(o.dtwist_nonlin, 0, ld, i_tw, v);
  if (wJ) st_tw(o.ddtwist, 0, ld, i_tw, v);
  if (wJl) st_tw(o.ddtwist_lin, 0, ld, i_tw, v);
  if (wJn) st_tw(o.ddtwist_nonlin, 0, ld, i_tw, v);

#pragma unroll
  for (int l = 0; l < (NJ_T > 0 ? NJ_T : nj); l++)
  {
    const JointDev& J = C.joint[l];
    double Rpc[9];
    V3 t;
    if (NJ_T > 0)
      joint_transform_sc(J, qv[NJ_T > 0 ? l : 0], sv[NJ_T > 0 ? l : 0], cv[NJ_T > 0 ? l : 0], Rpc, t);
    else
      joint_transform(J, ld_in(in.q, J.in, in.ld, i), Rpc, t);

    // computeScrews (primitives_impl.h:879): screw of joint l in the base frame uses the PARENT link rotation
    const V3 axb = rot(R, v3(J.axp));
    Tw s;
    s.l = (!NP && J.type == RDB_JOINT_PRISMATIC) ? axb : v3(0, 0, 0);
    s.a = (J.type == RDB_JOINT_REVOLUTE) ? axb : v3(0, 0, 0);

    // computeFrames (primitives_impl.h:869)
    const V3 d = rot(R, t);  // p_l - p_{l-1}
    p = p + d;
    double Rn[9];
    mul33(R, Rpc, Rn);
#pragma unroll
    for (int k = 0; k < 9; k++) R[k] = Rn[k];
    if (wTl)
    {
      if (eig) st_pose_eigen(Tl_e + 16 * (l + 1), R, p);
      else st_pose(o.T_links, (int64_t)12 * (l + 1), ld, i, R, p);
    }

    if (cJac) js.set(l, axb, p);

    // the rates of link l were requested one link earlier (unrolled kernels): the DRAM latency hides behind the previous link's arithmetic
    constexpr bool wantDD = (MASK & (K_DTWIST | K_DTWIST_LIN | K_TORQUE)) != 0 || cJer;
    constexpr bool wantDDD = (MASK & (K_DDTWIST | K_DDTWIST_LIN)) != 0;
    double dql, ddql, dddql;
    if (NJ_T > 0)
    {
      dql = dq_nx;
      ddql = ddq_nx;
      dddql = dddq_nx;
      if (l + 1 < NJ_T)
      {
        const int inn = C.joint[l + 1 < CAP ? l + 1 : 0].in;
        if (cVel) dq_nx = ld_in(in.dq, inn, in.ld, i);
        if (wantDD) ddq_nx = ld_in(in.ddq, inn, in.ld, i);
        if (wantDDD) dddq_nx = ld_in(in.dddq, inn, in.ld, i);
      }
    }
    else
    {
      dql = cVel ? ld_in(in.dq, J.in, in.ld, i) : 0.0;
      ddql = wantDD ? ld_in(in.ddq, J.in, in.ld, i) : 0.0;
      dddql = wantDDD ? ld_in(in.dddq, J.in, in.ld, i) : 0.0;
    }

    Tw vxs = tw0();
    if (cVel)
    {
      v = tw_axpy_s<NP>(transl(v, d), s, dql);  // primitives_impl.h:1007-1008
      vxs = NP ? Tw{cross(v.l, s.a), cross(v.a, s.a)} : scross(v, s);
      if (wV) st_tw(o.twist, l + 1, ld, i_tw, v);
    }
    if (MASK & K_DTWIST_LIN)
    {
      al = tw_axpy_s<NP>(transl(al, d), s, ddql);  // primitives_impl.h:1055-1056
      if (wAl) st_tw(o.dtwist_lin, l + 1, ld, i_tw, al);
    }
    if (MASK & K_DTWIST_NONLIN)
    {
      an = tw_axpy(transl(an, d), vxs, dql);  // primitives_impl.h:1074-1075
      if (wAn) st_tw(o.dtwist_nonlin, l + 1, ld, i_tw, an);
    }
    if (cAcc)
    {
      a = tw_axpy_s<NP>(tw_axpy(transl(a, d), vxs, dql), s, ddql);  // primitives_impl.h:1116-1117
      if (wA) st_tw(o.dtwist, l + 1, ld, i_tw, a);
    }
    if (MASK & K_DDTWIST_LIN)
    {
      jl = tw_axpy_s<NP>(transl(jl, d), s, dddql);  // primitives_impl.h:1148-1149
      if (wJl) st_tw(o.ddtwist_lin, l + 1, ld, i_tw, jl);
    }
    if (cJer)
    {
      // primitives_impl.h:1213-1218 / 1174-1178; the reference's 1x coefficient on (v x s) DDq is mirrored
      const Tw axs = NP ? Tw{cross(a.l, s.a), cross(a.a, s.a)} : scross(a, s);
      const Tw vvxs = scross(v, vxs);
      const Tw k = Tw{axs.l + vvxs.l, axs.a + vvxs.a};
      if (MASK & K_DDTWIST)
      {
        jf = tw_axpy(tw_axpy(tw_axpy_s<NP>(transl(jf, d), s, dddql), vxs, ddql), k, dql);
        if (wJ) st_tw(o.ddtwist, l + 1, ld, i_tw, jf);
      }
      if (MASK & K_DDTWIST_NONLIN)
      {
        jn = tw_axpy(tw_axpy(transl(jn, d), vxs, ddql), k, dql);
        if (wJn) st_tw(o.ddtwist_nonlin, l + 1, ld, i_tw, jn);
      }
    }

    if (MASK & K_TORQUE)
    {
      // getWrench (primitives_impl.h:1240-1250) for link l+1, then getJointTorque (1267-1271) as a forward
      // projection: tau_j = s_j . sum_{m>=j} dualTransl(w_m, p_j - p_m)   (spacevect_algebra.h:150-154)
      tau[l] = 0.0;
      const double* P = C.link[l].pi;
      const V3 mc = v3(P[1], P[2], P[3]);
      const V3 agl = rotT(R, a.l - v3(C.g));
      const V3 all = rotT(R, a.a);
      const V3 vl = rotT(R, v.l);
      const V3 wl = rotT(R, v.a);
      const V3 hl1 = cross_add(agl * P[0], all, mc);
      const V3 hl2 = cross_add(vl * P[0], wl, mc);
      const V3 Ial = v3(fma(P[4], all.x, fma(P[5], all.y, P[6] * all.z)), fma(P[5], all.x, fma(P[7], all.y, P[8] * all.z)),
                        fma(P[6], all.x, fma(P[8], all.y, P[9] * all.z)));
      const V3 Iw = v3(fma(P[4], wl.x, fma(P[5], wl.y, P[6] * wl.z)), fma(P[5], wl.x, fma(P[7], wl.y, P[8] * wl.z)),
                       fma(P[6], wl.x, fma(P[8], wl.y, P[9] * wl.z)));
      const V3 ha1 = cross_add(Ial, mc, agl);
      const V3 ha2 = cross_add(Iw, mc, vl);
      const V3 f = rot(R, cross_add(hl1, wl, hl2));
      const V3 n = rot(R, cross_add(cross_add(ha1, wl, ha2), vl, hl2));
#pragma unroll
      for (int j = 0; j <= l; j++)
      {
        // s_j . dualTransl(w, p_j - p): the force part for a prismatic joint, the moment about the joint origin for a revolute one
        const int tj = C.joint[j].type;
        if (tj == RDB_JOINT_REVOLUTE) tau[j] += dot(js.ab(j), cross_add(n, f, js.pj(j) - p));
        else if (!NP && tj == RDB_JOINT_PRISMATIC) tau[j] += dot(js.ab(j), f);
      }
    }
  }

  if ((MASK & K_TTOOL) && o.T_tool)
  {
    if (eig) st_pose_eigen(o.T_tool + i * 16, R, p);
    else st_pose(o.T_tool, 0, ld, i, R, p);
  }

  if ((MASK & K_JAC) && o.jacobian)
  {
    // getJacobian (primitives_impl.h:939-945): col = spatialTranslation(s_j, p_tool - p_j)
#pragma unroll
    for (int j = 0; j < (NJ_T > 0 ? NJ_T : nj); j++)
    {
      const int r = C.joint[j].in;
      if (r >= 0)
      {
        const int tj = C.joint[j].type;
        const V3 z = v3(0, 0, 0);
        const V3 abj = js.ab(j);
        const V3 lin = tj == RDB_JOINT_REVOLUTE ? cross(abj, p - js.pj(j)) : ((!NP && tj == RDB_JOINT_PRISMATIC) ? abj : z);
        st3(o.jacobian, (int64_t)6 * r, ld, i_jac, lin);
        st3(o.jacobian, (int64_t)6 * r + 3, ld, i_jac, tj == RDB_JOINT_REVOLUTE ? abj : z);
      }
    }
  }
  if (wTau)
  {
#pragma unroll
    for (int j = 0; j < (NJ_T > 0 ? NJ_T : nj); j++)
    {
      const int r = C.joint[j].in;
      if (r >= 0) st_out(o.torque, r, ld, i_tau, tau[j]);
    }
  }
  (void)n_in;
}

template <int NJ, unsigned MASK, bool NP = false>
__global__ void __launch_bounds__(RDB_BLOCK, RDB_KIN_MINB) kin_kernel(const __grid_constant__ ChainDev<NJ> C, const SamplesDev in, const KinOutDev o)
{
  extern __shared__ double kin_sm[];
  const int64_t i = (int64_t)blockIdx.x * RDB_BLOCK + threadIdx.x;
  if (i >= in.n) return;
  kin_body<NJ, MASK, NP>(C, in, o, i, kin_sm + threadIdx.x);
}

template <unsigned MASK>
__global__ void __launch_bounds__(RDB_BLOCK) kin_kernel_generic(const ChainDev<RDB_MAX_JOINTS>* __restrict__ C, const SamplesDev in,
                                                                const KinOutDev o)
{
  const int64_t i = (int64_t)blockIdx.x * RDB_BLOCK + threadIdx.x;
  if (i >= in.n) return;
  kin_body<0, MASK>(*C, in, o, i);
}

// =============================================================================================================
// synthetic inputs
// =============================================================================================================
__host__ __device__ inline uint64_t splitmix64(uint64_t x)
{
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__host__ __device__ inline double uniform_pm1(uint64_t seed, int64_t i, int stream_id, int plane)
{
  const uint64_t z = splitmix64(seed + ((uint64_t)i << 8) + ((uint64_t)stream_id << 6) + (uint64_t)plane);
  return 2.0 * ((double)(z >> 11) * (1.0 / 9007199254740992.0)) - 1.0;
}
__global__ void fill_uniform_kernel(double* x, int n_planes, int64_t n, int64_t ld, uint64_t seed, int stream_id)
{
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int j = 0; j < n_planes; j++) x[(int64_t)j * ld + i] = uniform_pm1(seed, i, stream_id, j);
}
void fill_uniform_host(double* x, int n_planes, int64_t n, int64_t ld, uint64_t seed, int stream_id)
{
  for (int j = 0; j < n_planes; j++)
    for (int64_t i = 0; i < n; i++) x[(int64_t)j * ld + i] = uniform_pm1(seed, i, stream_id, j);
}

// =============================================================================================================
// launchers
// =============================================================================================================
template <int NJ>
static ChainDev<NJ> narrow(const ChainDev<RDB_MAX_JOINTS>& h)
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

static inline unsigned grid_for(int64_t n) { return (unsigned)((n + RDB_BLOCK - 1) / RDB_BLOCK); }

#define RDB_FAST_NJ(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8)

template <int MODE>
static cudaError_t launch_dyn_mode(const ChainHost& ch, const SamplesDev& in, const DynOutDev& out, cudaStream_t st)
{
  if (in.n <= 0) return cudaSuccess;
  const unsigned grid = grid_for(in.n);
  // torque and inertia (and so forward dynamics) do not depend on how the parameters are split between rigidly attached links: those modes
  // walk the chain with the never-moving joints folded away and the parameters lumped (fold.cpp: fold_chain) -- C6 walks 6 links instead of 7
  const bool folded = !(MODE & DYN_REGRESSOR) && ch.gram.fold_version == ch.model_version && ch.gram.fold.nj >= 1;
  const ChainDev<RDB_MAX_JOINTS>& H = folded ? ch.gram.fold : ch.host;
  bool rev = folded;  // all-revolute specialisation (torque / inertia on the folded chain only)
  for (int j = 0; j < H.nj && rev; j++) rev = H.joint[j].type == RDB_JOINT_REVOLUTE;
  // regressor in the Eigen-record layout: staged stores (dyn_body REC); the tile is 32 x (10 n_act + 1) doubles per warp
  if ((MODE & DYN_REGRESSOR) != 0 && out.ps == 1 && out.ss_phi > 1 && H.nj <= 8)
  {
    const size_t smem = sizeof(double) * (RDB_BLOCK / 32) * 32 * (size_t)(10 * H.n_in + 1);
    switch (H.nj)
    {
#define X(N)                                                                                                                            \
  case N:                                                                                                                               \
  {                                                                                                                                     \
    auto kern = dyn_kernel<N, (MODE & DYN_REGRESSOR) ? MODE : DYN_REGRESSOR, false, true>;                                              \
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                                 \
    if (e != cudaSuccess) return e;                                                                                                     \
    kern<<<grid, RDB_BLOCK, smem, st>>>(narrow<N>(H), in, out);                                                                         \
    break;                                                                                                                              \
  }
      RDB_FAST_NJ(X)
#undef X
    }
    count_launch();
    return cudaGetLastError();
  }
  switch (H.nj)
  {
#define X(N)                                                                                                                    \
  case N:                                                                                                                       \
    if ((MODE & DYN_REGRESSOR) == 0 && rev)                                                                                     \
      dyn_kernel<N, (MODE & DYN_REGRESSOR) ? 0 : MODE, true><<<grid, RDB_BLOCK, 0, st>>>(narrow<N>(H), in, out);        \
    else                                                                                                                        \
      dyn_kernel<N, MODE><<<grid, RDB_BLOCK, 0, st>>>(narrow<N>(H), in, out);                                                      \
    break;
    RDB_FAST_NJ(X)
#undef X
    default:
      dyn_kernel_generic<MODE><<<grid, RDB_BLOCK, 0, st>>>(ch.dev, in, out);
  }
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_dyn(const ChainHost& ch, int mode, const SamplesDev& in, const DynOutDev& out, cudaStream_t st)
{
  switch (mode)
  {
    case DYN_REGRESSOR: return launch_dyn_mode<DYN_REGRESSOR>(ch, in, out, st);
    case DYN_REGRESSOR | DYN_TORQUE: return launch_dyn_mode<DYN_REGRESSOR | DYN_TORQUE>(ch, in, out, st);
    case DYN_TORQUE: return launch_dyn_mode<DYN_TORQUE>(ch, in, out, st);
    case DYN_INERTIA: return launch_dyn_mode<DYN_INERTIA>(ch, in, out, st);
    case DYN_FD: return launch_dyn_mode<DYN_FD>(ch, in, out, st);
  }
  return cudaErrorInvalidValue;
}
cudaError_t launch_dyn(const ChainHost& ch, int mode, const SamplesDev& in, double* phi, double* tau, double* M, int64_t ld_out,
                       cudaStream_t st)
{
  return launch_dyn(ch, mode, in, dyn_out_soa(phi, tau, M, ld_out), st);
}

template <unsigned MASK>
static cudaError_t launch_kin_mask(const ChainHost& ch, const SamplesDev& in, const KinOutDev& o, cudaStream_t st)
{
  if (in.n <= 0) return cudaSuccess;
  const unsigned grid = grid_for(in.n);
  bool np = true;  // no prismatic joint: the specialised kernels
  for (int j = 0; j < ch.host.nj; j++) np = np && ch.host.joint[j].type != RDB_JOINT_PRISMATIC;
  switch (ch.host.nj)
  {
#define X(N)                                                                                                        \
  case N:                                                                                                           \
    if (np) kin_kernel<N, MASK, true><<<grid, RDB_BLOCK, KinSm<N, MASK>::bytes, st>>>(narrow<N>(ch.host), in, o);   \
    else kin_kernel<N, MASK, false><<<grid, RDB_BLOCK, KinSm<N, MASK>::bytes, st>>>(narrow<N>(ch.host), in, o);     \
    break;
    RDB_FAST_NJ(X)
#undef X
    default:
      kin_kernel_generic<MASK><<<grid, RDB_BLOCK, 0, st>>>(ch.dev, in, o);
  }
  count_launch();
  return cudaGetLastError();
}

// compiled output combinations, smallest first; the launcher takes the first that covers the request
static constexpr unsigned KM_POSE = K_TTOOL | K_TLINKS;
static constexpr unsigned KM_POSE_JAC = K_TTOOL | K_TLINKS | K_JAC;
static constexpr unsigned KM_VEL = KM_POSE_JAC | K_TWIST;
static constexpr unsigned KM_ACC = KM_VEL | K_DTWIST | K_DTWIST_LIN | K_DTWIST_NONLIN;
static constexpr unsigned KM_CFG2 = K_TTOOL | K_JAC | K_TWIST | K_DTWIST | K_TORQUE;  // BASELINE.json configs[1]
static constexpr unsigned KM_JERK = K_TWIST | K_DTWIST | K_DDTWIST;                   // BASELINE.json configs[4]

cudaError_t launch_kin(const ChainHost& ch, unsigned want, const SamplesDev& in, const KinOutDev& o, cudaStream_t st)
{
#define TRY(M) \
  if ((want & ~(M)) == 0) return launch_kin_mask<M>(ch, in, o, st);
  TRY(KM_POSE)
  TRY(KM_POSE_JAC)
  TRY(KM_VEL)
  TRY(KM_CFG2)
  TRY(KM_JERK)
  TRY(KM_ACC)
#undef TRY
  return launch_kin_mask<K_ALL>(ch, in, o, st);
}

cudaError_t launch_fill_uniform(double* x, int n_planes, int64_t n, int64_t ld, uint64_t seed, int stream_id, cudaStream_t st)
{
  if (n <= 0) return cudaSuccess;
  fill_uniform_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, n_planes, n, ld, seed, stream_id);
  count_launch();
  return cudaGetLastError();
}

}  // namespace rdb
