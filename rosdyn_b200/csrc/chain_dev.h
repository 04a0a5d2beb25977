// chain_dev.h -- device-side image of a serial chain (POD, lives in the kernel-parameter constant bank).
//
// Everything a kernel needs about the model is q-independent and is precomputed on the host exactly as the
// reference's Joint::fromUrdf / Link::fromUrdf do (primitives_impl.h:50-72, 288-319, 399-417).  The fast
// kernels are templated on the number of chain joints NJ and receive ChainDev<NJ> BY VALUE as a
// __grid_constant__ parameter, so every model constant is a constant-bank operand of the DFMA that uses it
// (no register, no load).  Chains with more joints than the unrolled instantiations use the same code with
// runtime loops and a ChainDev<RDB_MAX_JOINTS> in global memory.
#pragma once
#include <stdint.h>

#include "../../include/rosdyn_b200.h"

namespace rdb
{

struct JointDev
{
  int32_t type;  // RDB_JOINT_*
  int32_t in;    // input plane of this joint or -1
  // R_pc(q) = A + sin(q) B + (1-cos q) C with A = R_pj, B = R_pj K, C = R_pj K^2 (row-major); this is the
  // reference's own factorisation (m_skew_axis_in_p / m_square_skew_axis_in_p, primitives_impl.h:43,70-71).
  double A[9], B[9], C[9];
  double t[3];    // t_pj
  double ax[3];   // unit axis in the joint (= child) frame; the child-frame screw is [0;ax] / [ax;0]
  double axp[3];  // axis in the parent frame, R_pj ax  (primitives_impl.h:69)
};

// the axis of every revolute joint of the folded chain, in the canonical frame of its link (fold.cpp); the REV generators of the fused
// kernels (gram_common.cuh) are written for it
constexpr double REV_AXIS[3] = {0.0, 0.0, 1.0};

struct LinkDev
{
  // the 10 standard inertial parameters about the link origin in link axes (primitives_impl.h:399-417):
  // m, m cx, m cy, m cz, Ixx, Ixy, Ixz, Iyy, Iyz, Izz ; spatial inertia I_cc = sum_p pi[p] E_p
  double pi[10];
};

template <int CAP>
struct ChainDev
{
  int32_t nj;    // chain joints incl. fixed
  int32_t n_in;  // input joints
  double g[3];
  JointDev joint[CAP];
  LinkDev link[CAP];  // link[l] = child link of joint l (the base link carries no parameters)
};

struct SamplesDev
{
  int64_t n, ld;
  const double *q, *dq, *ddq, *dddq;
};

// output selection bits of the kinematics kernel
enum : unsigned
{
  K_TTOOL = 1u << 0,
  K_TLINKS = 1u << 1,
  K_JAC = 1u << 2,
  K_TWIST = 1u << 3,
  K_DTWIST = 1u << 4,
  K_DTWIST_LIN = 1u << 5,
  K_DTWIST_NONLIN = 1u << 6,
  K_DDTWIST = 1u << 7,
  K_DDTWIST_LIN = 1u << 8,
  K_DDTWIST_NONLIN = 1u << 9,
  K_TORQUE = 1u << 10,
  K_ALL = (1u << 11) - 1
};

struct KinOutDev
{
  int64_t ld;
  double *T_tool, *T_links, *jacobian, *twist, *dtwist, *dtwist_lin, *dtwist_nonlin, *ddtwist, *ddtwist_lin, *ddtwist_nonlin, *torque;
  int32_t eigen;  // RDB_LAYOUT_EIGEN: per-sample records laid out as the reference's Eigen objects (see rosdyn_b200.h)
};

// outputs of the link-frame walker.  Element (plane p, sample i) of an array lives at  base + p * ps + i * ss_<array>:
// SoA planes: ps = ld, ss = 1;  Eigen records: ps = 1, ss = planes of the array (the record is the column-major Eigen matrix)
// Forward dynamics (DYN_FD) writes ddq into `tau`, reads the applied torques from tau_in [n_in][in.ld] (NULL = 0) and, when info is not
// NULL, writes info[i] (0, or 1 when M is not positive definite)
struct DynOutDev
{
  double *phi, *tau, *M;
  int64_t ps, ss_phi, ss_tau, ss_M;
  const double* tau_in = nullptr;
  int32_t* info = nullptr;
};
inline DynOutDev dyn_out_soa(double* phi, double* tau, double* M, int64_t ld) { return DynOutDev{phi, tau, M, ld, 1, 1, 1}; }

}  // namespace rdb
