// aux.cu -- the parts of rosdyn::Chain next to the hot path (SURVEY.md section 8a row a14 "external wrenches optional", 8f N4):
//   Chain::getWrench / getJointTorque with external wrenches   (primitives_impl.h:1225-1274)
//   Chain::getJacobianLink                                     (primitives_impl.h:951-979)
// One thread per sample, two passes over the chain exactly as the reference writes them (forward: frames, screws, twists,
// accelerations; backward: wrenches), per-link state in thread-local arrays.  These are not the throughput kernels (kernels.cu
// holds the forward-only register walkers for the hot entry points); they exist so that the whole getter surface is served.
#include <cuda_runtime.h>

#include "launch.h"
#include "spatial.cuh"

namespace rdb
{

struct AuxOutDev
{
  int64_t ld;
  const double* ext;   // [nL][6][ld_ext] external wrenches applied to the links, link frames, or nullptr
  int64_t ld_ext;
  double* torque;      // [n_in][ld]
  double* wrenches;    // [nL][6][ld]
  double* jac_link;    // [n_in*6][ld]
  int32_t link;        // link of jac_link
  int32_t k_before;    // active joints between the base and that link (size of m_parent_moveable_joints_of_link, primitives_impl.h:798-829)
};

template <int CAP, class ChainT>
__device__ __forceinline__ void aux_body(const ChainT& C, const SamplesDev& in, const AuxOutDev& o, int64_t i)
{
  const int nj = C.nj, nL = nj + 1;
  double R[CAP + 1][9];
  V3 p[CAP + 1], sl[CAP + 1], sa[CAP + 1], vl[CAP + 1], va[CAP + 1], al[CAP + 1], aa[CAP + 1];
  {
    const double I3[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int k = 0; k < 9; k++) R[0][k] = I3[k];
  }
  p[0] = sl[0] = sa[0] = vl[0] = va[0] = al[0] = aa[0] = v3(0, 0, 0);
  const bool dyn = o.torque || o.wrenches;
  // forward pass: computeFrames / computeScrews / getTwist / getDTwist (primitives_impl.h:863-882, 1004-1009, 1113-1118)
  for (int nl = 1; nl < nL; nl++)
  {
    const JointDev& J = C.joint[nl - 1];
    double Rpc[9];
    V3 t;
    joint_transform(J, ld_in(in.q, J.in, in.ld, i), Rpc, t);
    const V3 axb = rot(R[nl - 1], v3(J.axp));
    sl[nl] = (J.type == RDB_JOINT_PRISMATIC) ? axb : v3(0, 0, 0);
    sa[nl] = (J.type == RDB_JOINT_REVOLUTE) ? axb : v3(0, 0, 0);
    const V3 d = rot(R[nl - 1], t);
    p[nl] = p[nl - 1] + d;
    mul33(R[nl - 1], Rpc, R[nl]);
    if (dyn)
    {
      const double dq = ld_in(in.dq, J.in, in.ld, i), ddq = ld_in(in.ddq, J.in, in.ld, i);
      vl[nl] = axpy(cross_add(vl[nl - 1], va[nl - 1], d), sl[nl], dq);
      va[nl] = axpy(va[nl - 1], sa[nl], dq);
      const V3 xl = cross_add(cross(va[nl], sl[nl]), vl[nl], sa[nl]);  // spatialCrossProduct(v, s), spacevect_algebra.h:88-93
      const V3 xa = cross(va[nl], sa[nl]);
      al[nl] = axpy(axpy(cross_add(al[nl - 1], aa[nl - 1], d), xl, dq), sl[nl], ddq);
      aa[nl] = axpy(axpy(aa[nl - 1], xa, dq), sa[nl], ddq);
    }
  }
  if (dyn)
  {
    // backward pass: getWrench (primitives_impl.h:1231-1258)
    const V3 g = v3(C.g);
    V3 wf = v3(0, 0, 0), wn = v3(0, 0, 0);  // wrench of link nl+1 (force, torque) at its origin, base frame
    for (int nl = nL - 1; nl >= 0; nl--)
    {
      V3 f = v3(0, 0, 0), n = v3(0, 0, 0);
      if (nl > 0)
      {
        const double* P = C.link[nl - 1].pi;
        const double* Rl = R[nl];
        const V3 mc = v3(P[1], P[2], P[3]);
        const V3 a_l = rotT(Rl, al[nl]), a_a = rotT(Rl, aa[nl]), v_l = rotT(Rl, vl[nl]), v_a = rotT(Rl, va[nl]);
        // I_cc [x;y] = [ m x + y x mc ; mc x x + I0 y ]
        const V3 Ia_f = cross_add(a_l * P[0], a_a, mc);
        const V3 I0aa = v3(fma(P[4], a_a.x, fma(P[5], a_a.y, P[6] * a_a.z)), fma(P[5], a_a.x, fma(P[7], a_a.y, P[8] * a_a.z)),
                           fma(P[6], a_a.x, fma(P[8], a_a.y, P[9] * a_a.z)));
        const V3 Ia_n = cross_add(I0aa, mc, a_l);
        const V3 Iv_f = cross_add(v_l * P[0], v_a, mc);
        const V3 I0va = v3(fma(P[4], v_a.x, fma(P[5], v_a.y, P[6] * v_a.z)), fma(P[5], v_a.x, fma(P[7], v_a.y, P[8] * v_a.z)),
                           fma(P[6], v_a.x, fma(P[8], v_a.y, P[9] * v_a.z)));
        const V3 Iv_n = cross_add(I0va, mc, v_l);
        // + spatialDualCrossProduct(v, I v) = [ v_a x f ; v_a x n + v_l x f ]  (spacevect_algebra.h:108-113)
        const V3 fl = cross_add(Ia_f, v_a, Iv_f);
        const V3 nl_ = cross_add(cross_add(Ia_n, v_a, Iv_n), v_l, Iv_f);
        f = rot(Rl, fl);
        n = rot(Rl, nl_);
        // gravity wrench (primitives_impl.h:1249-1250): -m g ; -(R c) x (m g);  m c = mc
        f = f - g * P[0];
        n = n - cross(rot(Rl, mc), g);
      }
      if (o.ext)
      {
        // spatialTranformation(-ext, T_bl) -- the TWIST transform, as the reference applies it (primitives_impl.h:1255, SA.h:193-197)
        const double* e = o.ext + (int64_t)6 * nl * o.ld_ext + i;
        const V3 ef = v3(-__ldcs(e), -__ldcs(e + o.ld_ext), -__ldcs(e + 2 * o.ld_ext));
        const V3 en = v3(-__ldcs(e + 3 * o.ld_ext), -__ldcs(e + 4 * o.ld_ext), -__ldcs(e + 5 * o.ld_ext));
        const V3 Ren = rot(R[nl], en);
        f = f + cross_add(rot(R[nl], ef), Ren, p[nl]);
        n = n + Ren;
      }
      if (nl < nL - 1)
      {
        // + spatialDualTranslation(w[nl+1], p_nl - p_{nl+1})  (spacevect_algebra.h:150-154)
        f = f + wf;
        n = n + cross_add(wn, wf, p[nl] - p[nl + 1]);
      }
      wf = f;
      wn = n;
      if (o.wrenches)
      {
        st3(o.wrenches, (int64_t)6 * nl, o.ld, i, f);
        st3(o.wrenches, (int64_t)6 * nl + 3, o.ld, i, n);
      }
      if (o.torque && nl > 0)
      {
        const int r = C.joint[nl - 1].in;
        if (r >= 0) st_out(o.torque, r, o.ld, i, dot(f, sl[nl]) + dot(n, sa[nl]));  // primitives_impl.h:1267-1271
      }
    }
  }
  if (o.jac_link)
  {
    // getJacobianLink (primitives_impl.h:966-976): the first k_before ACTIVE joints (in input order, as the reference indexes
    // m_active_joints by the loop counter) give a column each; the others stay zero
    for (int j = 0; j < nj; j++)
    {
      const int r = C.joint[j].in;
      if (r < 0) continue;
      V3 lin = v3(0, 0, 0), ang = v3(0, 0, 0);
      if (r < o.k_before && C.joint[j].type != RDB_JOINT_FIXED)
      {
        lin = cross_add(sl[j + 1], sa[j + 1], p[o.link] - p[j + 1]);
        ang = sa[j + 1];
      }
      st3(o.jac_link, (int64_t)6 * r, o.ld, i, lin);
      st3(o.jac_link, (int64_t)6 * r + 3, o.ld, i, ang);
    }
  }
}

template <int NJ>
__global__ void __launch_bounds__(128) aux_kernel(const __grid_constant__ ChainDev<NJ> C, const SamplesDev in, const AuxOutDev o)
{
  const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (i >= in.n) return;
  aux_body<NJ>(C, in, o, i);
}
__global__ void __launch_bounds__(64) aux_kernel_generic(const ChainDev<RDB_MAX_JOINTS>* __restrict__ C, const SamplesDev in, const AuxOutDev o)
{
  const int64_t i = (int64_t)blockIdx.x * 64 + threadIdx.x;
  if (i >= in.n) return;
  aux_body<RDB_MAX_JOINTS>(*C, in, o, i);
}

cudaError_t launch_aux(const ChainHost& ch, const SamplesDev& in, const double* ext, int64_t ld_ext, double* torque, double* wrenches,
                       double* jac_link, int link, int64_t ld_out, cudaStream_t st)
{
  if (in.n <= 0) return cudaSuccess;
  AuxOutDev o{ld_out, ext, ld_ext, torque, wrenches, jac_link, link, 0};
  if (jac_link)
    for (int j = 0; j < link && j < ch.host.nj; j++)
      if (ch.host.joint[j].in >= 0) o.k_before++;
  if (ch.host.nj <= 8)
    aux_kernel<8><<<(unsigned)((in.n + 127) / 128), 128, 0, st>>>(narrow<8>(ch.host), in, o);
  else
    aux_kernel_generic<<<(unsigned)((in.n + 63) / 64), 64, 0, st>>>(ch.dev.get(), in, o);
  count_launch();
  return cudaGetLastError();
}

}  // namespace rdb
