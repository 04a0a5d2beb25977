// gram_common.cuh -- pieces shared by the fused regressor -> normal-equation kernels (gram_fused.cu: shared-memory slots filled directly by the
// generator warps; gram_ring.cu: generator warps decoupled from the slots through an L2-resident ring and TMA bulk copies): geometry of the
// augmented Gram matrix, mbarrier / DMMA wrappers, and the per-sample regressor generator.
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "launch.h"
#include "spatial.cuh"

namespace rdb
{

#ifndef GF_TSPLIT
#define GF_TSPLIT 2
#endif
#ifndef GF_ZCOL
#define GF_ZCOL 1  // all-revolute chains: drop the exact-zero mass column of a link on its own joint (GramGeom Z)
#endif
constexpr int GF_KSPLIT = 4;      // MMA warps that share the k-steps of a slot (one per SM sub-partition)
constexpr int GF_TS = GF_TSPLIT;  // 1: each MMA warp owns all tiles; 2: two warps per sub-partition split the tile rows by parity
constexpr int GF_MMA_WARPS = GF_KSPLIT * GF_TS;
constexpr int GF_MAX_SLOTS = 4;   // 32-sample slots in shared memory: as many as fit the 227 KB (3 for a 7-joint chain, 4 from 6 joints down);
                                  // 8 MMA + 4 generator warps = 3 warps per SM sub-partition is also what the 168-register budget allows
constexpr int GF_BAR_REDUCE = 1;  // named barrier of the final k-split reduction (0 is __syncthreads)

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void dmma884f(double& d0, double& d1, double a, double b)
{
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
// mbarriers in shared memory (one full / one empty per slot); arrive = release.cta, wait = acquire.cta
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b)
{
  asm volatile("{\n .reg .b64 st;\n mbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity)
{
  asm volatile(
      "{\n .reg .pred p;\n"
      "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      " @p bra D;\n bra W;\n"
      "D:\n}" ::"r"(smem_u32(b)),
      "r"(parity)
      : "memory");
}

// compile-time loop: f(std::integral_constant<int, B>) ... f(std::integral_constant<int, E - 1>), so that indices derived from the loop
// variable are constant expressions (accumulator arrays indexed through constexpr tables must stay in registers)
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f)
{
  if constexpr (B < E)
  {
    f(std::integral_constant<int, B>{});
    static_for<B + 1, E>(f);
  }
}

// geometry of the augmented Gram matrix and of a slot for a (folded) chain of NJ joints, all of them inputs.
// X = 1 (cross mode, extended model [Phi | Phi_c]): every row carries GX_COLS component columns of its own joint after the tau column.
constexpr int GX_COLS = 8;  // component columns per joint row (one 8-wide tile)
// Z = 1 (all-revolute chains, gram_ring.cu): the projection of a link on its OWN revolute joint has no mass term (the unit twist at birth is
// [0; axis], so Phi[j, 10 j + 0] == 0 exactly).  Inside every link block the mass column therefore comes LAST (p order 1..9, 0): the row of
// joint j then ends with an exact zero that is neither stored nor multiplied -- rowlen(j) = 10 (NJ - j), and position 10 NJ (the mass of the
// first moving link, an identically zero column of Phi) is never touched.
template <int NJ, int X = 0, int Z = 0>
struct GramGeom
{
  static constexpr int P = 10 * NJ;
  static constexpr int T = (P + 1 - Z + 7) / 8;   // tile columns of the augmented matrix
  static constexpr int NT = T * (T + 1) / 2;  // upper-triangular tiles
  static constexpr int KPW = 8 / GF_KSPLIT;   // k-steps (4 samples) of one MMA warp per joint row and slot
  static constexpr int NSTEPS = NJ * KPW;     // k-steps of one MMA warp per slot
  __host__ __device__ static constexpr int threads(int slots) { return 32 * (GF_MMA_WARPS + slots); }
  // offset (doubles) of the row of joint j inside a slot: [position][sample], only the positions 0 .. rowlen(j)-1 are stored
  __host__ __device__ static constexpr int rowbase(int j)
  {
    int o = 0;
    for (int i = 0; i < j; i++) o += (P + 1 - Z - 10 * i + (X ? GX_COLS : 0)) * 32;
    return o;
  }
  static constexpr int SLOT_DOUBLES = rowbase(NJ);
  __host__ __device__ static constexpr int tile(int I, int J) { return I * T - I * (I - 1) / 2 + (J - I); }
  // tile rows owned by an MMA warp: all (TS == 1) or the rows of parity `par` (TS == 2)
  __host__ __device__ static constexpr bool owns(int I, int ts, int par) { return ts == 1 || (I & 1) == par; }
  __host__ __device__ static constexpr int ntiles(int ts, int par)
  {
    int n = 0;
    for (int I = 0; I < T; I++)
      if (owns(I, ts, par)) n += T - I;
    return n;
  }
  __host__ __device__ static constexpr int local(int I, int J, int ts, int par)
  {
    int n = 0;
    for (int K = 0; K < I; K++)
      if (owns(K, ts, par)) n += T - K;
    return n + (J - I);
  }
  // Column order inside the kernel: POSITION 0 is tau, then the link blocks from the LAST link to the first (position of column 10 l + p:
  // 1 + 10 (NJ-1-l) + p).  The row of joint j is non-zero in the blocks of the links >= j, i.e. in the positions [0, rowlen(j)) -- a prefix,
  // aligned with the 8-wide tiles at its start, ragged only at its end: row j needs the tiles I, K < tj(j) (C6: 104 DMMA per 4 samples;
  // with the natural order, where a row starts at column 10 j in the middle of a tile, it was 109).
  __host__ __device__ static constexpr int pos(int l, int p) { return 1 + 10 * (NJ - 1 - l) + (Z ? (p == 0 ? 9 : p - 1) : p); }
  __host__ __device__ static constexpr int rowlen(int j) { return 1 + 10 * (NJ - j) - Z; }
  __host__ __device__ static constexpr int tj(int j) { return (rowlen(j) + 7) / 8; }
  // cross mode: per joint row j the tiles (regular tile I, component tile of joint j), I = 0 .. tj(j)-1, then (component, component)
  __host__ __device__ static constexpr int xtile(int j, int I)  // I == tj(j): the (component, component) tile
  {
    int n = 0;
    for (int k = 0; k < j; k++) n += tj(k) + 1;
    return n + I;
  }
  __host__ __device__ static constexpr int nxt()
  {
    int n = 0;
    for (int k = 0; k < NJ; k++) n += tj(k) + 1;
    return n;
  }
  static constexpr int NXT = nxt();
  __host__ __device__ static constexpr bool xowns(int j, int I, int ts, int par) { return ts == 1 || ((I == tj(j) ? j : I) & 1) == par; }
  __host__ __device__ static constexpr int xlocal(int j, int I, int ts, int par)
  {
    int n = 0;
    for (int k = 0; k <= j; k++)
      for (int K = 0; K <= tj(k); K++)
      {
        if (k == j && K == I) return n;
        if (xowns(k, K, ts, par)) n++;
      }
    return n;
  }
  __host__ __device__ static constexpr int nxtiles(int ts, int par)
  {
    int n = 0;
    for (int k = 0; k < NJ; k++)
      for (int K = 0; K <= tj(k); K++)
        if (xowns(k, K, ts, par)) n++;
    return n;
  }
};

// components of the joints of the folded chain (cross mode): the columns they contribute to the row of their joint, one entry per column
enum : int
{
  GXK_SAT = 1,    // FirstOrderPolynomialFriction column 0: clamp(omega / thr, -1, 1)           (friction_polynomial1.h:47-50)
  GXK_OMEGA = 2,  // column 1 of both friction models: omega = clamp(Dq, -vmax, vmax)
  GXK_SGN = 3,    // SecondOrderPolynomialFriction column 0: 0 / +-1 / omega / thr              (friction_polynomial2.h:44-53)
  GXK_SQ = 4,     // SecondOrderPolynomialFriction column 2: omega^2 * (that sign)
  GXK_Q = 5,      // IdealSpring column 0: q                                                    (ideal_spring.h:64-70)
  GXK_ONE = 6     // IdealSpring column 1: 1
};
struct GramComps
{
  int32_t ncols[8];
  int32_t kind[8][GX_COLS];
  double thr[8][GX_COLS], vmax[8][GX_COLS];
  double ithr[8][GX_COLS];  // 1 / thr (the normal equations multiply by it: a double division costs ~35 FP64 instructions; the materialised
                            // component regressor of components.cu keeps the reference's division)
};

// ---------------------------------------------------------------------------------------------- generator
template <int NJ>
struct GenIn
{
  double q[NJ], dq[NJ], ddq[NJ], sv[NJ], cv[NJ];
};
template <int NJ>
__device__ __forceinline__ void gen_load(const ChainDev<NJ>& C, const SamplesDev& in, int64_t i, GenIn<NJ>& x)
{
#pragma unroll
  for (int l = 0; l < NJ; l++)
  {
    x.q[l] = ld_in(in.q, C.joint[l].in, in.ld, i);
    x.dq[l] = ld_in(in.dq, C.joint[l].in, in.ld, i);
    x.ddq[l] = ld_in(in.ddq, C.joint[l].in, in.ld, i);
  }
}

// One sample per lane: all rows of getRegressor (+ getJointTorque) of sample i written to the slot.
// REV: every joint of the (folded) chain is revolute about e_z of its link frame -- the usual arm, in the canonical frames of fold.cpp.  The
// joint type and the axis are then compile-time facts: R = A' Rz(q) mixes two columns of A', the rates gain their e_z terms directly, the
// first transport of a joint's unit twist [0; e_z] is a row of R, and the projection of a link on its own joint has closed forms with two
// exact zeros (the mass and m c_z columns).
// Component columns of every joint row (element-wise in q_j, Dq_j; zero padded to one tile), written after the walk by ONE rolled loop over
// (joint, column): no call (a called function costs the walker its registers through the ABI -- it spilled 280 bytes per thread into an L1
// that the slots leave at ~20 KB), little code, and the walk stays one basic block.
template <int NJ>
__device__ __forceinline__ void gram_component_columns(const ChainDev<NJ>& C, const GramComps& comps, const SamplesDev& in, int64_t i,
                                                       double* __restrict__ slot, int lane)
{
  using G = GramGeom<NJ, 1>;
  // q_j / Dq_j are read again (L2 hits; keeping them in registers through the walk spills), ALL joints at once so that the loads overlap;
  // joint loop unrolled, column loop rolled: little code, no call
  double qv[NJ], dqv[NJ];
#pragma unroll
  for (int j = 0; j < NJ; j++)
  {
    qv[j] = ld_in(in.q, C.joint[j].in, in.ld, i);
    dqv[j] = ld_in(in.dq, C.joint[j].in, in.ld, i);
  }
  static_for<0, NJ>([&](auto jc) {
    constexpr int j = decltype(jc)::value;
    const double q = qv[j], dq = dqv[j];
    const int nc = comps.ncols[j];
    double* o = slot + G::rowbase(j) + G::rowlen(j) * 32;
#pragma unroll 1
    for (int c = 0; c < GX_COLS; c++)
    {
      double val = 0.0;
      if (c < nc)
      {
        const int kd = comps.kind[j][c];
        const double th = comps.thr[j][c], vm = comps.vmax[j][c];
        const double omega = fmin(fmax(dq, -vm), vm);
        if (kd == GXK_OMEGA) val = omega;
        else if (kd == GXK_Q) val = q;
        else if (kd == GXK_ONE) val = 1.0;
        else
        {
          const double r = omega * comps.ithr[j][c];
          if (kd == GXK_SAT) val = fmin(fmax(r, -1.0), 1.0);
          else
          {
            const double sg = omega == 0.0 ? 0.0 : (omega > th ? 1.0 : (omega < -th ? -1.0 : r));
            val = kd == GXK_SGN ? sg : omega * omega * sg;
          }
        }
      }
      o[c * 32 + (lane ^ (4 * (c & 3)))] = val;
    }
  });
}

// GLOBAL: the rows go to an L2-resident ring entry in global memory (st.global.cg: no L1 allocation) instead of a shared-memory slot
template <bool GLOBAL>
__device__ __forceinline__ void st_row(double* p, double v)
{
  if (GLOBAL) __stcg(p, v);
  else *p = v;
}

// LAZY: Dq / DDq of a link are loaded inside the walk (the compiler hoists them as far as registers allow) instead of being held in registers
// from before the wait for the output buffer: with two generator warps per sub-partition the latency hides behind the other warp
template <int NJ, bool REV, int X, int Z = 0, bool GLOBAL = false, bool LAZY = false>
__device__ __forceinline__ void gram_generate(const ChainDev<NJ>& C, const GramComps* comps, const GenIn<NJ>& x, const SamplesDev& in,
                                              const double* __restrict__ tau_meas, double* __restrict__ slot, int64_t i, int lane)
{
  static_assert(!Z || REV, "the zero mass column of a link on its own joint exists for revolute joints only");
  static_assert(REV_AXIS[0] == 0.0 && REV_AXIS[1] == 0.0 && REV_AXIS[2] == 1.0, "the REV walk below is written for the axis s = e_z");
  using G = GramGeom<NJ, X, Z>;
  constexpr int P = G::P;

  V3 U[NJ], S[NJ];
  double tau[NJ];
  V3 v = v3(0, 0, 0), w = v3(0, 0, 0), a = v3(0, 0, 0), al = v3(0, 0, 0);
  V3 g = v3(C.g);
#pragma unroll
  for (int l = 0; l < NJ; l++)
  {
    const JointDev& J = C.joint[l];
    const double dql = LAZY ? ld_in(in.dq, J.in, in.ld, i) : x.dq[l], ddql = LAZY ? ld_in(in.ddq, J.in, in.ld, i) : x.ddq[l];
    double R[9];
    const V3 t = REV || J.type != RDB_JOINT_PRISMATIC ? v3(J.t) : axpy(v3(J.t), v3(J.axp), x.q[l]);
    if (REV)
    {
#pragma unroll
      for (int k = 0; k < 3; k++)
      {
        R[3 * k] = fma(x.sv[l], J.A[3 * k + 1], x.cv[l] * J.A[3 * k]);
        R[3 * k + 1] = fma(-x.sv[l], J.A[3 * k], x.cv[l] * J.A[3 * k + 1]);
        R[3 * k + 2] = J.A[3 * k + 2];
      }
    }
    else if (J.type == RDB_JOINT_REVOLUTE)
    {
      const double c1 = 1.0 - x.cv[l];
#pragma unroll
      for (int k = 0; k < 9; k++) R[k] = fma(c1, J.C[k], fma(x.sv[l], J.B[k], J.A[k]));
    }
    else
    {
#pragma unroll
      for (int k = 0; k < 9; k++) R[k] = J.A[k];
    }
    v = rotT(R, cross_add(v, w, t));
    w = rotT(R, w);
    a = rotT(R, cross_add(a, al, t));
    al = rotT(R, al);
    g = rotT(R, g);
    if (REV)
    {
      // s = e_z:  w += s Dq,  a += (v x s) Dq,  al += (w x s) Dq + s DDq
      w.z += dql;
      a.x = fma(v.y, dql, a.x);
      a.y = fma(-v.x, dql, a.y);
      al.x = fma(w.y, dql, al.x);
      al.y = fma(-w.x, dql, al.y);
      al.z += ddql;
    }
    else
    {
      const V3 axj = v3(J.ax);
      const V3 su = J.type == RDB_JOINT_PRISMATIC ? axj : v3(0, 0, 0);
      const V3 ss = J.type == RDB_JOINT_REVOLUTE ? axj : v3(0, 0, 0);
      v = axpy(v, su, dql);
      w = axpy(w, ss, dql);
      const V3 xl = cross_add(cross(w, su), v, ss);
      const V3 xa = cross(w, ss);
      a = axpy(axpy(a, xl, dql), su, ddql);
      al = axpy(axpy(al, xa, dql), ss, ddql);
      U[l] = su;
      S[l] = ss;
    }
#pragma unroll
    for (int j = 0; j < l; j++)
    {
      if (REV && j == l - 1)  // [0; e_z] of joint l-1 moved to link l: S = R^T e_z, U = R^T (e_z x t)
      {
        S[j] = v3(R[6], R[7], R[8]);
        U[j] = v3(fma(t.x, R[3], -(t.y * R[0])), fma(t.x, R[4], -(t.y * R[1])), fma(t.x, R[5], -(t.y * R[2])));
      }
      else
      {
        U[j] = rotT(R, cross_add(U[j], S[j], t));
        S[j] = rotT(R, S[j]);
      }
    }
    tau[l] = 0.0;
    const double* Pl = C.link[l].pi;
    const V3 fm = cross_add(a - g, w, v);
#pragma unroll
    for (int j = 0; j <= l; j++)
    {
      const bool own = REV && j == l;  // unit twist [0; e_z]: u = 0, h = fm x e_z, rho = e_z x w
      double e[10];
      if (own)
      {
        e[0] = 0.0;
        e[1] = fm.y;
        e[2] = -fm.x;
        e[3] = 0.0;
        e[7] = w.x * w.y;
        e[4] = -e[7];
        e[5] = fma(w.x, w.x, -(w.y * w.y));
        e[6] = fma(-w.y, w.z, al.x);
        e[8] = fma(w.x, w.z, al.y);
        e[9] = al.z;
      }
      else
      {
        const V3 u = U[j], s = S[j];
        const V3 h = cross_add(cross_add(cross(u, al), w, cross(w, u)), fm, s);
        const V3 rho = cross(s, w);
        e[0] = dot(u, fm);
        e[1] = h.x;
        e[2] = h.y;
        e[3] = h.z;
        e[4] = fma(s.x, al.x, rho.x * w.x);
        e[5] = fma(s.x, al.y, fma(s.y, al.x, fma(rho.x, w.y, rho.y * w.x)));
        e[6] = fma(s.x, al.z, fma(s.z, al.x, fma(rho.x, w.z, rho.z * w.x)));
        e[7] = fma(s.y, al.y, rho.y * w.y);
        e[8] = fma(s.y, al.z, fma(s.z, al.y, fma(rho.y, w.z, rho.z * w.y)));
        e[9] = fma(s.z, al.z, rho.z * w.z);
      }
      // tau_j += Phi_{j,l,:} . pi_l in two independent chains (the exact zeros of the own joint are not multiplied)
      double t0 = tau[j], t1 = e[1] * Pl[1];
#pragma unroll
      for (int p = 0; p < 10; p += 2)
        if (!(own && p == 0)) t0 = fma(e[p], Pl[p], t0);
#pragma unroll
      for (int p = 3; p < 10; p += 2)
        if (!(own && p == 3)) t1 = fma(e[p], Pl[p], t1);
      tau[j] = t0 + t1;
      double* o = slot + G::rowbase(j);
#pragma unroll
      for (int p = 0; p < 10; p++)
        if (!(Z && own && p == 0))  // Z: the exact zero at the end of the row is not stored
          st_row<GLOBAL>(o + G::pos(l, p) * 32 + (lane ^ (4 * (G::pos(l, p) & 3))), e[p]);
    }
  }
#pragma unroll
  for (int j = 0; j < NJ; j++)
  {
    const double tv = tau_meas ? __ldcs(tau_meas + (int64_t)C.joint[j].in * in.ld + i) : tau[j];
    st_row<GLOBAL>(slot + G::rowbase(j) + lane, tv);  // position 0
  }
  if (X) gram_component_columns<NJ>(C, *comps, in, i, slot, lane);
}

// lanes past the end of the batch (last group only): their rows become exact zeros
template <int NJ, int X, int Z = 0, bool GLOBAL = false>
__device__ __noinline__ void gram_zero_lane(double* __restrict__ slot, int lane)
{
  using G = GramGeom<NJ, X, Z>;
  for (int j = 0; j < NJ; j++)
  {
    for (int c = 0; c < G::rowlen(j); c++) st_row<GLOBAL>(slot + G::rowbase(j) + c * 32 + (lane ^ (4 * (c & 3))), 0.0);
    if (X)
      for (int c = 0; c < GX_COLS; c++) st_row<GLOBAL>(slot + G::rowbase(j) + (G::rowlen(j) + c) * 32 + (lane ^ (4 * (c & 3))), 0.0);
  }
}

}  // namespace rdb
