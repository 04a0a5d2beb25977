// gram_common.cuh -- pieces shared by the fused regressor -> normal-equation kernels (gram_fused.cuh): geometry of the augmented Gram
// matrix and of a slot, the DMMA wrapper, and the per-sample regressor generator.
// The header is also compiled at run time by NVRTC (gram_jit.cpp), which has no system headers: it needs chain_dev.h and spatial.cuh only.
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#endif

#include "chain_dev.h"
#include "spatial.cuh"

namespace rdb
{

constexpr int GF_KSPLIT = 4;                   // MMA warps that share the k-steps of a slot (one per SM sub-partition)
constexpr int GF_MMA_WARPS = 2 * GF_KSPLIT;    // two per sub-partition: they split the tile rows by parity
constexpr int GF_GENS = GF_KSPLIT;             // generator warps: one per sub-partition, whatever the number of slots
constexpr int GF_THREADS = 32 * (GF_MMA_WARPS + GF_GENS);
constexpr int GF_MAX_SLOTS = 4;   // 32-sample slots in shared memory: as many as fit the 227 KB (3 for a 7-joint chain, 4 from 6 joints down);
                                  // 8 MMA + 4 generator warps = 3 warps per SM sub-partition is also what the 168-register budget allows
constexpr int GF_BAR_REDUCE = 1;  // named barrier of the final k-split reduction (0 is __syncthreads)

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void dmma884f(double& d0, double& d1, double a, double b)
{
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int V>
struct ic
{
  static constexpr int value = V;
};
// compile-time loop: f(ic<B>) ... f(ic<E - 1>), so that indices derived from the loop variable are constant expressions (accumulator arrays
// indexed through constexpr tables must stay in registers)
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f)
{
  if constexpr (B < E)
  {
    f(ic<B>{});
    static_for<B + 1, E>(f);
  }
}

// geometry of the augmented Gram matrix and of a slot for a (folded) chain of NJ joints, all of them inputs.
constexpr int GX_COLS = 8;  // component columns per joint row (extended model: one 8-wide cross tile)
// Z = 1 (all-revolute chains, extended model): the projection of a link on its OWN revolute joint has no mass term (the unit
// twist at birth is [0; axis], so Phi[j, 10 j + 0] == 0 exactly).  Inside every link block the mass column therefore comes LAST (p order
// 1..9, 0): the row of joint j then ends with an exact zero that is neither stored nor multiplied -- rowlen(j) = 10 (NJ - j), and position
// 10 NJ (the mass of the first moving link, an identically zero column of Phi) is never touched.
// Z = 2 (all-revolute chains, rigid-body model) drops every column that the REV walk (gram_walk_rev) makes an exact zero:
//   * the own-joint projection [0; e_z] has m c_z == 0 as well as m == 0 (gram_walk_rev, branch j == l);
//   * the first moving link sits on the fixed base: there v = a = 0, w = (0, 0, Dq_0), alpha = (0, 0, DDq_0), so of its own-joint closed
//     forms only I_zz = alpha_z, m c_x = fm_y and m c_y = -fm_x are not exact zeros (I_xx, I_xy, I_xz, I_yy, I_yz are -w_x w_y,
//     w_x^2 - w_y^2, fma(-w_y, w_z, alpha_x), w_x w_y, fma(w_x, w_z, alpha_y) with w_x = w_y = alpha_x = alpha_y = 0).  Link 0 appears in
//     row 0 only, so these seven are identically zero columns of Phi and have no position at all.
// Inside every link block the order is I_zz, m c_x, m c_y, I_xx .. I_yz, m c_z, m (inblk): the own block of row j >= 1 is the first 8
// positions of its block, that of row 0 the first 3.  tau is no column of the tiles either (TC == 0): its row sits behind the regressor rows
// of the slot and the MMA warps accumulate Phi^T tau and tau^T tau by DFMA on the fragments they load for the DMMAs (gram_tau_step):
// rowlen(0) = 10 (NJ - 1) + 3, rowlen(j >= 1) = 10 (NJ - j) - 2, C6 81 instead of 98 DMMA per 4 samples (90 with tau as tile column 0).
template <int NJ, int Z = 0>
struct GramGeom
{
  static constexpr int P = 10 * NJ;
  static constexpr int TC = Z == 2 ? 0 : 1;  // tau positions in front of the link blocks (position 0 when TC == 1)
  // place of parameter p (m, m c_xyz, I_xx, I_xy, I_xz, I_yy, I_yz, I_zz) inside its link block, and back
  __host__ __device__ static constexpr int inblk(int p)
  {
    constexpr int zord[10] = {9, 1, 2, 8, 3, 4, 5, 6, 7, 0};
    return Z == 2 ? zord[p] : (Z == 1 ? (p == 0 ? 9 : p - 1) : p);
  }
  __host__ __device__ static constexpr int param_at(int q)
  {
    constexpr int zinv[10] = {9, 1, 2, 4, 5, 6, 7, 8, 3, 0};
    return Z == 2 ? zinv[q] : (Z == 1 ? (q == 9 ? 0 : q + 1) : q);
  }
  // Column order inside the kernel: tau (TC == 1: POSITION 0), then the link blocks from the LAST link to the first (position of column
  // 10 l + p: TC + 10 (NJ-1-l) + inblk(p)).  The row of joint j is non-zero in the blocks of the links >= j, i.e. in the positions
  // [0, rowlen(j)) -- a prefix, aligned with the 8-wide tiles at its start, ragged only at its end: row j needs the tiles I, K < tj(j)
  // (with the natural order, where a row starts at column 10 j in the middle of a tile, C6 took 109 DMMA per 4 samples).
  __host__ __device__ static constexpr int pos(int l, int p) { return TC + 10 * (NJ - 1 - l) + inblk(p); }
  // is column 10 l + p of the row of joint j (l >= j) stored, i.e. not one of the exact zeros the layout drops
  __host__ __device__ static constexpr bool stored(int j, int l, int p)
  {
    if (j != l || Z == 0) return true;
    if (Z == 1) return p != 0;
    return l == 0 ? (p == 1 || p == 2 || p == 9) : (p != 0 && p != 3);
  }
  __host__ __device__ static constexpr int rowlen(int j)
  {
    return Z == 2 ? TC + 10 * (NJ - 1 - j) + (j == 0 ? 3 : 8) : 1 + 10 * (NJ - j) - Z;
  }
  static constexpr int NPOS = rowlen(0);  // positions that exist
  // parameter column at a position (P: tau), and whether a parameter column has a position (else it is identically zero in Phi)
  __host__ __device__ static constexpr int col_of(int q) { return q < TC ? P : 10 * (NJ - 1 - (q - TC) / 10) + param_at((q - TC) % 10); }
  __host__ __device__ static constexpr bool has_pos(int c) { return c / 10 > 0 || stored(0, 0, c % 10); }
  static constexpr int T = (NPOS + 7) / 8;    // tile columns of the augmented matrix
  static constexpr int NT = T * (T + 1) / 2;  // upper-triangular tiles
  static constexpr int NF = T + 1 - TC;       // values a lane loads per k-step: one per tile column, then (TC == 0) the tau of its sample
  // per-CTA partial: the NT tiles (64 doubles each), then with TC == 0 b by position (8 T) and tau^T tau
  static constexpr int PARTIAL = NT * 64 + (TC ? 0 : 8 * T + 1);
  static constexpr int KPW = 8 / GF_KSPLIT;   // k-steps (4 samples) of one MMA warp per joint row and slot
  static constexpr int NSTEPS = NJ * KPW;     // k-steps of one MMA warp per slot
  // offset (doubles) of the row of joint j inside a slot: [position][sample], only the positions 0 .. rowlen(j)-1 are stored
  __host__ __device__ static constexpr int rowbase(int j)
  {
    int o = 0;
    for (int i = 0; i < j; i++) o += rowlen(i) * 32;
    return o;
  }
  // offset of the tau row of joint j: position 0 of its row, or (TC == 0) behind all rows, [joint][sample]
  __host__ __device__ static constexpr int taubase(int j) { return TC ? rowbase(j) : rowbase(NJ) + 32 * j; }
  static constexpr int SLOT_DOUBLES = rowbase(NJ) + (TC ? 0 : 32 * NJ);
  __host__ __device__ static constexpr int tile(int I, int J) { return I * T - I * (I - 1) / 2 + (J - I); }
  // tile rows owned by an MMA warp: the rows of parity `par`
  __host__ __device__ static constexpr bool owns(int I, int par) { return (I & 1) == par; }
  __host__ __device__ static constexpr int ntiles(int par)  // at least 1: a warp may own no tile row (T == 1), arrays need a size
  {
    int n = 0;
    for (int I = 0; I < T; I++)
      if (owns(I, par)) n += T - I;
    return n > 0 ? n : 1;
  }
  __host__ __device__ static constexpr int local(int I, int J, int par)
  {
    int n = 0;
    for (int K = 0; K < I; K++)
      if (owns(K, par)) n += T - K;
    return n + (J - I);
  }
  // TC == 0: DFMA accumulators of an MMA warp -- b at position 8 I + g for each tile row I it owns (lane (g, t): the samples t mod 4), then
  // in the par 0 warps tau^T tau; bown(I): the accumulator of tile row I
  __host__ __device__ static constexpr int bown(int I, int par)
  {
    int n = 0;
    for (int K = 0; K < I; K++)
      if (owns(K, par)) n++;
    return n;
  }
  __host__ __device__ static constexpr int nbacc(int par) { return TC || (par != 0 && bown(T, par) == 0) ? 1 : bown(T, par) + (par == 0 ? 1 : 0); }
  __host__ __device__ static constexpr int tj(int j) { return (rowlen(j) + 7) / 8; }
  // extended model: per joint row j the cross tiles (regular tile I, component tile of joint j), I = 0 .. tj(j)-1, then (component, component)
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
  __host__ __device__ static constexpr bool xowns(int j, int I, int par) { return ((I == tj(j) ? j : I) & 1) == par; }
  __host__ __device__ static constexpr int xlocal(int j, int I, int par)
  {
    int n = 0;
    for (int k = 0; k <= j; k++)
      for (int K = 0; K <= tj(k); K++)
      {
        if (k == j && K == I) return n;
        if (xowns(k, K, par)) n++;
      }
    return n;
  }
  __host__ __device__ static constexpr int nxtiles(int par)
  {
    int n = 0;
    for (int k = 0; k < NJ; k++)
      for (int K = 0; K <= tj(k); K++)
        if (xowns(k, K, par)) n++;
    return n;
  }
};

// components of the joints of the folded chain (extended model): the columns they contribute to the row of their joint, one entry per column
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

// ---------------------------------------------------------------------------------------------- model constants and typed arithmetic
// The walk reads the model (A' and t' of every folded joint, the lumped parameters pi', gravity) through kc<M, ...>.  RtModel: the
// __grid_constant__ ChainDev of the kernel, values ptxas cannot see (the precompiled kernels).  Any other M is a type generated at run time
// for one chain (gram_jit.cpp) whose constexpr M::val(field, link, k) holds the exact values: kc then returns Zr for an exact 0, Un<+-1> for
// an exact +-1 and the value itself otherwise, and the t* operations below drop a product with Zr and turn one with Un into a pass-through or
// a negation.  Everything else is the same operation in the same order as with RtModel (no reassociation, no snapping of tiny values), so for
// finite inputs the results are bit-identical up to the sign of exact zeros.  The t* operations use the _rn intrinsics, which are never
// contracted: a product that loses its addend must not be fused into a later addition that the precompiled kernel rounds separately.
struct RtModel
{
  static constexpr bool RUNTIME = true;
};
enum : int
{
  MK_A = 0,   // A'[link][0..8]
  MK_T = 1,   // t'[link][0..2]
  MK_PI = 2,  // pi'[link][0..9]
  MK_G = 3    // g[0..2]
};
struct Zr
{
};
template <int S>
struct Un
{
};
template <class T>
struct tv_unit
{
  static constexpr int s = 0;
};
template <int S>
struct tv_unit<Un<S>>
{
  static constexpr int s = S;
};
template <class T>
struct tv_zero
{
  static constexpr bool v = false;
};
template <>
struct tv_zero<Zr>
{
  static constexpr bool v = true;
};

template <class M, int F, int L, int K, int NJ>
__device__ __forceinline__ auto kc(const ChainDev<NJ>& C)
{
  if constexpr (M::RUNTIME)
  {
    if constexpr (F == MK_A) return C.joint[L].A[K];
    else if constexpr (F == MK_T) return C.joint[L].t[K];
    else if constexpr (F == MK_PI) return C.link[L].pi[K];
    else return C.g[K];
  }
  else
  {
    constexpr double v = M::val(F, L, K);
    if constexpr (v == 0.0) return Zr{};
    else if constexpr (v == 1.0) return Un<1>{};
    else if constexpr (v == -1.0) return Un<-1>{};
    else return v;
  }
}

template <class A>
__device__ __forceinline__ double tv_d(A a)
{
  if constexpr (tv_zero<A>::v) return 0.0;
  else if constexpr (tv_unit<A>::s != 0) return (double)tv_unit<A>::s;
  else return a;
}
template <class A>
__device__ __forceinline__ auto tneg(A a)
{
  if constexpr (tv_zero<A>::v) return Zr{};
  else if constexpr (tv_unit<A>::s != 0) return Un<-tv_unit<A>::s>{};
  else return -a;
}
template <class A, class B>
__device__ __forceinline__ auto tmul(A a, B b)
{
  constexpr int ua = tv_unit<A>::s, ub = tv_unit<B>::s;
  if constexpr (tv_zero<A>::v || tv_zero<B>::v) return Zr{};
  else if constexpr (ua != 0 && ub != 0) return Un<ua * ub>{};
  else if constexpr (ua != 0) return ua > 0 ? b : -b;
  else if constexpr (ub != 0) return ub > 0 ? a : -a;
  else return __dmul_rn(a, b);
}
template <class A, class B>
__device__ __forceinline__ auto tadd(A a, B b)
{
  if constexpr (tv_zero<A>::v) return b;
  else if constexpr (tv_zero<B>::v) return a;
  else return __dadd_rn(tv_d(a), tv_d(b));
}
// fma(a, b, c): with c == 0 the rounded product, with a or b == +-1 the rounded sum
template <class A, class B, class C>
__device__ __forceinline__ auto tfma(A a, B b, C c)
{
  using P = decltype(tmul(a, b));
  if constexpr (tv_zero<P>::v) return c;
  else if constexpr (tv_zero<C>::v) return tmul(a, b);
  else if constexpr (tv_unit<A>::s != 0 || tv_unit<B>::s != 0) return tadd(tmul(a, b), c);
  else return __fma_rn(a, b, tv_d(c));
}

template <class X, class Y, class W>
struct T3
{
  X x;
  Y y;
  W z;
};
template <class X, class Y, class W>
__device__ __forceinline__ T3<X, Y, W> mk3(X x, Y y, W z)
{
  return T3<X, Y, W>{x, y, z};
}
// the operations of spatial.cuh, in the same order, on typed vectors (V3 or T3)
template <class A, class B>
__device__ __forceinline__ auto tsub(const A& a, const B& b)
{
  return mk3(tadd(a.x, tneg(b.x)), tadd(a.y, tneg(b.y)), tadd(a.z, tneg(b.z)));
}
template <class A, class B>
__device__ __forceinline__ auto tdot(const A& a, const B& b)
{
  return tfma(a.x, b.x, tfma(a.y, b.y, tmul(a.z, b.z)));
}
template <class A, class B>
__device__ __forceinline__ auto tcross(const A& a, const B& b)
{
  return mk3(tfma(a.y, b.z, tneg(tmul(a.z, b.y))), tfma(a.z, b.x, tneg(tmul(a.x, b.z))), tfma(a.x, b.y, tneg(tmul(a.y, b.x))));
}
template <class Cv, class A, class B>
__device__ __forceinline__ auto tcross_add(const Cv& c, const A& a, const B& b)
{
  return mk3(tfma(a.y, b.z, tfma(tneg(a.z), b.y, c.x)), tfma(a.z, b.x, tfma(tneg(a.x), b.z, c.y)), tfma(a.x, b.y, tfma(tneg(a.y), b.x, c.z)));
}
// R^T a, R given by its rows R.x, R.y, R.z
template <class R, class A>
__device__ __forceinline__ auto trotT(const R& r, const A& a)
{
  return mk3(tfma(r.x.x, a.x, tfma(r.y.x, a.y, tmul(r.z.x, a.z))), tfma(r.x.y, a.x, tfma(r.y.y, a.y, tmul(r.z.y, a.z))),
             tfma(r.x.z, a.x, tfma(r.y.z, a.y, tmul(r.z.z, a.z))));
}

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

// the projection Phi[j, block of link L] = e of joint j's unit twist (u, s) moved to link L: tau_j += e . pi_L in two independent chains,
// e stored into the row of joint j.  OWN: the projection of a revolute link on its own joint (e[0] == e[3] == 0, typed Zr, not multiplied).
template <class M, int NJ, int Z, int L, int J, bool OWN, class E0, class E1, class E2, class E3, class E4, class E5, class E6,
          class E7, class E8, class E9>
__device__ __forceinline__ void gram_emit(const ChainDev<NJ>& C, double (&tau)[NJ], double* __restrict__ slot, int lane, E0 e0, E1 e1, E2 e2, E3 e3,
                                          E4 e4, E5 e5, E6 e6, E7 e7, E8 e8, E9 e9)
{
  using G = GramGeom<NJ, Z>;
  auto P = [&](auto pc) { return kc<M, MK_PI, L, decltype(pc)::value>(C); };
  auto t0a = [&] {  // joint L's torque starts here: from +0.0 as the precompiled kernel always did, from nothing with a compile-time model
    if constexpr (J == L && M::RUNTIME) return 0.0;
    else if constexpr (J == L) return Zr{};
    else return tau[J];
  }();
  const auto t0 = tfma(e8, P(ic<8>{}), tfma(e6, P(ic<6>{}), tfma(e4, P(ic<4>{}), tfma(e2, P(ic<2>{}), tfma(e0, P(ic<0>{}), t0a)))));
  const auto t1 = tfma(e9, P(ic<9>{}), tfma(e7, P(ic<7>{}), tfma(e5, P(ic<5>{}), tfma(e3, P(ic<3>{}), tmul(e1, P(ic<1>{}))))));
  tau[J] = tv_d(tadd(t0, t1));
  double* o = slot + G::rowbase(J);
  const double e[10] = {tv_d(e0), tv_d(e1), tv_d(e2), tv_d(e3), tv_d(e4), tv_d(e5), tv_d(e6), tv_d(e7), tv_d(e8), tv_d(e9)};
#pragma unroll
  for (int p = 0; p < 10; p++)
    if (G::stored(J, L, p))  // the exact zeros the layout drops are not stored
      o[G::pos(L, p) * 32 + (lane ^ (4 * (G::pos(L, p) & 3)))] = e[p];
}
template <class M, int NJ, int Z, int L, int J, class U, class S, class Fm, class W, class Al>
__device__ __forceinline__ void gram_project(const ChainDev<NJ>& C, double (&tau)[NJ], double* __restrict__ slot, int lane, const U& u, const S& s,
                                             const Fm& fm, const W& w, const Al& al)
{
  const auto h = tcross_add(tcross_add(tcross(u, al), w, tcross(w, u)), fm, s);
  const auto rho = tcross(s, w);
  gram_emit<M, NJ, Z, L, J, false>(
      C, tau, slot, lane, tdot(u, fm), h.x, h.y, h.z, tfma(s.x, al.x, tmul(rho.x, w.x)),
      tfma(s.x, al.y, tfma(s.y, al.x, tfma(rho.x, w.y, tmul(rho.y, w.x)))), tfma(s.x, al.z, tfma(s.z, al.x, tfma(rho.x, w.z, tmul(rho.z, w.x)))),
      tfma(s.y, al.y, tmul(rho.y, w.y)), tfma(s.y, al.z, tfma(s.z, al.y, tfma(rho.y, w.z, tmul(rho.z, w.y)))), tfma(s.z, al.z, tmul(rho.z, w.z)));
}

// One sample per lane: all rows of getRegressor (+ getJointTorque) of sample i written to the slot.
// REV: every joint of the (folded) chain is revolute about e_z of its link frame -- the usual arm, in the canonical frames of fold.cpp.  The
// joint type and the axis are then compile-time facts: R = A' Rz(q) mixes two columns of A', the rates gain their e_z terms directly, the
// first transport of a joint's unit twist [0; e_z] is a row of R, and the projection of a link on its own joint has closed forms with two
// exact zeros (the mass and m c_z columns).  M: where the model constants come from (RtModel, or a run-time generated model type).
// With a compile-time model the walk's state stays typed as well (T3 of double / Zr / Un): the base at rest, gravity, the rate terms and the
// carried unit twists keep the exact zeros and ones they inherit from the model, so their products are not issued either.  The types change
// from link to link, hence one function instantiation per link (gram_rev_link) that takes the state by value, and the carried twists of the
// earlier joints as a pack that grows by one per link (RevTwists).  With RtModel every component is a double and the code is the
// precompiled walk.

// the unit twists (U_j, S_j) of joints 0 .. N-1 moved to the current link: the last joint in front, the earlier ones in `rest`
struct RevTwistsEnd
{
  static constexpr int N = 0;
};
template <class U, class S, class Rest>
struct RevTwists
{
  static constexpr int N = Rest::N + 1;
  U u;
  S s;
  Rest rest;
};
template <class U, class S, class Rest>
__device__ __forceinline__ RevTwists<U, S, Rest> mk_twists(const U& u, const S& s, const Rest& rest)
{
  return RevTwists<U, S, Rest>{u, s, rest};
}
// every twist of the pack moved one link further: U = R^T (U + S x t), S = R^T S
template <class R, class T, class P>
__device__ __forceinline__ auto rev_transport(const R& r, const T& t, const P& p)
{
  if constexpr (P::N == 0) return p;
  else
  {
    const auto rest = rev_transport(r, t, p.rest);
    return mk_twists(trotT(r, tcross_add(p.u, p.s, t)), trotT(r, p.s), rest);
  }
}
// the projections of link L on the joints of the pack (joint P::N - 1 in front)
template <class M, int NJ, int Z, int L, class P, class Fm, class W, class Al>
__device__ __forceinline__ void rev_project(const ChainDev<NJ>& C, double (&tau)[NJ], double* __restrict__ slot, int lane, const P& p, const Fm& fm,
                                            const W& w, const Al& al)
{
  if constexpr (P::N > 0)
  {
    rev_project<M, NJ, Z, L>(C, tau, slot, lane, p.rest, fm, w, al);
    gram_project<M, NJ, Z, L, P::N - 1>(C, tau, slot, lane, p.u, p.s, fm, w, al);
  }
}

// link L of the REV walk: v, w, a, al, g of link L-1 (L == 0: the base at rest and the model's gravity) and the twists of joints 0 .. L-2
// moved to link L-1
template <int L, int NJ, class M, int Z, class V, class W, class A, class Al, class G, class P>
__device__ __forceinline__ void gram_rev_link(const ChainDev<NJ>& C, const GenIn<NJ>& x, double* __restrict__ slot, int lane, double (&tau)[NJ],
                                              const V& vp, const W& wp, const A& ap, const Al& alp, const G& gp, const P& twists)
{
  if constexpr (L < NJ)
  {
    const double dql = x.dq[L], ddql = x.ddq[L];
    const double sl = x.sv[L], cl = x.cv[L];
    const auto t = mk3(kc<M, MK_T, L, 0>(C), kc<M, MK_T, L, 1>(C), kc<M, MK_T, L, 2>(C));
    // R = A' Rz(q), row k: (fma(s, A'[k][1], c A'[k][0]), fma(-s, A'[k][0], c A'[k][1]), A'[k][2])
    auto row = [&](auto kc_) {
      constexpr int k = decltype(kc_)::value;
      const auto a0 = kc<M, MK_A, L, 3 * k>(C);
      const auto a1 = kc<M, MK_A, L, 3 * k + 1>(C);
      return mk3(tfma(sl, a1, tmul(cl, a0)), tfma(-sl, a0, tmul(cl, a1)), kc<M, MK_A, L, 3 * k + 2>(C));
    };
    const auto R = mk3(row(ic<0>{}), row(ic<1>{}), row(ic<2>{}));
    const auto v = trotT(R, tcross_add(vp, wp, t));
    const auto wr = trotT(R, wp);
    const auto ar = trotT(R, tcross_add(ap, alp, t));
    const auto alr = trotT(R, alp);
    const auto g = trotT(R, gp);
    // s = e_z:  w += s Dq,  a += (v x s) Dq,  al += (w x s) Dq + s DDq
    const auto w = mk3(wr.x, wr.y, tadd(wr.z, dql));
    const auto a = mk3(tfma(v.y, dql, ar.x), tfma(tneg(v.x), dql, ar.y), ar.z);
    const auto al = mk3(tfma(w.y, dql, alr.x), tfma(tneg(w.x), dql, alr.y), tadd(alr.z, ddql));
    // [0; e_z] of joint L-1 moved to link L: S = R^T e_z, U = R^T (e_z x t), in front of the earlier joints' twists moved on
    const auto moved = [&] {
      if constexpr (L == 0) return twists;
      else
        return mk_twists(mk3(tfma(t.x, R.y.x, tneg(tmul(t.y, R.x.x))), tfma(t.x, R.y.y, tneg(tmul(t.y, R.x.y))),
                             tfma(t.x, R.y.z, tneg(tmul(t.y, R.x.z)))),
                         R.z, rev_transport(R, t, twists));
    }();
    const auto fm = tcross_add(tsub(a, g), w, v);
    rev_project<M, NJ, Z, L>(C, tau, slot, lane, moved, fm, w, al);
    // own joint, unit twist [0; e_z]: u = 0, h = fm x e_z, rho = e_z x w
    const auto e7 = tmul(w.x, w.y);
    gram_emit<M, NJ, Z, L, L, true>(C, tau, slot, lane, Zr{}, fm.y, tneg(fm.x), Zr{}, tneg(e7), tfma(w.x, w.x, tneg(tmul(w.y, w.y))),
                                    tfma(tneg(w.y), w.z, al.x), e7, tfma(w.x, w.z, al.y), al.z);
    gram_rev_link<L + 1, NJ, M, Z>(C, x, slot, lane, tau, v, w, a, al, g, moved);
  }
}

template <int NJ, class M, int Z>
__device__ __forceinline__ void gram_walk_rev(const ChainDev<NJ>& C, const GenIn<NJ>& x, double* __restrict__ slot, int lane, double (&tau)[NJ])
{
  static_assert(REV_AXIS[0] == 0.0 && REV_AXIS[1] == 0.0 && REV_AXIS[2] == 1.0, "the REV walk below is written for the axis s = e_z");
  // the base is at rest: v = w = a = al = 0 (with RtModel doubles of +0.0, like every other value there)
  const auto z = [] {
    if constexpr (M::RUNTIME) return 0.0;
    else return Zr{};
  }();
  const auto z3 = mk3(z, z, z);
  gram_rev_link<0, NJ, M, Z>(C, x, slot, lane, tau, z3, z3, z3, z3, mk3(kc<M, MK_G, 0, 0>(C), kc<M, MK_G, 0, 1>(C), kc<M, MK_G, 0, 2>(C)),
                             RevTwistsEnd{});
}

// any joint types and axes (the constant-bank model)
template <int NJ, int Z>
__device__ __forceinline__ void gram_walk_gen(const ChainDev<NJ>& C, const GenIn<NJ>& x, double* __restrict__ slot, int lane, double (&tau)[NJ])
{
  using G = GramGeom<NJ, Z>;
  V3 U[NJ], S[NJ];
  V3 v = v3(0, 0, 0), w = v3(0, 0, 0), a = v3(0, 0, 0), al = v3(0, 0, 0);
  V3 g = v3(C.g);
#pragma unroll
  for (int l = 0; l < NJ; l++)
  {
    const JointDev& J = C.joint[l];
    const double dql = x.dq[l], ddql = x.ddq[l];
    double R[9];
    const V3 t = J.type != RDB_JOINT_PRISMATIC ? v3(J.t) : axpy(v3(J.t), v3(J.axp), x.q[l]);
    if (J.type == RDB_JOINT_REVOLUTE)
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
#pragma unroll
    for (int j = 0; j < l; j++)
    {
      U[j] = rotT(R, cross_add(U[j], S[j], t));
      S[j] = rotT(R, S[j]);
    }
    tau[l] = 0.0;
    const double* Pl = C.link[l].pi;
    const V3 fm = cross_add(a - g, w, v);
#pragma unroll
    for (int j = 0; j <= l; j++)
    {
      const V3 u = U[j], s = S[j];
      const V3 h = cross_add(cross_add(cross(u, al), w, cross(w, u)), fm, s);
      const V3 rho = cross(s, w);
      double e[10];
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
      // tau_j += Phi_{j,l,:} . pi_l in two independent chains
      double t0 = tau[j], t1 = e[1] * Pl[1];
#pragma unroll
      for (int p = 0; p < 10; p += 2) t0 = fma(e[p], Pl[p], t0);
#pragma unroll
      for (int p = 3; p < 10; p += 2) t1 = fma(e[p], Pl[p], t1);
      tau[j] = t0 + t1;
      double* o = slot + G::rowbase(j);
#pragma unroll
      for (int p = 0; p < 10; p++) o[G::pos(l, p) * 32 + (lane ^ (4 * (G::pos(l, p) & 3)))] = e[p];
    }
  }
}

template <int NJ, bool REV, int Z, class M>
__device__ __forceinline__ void gram_generate(const ChainDev<NJ>& C, const GenIn<NJ>& x, const SamplesDev& in, const double* __restrict__ tau_meas,
                                              double* __restrict__ slot, int64_t i, int lane)
{
  static_assert(!Z || REV, "the zero mass column of a link on its own joint exists for revolute joints only");
  static_assert(REV || M::RUNTIME, "compile-time models are built for the REV walk");
  using G = GramGeom<NJ, Z>;
  double tau[NJ];
  if constexpr (REV) gram_walk_rev<NJ, M, Z>(C, x, slot, lane, tau);
  else gram_walk_gen<NJ, Z>(C, x, slot, lane, tau);
#pragma unroll
  for (int j = 0; j < NJ; j++)
  {
    const double tv = tau_meas ? __ldcs(tau_meas + (int64_t)C.joint[j].in * in.ld + i) : tau[j];
    slot[G::taubase(j) + lane] = tv;
  }
}

// lanes past the end of the batch (last group only): their rows become exact zeros
template <int NJ, int Z>
__device__ __noinline__ void gram_zero_lane(double* __restrict__ slot, int lane)
{
  using G = GramGeom<NJ, Z>;
  for (int j = 0; j < NJ; j++)
  {
    for (int c = 0; c < G::rowlen(j); c++) slot[G::rowbase(j) + c * 32 + (lane ^ (4 * (c & 3)))] = 0.0;
    if (!G::TC) slot[G::taubase(j) + lane] = 0.0;
  }
}

}  // namespace rdb
