// Device-side recursive Newton-Euler inverse dynamics (reference dynamics/dynamics.py:109-157,
// Modern Robotics Eq. 8.50-8.54, twists in [v; w] order).
//
//   fast path   : fast_rnea<T, Desc>()   -- structure fixed at compile time (rbm_typed.cuh), one
//                 sample per thread, whole chain state in registers.
//   generic path: generic_rnea<T, NJ>()  -- any model, parameters read from shared memory.
#pragma once
#include "rbm_model.cuh"
#include "rbm_trig.cuh"
#include "rbm_typed.cuh"

namespace rbm {

// =================================================================================================
// Structure descriptors
// =================================================================================================
enum JointKind : int { JOINT_PZ = 0, JOINT_RZ = 1 };          // prismatic along +z / revolute about +z
enum InertiaKind : int { INERTIA_ISO = 0, INERTIA_RIGID = 1 }; // diag(m,m,m,I,I,I) / general rigid body

template <int JK, class Perm, bool HasT, int IK>
struct LinkD {
  static constexpr int jk = JK;
  using perm = Perm;               // home rotation hposes_body_parent[i+1].R as a signed permutation
  static constexpr bool has_t = HasT;  // home translation non-zero?
  static constexpr int ik = IK;
};

// The reference's manipulator (xml_models/manipulators/sequential.xml:13-39): x/y/z gantry then a
// roll/pitch/yaw wrist, every joint about its own +z, body eulers single-axis +-90 deg, all body and
// joint positions zero, links 1-5 an 8 kg isotropic block, link 6 the block plus attachment + object
// (core/simulate.py:129-137).  Home rotations below are hposes_lj_kj[1..6].R (core/simulate.py:140-146).
template <int IK15>
struct SequentialDesc {
  using L0 = LinkD<JOINT_PZ, SPerm<-3, 2, 1>, false, IK15>;
  using L1 = LinkD<JOINT_PZ, SPerm<1, -3, 2>, false, IK15>;
  using L2 = LinkD<JOINT_PZ, SPerm<3, 2, -1>, false, IK15>;
  using L3 = LinkD<JOINT_RZ, SPerm<1, 3, -2>, false, IK15>;
  using L4 = LinkD<JOINT_RZ, SPerm<-3, 2, 1>, false, IK15>;
  using L5 = LinkD<JOINT_RZ, SPerm<1, -3, 2>, false, INERTIA_RIGID>;
  // Does tau depend on q_j at all?  For the three leading prismatic joints it does not: a joint translation enters only
  // through p_j x (.) terms -- forward with the parent's angular velocity / acceleration (structurally zero: every earlier
  // joint is prismatic too) and backward in the MOMENT transported to links 0..2, which no prismatic joint force reads.
  // (The same dead-code argument is what lets nvcc drop those terms from the kernel.)  Used by the linearisation to skip
  // finite differences that are identically zero; verified against the oracle in tests/test_gpu_linearize.py.
  static constexpr bool q_matters(int j) { return j >= 3; }
  // Does tau depend on qd_j?  Not for the gantry joints either: a constant translation velocity of the whole wrist is a Galilean
  // boost (no rotation precedes those joints), so its contributions to G dV and ad(V)^T G V cancel identically -- numerically to
  // ~1e-13 in the oracle.  The cancellation is between separately rounded terms, so the typed algebra cannot see it; it is
  // declared here and checked against the oracle (tests/test_gpu_linearize.py::test_structure_of_the_euler_map).
  static constexpr bool qd_matters(int j) { return j >= 3; }
};
using SeqIso = SequentialDesc<INERTIA_ISO>;
using SeqRigid = SequentialDesc<INERTIA_RIGID>;

// =================================================================================================
// Fast path
// =================================================================================================
template <class VV, class WW, class AA, class LL, class PP, class BF, class BM>
struct LinkOut {
  VV v;   // linear part of the twist V_i
  WW w;   // angular part
  AA a;   // linear part of dV_i
  LL l;   // angular part
  PP p;   // translation of T_i = T_{i,i-1}
  BF bf;  // body wrench  G_i dV_i - ad(V_i)^T G_i V_i, force part
  BM bm;  // moment part
};
template <class VV, class WW, class AA, class LL, class PP, class BF, class BM>
RBM_HD LinkOut<VV, WW, AA, LL, PP, BF, BM> mk_link(VV v, WW w, AA a, LL l, PP p, BF bf, BM bm) {
  return {v, w, a, l, p, bf, bm};
}

// R_i x  with  R_i = Rz(-q) * P  (revolute)  or  P  (prismatic)
template <class L, class T, class V>
RBM_HD auto link_rot(T c, T s, const V& x) {
  auto y = sp_apply<typename L::perm>(x);
  if constexpr (L::jk == JOINT_RZ) return rotz_neg(c, s, y);
  else return y;
}
// R_i^T x
template <class L, class T, class V>
RBM_HD auto link_rot_T(T c, T s, const V& x) {
  if constexpr (L::jk == JOINT_RZ) return sp_apply_T<typename L::perm>(rotz_pos(c, s, x));
  else return sp_apply_T<typename L::perm>(x);
}

// b_i = G_i dV_i - ad(V_i)^T G_i V_i  (the two inertia terms of Eq. 8.53)
template <class L, int I, class T, class VV, class WW, class AA, class LL, class PP>
RBM_HD auto fwd_wrench(const FastParams<T>& P, const VV& v, const WW& w, const AA& a, const LL& l, const PP& p) {
  const T m = P.mass[I];
  if constexpr (L::ik == INERTIA_ISO) {
    // G = diag(m,m,m,J,J,J):  b = [ m (a + w x v) ;  J l ]   (w x Jw = 0, v x mv = 0)
    auto bf = scale(m, a + cross(w, v));
    auto bm = scale(P.I[I][0], l);
    return mk_link(v, w, a, l, p, bf, bm);
  } else {
    // G = [[m 1, -[h]x], [[h]x, Ibar]]
    auto h = ld3(P.h[I]);
    auto pl = scale(m, v) + cross(w, h);              // linear momentum
    auto pa = cross(h, v) + sym3_mul(P.I[I], w);      // angular momentum about the frame origin
    auto bf = scale(m, a) + cross(l, h) + cross(w, pl);
    auto bm = cross(h, a) + sym3_mul(P.I[I], l) + cross(v, pl) + cross(w, pa);
    return mk_link(v, w, a, l, p, bf, bm);
  }
}

// One forward step (Eq. 8.50-8.52) plus the link's body wrench.
template <class L, int I, class T, class QD, class QDD, class VV, class WW, class AA, class LL>
RBM_HD auto fwd_link(const FastParams<T>& P, T q, QD qd, QDD qdd, T c, T s, const VV& vp, const WW& wp, const AA& ap, const LL& lp) {
  // translation of T_i = exp(-S q) * M_i
  auto tm = [&] {
    if constexpr (L::has_t) return ld3(P.tm[I]);
    else return Z3{};
  }();
  auto p = [&] {
    if constexpr (L::jk == JOINT_RZ) {
      if constexpr (L::has_t) return rotz_neg(c, s, tm);
      else return Z3{};
    } else {
      return tm + mk3(Z{}, Z{}, -q);
    }
  }();
  auto Rw = link_rot<L>(c, s, wp);
  auto Rl = link_rot<L>(c, s, lp);
  auto Rv = link_rot<L>(c, s, vp) + cross(p, Rw);   // Ad(T) acting on [v; w]
  auto Ra = link_rot<L>(c, s, ap) + cross(p, Rl);
  if constexpr (L::jk == JOINT_RZ) {
    auto w = Rw + mk3(Z{}, Z{}, qd);                                  // Eq. 8.51
    auto v = Rv;
    auto l = Rl + scale(qd, cross_e3(w)) + mk3(Z{}, Z{}, qdd);        // Eq. 8.52: ad(V) S qd + S qdd
    auto a = Ra + scale(qd, cross_e3(v));
    return fwd_wrench<L, I>(P, v, w, a, l, p);
  } else {
    auto w = Rw;
    auto v = Rv + mk3(Z{}, Z{}, qd);
    auto l = Rl;
    auto a = Ra + scale(qd, cross_e3(w)) + mk3(Z{}, Z{}, qdd);
    return fwd_wrench<L, I>(P, v, w, a, l, p);
  }
}

// One backward step (Eq. 8.53): F_i = Ad(T_{i+1})^T F_{i+1} + b_i, where (c, s, p) belong to link i+1.
template <class Lnext, class T, class PP, class FF, class MM, class BF, class BM>
RBM_HD auto bwd_link(T c, T s, const PP& p, const FF& f, const MM& mo, const BF& bf, const BM& bm) {
  auto fo = link_rot_T<Lnext>(c, s, f) + bf;
  auto mo2 = link_rot_T<Lnext>(c, s, mo - cross(p, f)) + bm;
  struct R { decltype(fo) f; decltype(mo2) m; };
  return R{fo, mo2};
}

template <class T>
struct FastResult {
  T tau[6];
  T v[3], w[3], a[3], l[3];  // twist and twist rate of the last link (V_6, dV_6)
};

template <class T> RBM_HD void sincos_t(T x, T* s, T* c) { sincos_one(x, s, c); }  // rbm_trig.cuh

// sin / cos of the revolute joint angles of descriptor D (prismatic entries stay c = 1, s = 0); the angles are evaluated as
// one group so that their polynomial chains interleave (rbm_trig.cuh)
template <class T, class D>
RBM_HD void fast_sincos(const T (&q)[6], T (&c)[6], T (&s)[6]) {
  constexpr bool hinge[6] = {D::L0::jk == JOINT_RZ, D::L1::jk == JOINT_RZ, D::L2::jk == JOINT_RZ,
                             D::L3::jk == JOINT_RZ, D::L4::jk == JOINT_RZ, D::L5::jk == JOINT_RZ};
  constexpr int NH = hinge[0] + hinge[1] + hinge[2] + hinge[3] + hinge[4] + hinge[5];
#pragma unroll
  for (int i = 0; i < 6; ++i) { c[i] = T(1); s[i] = T(0); }
  if constexpr (NH > 0) {
    T x[NH], sn[NH], cs[NH];
    int k = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (hinge[i]) x[k++] = q[i];
    sincos_group<NH, T>(x, sn, cs);
    k = 0;
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (hinge[i]) { s[i] = sn[k]; c[i] = cs[k]; ++k; }
  }
}

// TWIST = false: the caller reads tau only, so the joint velocities tau does not depend on (!D::qd_matters) are structural zeros --
// their loads and their share of the recursion disappear.  FastResult::v/w/a/l are then NOT the physical twist of the last link
// (they miss the Galilean boost of the gantry velocities).
template <class T, class D, bool WANT_TAU, bool VEL = true, bool GRAV = true, bool ACC = true, int ONEHOT = -1, bool TWIST = true>
RBM_HD void fast_rnea_core(const FastParams<T>& P, const T* g, const T (&q)[6], const T (&c)[6], const T (&s)[6], const T (&qd)[6],
                           const T (&qdd)[6], FastResult<T>& out);

// Joint sines / cosines supplied by the caller (the linearisation re-uses them across its many evaluations).
template <class T, class D, bool WANT_TAU, bool TWIST = true>
RBM_HD void fast_rnea_cs(const FastParams<T>& P, const T (&q)[6], const T (&c)[6], const T (&s)[6], const T (&qd)[6], const T (&qdd)[6],
                         FastResult<T>& out) {
  fast_rnea_core<T, D, WANT_TAU, true, true, true, -1, TWIST>(P, P.g, q, c, s, qd, qdd, out);
}

// Full RNEA for one sample.  WANT_TAU = false leaves the backward sweep out (regressor kernels).
template <class T, class D, bool WANT_TAU>
RBM_HD void fast_rnea(const FastParams<T>& P, const T (&q)[6], const T (&qd)[6], const T (&qdd)[6], FastResult<T>& out) {
  T c[6], s[6];
  fast_sincos<T, D>(q, c, s);
  fast_rnea_cs<T, D, WANT_TAU>(P, q, c, s, qd, qdd, out);
}

// What the inverse-dynamics kernels return for one sample: tau from the TWIST = false recursion and, with OUT_TWIST, V_6 / dV_6 from a
// second forward sweep that keeps every joint velocity.  tau is the same arithmetic whether or not the twist is asked for, so the two
// forms return the same bits.
template <class T, class D, bool OUT_TWIST>
RBM_HD void fast_rnea_tau(const FastParams<T>& P, const T (&q)[6], const T (&qd)[6], const T (&qdd)[6], FastResult<T>& out) {
  T c[6], s[6];
  fast_sincos<T, D>(q, c, s);
  fast_rnea_cs<T, D, true, false>(P, q, c, s, qd, qdd, out);
  if constexpr (OUT_TWIST) fast_rnea_cs<T, D, false>(P, q, c, s, qd, qdd, out);  // overwrites v/w/a/l only
}

// The recursion itself; `g` is the linear part of the base acceleration (P.g, or zeros when the joint-space inertia
// matrix is being extracted column by column).
// VEL = false treats every joint velocity as a structural zero, GRAV = false the base acceleration and ACC = false every joint
// acceleration: (VEL off, GRAV off) is the acceleration-only evaluation whose columns are the joint-space inertia matrix,
// (ACC off, GRAV off) the velocity-product term C(q, qd) alone.  ONEHOT = j >= 0 (with VEL and GRAV off) evaluates qdd = e_j with every
// other joint acceleration a STRUCTURAL zero: column j of the inertia matrix, where the links before j carry no motion at all and the
// typed algebra removes their share of the recursion (the linearisation builds M this way: about half the work of six general columns).
template <class T, class D, bool WANT_TAU, bool VEL, bool GRAV, bool ACC, int ONEHOT, bool TWIST>
RBM_HD void fast_rnea_core(const FastParams<T>& P, const T* g, const T (&q)[6], const T (&c)[6], const T (&s)[6], const T (&qd)[6],
                           const T (&qdd)[6], FastResult<T>& out) {
  // base: twist_0 = 0, dtwist_0 = [g; 0]  (core/simulate.py:149,154-155)
  auto v0 = Z3{};
  auto w0 = Z3{};
  auto a0 = [&] {
    if constexpr (GRAV) return ld3(g);
    else return Z3{};
  }();
  auto l0 = Z3{};
  auto vel = [&](auto I) {
    if constexpr (VEL && (TWIST || D::qd_matters(decltype(I)::value))) return qd[decltype(I)::value];
    else return Z{};
  };
  auto acc = [&](auto I) {
    if constexpr (ONEHOT >= 0) {
      if constexpr (decltype(I)::value == ONEHOT) return T(1);
      else return Z{};
    } else if constexpr (ACC) return qdd[decltype(I)::value];
    else return Z{};
  };
  using std::integral_constant;
  auto k0 = fwd_link<typename D::L0, 0>(P, q[0], vel(integral_constant<int, 0>{}), acc(integral_constant<int, 0>{}), c[0], s[0], v0, w0, a0, l0);
  auto k1 = fwd_link<typename D::L1, 1>(P, q[1], vel(integral_constant<int, 1>{}), acc(integral_constant<int, 1>{}), c[1], s[1], k0.v, k0.w, k0.a, k0.l);
  auto k2 = fwd_link<typename D::L2, 2>(P, q[2], vel(integral_constant<int, 2>{}), acc(integral_constant<int, 2>{}), c[2], s[2], k1.v, k1.w, k1.a, k1.l);
  auto k3 = fwd_link<typename D::L3, 3>(P, q[3], vel(integral_constant<int, 3>{}), acc(integral_constant<int, 3>{}), c[3], s[3], k2.v, k2.w, k2.a, k2.l);
  auto k4 = fwd_link<typename D::L4, 4>(P, q[4], vel(integral_constant<int, 4>{}), acc(integral_constant<int, 4>{}), c[4], s[4], k3.v, k3.w, k3.a, k3.l);
  auto k5 = fwd_link<typename D::L5, 5>(P, q[5], vel(integral_constant<int, 5>{}), acc(integral_constant<int, 5>{}), c[5], s[5], k4.v, k4.w, k4.a, k4.l);

  out.v[0] = to_scalar<T>(k5.v.x); out.v[1] = to_scalar<T>(k5.v.y); out.v[2] = to_scalar<T>(k5.v.z);
  out.w[0] = to_scalar<T>(k5.w.x); out.w[1] = to_scalar<T>(k5.w.y); out.w[2] = to_scalar<T>(k5.w.z);
  out.a[0] = to_scalar<T>(k5.a.x); out.a[1] = to_scalar<T>(k5.a.y); out.a[2] = to_scalar<T>(k5.a.z);
  out.l[0] = to_scalar<T>(k5.l.x); out.l[1] = to_scalar<T>(k5.l.y); out.l[2] = to_scalar<T>(k5.l.z);

  if constexpr (WANT_TAU) {
    // backward sweep; wrench_tip = 0 and pose_tip_ee = I (dynamics/dynamics.py:116-117) => F_6 = b_6
    auto pick = [](auto Ld, const auto& f, const auto& m) {
      using L = decltype(Ld);
      if constexpr (L::jk == JOINT_RZ) return to_scalar<T>(m.z);
      else return to_scalar<T>(f.z);
    };
    auto f5 = k5.bf;
    auto m5 = k5.bm;
    out.tau[5] = pick(typename D::L5{}, f5, m5);
    auto F4 = bwd_link<typename D::L5>(c[5], s[5], k5.p, f5, m5, k4.bf, k4.bm);
    out.tau[4] = pick(typename D::L4{}, F4.f, F4.m);
    auto F3 = bwd_link<typename D::L4>(c[4], s[4], k4.p, F4.f, F4.m, k3.bf, k3.bm);
    out.tau[3] = pick(typename D::L3{}, F3.f, F3.m);
    auto F2 = bwd_link<typename D::L3>(c[3], s[3], k3.p, F3.f, F3.m, k2.bf, k2.bm);
    out.tau[2] = pick(typename D::L2{}, F2.f, F2.m);
    auto F1 = bwd_link<typename D::L2>(c[2], s[2], k2.p, F2.f, F2.m, k1.bf, k1.bm);
    out.tau[1] = pick(typename D::L1{}, F1.f, F1.m);
    auto F0 = bwd_link<typename D::L1>(c[1], s[1], k1.p, F1.f, F1.m, k0.bf, k0.bm);
    out.tau[0] = pick(typename D::L0{}, F0.f, F0.m);
  }
}

// =================================================================================================
// Generic path (parameters in shared memory, layout in rbm_model.cuh)
// =================================================================================================
template <class T> struct G3 { T x, y, z; };
template <class T> RBM_HD G3<T> g3(const T* p) { return {p[0], p[1], p[2]}; }
template <class T> RBM_HD G3<T> operator+(G3<T> a, G3<T> b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
template <class T> RBM_HD G3<T> operator-(G3<T> a, G3<T> b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
template <class T> RBM_HD G3<T> operator*(T s, G3<T> a) { return {s * a.x, s * a.y, s * a.z}; }
template <class T> RBM_HD G3<T> gcross(G3<T> a, G3<T> b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
template <class T> RBM_HD G3<T> mat_vec(const T* R, G3<T> v) {  // row-major 3x3
  return {R[0] * v.x + R[1] * v.y + R[2] * v.z, R[3] * v.x + R[4] * v.y + R[5] * v.z, R[6] * v.x + R[7] * v.y + R[8] * v.z};
}
template <class T> RBM_HD G3<T> matT_vec(const T* R, G3<T> v) {
  return {R[0] * v.x + R[3] * v.y + R[6] * v.z, R[1] * v.x + R[4] * v.y + R[7] * v.z, R[2] * v.x + R[5] * v.y + R[8] * v.z};
}

template <class T> RBM_HD T abs_t(T x) { return x < T(0) ? -x : x; }

// T_i = SE3.exp(-S q) . M_i  (dynamics.py:126).  The exponential (liegroups' Rodrigues / left-Jacobian formulas) and the product with
// the home pose are folded at model creation into R = c RA + s RB + RC, p = c PA + s PB + q PC + PD (rbm_model.cuh): 27 FMAs and one
// sincos per revolute joint, no division, no composition at run time; a prismatic joint costs 3 FMAs.  The branch on the joint kind
// depends on the model only (warp-uniform; a constant-bank compare in the unrolled kernel).
template <class T>
RBM_HD void joint_trig(const T* J /* per-joint param block */, T q, T& s, T& c) {
  const T nw = J[GJ_NW];
  if (nw == T(0)) { s = T(0); c = T(1); return; }
  sincos_t(q * nw, &s, &c);
}
template <class T>
RBM_HD void joint_pose(const T* J, T q, T s, T c, T* R, T* p) {
  if (J[GJ_NW] == T(0)) {
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = J[GJ_RC + k];
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] = J[GJ_PD + k] + q * J[GJ_PC + k];
    return;
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) R[k] = J[GJ_RC + k] + c * J[GJ_RA + k] + s * J[GJ_RB + k];
#pragma unroll
  for (int k = 0; k < 3; ++k) p[k] = J[GJ_PD + k] + q * J[GJ_PC + k] + c * J[GJ_PA + k] + s * J[GJ_PB + k];
}

// Ad(T) [v; w] = [R v + p x (R w); R w]
template <class T>
RBM_HD void adjoint_apply(const T* R, G3<T> p, G3<T> v, G3<T> w, G3<T>& vo, G3<T>& wo) {
  wo = mat_vec(R, w);
  vo = mat_vec(R, v) + gcross(p, wo);
}
// Ad(T)^T [f; m] = [R^T f; R^T (m - p x f)]
template <class T>
RBM_HD void adjointT_apply(const T* R, G3<T> p, G3<T> f, G3<T> m, G3<T>& fo, G3<T>& mo) {
  fo = matT_vec(R, f);
  mo = matT_vec(R, m - gcross(p, f));
}

// Generic RNEA for one sample.  NJ > 0: compile-time joint count (loops unroll, state in registers, `sp` may be a constant-bank
// kernel argument so every model constant is an FMA operand); NJ == 0: run-time count (per-link state lives in local memory).
// The body wrench b_i = G_i dV_i - ad(V_i)^T G_i V_i is formed during the forward sweep; of the link transforms only (sin, cos) of the
// joint are kept -- the backward sweep re-forms (R_i, p_i) from them (27 FMAs) instead of holding 12 numbers per link live, which is
// what made the unrolled fp64 kernel spill at 254 registers.  Optional full-state outputs mirror the reference's return value
// (tau, poses, twists, dtwists) for the scalar drop-in API.
template <class T, int NJ>
RBM_HD void generic_rnea(const T* __restrict__ sp, const T* __restrict__ base /* [V0 | dV0 | Ftip], normally == sp */, int nj_rt, const T* q, const T* qd, const T* qdd, T* tau,
                                             T* poses /* [nj][12] or null */, T* twists /* [nj+1][6] or null */, T* dtwists /* idem */,
                                             T* Vlast /* [6] or null */, T* dVlast /* [6] or null */) {
  constexpr int MAXJ = NJ > 0 ? NJ : RBM_MAX_JOINTS;
  const int nj = NJ > 0 ? NJ : nj_rt;
  T sn[MAXJ], cs[MAXJ];
  T bs[MAXJ][6];
  G3<T> v = g3(base + GP_V0), w = g3(base + GP_V0 + 3);
  G3<T> a = g3(base + GP_DV0), l = g3(base + GP_DV0 + 3);
  if (twists) {
    twists[0] = v.x; twists[1] = v.y; twists[2] = v.z; twists[3] = w.x; twists[4] = w.y; twists[5] = w.z;
    dtwists[0] = a.x; dtwists[1] = a.y; dtwists[2] = a.z; dtwists[3] = l.x; dtwists[4] = l.y; dtwists[5] = l.z;
  }
#pragma unroll
  for (int i = 0; i < nj; ++i) {
    const T* J = sp + GP_HEAD + GJ_STRIDE * i;
    T R[9], pp[3];
    joint_trig(J, q[i], sn[i], cs[i]);
    joint_pose(J, q[i], sn[i], cs[i], R, pp);
    G3<T> p = g3(pp);
    G3<T> sv = g3(J + GJ_S), sw = g3(J + GJ_S + 3);
    G3<T> vn, wn, an, ln;
    adjoint_apply(R, p, v, w, vn, wn);
    adjoint_apply(R, p, a, l, an, ln);
    v = vn + qd[i] * sv;  // Eq. 8.51
    w = wn + qd[i] * sw;
    // Eq. 8.52: ad(V) S = [w x s_v + v x s_w ; w x s_w]
    a = an + qd[i] * (gcross(w, sv) + gcross(v, sw)) + qdd[i] * sv;
    l = ln + qd[i] * gcross(w, sw) + qdd[i] * sw;
    const T V6[6] = {v.x, v.y, v.z, w.x, w.y, w.z};
    const T dV6[6] = {a.x, a.y, a.z, l.x, l.y, l.z};
    if (poses) {
#pragma unroll
      for (int k = 0; k < 9; ++k) poses[12 * i + k] = R[k];
      poses[12 * i + 9] = pp[0]; poses[12 * i + 10] = pp[1]; poses[12 * i + 11] = pp[2];
    }
    if (twists) {
#pragma unroll
      for (int k = 0; k < 6; ++k) { twists[6 * (i + 1) + k] = V6[k]; dtwists[6 * (i + 1) + k] = dV6[k]; }
    }
    if (tau) {
      const T* G = J + GJ_G;
      T h[6], gd[6];  // momentum G V and inertial force G dV
      if (J[GJ_RIGID] != T(0)) {
        // G = [[m 1, -[c]x], [[c]x, I]] (every physical link; warp-uniform branch): 10 numbers instead of a dense 6x6 product
        const T m = G[0];
        const G3<T> cm = {G[6 * 5 + 1], G[6 * 3 + 2], G[6 * 4 + 0]};  // first moment m c from the lower-left block [c]x
        const T I[6] = {G[6 * 3 + 3], G[6 * 4 + 4], G[6 * 5 + 5], G[6 * 3 + 4], G[6 * 4 + 5], G[6 * 5 + 3]};  // xx yy zz xy yz zx
        auto sym = [&](G3<T> x) -> G3<T> { return {I[0] * x.x + I[3] * x.y + I[5] * x.z, I[3] * x.x + I[1] * x.y + I[4] * x.z, I[5] * x.x + I[4] * x.y + I[2] * x.z}; };
        const G3<T> hf = m * v + gcross(w, cm), hm = gcross(cm, v) + sym(w);
        const G3<T> gf = m * a + gcross(l, cm), gm = gcross(cm, a) + sym(l);
        h[0] = hf.x; h[1] = hf.y; h[2] = hf.z; h[3] = hm.x; h[4] = hm.y; h[5] = hm.z;
        gd[0] = gf.x; gd[1] = gf.y; gd[2] = gf.z; gd[3] = gm.x; gd[4] = gm.y; gd[5] = gm.z;
      } else {
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          T sh = T(0), sg = T(0);
#pragma unroll
          for (int k = 0; k < 6; ++k) { sh += G[6 * r + k] * V6[k]; sg += G[6 * r + k] * dV6[k]; }
          h[r] = sh; gd[r] = sg;
        }
      }
      // -ad(V)^T [hf; hm] = [w x hf ; v x hf + w x hm]
      G3<T> hf = g3(h), hm = g3(h + 3);
      G3<T> bf = g3(gd) + gcross(w, hf);
      G3<T> bm = g3(gd + 3) + gcross(v, hf) + gcross(w, hm);
      bs[i][0] = bf.x; bs[i][1] = bf.y; bs[i][2] = bf.z; bs[i][3] = bm.x; bs[i][4] = bm.y; bs[i][5] = bm.z;
    }
  }
  if (Vlast) {
    Vlast[0] = v.x; Vlast[1] = v.y; Vlast[2] = v.z; Vlast[3] = w.x; Vlast[4] = w.y; Vlast[5] = w.z;
    dVlast[0] = a.x; dVlast[1] = a.y; dVlast[2] = a.z; dVlast[3] = l.x; dVlast[4] = l.y; dVlast[5] = l.z;
  }
  if (!tau) return;
  G3<T> f = g3(base + GP_FTIP), m = g3(base + GP_FTIP + 3);
#pragma unroll
  for (int i = nj - 1; i >= 0; --i) {
    const T* J = sp + GP_HEAD + GJ_STRIDE * i;
    G3<T> fo, mo;
    if (i == nj - 1) {  // tip transform (dynamics.py:136-137)
      adjointT_apply(sp + GP_TIPR, g3(sp + GP_TIPT), f, m, fo, mo);
    } else {  // T_{i+1} again, from the joint's (sin, cos)
      T R[9], pp[3];
      joint_pose(J + GJ_STRIDE, q[i + 1], sn[i + 1], cs[i + 1], R, pp);
      adjointT_apply(R, g3(pp), f, m, fo, mo);   // Eq. 8.53
    }
    f = fo + g3(bs[i]);
    m = mo + g3(bs[i] + 3);
    tau[i] = f.x * J[GJ_S] + f.y * J[GJ_S + 1] + f.z * J[GJ_S + 2] + m.x * J[GJ_S + 3] + m.y * J[GJ_S + 4] + m.z * J[GJ_S + 5];  // Eq. 8.54
  }
}

// =================================================================================================
// Sensor-frame twists (core/simulate.py:202-209) and regressor rows (dynamics/dynamics.py:215-249)
// =================================================================================================
// V_s = Ad(T_sen) V ; dV_s = Ad(T_sen) dV.  The reference also adds ad(V_s) Ad(T_sen) V = ad(V_s) V_s,
// which is identically zero (its floating-point residue there is ~1e-17); it is not evaluated here.
template <class T>
RBM_HD void sensor_twists(const T* R, const T* t, const T* V, const T* dV, T* Vs, T* dVs) {
  G3<T> p = g3(t), vo, wo;
  adjoint_apply(R, p, g3(V), g3(V + 3), vo, wo);
  Vs[0] = vo.x; Vs[1] = vo.y; Vs[2] = vo.z; Vs[3] = wo.x; Vs[4] = wo.y; Vs[5] = wo.z;
  adjoint_apply(R, p, g3(dV), g3(dV + 3), vo, wo);
  dVs[0] = vo.x; dVs[1] = vo.y; dVs[2] = vo.z; dVs[3] = wo.x; dVs[4] = wo.y; dVs[5] = wo.z;
}

// Non-zero blocks of the 6x10 regressor:  top (rows 0-2, cols 0-3) = [x | [dw]x + [w]x[w]x],
// bot (rows 3-5, cols 1-9) = [-[x]x | bullet(dw) + [w]x bullet(w)]   with x = dv + w x v.
// Two stages so that the Gram kernels can carry just (x, w, dw) -- 9 scalars -- from one sample to the next.
template <class T>
RBM_HD void regressor_x(const T* V, const T* dV, T (&x)[3]) {
  const T vx = V[0], vy = V[1], vz = V[2], wx = V[3], wy = V[4], wz = V[5];
  x[0] = dV[0] + (wy * vz - wz * vy);
  x[1] = dV[1] + (wz * vx - wx * vz);
  x[2] = dV[2] + (wx * vy - wy * vx);
}
template <class T>
RBM_HD void regressor_blocks_xwl(const T (&x)[3], const T* w, const T* l, T (&top)[3][4], T (&bot)[3][9]) {
  const T wx = w[0], wy = w[1], wz = w[2];
  const T xx = wx * wx, yy = wy * wy, zz = wz * wz, xy = wx * wy, yz = wy * wz, zx = wz * wx;
  const T lx = l[0], ly = l[1], lz = l[2];
  const T x0 = x[0], x1 = x[1], x2 = x[2];
  top[0][0] = x0; top[0][1] = -(yy + zz); top[0][2] = xy - lz;     top[0][3] = zx + ly;
  top[1][0] = x1; top[1][1] = xy + lz;    top[1][2] = -(xx + zz);  top[1][3] = yz - lx;
  top[2][0] = x2; top[2][1] = zx - ly;    top[2][2] = yz + lx;     top[2][3] = -(xx + yy);
  // -[x]x
  bot[0][0] = T(0); bot[0][1] = x2;   bot[0][2] = -x1;
  bot[1][0] = -x2;  bot[1][1] = T(0); bot[1][2] = x0;
  bot[2][0] = x1;   bot[2][1] = -x0;  bot[2][2] = T(0);
  // bullet(dw) + [w]x bullet(w), columns ixx iyy izz ixy iyz izx
  bot[0][3] = lx;   bot[0][4] = -yz;  bot[0][5] = yz;   bot[0][6] = ly - zx; bot[0][7] = yy - zz; bot[0][8] = lz + xy;
  bot[1][3] = zx;   bot[1][4] = ly;   bot[1][5] = -zx;  bot[1][6] = lx + yz; bot[1][7] = lz - xy; bot[1][8] = zz - xx;
  bot[2][3] = -xy;  bot[2][4] = xy;   bot[2][5] = lz;   bot[2][6] = xx - yy; bot[2][7] = ly + zx; bot[2][8] = lx - yz;
}
template <class T>
RBM_HD void regressor_blocks(const T* V, const T* dV, T (&top)[3][4], T (&bot)[3][9]) {
  T x[3];
  regressor_x(V, dV, x);
  regressor_blocks_xwl(x, V + 3, dV + 3, top, bot);
}

// ---- planner-driven inputs (planners/joint_position_planner.py:86-131): the quintic profile is evaluated in double in the step
// variable k
template <class T>
struct PlanArg {
  double coeffs[6];          // s(k) = c0 k^5 + c1 k^4 + ... + c5   (normalised profile in the step variable k)
  double inv_dt, inv_dt2;    // 1 / timestep, 1 / timestep^2
  double step0, stride;      // sample s evaluates step k = step0 + s * stride
  T disp[RBM_MAX_JOINTS];    // displacement per joint
  T offset[RBM_MAX_JOINTS];  // pos_offset per joint
};

template <class T>
RBM_HD void plan_profile(const PlanArg<T>& pl, int64_t s, T& sp, T& sv, T& sa) {
  const double k = pl.step0 + (double)s * pl.stride;
  const double k2 = k * k, k3 = k2 * k, k4 = k3 * k, k5 = k4 * k;
  const double* c = pl.coeffs;
  sp = (T)(c[0] * k5 + c[1] * k4 + c[2] * k3 + c[3] * k2 + c[4] * k + c[5]);                                  // :120,125
  sv = (T)((5.0 * c[0] * k4 + 4.0 * c[1] * k3 + 3.0 * c[2] * k2 + 2.0 * c[3] * k + c[4]) * pl.inv_dt);        // :121,126
  sa = (T)((20.0 * c[0] * k3 + 12.0 * c[1] * k2 + 6.0 * c[2] * k + 2.0 * c[3]) * pl.inv_dt2);                 // :122-123,127
}


}  // namespace rbm
