// Joint-torque payload regressor: per-sample arithmetic of the payload kernels (rbm_regressor.cu), __host__ __device__ so that the
// host harness instantiates the same code.
//
// `model` is the robot WITHOUT the payload; phi holds the payload's 10 inertial parameters in the sensor frame of the model's
// pose_sen_Rt, in the order and frame of the F/T route.  RNEA is linear in the link inertias, so
//   tau(q, qd, qdd) = tau0(q, qd, qdd) + Phi(q, qd, qdd) phi,      Phi = J_s^T Y_s   (nj x 10)
// tau0 is the model's own inverse dynamics, Y_s = Y(V_s, dV_s) the sensor-frame regressor of the F/T route and J_s the Jacobian of
// the last link expressed in the sensor frame (column j = joint j's screw seen from the sensor): the payload loads the last link
// with the wrench Ad(T_sen)^T Y_s phi, and a wrench W_s at the sensor does the joint work J_s^T W_s.
//
// Structure of the sequential (fast-path) models, checked against the oracle by tests/test_payload_identification.py:
//   * rows 0..2 (prismatic gantry joints) read only the force of the payload's wrench, which depends on m and m c alone: those rows
//     are structurally zero in columns 4..9 (true of any prismatic joint: its Jacobian column has no angular part);
//   * Y_s depends on x = dv + w x v, w and dw only, which the gantry-velocity boost leaves unchanged (dv moves by -w x dv), and
//     the Jacobian does not depend on q[0..2]: Phi and tau0 come from the tau-only (TWIST = false) recursion, which reads neither
//     q[0..2] nor qd[0..2].
#pragma once
#include "rbm_gram.cuh"
#include "rbm_rnea.cuh"

namespace rbm {

template <class D>
RBM_HD constexpr bool fast_prismatic(int j) {
  return (j == 0 ? D::L0::jk : j == 1 ? D::L1::jk : j == 2 ? D::L2::jk : j == 3 ? D::L3::jk : j == 4 ? D::L4::jk : D::L5::jk) == JOINT_PZ;
}

// Phi[c] = Js_lin . Y_s[force rows][c] + Js_ang . Y_s[torque rows][c]; a prismatic joint's column has no angular part
template <class T>
RBM_HD void payload_row(const T (&ls)[3], const T (&as)[3], bool prismatic, const T (&top)[3][4], const T (&bot)[3][9], T (&phi)[10]) {
#pragma unroll
  for (int c = 0; c < 4; ++c) phi[c] = ls[0] * top[0][c] + ls[1] * top[1][c] + ls[2] * top[2][c];
#pragma unroll
  for (int c = 4; c < 10; ++c) phi[c] = T(0);
  if (prismatic) return;
#pragma unroll
  for (int c = 1; c < 10; ++c)
#pragma unroll
    for (int r = 0; r < 3; ++r)
      if (bot_nz(r, c - 1)) phi[c] += as[r] * bot[r][c - 1];
}

// Column J of the last link's Jacobian J_6 (dV_6 for qdd = e_J with no velocity and no gravity): the one-hot form of the forward
// recursion, in which the links before J carry no motion and the typed algebra drops them.
template <class T, class D, int J>
RBM_HD void fast_jacobian_col(const FastParams<T>& P, const T (&q)[6], const T (&c)[6], const T (&s)[6], T (&lin)[3], T (&ang)[3]) {
  FastResult<T> r;
  fast_rnea_core<T, D, false, false, false, true, J, true>(P, P.g, q, c, s, q, q, r);  // qd / qdd are not read
#pragma unroll
  for (int k = 0; k < 3; ++k) { lin[k] = r.a[k]; ang[k] = r.l[k]; }
}

// Fast paths: tau0 (bit-identical to the rbm_rnea_* kernels: the same fast_rnea_tau arithmetic), then emit(j, Phi[j]) for j = 0..5,
// one row at a time so that a caller accumulating the rows never holds the whole 6 x 10 block.  q[0..2] and qd[0..2] are never read.
template <class T, class D, bool SEN_DIAG, class Emit>
RBM_HD void payload_fast(const FastParams<T>& P, const T (&q)[6], const T (&qd)[6], const T (&qdd)[6], T (&tau0)[6], Emit&& emit) {
  T c[6], s[6];
  fast_sincos<T, D>(q, c, s);
  FastResult<T> r;
  fast_rnea_cs<T, D, true, false>(P, q, c, s, qd, qdd, r);  // == fast_rnea_tau<T, D, false>
#pragma unroll
  for (int j = 0; j < 6; ++j) tau0[j] = r.tau[j];
  // Y_s from the same sweep: its (v, w, a, l) miss the gantry-velocity boost, which leaves x, w and dw unchanged
  T V[6], dV[6], Vs[6], dVs[6];
#pragma unroll
  for (int k = 0; k < 3; ++k) { V[k] = r.v[k]; V[3 + k] = r.w[k]; dV[k] = r.a[k]; dV[3 + k] = r.l[k]; }
  if constexpr (SEN_DIAG) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const T d = P.senR[4 * k];
      Vs[k] = d * V[k]; Vs[3 + k] = d * V[3 + k];
      dVs[k] = d * dV[k]; dVs[3 + k] = d * dV[3 + k];
    }
  } else {
    sensor_twists(P.senR, P.sent, V, dV, Vs, dVs);
  }
  T x[3], top[3][4], bot[3][9];
  regressor_x(Vs, dVs, x);
  regressor_blocks_xwl(x, Vs + 3, dVs + 3, top, bot);
  auto row = [&](auto Jc) {
    constexpr int J = decltype(Jc)::value;
    constexpr bool prism = fast_prismatic<D>(J);
    T lin[3], ang[3], ls[3], as[3];
    fast_jacobian_col<T, D, J>(P, q, c, s, lin, ang);
    if constexpr (SEN_DIAG) {
#pragma unroll
      for (int k = 0; k < 3; ++k) { const T d = P.senR[4 * k]; ls[k] = d * lin[k]; as[k] = d * ang[k]; }
    } else if constexpr (prism) {  // J_s = Ad(T_sen) J_6 = [R lin; 0]
      const G3<T> v = mat_vec(P.senR, g3(lin));
      ls[0] = v.x; ls[1] = v.y; ls[2] = v.z;
      as[0] = as[1] = as[2] = T(0);
    } else {
      G3<T> v, w;
      adjoint_apply(P.senR, g3(P.sent), g3(lin), g3(ang), v, w);
      ls[0] = v.x; ls[1] = v.y; ls[2] = v.z; as[0] = w.x; as[1] = w.y; as[2] = w.z;
    }
    T phi[10];
    payload_row(ls, as, prism, top, bot, phi);
    emit(J, phi);
  };
  using std::integral_constant;
  row(integral_constant<int, 0>{}); row(integral_constant<int, 1>{}); row(integral_constant<int, 2>{});
  row(integral_constant<int, 3>{}); row(integral_constant<int, 4>{}); row(integral_constant<int, 5>{});
}

// Generic path (any chain of up to RBM_MAX_JOINTS joints, parameters `sp` in the rbm_model.cuh layout): tau0 from generic_rnea, then
// a wrench-only backward propagation of the six unit sensor wrenches over the re-formed link poses gives row i of J_s^T, and
// emit(i, Phi[i]) receives the rows from the last joint to the first.
template <class T, class Emit>
RBM_HD void payload_generic(const T* sp, int nj, const T* q, const T* qd, const T* qdd, T* tau0, Emit&& emit) {
  T V[6], dV[6], Vs[6], dVs[6], top[3][4], bot[3][9];
  generic_rnea<T, 0>(sp, sp, nj, q, qd, qdd, tau0, nullptr, nullptr, nullptr, V, dV);
  const T* Rs = sp + GP_SENR;
  const G3<T> ts = g3(sp + GP_SENT);
  sensor_twists(Rs, sp + GP_SENT, V, dV, Vs, dVs);
  regressor_blocks(Vs, dVs, top, bot);
  // unit wrench e_r at the sensor, seen by the last link: Ad(T_sen)^T e_r.  The wrenches are walked one at a time (run-time loops):
  // with 36 of them live beside the Gram kernel's 66 fp64 accumulators the unrolled form spills.
  T F[6][6];
#pragma unroll 1
  for (int r = 0; r < 6; ++r) {
    const G3<T> e = {T(r % 3 == 0), T(r % 3 == 1), T(r % 3 == 2)}, z = {T(0), T(0), T(0)};
    G3<T> fo, mo;
    adjointT_apply(Rs, ts, r < 3 ? e : z, r < 3 ? z : e, fo, mo);
    F[r][0] = fo.x; F[r][1] = fo.y; F[r][2] = fo.z; F[r][3] = mo.x; F[r][4] = mo.y; F[r][5] = mo.z;
  }
#pragma unroll 1
  for (int i = nj - 1; i >= 0; --i) {
    const T* J = sp + GP_HEAD + GJ_STRIDE * i;
    T R[9], pp[3];
    if (i < nj - 1) {  // F_i = Ad(T_{i+1})^T F_{i+1}   (Eq. 8.53 without the body wrenches)
      T sn, cs;
      joint_trig(J + GJ_STRIDE, q[i + 1], sn, cs);
      joint_pose(J + GJ_STRIDE, q[i + 1], sn, cs, R, pp);
    }
    T row[6];  // joint i's torque per unit sensor wrench e_r
#pragma unroll 1
    for (int r = 0; r < 6; ++r) {
      G3<T> f = g3(F[r]), m = g3(F[r] + 3);
      if (i < nj - 1) {
        G3<T> fo, mo;
        adjointT_apply(R, g3(pp), f, m, fo, mo);
        f = fo; m = mo;
        F[r][0] = f.x; F[r][1] = f.y; F[r][2] = f.z; F[r][3] = m.x; F[r][4] = m.y; F[r][5] = m.z;
      }
      row[r] = f.x * J[GJ_S] + f.y * J[GJ_S + 1] + f.z * J[GJ_S + 2] + m.x * J[GJ_S + 3] + m.y * J[GJ_S + 4] + m.z * J[GJ_S + 5];
    }
    const T ls[3] = {row[0], row[1], row[2]}, as[3] = {row[3], row[4], row[5]};
    T phi[10];
    payload_row(ls, as, false, top, bot, phi);
    emit(i, phi);
  }
}

}  // namespace rbm
