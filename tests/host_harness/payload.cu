// TEST INFRASTRUCTURE ONLY (never part of librbm_b200.so): the host instantiation of the joint-torque payload regressor
// (csrc/rbm_payload.cuh) and of its Gram accumulation (payload_accumulate_row / payload_pack_entry, csrc/rbm_gram.cuh), the per-sample
// code of k_payload_regressor and k_payload_gram.  Built and loaded by tests/test_payload_identification.py.
// Layouts are the kernels': q, qd, qdd, tau [nj][n];  Phi [n][nj][10];  tau0 [nj][n].
#include <cstdint>

#include "rbm_payload.cuh"

using namespace rbm;

namespace {
template <class T>
FastParams<T> convert(const double* fp) {
  FastParams<T> P;
  T* dst = reinterpret_cast<T*>(&P);
  for (size_t i = 0; i < sizeof(FastParams<double>) / sizeof(double); ++i) dst[i] = (T)fp[i];
  return P;
}

// body(s, j, phi_row, tau0_j) for every sample s and joint j
template <class T, class F>
int for_each_row(int path, const double* fp, const double* gp64, int nj, const T* q, const T* qd, const T* qdd, int64_t n, F&& body) {
  if (path == PATH_SEQ_ISO || path == PATH_SEQ_RIGID) {
    if (nj != 6) return -1;
    const FastParams<T> P = convert<T>(fp);
    for (int64_t s = 0; s < n; ++s) {
      T rq[6], rqd[6], rqdd[6], tau0[6];
      for (int j = 0; j < 6; ++j) { rq[j] = q[j * n + s]; rqd[j] = qd[j * n + s]; rqdd[j] = qdd[j * n + s]; }
      auto row = [&](int j, const T (&phi)[10]) { body(s, j, phi, tau0[j], fast_prismatic<SeqIso>(j)); };
      const bool diag = P.sen_diag != T(0);
      if (path == PATH_SEQ_ISO) diag ? payload_fast<T, SeqIso, true>(P, rq, rqd, rqdd, tau0, row) : payload_fast<T, SeqIso, false>(P, rq, rqd, rqdd, tau0, row);
      else diag ? payload_fast<T, SeqRigid, true>(P, rq, rqd, rqdd, tau0, row) : payload_fast<T, SeqRigid, false>(P, rq, rqd, rqdd, tau0, row);
    }
    return 0;
  }
  if (nj < 1 || nj > RBM_MAX_JOINTS) return -1;
  T gp[GP_HEAD + GJ_STRIDE * RBM_MAX_JOINTS];
  for (int i = 0; i < GP_HEAD + GJ_STRIDE * nj; ++i) gp[i] = (T)gp64[i];
  for (int64_t s = 0; s < n; ++s) {
    T rq[RBM_MAX_JOINTS], rqd[RBM_MAX_JOINTS], rqdd[RBM_MAX_JOINTS], tau0[RBM_MAX_JOINTS] = {};
    for (int j = 0; j < nj; ++j) { rq[j] = q[j * n + s]; rqd[j] = qd[j * n + s]; rqdd[j] = qdd[j * n + s]; }
    payload_generic<T>(gp, nj, rq, rqd, rqdd, tau0, [&](int i, const T (&phi)[10]) { body(s, i, phi, tau0[i], false); });
  }
  return 0;
}

template <class T>
int payload(int path, const double* fp, const double* gp, int nj, const T* q, const T* qd, const T* qdd, T* Phi, T* tau0, int64_t n) {
  return for_each_row<T>(path, fp, gp, nj, q, qd, qdd, n, [&](int64_t s, int j, const T (&phi)[10], T t0, bool) {
    for (int c = 0; c < 10; ++c) Phi[(s * nj + j) * 10 + c] = phi[c];
    tau0[j * n + s] = t0;
  });
}
}  // namespace

extern "C" {
int h_payload_f64(int path, const double* fp, const double* gp, int nj, const double* q, const double* qd, const double* qdd, double* Phi, double* tau0,
                  int64_t n) {
  return payload<double>(path, fp, gp, nj, q, qd, qdd, Phi, tau0, n);
}
int h_payload_f32(int path, const double* fp, const double* gp, int nj, const float* q, const float* qd, const float* qdd, float* Phi, float* tau0,
                  int64_t n) {
  return payload<float>(path, fp, gp, nj, q, qd, qdd, Phi, tau0, n);
}
// the 112-double pack [Phi^T Phi | Phi^T r | r^T r | n] with r = tau - tau0
int h_payload_gram_f64(int path, const double* fp, const double* gp, int nj, const double* q, const double* qd, const double* qdd, const double* tau,
                       double* pack, int64_t n) {
  double acc[kPayAcc] = {0};
  const int rc = for_each_row<double>(path, fp, gp, nj, q, qd, qdd, n, [&](int64_t s, int j, const double (&phi)[10], double t0, bool prismatic) {
    payload_accumulate_row(acc, phi, tau[j * n + s] - t0, prismatic);
  });
  if (rc) return rc;
  for (int t = 0; t < 111; ++t) pack[t] = payload_pack_entry(acc, t);
  pack[111] = (double)n;
  return 0;
}
}  // extern "C"
