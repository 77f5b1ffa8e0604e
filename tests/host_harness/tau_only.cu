// TEST INFRASTRUCTURE ONLY (never part of librbm_b200.so): the host instantiation of the tau-only fast recursion,
// fast_rnea_core<..., TWIST = false> (csrc/rbm_rnea.cuh), which the inverse-dynamics kernels compute tau with.  Built and loaded by
// tests/test_rnea_tau_only.py, beside the full evaluation of harness.cu.
#include <cstdint>

#include "rbm_rnea.cuh"

using namespace rbm;

namespace {
template <class T, class D>
void run_tau_only(const FastParams<T>& P, const T* traj, T* tau, int64_t n) {
  for (int64_t s = 0; s < n; ++s) {
    T q[6], qd[6], qdd[6], c[6], sn[6];
    for (int j = 0; j < 6; ++j) { q[j] = traj[s * 18 + j]; qd[j] = traj[s * 18 + 6 + j]; qdd[j] = traj[s * 18 + 12 + j]; }
    fast_sincos<T, D>(q, c, sn);
    FastResult<T> r;
    fast_rnea_cs<T, D, true, false>(P, q, c, sn, qd, qdd, r);
    for (int j = 0; j < 6; ++j) tau[s * 6 + j] = r.tau[j];
  }
}

template <class T>
int dispatch(int path, const double* fp, const T* traj, T* tau, int64_t n) {
  FastParams<T> P;
  T* dst = reinterpret_cast<T*>(&P);
  for (size_t i = 0; i < sizeof(FastParams<double>) / sizeof(double); ++i) dst[i] = (T)fp[i];
  if (path == PATH_SEQ_ISO) run_tau_only<T, SeqIso>(P, traj, tau, n);
  else if (path == PATH_SEQ_RIGID) run_tau_only<T, SeqRigid>(P, traj, tau, n);
  else return -1;
  return 0;
}
}  // namespace

extern "C" {
int h_fast_rnea_tau_only_f64(int path, const double* fast_params, const double* traj, double* tau, int64_t n) {
  return dispatch<double>(path, fast_params, traj, tau, n);
}
int h_fast_rnea_tau_only_f32(int path, const double* fast_params, const float* traj, float* tau, int64_t n) {
  return dispatch<float>(path, fast_params, traj, tau, n);
}
}  // extern "C"
