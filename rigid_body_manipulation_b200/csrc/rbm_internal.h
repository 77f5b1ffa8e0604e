// Host-side internals shared by the translation units of librbm_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rbm_b200.h"
#include "rbm_model.cuh"

struct rbm_model {
  int nj = 0;
  int path = rbm::PATH_GENERIC;
  int device = 0;
  bool no_tma = false;  // RBM_FLAG_NO_TMA: keep to the direct-load kernels (A/B comparisons, debugging)
  std::vector<double> gp64;  // generic packed parameters (rbm_model.cuh layout), host copies
  std::vector<float> gp32;
  double* d_gp64 = nullptr;  // device copies, staged into shared memory by every block
  float* d_gp32 = nullptr;
  rbm::FastParams<double> fp64;
  rbm::FastParams<float> fp32;
  // staging for the *_host entry points (allocated on first use, grow-only, guarded by pipe_mu)
  static constexpr int kPipeSlots = 3;
  mutable std::mutex pipe_mu;
  mutable cudaStream_t pipe_st[kPipeSlots] = {nullptr, nullptr, nullptr};
  mutable void* pipe_in[kPipeSlots] = {nullptr, nullptr, nullptr};
  mutable void* pipe_out[kPipeSlots] = {nullptr, nullptr, nullptr};
  mutable size_t pipe_in_bytes = 0, pipe_out_bytes = 0;
  // scratch of the small-batch host entry point rbm_rnea_full_host_f64 (device + pinned host mirror)
  mutable double* full_dev = nullptr;
  mutable double* full_pinned = nullptr;
  mutable size_t full_doubles = 0;
};

namespace rbm {

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);

#define RBM_CUDA_TRY(expr)                                   \
  do {                                                       \
    cudaError_t _e = (expr);                                 \
    if (_e != cudaSuccess) return ::rbm::cuda_fail(_e, #expr); \
  } while (0)

// Makes `device` current for the scope and restores the caller's device afterwards (the library never leaves the calling
// thread's current device changed; all model-bound entry points launch on the model's device).
class DeviceGuard {
 public:
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev_) != cudaSuccess) prev_ = -1;
    if (prev_ != device) {
      status_ = cudaSetDevice(device);
      switched_ = status_ == cudaSuccess;
    }
  }
  ~DeviceGuard() {
    if (switched_ && prev_ >= 0) cudaSetDevice(prev_);
  }
  cudaError_t status() const { return status_; }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;

 private:
  int prev_ = -1;
  bool switched_ = false;
  cudaError_t status_ = cudaSuccess;
};

template <class T> struct ModelView;
template <> struct ModelView<double> {
  static const double* generic(const rbm_model* m) { return m->d_gp64; }
  static const double* generic_host(const rbm_model* m) { return m->gp64.data(); }
  static const FastParams<double>& fast(const rbm_model* m) { return m->fp64; }
};
template <> struct ModelView<float> {
  static const float* generic(const rbm_model* m) { return m->d_gp32; }
  static const float* generic_host(const rbm_model* m) { return m->gp32.data(); }
  static const FastParams<float>& fast(const rbm_model* m) { return m->fp32; }
};

// launchers (rbm_rnea.cu)
template <class T>
int launch_rnea_soa(const rbm_model* m, const T* q, const T* qd, const T* qdd, T* tau, T* V, T* dV, int64_t n, int64_t ld, cudaStream_t st);
template <class T>
int launch_rnea_aos(const rbm_model* m, const T* traj, T* tau, int64_t n, cudaStream_t st);
template <class T>
int launch_rnea_planned(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0, double stride,
                        T* tau, T* traj, int64_t n, int64_t ld, cudaStream_t st);
template <class T>
int launch_rnea_full(const rbm_model* m, const T* traj, T* tau, T* poses, T* twists, T* dtwists, int64_t n, cudaStream_t st);


// launchers (rbm_regressor.cu)
int gram_grid(const rbm_model* m, int64_t n, int per_sm);
template <class T>
int launch_regressor_rows(const T* tw, const T* dtw, T* Y, int64_t n, cudaStream_t st);
template <class T>
int launch_sensor_twists(const double* pose_Rt, const T* tw, const T* dtw, T* tws, T* dtws, int64_t n, cudaStream_t st);
template <class T>
int launch_regressor_from_traj(const rbm_model* m, const T* q, const T* qd, const T* qdd, T* Y, T* Vs, T* dVs, const T* phi, T* F, int64_t n, int64_t ld,
                               cudaStream_t st);
template <class T>
int launch_regressor_gram(const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* f, double* pack, double* partials, int64_t n, int64_t ld,
                          cudaStream_t st);
template <class T>
int launch_regressor_gram_grouped(const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* f, int64_t frame_stride, int64_t f_frame_stride,
                                  int64_t n_frames, double* packs, int64_t n_groups, int64_t ld, int64_t ld_out, cudaStream_t st);

// launcher (rbm_linearize.cu)
template <class T>
int launch_linearize(const rbm_model* m, const T* q, const T* qd, const T* u, double dt, double eps, int centered, T* A, T* B, T* qdd, int64_t n,
                     int64_t ld, cudaStream_t st);

template <class T>
int launch_forward_dynamics(const rbm_model* m, const T* q, const T* qd, const T* u, double dt, T* qdd, T* q_next, T* qd_next, int64_t n, int64_t ld,
                            cudaStream_t st);

int launch_closed_loop(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double plan_timestep, double step0,
                       int n_steps, const double* K, const double* phi, double dt, double fps, double div, const double* q0, const double* qd0,
                       double* frames, int max_frames, int* frame_steps, int* n_frames, double* final_state, int64_t n, int64_t ld, cudaStream_t st);

// launchers (rbm_setup.cu)
int launch_transfer_simat(const double* poses, const double* simats, double* out, int64_t n, int pose_stride, int simat_stride, int mode, cudaStream_t st);
int launch_transfer_imat(const double* poses, const double* imats, const double* mass, double* out, int64_t n, cudaStream_t st);
int launch_spatial_inertia(const double* mass, const double* diag, double* out, int64_t n, cudaStream_t st);
int launch_compose(const double* trans, const double* rot, int rot_len, double* out, int* status, int64_t n, cudaStream_t st);
int launch_point_motion(const double* tw, const double* dtw, const double* pts, double* linvel, double* linacc, int64_t n, cudaStream_t st);

}  // namespace rbm
