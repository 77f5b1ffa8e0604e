// extern "C" boundary of librbm_b200.so (declared in include/rbm_b200.h) and the host-side model analysis.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>

#include "rbm_internal.h"

namespace rbm {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int cuda_fail(cudaError_t e, const char* what) {
  g_last_error = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
  return RBM_ERR_CUDA;
}

static int invalid(const std::string& msg) {
  g_last_error = msg;
  return RBM_ERR_INVALID;
}

// ---------------------------------------------------------------------------------------------
// structure analysis: does the model match the compile-time descriptor of rbm_rnea.cuh?
// ---------------------------------------------------------------------------------------------
// Entries produced by quaternion round trips are exact up to ~2e-16; anything within kSnap of the
// descriptor's 0 / +-1 pattern is treated as the pattern (perturbs tau by <= ~1e-13 relative, four orders
// below the 1e-9 parity bar; RBM_FLAG_FORCE_GENERIC keeps the unsnapped constants).
static const double kSnap = 1e-13;

static const int kSeqPerm[6][3] = {{-3, 2, 1}, {1, -3, 2}, {3, 2, -1}, {1, 3, -2}, {-3, 2, 1}, {1, -3, 2}};
static const int kSeqHinge[6] = {0, 0, 0, 1, 1, 1};

static bool near(double a, double b, double tol = kSnap) { return std::fabs(a - b) <= tol; }

static bool rotation_is_perm(const double* R, const int* perm) {
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      const int col = std::abs(perm[r]) - 1;
      const double want = (c == col) ? (perm[r] > 0 ? 1.0 : -1.0) : 0.0;
      if (!near(R[3 * r + c], want)) return false;
    }
  return true;
}

struct RigidForm {
  double m, h[3], I[6];
  bool iso;  // h == 0 and I == J * identity
};

// G == [[m 1, -[h]x], [[h]x, Ibar]] with Ibar symmetric?
static bool rigid_form(const double* G, RigidForm* out) {
  double scale = 0.0;
  for (int i = 0; i < 36; ++i) scale = std::fmax(scale, std::fabs(G[i]));
  const double tol = 1e-12 * std::fmax(scale, 1e-300);
  const double m = G[0];
  auto g = [&](int r, int c) { return G[6 * r + c]; };
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c)
      if (!near(g(r, c), r == c ? m : 0.0, tol)) return false;
  const double hx = g(5, 1), hy = g(3, 2), hz = g(4, 0);
  const double hxm[3][3] = {{0, -hz, hy}, {hz, 0, -hx}, {-hy, hx, 0}};
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      if (!near(g(3 + r, c), hxm[r][c], tol)) return false;
      if (!near(g(r, 3 + c), -hxm[r][c], tol)) return false;
      if (!near(g(3 + r, 3 + c), g(3 + c, 3 + r), tol)) return false;
    }
  out->m = m;
  out->h[0] = hx; out->h[1] = hy; out->h[2] = hz;
  out->I[0] = g(3, 3); out->I[1] = g(4, 4); out->I[2] = g(5, 5);
  out->I[3] = g(3, 4); out->I[4] = g(4, 5); out->I[5] = g(5, 3);
  out->iso = near(hx, 0, tol) && near(hy, 0, tol) && near(hz, 0, tol) && near(out->I[0], out->I[1], tol) && near(out->I[0], out->I[2], tol) &&
             near(out->I[3], 0, tol) && near(out->I[4], 0, tol) && near(out->I[5], 0, tol);
  return true;
}

static int detect_path(int nj, const double* hposes_Rt, const double* simats, const double* uscrews, const double* twist_0,
                       const double* dtwist_0, const double* wrench_tip, const double* pose_tip, FastParams<double>* fp) {
  if (nj != 6) return PATH_GENERIC;
  for (int k = 0; k < 6; ++k)
    if (twist_0[k] != 0.0 || (wrench_tip && wrench_tip[k] != 0.0)) return PATH_GENERIC;
  for (int k = 3; k < 6; ++k)
    if (dtwist_0[k] != 0.0) return PATH_GENERIC;
  if (pose_tip) {
    static const int ident[3] = {1, 2, 3};
    if (!rotation_is_perm(pose_tip, ident)) return PATH_GENERIC;
    for (int k = 9; k < 12; ++k)
      if (!near(pose_tip[k], 0.0)) return PATH_GENERIC;
  }
  bool all_iso15 = true;
  for (int i = 0; i < 6; ++i) {
    const double* S = uscrews + 6 * i;
    for (int k = 0; k < 6; ++k) {
      const double want = (k == (kSeqHinge[i] ? 5 : 2)) ? 1.0 : 0.0;
      if (!near(S[k], want)) return PATH_GENERIC;
    }
    const double* H = hposes_Rt + 12 * (i + 1);
    if (!rotation_is_perm(H, kSeqPerm[i])) return PATH_GENERIC;
    for (int k = 9; k < 12; ++k)
      if (!near(H[k], 0.0)) return PATH_GENERIC;
    RigidForm rf;
    if (!rigid_form(simats + 36 * (i + 1), &rf)) return PATH_GENERIC;
    fp->mass[i] = rf.m;
    for (int k = 0; k < 3; ++k) { fp->h[i][k] = rf.h[k]; fp->tm[i][k] = 0.0; }
    for (int k = 0; k < 6; ++k) fp->I[i][k] = rf.I[k];
    if (i < 5 && !rf.iso) all_iso15 = false;
  }
  for (int k = 0; k < 3; ++k) fp->g[k] = dtwist_0[k];
  return all_iso15 ? PATH_SEQ_ISO : PATH_SEQ_RIGID;
}

template <class T>
static void convert_fast(const FastParams<double>& a, FastParams<T>* b) {
  const double* src = reinterpret_cast<const double*>(&a);
  T* dst = reinterpret_cast<T*>(b);
  for (size_t i = 0; i < sizeof(FastParams<double>) / sizeof(double); ++i) dst[i] = (T)src[i];
}

}  // namespace rbm

// ---- host end-to-end paths ---------------------------------------------------------------------
// Three-slot pipeline shared by the *_host entry points: slot k owns a stream and a device staging pair (in, out); chunk i runs
// H2D -> kernel -> D2H on stream (i % 3), so the upload of one chunk, the kernel of the previous and the download of the one
// before overlap.  One cudaMemcpyAsync / cudaMemcpy2DAsync per array and chunk (no batched-memcpy API).
namespace rbm {

static int ensure_pipe(const rbm_model* m, size_t in_bytes, size_t out_bytes) {
  constexpr int kSlots = rbm_model::kPipeSlots;
  for (int k = 0; k < kSlots; ++k)
    if (!m->pipe_st[k]) RBM_CUDA_TRY(cudaStreamCreateWithFlags(&m->pipe_st[k], cudaStreamNonBlocking));
  if (in_bytes > m->pipe_in_bytes || out_bytes > m->pipe_out_bytes) {
    if (in_bytes < m->pipe_in_bytes) in_bytes = m->pipe_in_bytes;
    if (out_bytes < m->pipe_out_bytes) out_bytes = m->pipe_out_bytes;
    for (int k = 0; k < kSlots; ++k) {
      RBM_CUDA_TRY(cudaStreamSynchronize(m->pipe_st[k]));
      if (m->pipe_in[k]) cudaFree(m->pipe_in[k]);
      if (m->pipe_out[k]) cudaFree(m->pipe_out[k]);
      m->pipe_in[k] = m->pipe_out[k] = nullptr;
    }
    m->pipe_in_bytes = m->pipe_out_bytes = 0;
    for (int k = 0; k < kSlots; ++k) {
      RBM_CUDA_TRY(cudaMalloc(&m->pipe_in[k], in_bytes ? in_bytes : 16));
      RBM_CUDA_TRY(cudaMalloc(&m->pipe_out[k], out_bytes ? out_bytes : 16));
      // rows that a kernel path never reads are never uploaded either (rbm_rnea_host_soa_*): keep them defined
      RBM_CUDA_TRY(cudaMemsetAsync(m->pipe_in[k], 0, in_bytes ? in_bytes : 16, m->pipe_st[k]));
    }
    m->pipe_in_bytes = in_bytes;
    m->pipe_out_bytes = out_bytes;
  }
  return RBM_OK;
}

// drains the pipeline; on any failure the streams are drained BEFORE returning: copies of earlier chunks may still be reading the
// caller's input / writing its output, and the caller may release those buffers as soon as the entry point returns
static int drain_pipe(const rbm_model* m, int rc, const char* who) {
  for (int k = 0; k < rbm_model::kPipeSlots; ++k) {
    if (!m->pipe_st[k]) continue;
    cudaError_t e = cudaStreamSynchronize(m->pipe_st[k]);
    if (e != cudaSuccess && rc == RBM_OK) rc = cuda_fail(e, who);
  }
  return rc;
}

template <class T>
int rnea_host(const rbm_model* m, const T* traj_host, T* tau_host, int64_t n, int64_t chunk) {
  if (!m) return invalid("rbm_rnea_host: model is NULL");
  if (n < 0) return invalid("rbm_rnea_host: n < 0");
  if (n == 0) return RBM_OK;
  if (!traj_host || !tau_host) return invalid("rbm_rnea_host: NULL buffer");
  const int nj = m->nj;
  if (chunk <= 0) chunk = 1 << 16;  // measured best on B200 + PCIe Gen5 (tools/bench_e2e_chunk.py): short pipeline fill, copies still large
  if (chunk > n) chunk = n;
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  std::lock_guard<std::mutex> lock(m->pipe_mu);
  constexpr int kSlots = rbm_model::kPipeSlots;
  if (int rc0 = ensure_pipe(m, sizeof(T) * chunk * 3 * nj, sizeof(T) * chunk * nj)) return rc0;
  int rc = RBM_OK;
  int slot = 0;
  for (int64_t s0 = 0; s0 < n && rc == RBM_OK; s0 += chunk, slot = (slot + 1) % kSlots) {
    const int64_t cnt = (n - s0 < chunk) ? (n - s0) : chunk;
    cudaStream_t st = m->pipe_st[slot];
    T* d_in = static_cast<T*>(m->pipe_in[slot]);
    T* d_out = static_cast<T*>(m->pipe_out[slot]);
    // stream order makes the slot safe to reuse: its previous D2H precedes this H2D on the same stream
    cudaError_t e = cudaMemcpyAsync(d_in, traj_host + s0 * 3 * nj, sizeof(T) * cnt * 3 * nj, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) { rc = cuda_fail(e, "rbm_rnea_host (H2D)"); break; }
    rc = launch_rnea_aos<T>(m, d_in, d_out, cnt, st);
    if (rc != RBM_OK) break;
    e = cudaMemcpyAsync(tau_host + s0 * nj, d_out, sizeof(T) * cnt * nj, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) { rc = cuda_fail(e, "rbm_rnea_host (D2H)"); break; }
  }
  return drain_pipe(m, rc, "rbm_rnea_host (synchronize)");
}

// Chunk of the SoA / planner-driven pipelines: a quarter of the batch, between 2^16 and 2^19 samples (measured on B200 + PCIe Gen5,
// tools/bench_e2e_chunk.py -> profiles/r2_e2e_chunk.jsonl: four to sixteen chunks keep fill / drain short while every strided copy
// still moves >= 0.5 MB per row).
static int64_t default_chunk(int64_t n) {
  int64_t c = n / 4;
  if (c < (int64_t)1 << 16) c = (int64_t)1 << 16;
  if (c > (int64_t)1 << 19) c = (int64_t)1 << 19;
  return c;
}

// which rows of (q, qd, qdd) the inverse-dynamics kernel of this model reads: [3][nj], 1 = live.  twists: V_6 / dV_6 are asked for too.
static void live_inputs(const rbm_model* m, int32_t* mask, bool twists) {
  for (int i = 0; i < 3 * m->nj; ++i) mask[i] = 1;
  if (m->path == PATH_GENERIC) return;
  // sequential structure (SequentialDesc::q_matters): tau, V_6 and dV_6 do not depend on the three gantry positions
  for (int j = 0; j < 3; ++j) mask[j] = 0;
  // SequentialDesc::qd_matters: tau does not depend on the three gantry velocities either (V_6 does)
  if (!twists)
    for (int j = 0; j < 3; ++j) mask[m->nj + j] = 0;
}

// SoA host entry: q, qd, qdd [nj][ld] on the host -> tau [nj][ld] on the host.  Dead rows stay on the host.
template <class T>
int rnea_host_soa(const rbm_model* m, const T* q_host, const T* qd_host, const T* qdd_host, T* tau_host, int64_t n, int64_t ld, int64_t chunk) {
  if (!m) return invalid("rbm_rnea_host_soa: model is NULL");
  if (n < 0) return invalid("rbm_rnea_host_soa: n < 0");
  if (n == 0) return RBM_OK;
  if (!q_host || !qd_host || !qdd_host || !tau_host) return invalid("rbm_rnea_host_soa: NULL buffer");
  if (ld < n) return invalid("rbm_rnea_host_soa: ld < n");
  const int nj = m->nj;
  if (chunk <= 0) chunk = default_chunk(n);
  if (chunk > n) chunk = n;
  chunk = (chunk + 1) & ~int64_t(1);  // even device pitch: keeps the fp32 two-samples-per-thread kernel eligible
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  std::lock_guard<std::mutex> lock(m->pipe_mu);
  constexpr int kSlots = rbm_model::kPipeSlots;
  if (int rc0 = ensure_pipe(m, sizeof(T) * chunk * 3 * nj, sizeof(T) * chunk * nj)) return rc0;
  int32_t live[3 * RBM_MAX_JOINTS];
  live_inputs(m, live, false);
  const T* src[3] = {q_host, qd_host, qdd_host};
  int rc = RBM_OK;
  int slot = 0;
  for (int64_t s0 = 0; s0 < n && rc == RBM_OK; s0 += chunk, slot = (slot + 1) % kSlots) {
    const int64_t cnt = (n - s0 < chunk) ? (n - s0) : chunk;
    cudaStream_t st = m->pipe_st[slot];
    T* d_in = static_cast<T*>(m->pipe_in[slot]);   // [3][nj][chunk]
    T* d_out = static_cast<T*>(m->pipe_out[slot]); // [nj][chunk]
    for (int a = 0; a < 3 && rc == RBM_OK; ++a) {
      // maximal runs of live rows of array a: one strided 2-D copy each (row = cnt samples, host pitch ld, device pitch chunk)
      for (int j = 0; j < nj;) {
        if (!live[a * nj + j]) { ++j; continue; }
        int j1 = j;
        while (j1 < nj && live[a * nj + j1]) ++j1;
        cudaError_t e = cudaMemcpy2DAsync(d_in + ((int64_t)a * nj + j) * chunk, sizeof(T) * chunk, src[a] + (int64_t)j * ld + s0, sizeof(T) * ld,
                                          sizeof(T) * cnt, (size_t)(j1 - j), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) { rc = cuda_fail(e, "rbm_rnea_host_soa (H2D)"); break; }
        j = j1;
      }
    }
    if (rc != RBM_OK) break;
    rc = launch_rnea_soa<T>(m, d_in, d_in + (int64_t)nj * chunk, d_in + (int64_t)2 * nj * chunk, d_out, nullptr, nullptr, cnt, chunk, st);
    if (rc != RBM_OK) break;
    cudaError_t e = cudaMemcpy2DAsync(tau_host + s0, sizeof(T) * ld, d_out, sizeof(T) * chunk, sizeof(T) * cnt, (size_t)nj, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) { rc = cuda_fail(e, "rbm_rnea_host_soa (D2H)"); break; }
  }
  return drain_pipe(m, rc, "rbm_rnea_host_soa (synchronize)");
}

// planner-driven host entry: nothing uploaded, tau [nj][ld] downloaded
template <class T>
int rnea_planned_host(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0, double stride,
                      T* tau_host, int64_t n, int64_t ld, int64_t chunk) {
  if (!m) return invalid("rbm_rnea_planned_host: model is NULL");
  if (n < 0) return invalid("rbm_rnea_planned_host: n < 0");
  if (n == 0) return RBM_OK;
  if (!coeffs || !disp || !offset || !tau_host) return invalid("rbm_rnea_planned_host: NULL pointer");
  if (ld < n) return invalid("rbm_rnea_planned_host: ld < n");
  if (!(timestep > 0.0)) return invalid("rbm_rnea_planned_host: timestep must be positive");
  const int nj = m->nj;
  if (chunk <= 0) chunk = default_chunk(n);
  if (chunk > n) chunk = n;
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  std::lock_guard<std::mutex> lock(m->pipe_mu);
  constexpr int kSlots = rbm_model::kPipeSlots;
  if (int rc0 = ensure_pipe(m, 0, sizeof(T) * chunk * nj)) return rc0;
  int rc = RBM_OK;
  int slot = 0;
  for (int64_t s0 = 0; s0 < n && rc == RBM_OK; s0 += chunk, slot = (slot + 1) % kSlots) {
    const int64_t cnt = (n - s0 < chunk) ? (n - s0) : chunk;
    cudaStream_t st = m->pipe_st[slot];
    T* d_out = static_cast<T*>(m->pipe_out[slot]);
    rc = launch_rnea_planned<T>(m, coeffs, disp, offset, timestep, step0 + (double)s0 * stride, stride, d_out, nullptr, cnt, chunk, st);
    if (rc != RBM_OK) break;
    cudaError_t e = cudaMemcpy2DAsync(tau_host + s0, sizeof(T) * ld, d_out, sizeof(T) * chunk, sizeof(T) * cnt, (size_t)nj, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) { rc = cuda_fail(e, "rbm_rnea_planned_host (D2H)"); break; }
  }
  return drain_pipe(m, rc, "rbm_rnea_planned_host (synchronize)");
}
}  // namespace rbm


using namespace rbm;

extern "C" {

const char* rbm_version(void) { return "rbm_b200 0.1 (sm_100a)"; }
const char* rbm_last_error_string(void) { return g_last_error.c_str(); }

int rbm_device_pci_bus_id(int device, char* out, int len) {
  if (!out || len < 13) return invalid("rbm_device_pci_bus_id: need a buffer of at least 13 bytes");
  RBM_CUDA_TRY(cudaDeviceGetPCIBusId(out, len, device));
  return RBM_OK;
}

int rbm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

}  // extern "C"

namespace {
// Device-free part of model creation: validation, generic packing, structure analysis.  Fills everything of `m` except the
// device buffers.
int analyze_model(const char* who, int nj, const double* hposes_Rt, const double* simats, const double* uscrews, const double* twist_0,
                  const double* dtwist_0, const double* wrench_tip, const double* pose_tip_Rt, const double* pose_sen_Rt, unsigned flags,
                  rbm_model* m) {
  const std::string w(who);
  if (nj < 1) return invalid(w + ": nj must be >= 1");
  if (nj > RBM_MAX_JOINTS) {
    set_error(w + ": nj exceeds RBM_MAX_JOINTS (16)");
    return RBM_ERR_UNSUPPORTED;
  }
  if (!hposes_Rt || !simats || !uscrews || !twist_0 || !dtwist_0) return invalid(w + ": NULL constant array");
  const int np = generic_param_count(nj);
  for (int i = 0; i < (nj + 1) * 12; ++i)
    if (!std::isfinite(hposes_Rt[i])) return invalid(w + ": non-finite home pose");
  for (int i = 0; i < (nj + 1) * 36; ++i)
    if (!std::isfinite(simats[i])) return invalid(w + ": non-finite spatial inertia");
  for (int i = 0; i < nj * 6; ++i)
    if (!std::isfinite(uscrews[i])) return invalid(w + ": non-finite screw");
  m->nj = nj;
  m->no_tma = (flags & RBM_FLAG_NO_TMA) != 0;
  m->gp64.assign(np, 0.0);
  double* g = m->gp64.data();
  static const double ident[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
  std::memcpy(g + GP_V0, twist_0, 6 * sizeof(double));
  std::memcpy(g + GP_DV0, dtwist_0, 6 * sizeof(double));
  if (wrench_tip) std::memcpy(g + GP_FTIP, wrench_tip, 6 * sizeof(double));
  std::memcpy(g + GP_TIPR, pose_tip_Rt ? pose_tip_Rt : ident, 12 * sizeof(double));
  std::memcpy(g + GP_SENR, pose_sen_Rt ? pose_sen_Rt : ident, 12 * sizeof(double));
  for (int i = 0; i < nj; ++i) {
    double* J = g + GP_HEAD + GJ_STRIDE * i;
    const double* hR = hposes_Rt + 12 * (i + 1);
    const double* ht = hR + 9;
    const double* sv = uscrews + 6 * i;
    const double* sw = sv + 3;
    std::memcpy(J + GJ_S, sv, 6 * sizeof(double));
    const double wn = std::sqrt(sw[0] * sw[0] + sw[1] * sw[1] + sw[2] * sw[2]);
    J[GJ_NW] = -wn;
    if (wn == 0.0) {  // prismatic: R = hR, p = ht - q v
      for (int k = 0; k < 9; ++k) J[GJ_RC + k] = hR[k];
      for (int k = 0; k < 3; ++k) { J[GJ_PC + k] = -sv[k]; J[GJ_PD + k] = ht[k]; }
    } else {
      // fold the exponential's constants (layout comment in rbm_model.cuh)
      const double a[3] = {sw[0] / wn, sw[1] / wn, sw[2] / wn}, r[3] = {sv[0] / wn, sv[1] / wn, sv[2] / wn};
      auto cross = [](const double* x, const double* y, double* o) {
        o[0] = x[1] * y[2] - x[2] * y[1]; o[1] = x[2] * y[0] - x[0] * y[2]; o[2] = x[0] * y[1] - x[1] * y[0];
      };
      for (int c = 0; c < 3; ++c) {  // column c of hR
        const double col[3] = {hR[c], hR[3 + c], hR[6 + c]};
        const double ac = a[0] * col[0] + a[1] * col[1] + a[2] * col[2];
        double xc[3];
        cross(a, col, xc);
        for (int rr = 0; rr < 3; ++rr) {
          J[GJ_RC + 3 * rr + c] = a[rr] * ac;
          J[GJ_RA + 3 * rr + c] = col[rr] - a[rr] * ac;
          J[GJ_RB + 3 * rr + c] = xc[rr];
        }
      }
      const double at = a[0] * ht[0] + a[1] * ht[1] + a[2] * ht[2], ar = a[0] * r[0] + a[1] * r[1] + a[2] * r[2];
      const double av = a[0] * sv[0] + a[1] * sv[1] + a[2] * sv[2];
      double axr[3], axt[3];
      cross(a, r, axr);
      cross(a, ht, axt);
      for (int k = 0; k < 3; ++k) {
        J[GJ_PA + k] = ht[k] - a[k] * at - axr[k];
        J[GJ_PB + k] = axt[k] + r[k] - ar * a[k];
        J[GJ_PC + k] = -av * a[k];
        J[GJ_PD + k] = a[k] * at + axr[k];
      }
    }
    std::memcpy(J + GJ_G, simats + 36 * (i + 1), 36 * sizeof(double));
    RigidForm rf;
    J[GJ_RIGID] = rigid_form(simats + 36 * (i + 1), &rf) ? 1.0 : 0.0;
  }
  m->gp32.resize(np);
  for (int i = 0; i < np; ++i) m->gp32[i] = (float)g[i];

  std::memset(&m->fp64, 0, sizeof(m->fp64));
  m->path = PATH_GENERIC;
  if (!(flags & RBM_FLAG_FORCE_GENERIC))
    m->path = detect_path(nj, hposes_Rt, simats, uscrews, twist_0, dtwist_0, wrench_tip, pose_tip_Rt, &m->fp64);
  std::memcpy(m->fp64.senR, g + GP_SENR, 9 * sizeof(double));
  std::memcpy(m->fp64.sent, g + GP_SENT, 3 * sizeof(double));
  {  // sensor pose with a diagonal rotation and no offset (snapped like the home rotations): Ad(T) acts component-wise
    bool diag = m->path != PATH_GENERIC;
    for (int r = 0; r < 3 && diag; ++r) {
      for (int c = 0; c < 3; ++c) {
        const double v = m->fp64.senR[3 * r + c];
        if (r == c ? !(near(v, 1.0) || near(v, -1.0)) : !near(v, 0.0)) diag = false;
      }
      if (!near(m->fp64.sent[r], 0.0)) diag = false;
    }
    m->fp64.sen_diag = diag ? 1.0 : 0.0;
    if (diag)
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) m->fp64.senR[3 * r + c] = r == c ? (m->fp64.senR[3 * r + c] > 0 ? 1.0 : -1.0) : 0.0;
  }
  convert_fast(m->fp64, &m->fp32);
  return RBM_OK;
}
}  // namespace

extern "C" {

int rbm_fast_param_count(void) { return (int)(sizeof(FastParams<double>) / sizeof(double)); }
int rbm_generic_param_count(int nj) { return (nj < 1 || nj > RBM_MAX_JOINTS) ? RBM_ERR_INVALID : generic_param_count(nj); }

int rbm_model_analyze(int nj, const double* hposes_Rt, const double* simats, const double* uscrews, const double* twist_0, const double* dtwist_0,
                      const double* wrench_tip, const double* pose_tip_Rt, const double* pose_sen_Rt, unsigned flags, int* kernel_path,
                      double* fast_params, double* generic_params) {
  rbm_model tmp;
  int rc = analyze_model("rbm_model_analyze", nj, hposes_Rt, simats, uscrews, twist_0, dtwist_0, wrench_tip, pose_tip_Rt, pose_sen_Rt, flags, &tmp);
  if (rc != RBM_OK) return rc;
  if (kernel_path) *kernel_path = tmp.path;
  if (fast_params) std::memcpy(fast_params, &tmp.fp64, sizeof(tmp.fp64));
  if (generic_params) std::memcpy(generic_params, tmp.gp64.data(), tmp.gp64.size() * sizeof(double));
  return RBM_OK;
}

int rbm_model_create(int nj, const double* hposes_Rt, const double* simats, const double* uscrews, const double* twist_0,
                     const double* dtwist_0, const double* wrench_tip, const double* pose_tip_Rt, const double* pose_sen_Rt,
                     unsigned flags, int device, rbm_model** out) {
  if (!out) return invalid("rbm_model_create: out is NULL");
  *out = nullptr;
  rbm_model* m = new (std::nothrow) rbm_model();
  if (!m) return invalid("rbm_model_create: out of host memory");
  int rc = analyze_model("rbm_model_create", nj, hposes_Rt, simats, uscrews, twist_0, dtwist_0, wrench_tip, pose_tip_Rt, pose_sen_Rt, flags, m);
  if (rc != RBM_OK) {
    delete m;
    return rc;
  }
  m->device = device;
  const int np = generic_param_count(nj);
  DeviceGuard guard(device);
  cudaError_t e = guard.status();
  if (e == cudaSuccess) e = cudaMalloc(&m->d_gp64, np * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&m->d_gp32, np * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(m->d_gp64, m->gp64.data(), np * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(m->d_gp32, m->gp32.data(), np * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    rc = cuda_fail(e, "rbm_model_create (device allocation / upload)");
    cudaGetLastError();
    rbm_model_destroy(m);
    return rc;
  }
  *out = m;
  return RBM_OK;
}

void rbm_model_destroy(rbm_model* m) {
  if (!m) return;
  if (m->full_dev) cudaFree(m->full_dev);
  if (m->full_pinned) cudaFreeHost(m->full_pinned);
  for (int k = 0; k < rbm_model::kPipeSlots; ++k) {
    if (m->pipe_st[k]) cudaStreamDestroy(m->pipe_st[k]);
    if (m->pipe_in[k]) cudaFree(m->pipe_in[k]);
    if (m->pipe_out[k]) cudaFree(m->pipe_out[k]);
  }
  if (m->d_gp64) cudaFree(m->d_gp64);
  if (m->d_gp32) cudaFree(m->d_gp32);
  delete m;
}

int rbm_model_num_joints(const rbm_model* m) { return m ? m->nj : RBM_ERR_INVALID; }
int rbm_model_kernel_path(const rbm_model* m) { return m ? m->path : RBM_ERR_INVALID; }

#define RBM_CHECK_BATCH(name)                                                         \
  if (!m) return invalid(name ": model is NULL");                                    \
  if (n < 0) return invalid(name ": n < 0");                                         \
  if (n == 0) return RBM_OK;                                                         \
  DeviceGuard rbm_guard_(m->device);                                                 \
  RBM_CUDA_TRY(rbm_guard_.status());

int rbm_rnea_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, double* tau, double* twist_last,
                 double* dtwist_last, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_f64")
  if (!q || !qd || !qdd || !tau) return invalid("rbm_rnea_f64: NULL batch pointer");
  if (ld < n) return invalid("rbm_rnea_f64: ld < n");
  if ((twist_last == nullptr) != (dtwist_last == nullptr)) return invalid("rbm_rnea_f64: twist_last and dtwist_last go together");
  return launch_rnea_soa<double>(m, q, qd, qdd, tau, twist_last, dtwist_last, n, ld, (cudaStream_t)stream);
}

int rbm_rnea_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, float* tau, float* twist_last,
                 float* dtwist_last, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_f32")
  if (!q || !qd || !qdd || !tau) return invalid("rbm_rnea_f32: NULL batch pointer");
  if (ld < n) return invalid("rbm_rnea_f32: ld < n");
  if ((twist_last == nullptr) != (dtwist_last == nullptr)) return invalid("rbm_rnea_f32: twist_last and dtwist_last go together");
  return launch_rnea_soa<float>(m, q, qd, qdd, tau, twist_last, dtwist_last, n, ld, (cudaStream_t)stream);
}

int rbm_rnea_aos_f64(const rbm_model* m, const double* traj, double* tau, int64_t n, void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_aos_f64")
  if (!traj || !tau) return invalid("rbm_rnea_aos_f64: NULL batch pointer");
  return launch_rnea_aos<double>(m, traj, tau, n, (cudaStream_t)stream);
}

int rbm_rnea_aos_f32(const rbm_model* m, const float* traj, float* tau, int64_t n, void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_aos_f32")
  if (!traj || !tau) return invalid("rbm_rnea_aos_f32: NULL batch pointer");
  return launch_rnea_aos<float>(m, traj, tau, n, (cudaStream_t)stream);
}

int rbm_rnea_planned_f64(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0, double stride,
                         double* tau, double* traj, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_planned_f64")
  if (!coeffs || !disp || !offset || !tau) return invalid("rbm_rnea_planned_f64: NULL pointer");
  if (ld < n) return invalid("rbm_rnea_planned_f64: ld < n");
  if (!(timestep > 0.0)) return invalid("rbm_rnea_planned_f64: timestep must be positive");
  return launch_rnea_planned<double>(m, coeffs, disp, offset, timestep, step0, stride, tau, traj, n, ld, (cudaStream_t)stream);
}

int rbm_rnea_planned_f32(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0, double stride,
                         float* tau, float* traj, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_planned_f32")
  if (!coeffs || !disp || !offset || !tau) return invalid("rbm_rnea_planned_f32: NULL pointer");
  if (ld < n) return invalid("rbm_rnea_planned_f32: ld < n");
  if (!(timestep > 0.0)) return invalid("rbm_rnea_planned_f32: timestep must be positive");
  return launch_rnea_planned<float>(m, coeffs, disp, offset, timestep, step0, stride, tau, traj, n, ld, (cudaStream_t)stream);
}

int rbm_rnea_full_f64(const rbm_model* m, const double* traj, double* tau, double* poses, double* twists, double* dtwists, int64_t n,
                      void* stream) {
  RBM_CHECK_BATCH("rbm_rnea_full_f64")
  if (!traj || !tau) return invalid("rbm_rnea_full_f64: NULL batch pointer");
  if ((twists == nullptr) != (dtwists == nullptr)) return invalid("rbm_rnea_full_f64: twists and dtwists go together");
  return launch_rnea_full<double>(m, traj, tau, poses, twists, dtwists, n, (cudaStream_t)stream);
}

int rbm_rnea_host_f64(const rbm_model* m, const double* traj_host, double* tau_host, int64_t n, int64_t chunk) {
  return rnea_host<double>(m, traj_host, tau_host, n, chunk);
}
int rbm_rnea_host_f32(const rbm_model* m, const float* traj_host, float* tau_host, int64_t n, int64_t chunk) {
  return rnea_host<float>(m, traj_host, tau_host, n, chunk);
}

int rbm_rnea_host_soa_f64(const rbm_model* m, const double* q_host, const double* qd_host, const double* qdd_host, double* tau_host, int64_t n,
                          int64_t ld, int64_t chunk) {
  return rnea_host_soa<double>(m, q_host, qd_host, qdd_host, tau_host, n, ld, chunk);
}
int rbm_rnea_host_soa_f32(const rbm_model* m, const float* q_host, const float* qd_host, const float* qdd_host, float* tau_host, int64_t n, int64_t ld,
                          int64_t chunk) {
  return rnea_host_soa<float>(m, q_host, qd_host, qdd_host, tau_host, n, ld, chunk);
}
int rbm_rnea_planned_host_f64(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0,
                              double stride, double* tau_host, int64_t n, int64_t ld, int64_t chunk) {
  return rnea_planned_host<double>(m, coeffs, disp, offset, timestep, step0, stride, tau_host, n, ld, chunk);
}
int rbm_rnea_planned_host_f32(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0,
                              double stride, float* tau_host, int64_t n, int64_t ld, int64_t chunk) {
  return rnea_planned_host<float>(m, coeffs, disp, offset, timestep, step0, stride, tau_host, n, ld, chunk);
}
int rbm_model_live_inputs(const rbm_model* m, int32_t* mask) {
  if (!m || !mask) return invalid("rbm_model_live_inputs: NULL argument");
  live_inputs(m, mask, true);
  return RBM_OK;
}


// Small-batch host convenience behind the scalar drop-in `dynamics.inverse`: host traj in, every output of the reference's
// return value out, with one H2D copy, one launch and one D2H copy through scratch owned by the model.
int rbm_rnea_full_host_f64(const rbm_model* m, const double* traj_host, double* tau_host, double* poses_host, double* twists_host,
                           double* dtwists_host, int64_t n) {
  RBM_CHECK_BATCH("rbm_rnea_full_host_f64")
  if (!traj_host || !tau_host) return invalid("rbm_rnea_full_host_f64: NULL buffer");
  if ((twists_host == nullptr) != (dtwists_host == nullptr)) return invalid("rbm_rnea_full_host_f64: twists and dtwists go together");
  const int nj = m->nj;
  const size_t n_in = (size_t)n * 3 * nj, n_tau = (size_t)n * nj, n_pose = (size_t)n * nj * 12, n_tw = (size_t)n * (nj + 1) * 6;
  const size_t total = n_in + n_tau + n_pose + 2 * n_tw;
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  std::lock_guard<std::mutex> lock(m->pipe_mu);
  if (total > m->full_doubles) {
    if (m->full_dev) cudaFree(m->full_dev);
    if (m->full_pinned) cudaFreeHost(m->full_pinned);
    m->full_dev = nullptr;
    m->full_pinned = nullptr;
    m->full_doubles = 0;
    const size_t cap = total < 4096 ? 4096 : total;
    RBM_CUDA_TRY(cudaMalloc(&m->full_dev, cap * sizeof(double)));
    RBM_CUDA_TRY(cudaMallocHost(&m->full_pinned, cap * sizeof(double)));
    m->full_doubles = cap;
  }
  if (!m->pipe_st[0]) RBM_CUDA_TRY(cudaStreamCreateWithFlags(&m->pipe_st[0], cudaStreamNonBlocking));
  cudaStream_t st = m->pipe_st[0];
  double* d_in = m->full_dev;
  double* d_out = m->full_dev + n_in;
  std::memcpy(m->full_pinned, traj_host, n_in * sizeof(double));
  RBM_CUDA_TRY(cudaMemcpyAsync(d_in, m->full_pinned, n_in * sizeof(double), cudaMemcpyHostToDevice, st));
  int rc = launch_rnea_full<double>(m, d_in, d_out, d_out + n_tau, d_out + n_tau + n_pose, d_out + n_tau + n_pose + n_tw, n, st);
  if (rc != RBM_OK) return rc;
  double* h_out = m->full_pinned + n_in;
  RBM_CUDA_TRY(cudaMemcpyAsync(h_out, d_out, (total - n_in) * sizeof(double), cudaMemcpyDeviceToHost, st));
  RBM_CUDA_TRY(cudaStreamSynchronize(st));
  std::memcpy(tau_host, h_out, n_tau * sizeof(double));
  if (poses_host) std::memcpy(poses_host, h_out + n_tau, n_pose * sizeof(double));
  if (twists_host) {
    std::memcpy(twists_host, h_out + n_tau + n_pose, n_tw * sizeof(double));
    std::memcpy(dtwists_host, h_out + n_tau + n_pose + n_tw, n_tw * sizeof(double));
  }
  return RBM_OK;
}

// ---- regressor / identification ------------------------------------------------------------------
int rbm_regressor_rows_f64(const double* twists, const double* dtwists, double* Y, int64_t n, void* stream) {
  if (n < 0) return invalid("rbm_regressor_rows_f64: n < 0");
  if (n == 0) return RBM_OK;
  if (!twists || !dtwists || !Y) return invalid("rbm_regressor_rows_f64: NULL pointer");
  return launch_regressor_rows<double>(twists, dtwists, Y, n, (cudaStream_t)stream);
}

int rbm_sensor_twists_f64(const double* pose_Rt, const double* twists, const double* dtwists, double* twists_sen, double* dtwists_sen, int64_t n,
                          void* stream) {
  if (n < 0) return invalid("rbm_sensor_twists_f64: n < 0");
  if (n == 0) return RBM_OK;
  if (!pose_Rt || !twists || !dtwists || !twists_sen || !dtwists_sen) return invalid("rbm_sensor_twists_f64: NULL pointer");
  return launch_sensor_twists<double>(pose_Rt, twists, dtwists, twists_sen, dtwists_sen, n, (cudaStream_t)stream);
}

}  // extern "C"

namespace {
template <class T>
int regressor_from_traj(const char* name, const rbm_model* m, const T* q, const T* qd, const T* qdd, T* Y, T* Vs, T* dVs, const T* phi, T* F, int64_t n,
                        int64_t ld, void* stream) {
  if (!m) return invalid(std::string(name) + ": model is NULL");
  if (n < 0) return invalid(std::string(name) + ": n < 0");
  if (n == 0) return RBM_OK;
  if (!q || !qd || !qdd) return invalid(std::string(name) + ": NULL batch pointer");
  if (ld < n) return invalid(std::string(name) + ": ld < n");
  if ((Vs == nullptr) != (dVs == nullptr)) return invalid(std::string(name) + ": twist_sen and dtwist_sen go together");
  if ((phi == nullptr) != (F == nullptr)) return invalid(std::string(name) + ": phi and wrench go together");
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  return launch_regressor_from_traj<T>(m, q, qd, qdd, Y, Vs, dVs, phi, F, n, ld, (cudaStream_t)stream);
}
template <class T>
int regressor_gram(const char* name, const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* f, double* pack, void* ws, size_t ws_bytes,
                   int64_t n, int64_t ld, void* stream) {
  if (!m) return invalid(std::string(name) + ": model is NULL");
  if (n < 0) return invalid(std::string(name) + ": n < 0");
  if (!pack || !ws) return invalid(std::string(name) + ": NULL gram_pack / workspace");
  if (n > 0 && (!q || !qd || !qdd || !f)) return invalid(std::string(name) + ": NULL batch pointer");
  if (ld < n) return invalid(std::string(name) + ": ld < n");
  if (ws_bytes < rbm_gram_workspace_bytes(m, n)) return invalid(std::string(name) + ": workspace too small (see rbm_gram_workspace_bytes)");
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  return launch_regressor_gram<T>(m, q, qd, qdd, f, pack, static_cast<double*>(ws), n, ld, (cudaStream_t)stream);
}
template <class T>
int payload_regressor(const char* name, const rbm_model* m, const T* q, const T* qd, const T* qdd, T* Phi, T* tau0, int64_t n, int64_t ld, void* stream) {
  if (!m) return invalid(std::string(name) + ": model is NULL");
  if (n < 0) return invalid(std::string(name) + ": n < 0");
  if (n == 0) return RBM_OK;
  if (!q || !qd || !qdd) return invalid(std::string(name) + ": NULL batch pointer");
  if (ld < n) return invalid(std::string(name) + ": ld < n");
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  return launch_payload_regressor<T>(m, q, qd, qdd, Phi, tau0, n, ld, (cudaStream_t)stream);
}
template <class T>
int payload_gram(const char* name, const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* tau, double* pack, void* ws, size_t ws_bytes,
                 int64_t n, int64_t ld, void* stream) {
  if (!m) return invalid(std::string(name) + ": model is NULL");
  if (n < 0) return invalid(std::string(name) + ": n < 0");
  if (!pack || !ws) return invalid(std::string(name) + ": NULL gram_pack / workspace");
  if (n > 0 && (!q || !qd || !qdd || !tau)) return invalid(std::string(name) + ": NULL batch pointer");
  if (ld < n) return invalid(std::string(name) + ": ld < n");
  if (ws_bytes < rbm_gram_workspace_bytes(m, n)) return invalid(std::string(name) + ": workspace too small (see rbm_gram_workspace_bytes)");
  DeviceGuard guard(m->device);
  RBM_CUDA_TRY(guard.status());
  return launch_payload_gram<T>(m, q, qd, qdd, tau, pack, static_cast<double*>(ws), n, ld, (cudaStream_t)stream);
}
}  // namespace

extern "C" {

int rbm_regressor_from_traj_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, double* Y, double* twist_sen,
                                double* dtwist_sen, const double* phi, double* wrench, int64_t n, int64_t ld, void* stream) {
  return regressor_from_traj<double>("rbm_regressor_from_traj_f64", m, q, qd, qdd, Y, twist_sen, dtwist_sen, phi, wrench, n, ld, stream);
}
int rbm_regressor_from_traj_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, float* Y, float* twist_sen, float* dtwist_sen,
                                const float* phi, float* wrench, int64_t n, int64_t ld, void* stream) {
  return regressor_from_traj<float>("rbm_regressor_from_traj_f32", m, q, qd, qdd, Y, twist_sen, dtwist_sen, phi, wrench, n, ld, stream);
}

size_t rbm_gram_workspace_bytes(const rbm_model* m, int64_t n) {
  if (!m) return 0;
  return sizeof(double) * 70 * (size_t)gram_grid(m, n < 0 ? 0 : n, 2);  // upper bound over dtypes
}
int rbm_regressor_gram_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, const double* f, double* gram_pack,
                           void* workspace, size_t workspace_bytes, int64_t n, int64_t ld, void* stream) {
  return regressor_gram<double>("rbm_regressor_gram_f64", m, q, qd, qdd, f, gram_pack, workspace, workspace_bytes, n, ld, stream);
}
int rbm_regressor_gram_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, const float* f, double* gram_pack, void* workspace,
                           size_t workspace_bytes, int64_t n, int64_t ld, void* stream) {
  return regressor_gram<float>("rbm_regressor_gram_f32", m, q, qd, qdd, f, gram_pack, workspace, workspace_bytes, n, ld, stream);
}

int rbm_payload_regressor_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, double* Phi, double* tau0, int64_t n, int64_t ld,
                              void* stream) {
  return payload_regressor<double>("rbm_payload_regressor_f64", m, q, qd, qdd, Phi, tau0, n, ld, stream);
}
int rbm_payload_regressor_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, float* Phi, float* tau0, int64_t n, int64_t ld,
                              void* stream) {
  return payload_regressor<float>("rbm_payload_regressor_f32", m, q, qd, qdd, Phi, tau0, n, ld, stream);
}
int rbm_payload_gram_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, const double* tau, double* gram_pack, void* workspace,
                         size_t workspace_bytes, int64_t n, int64_t ld, void* stream) {
  return payload_gram<double>("rbm_payload_gram_f64", m, q, qd, qdd, tau, gram_pack, workspace, workspace_bytes, n, ld, stream);
}
int rbm_payload_gram_f32(const rbm_model* m, const float* q, const float* qd, const float* qdd, const float* tau, double* gram_pack, void* workspace,
                         size_t workspace_bytes, int64_t n, int64_t ld, void* stream) {
  return payload_gram<float>("rbm_payload_gram_f32", m, q, qd, qdd, tau, gram_pack, workspace, workspace_bytes, n, ld, stream);
}

int rbm_regressor_gram_grouped_f64(const rbm_model* m, const double* q, const double* qd, const double* qdd, const double* f, int64_t frame_stride,
                                   int64_t f_frame_stride, int64_t n_frames, double* gram_packs, int64_t n_groups, int64_t ld, int64_t ld_out, void* stream) {
  const int64_t n = n_groups;
  RBM_CHECK_BATCH("rbm_regressor_gram_grouped_f64")
  if (!q || !qd || !qdd || !f || !gram_packs) return invalid("rbm_regressor_gram_grouped_f64: NULL pointer");
  if (n_frames < 0 || frame_stride < 0 || f_frame_stride < 0) return invalid("rbm_regressor_gram_grouped_f64: n_frames / frame_stride < 0");
  if (ld < n_groups || ld_out < n_groups) return invalid("rbm_regressor_gram_grouped_f64: ld / ld_out < n_groups");
  return launch_regressor_gram_grouped<double>(m, q, qd, qdd, f, frame_stride, f_frame_stride, n_frames, gram_packs, n_groups, ld, ld_out, (cudaStream_t)stream);
}

int rbm_linearize_f64(const rbm_model* m, const double* q, const double* qd, const double* u, double dt, double eps, int centered, double* A,
                      double* B, double* qdd, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_linearize_f64")
  if (!q || !qd || !A || !B) return invalid("rbm_linearize_f64: NULL batch pointer");
  if (ld < n) return invalid("rbm_linearize_f64: ld < n");
  if (!(dt > 0.0) || !(eps > 0.0)) return invalid("rbm_linearize_f64: dt and eps must be positive");
  return launch_linearize<double>(m, q, qd, u, dt, eps, centered, A, B, qdd, n, ld, (cudaStream_t)stream);
}

int rbm_forward_dynamics_f64(const rbm_model* m, const double* q, const double* qd, const double* u, double dt, double* qdd, double* q_next,
                             double* qd_next, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_forward_dynamics_f64")
  if (!q || !qd) return invalid("rbm_forward_dynamics_f64: NULL batch pointer");
  if (!qdd && !q_next) return invalid("rbm_forward_dynamics_f64: no output requested");
  if ((q_next == nullptr) != (qd_next == nullptr)) return invalid("rbm_forward_dynamics_f64: q_next and qd_next go together");
  if (q_next && !(dt > 0.0)) return invalid("rbm_forward_dynamics_f64: dt must be positive");
  if (ld < n) return invalid("rbm_forward_dynamics_f64: ld < n");
  return launch_forward_dynamics<double>(m, q, qd, u, dt, qdd, q_next, qd_next, n, ld, (cudaStream_t)stream);
}

int rbm_closed_loop_f64(const rbm_model* m, const double* plan_coeffs, const double* displacement, const double* pos_offset, double plan_timestep,
                        double init_step, int64_t n_steps, const double* gain, const double* phi_sensed, double dt, double fps,
                        double pos_residual_divisor, const double* q0, const double* qd0, double* frames, int64_t max_frames, int32_t* frame_steps,
                        int32_t* n_frames, double* final_state, int64_t n, int64_t ld, void* stream) {
  RBM_CHECK_BATCH("rbm_closed_loop_f64")
  if (!plan_coeffs || !displacement || !pos_offset) return invalid("rbm_closed_loop_f64: NULL planner description");
  if (!gain || !phi_sensed || !q0) return invalid("rbm_closed_loop_f64: NULL gain / phi_sensed / q0");
  if (n_steps < 0 || n_steps > (int64_t)1 << 30) return invalid("rbm_closed_loop_f64: n_steps out of range");
  if (max_frames < 0 || max_frames > (int64_t)1 << 30 || (max_frames > 0 && !frames)) return invalid("rbm_closed_loop_f64: frames / max_frames");
  if (!(dt > 0.0) || !(plan_timestep > 0.0) || !(fps >= 0.0) || pos_residual_divisor == 0.0) return invalid("rbm_closed_loop_f64: dt, plan_timestep > 0, fps >= 0, divisor != 0");
  if (ld < n) return invalid("rbm_closed_loop_f64: ld < n");
  return launch_closed_loop(m, plan_coeffs, displacement, pos_offset, plan_timestep, init_step, (int)n_steps, gain, phi_sensed, dt, fps,
                            pos_residual_divisor, q0, qd0, frames, (int)max_frames, frame_steps, n_frames, final_state, n, ld, (cudaStream_t)stream);
}

// ---- frame algebra helpers ------------------------------------------------------------------------
#define RBM_SIMPLE_CHECK(name, cond)                       \
  if (n < 0) return invalid(name ": n < 0");               \
  if (n == 0) return RBM_OK;                               \
  if (!(cond)) return invalid(name ": NULL pointer");

int rbm_transfer_simat_f64(const double* poses_Rt, const double* simats, double* out, int64_t n, void* stream) {
  RBM_SIMPLE_CHECK("rbm_transfer_simat_f64", poses_Rt && simats && out)
  return launch_transfer_simat(poses_Rt, simats, out, n, 12, 36, 0, (cudaStream_t)stream);
}
int rbm_coordinate_transfer_simat_f64(const double* poses_Rt, const double* simats, double* out, int64_t n, void* stream) {
  RBM_SIMPLE_CHECK("rbm_coordinate_transfer_simat_f64", poses_Rt && simats && out)
  return launch_transfer_simat(poses_Rt, simats, out, n, 12, 36, 1, (cudaStream_t)stream);
}
int rbm_coordinate_transfer_imat_f64(const double* poses_Rt, const double* imats, const double* mass, double* out, int64_t n, void* stream) {
  RBM_SIMPLE_CHECK("rbm_coordinate_transfer_imat_f64", poses_Rt && imats && mass && out)
  return launch_transfer_imat(poses_Rt, imats, mass, out, n, (cudaStream_t)stream);
}
int rbm_spatial_inertia_f64(const double* mass, const double* diag, double* out, int64_t n, void* stream) {
  RBM_SIMPLE_CHECK("rbm_spatial_inertia_f64", mass && diag && out)
  return launch_spatial_inertia(mass, diag, out, n, (cudaStream_t)stream);
}
int rbm_compose_f64(const double* trans, const double* rot, int rot_len, double* poses_Rt, int32_t* status, int64_t n, void* stream) {
  if (rot_len != 4 && rot_len != 9) return invalid("rbm_compose_f64: rot_len must be 4 (wxyz quaternion) or 9 (rotation matrix)");
  RBM_SIMPLE_CHECK("rbm_compose_f64", trans && rot && poses_Rt && status)
  return launch_compose(trans, rot, rot_len, poses_Rt, status, n, (cudaStream_t)stream);
}
int rbm_point_motion_f64(const double* twists, const double* dtwists, const double* points, double* linvel, double* linacc, int64_t n, void* stream) {
  RBM_SIMPLE_CHECK("rbm_point_motion_f64", twists && points && (linvel || linacc) && (!linacc || dtwists))
  return launch_point_motion(twists, dtwists, points, linvel, linacc, n, (cudaStream_t)stream);
}

}  // extern "C"
