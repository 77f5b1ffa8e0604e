// Batched inverse-dynamics kernels and their launchers (sm_100a).
//
// One sample per thread; consecutive threads own consecutive samples, so every SoA stream
// (q_j, qd_j, qdd_j, tau_j) is read / written as fully coalesced 128-byte lines and nothing is
// re-read.  Rows the result does not depend on are not loaded (SoaRows): a tau-only launch on the
// sequential structure moves 18 * sizeof(T) bytes per sample of the 24 the rows hold.
#include <atomic>
#include <cstdlib>
#include <cstring>

#include "rbm_async.cuh"
#include "rbm_internal.h"
#include "rbm_rnea.cuh"

namespace rbm {

constexpr int kBlock = 128;

// griddepcontrol (sm_90+): no-ops when the kernel was not launched with the programmatic-serialisation attribute
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_prior_grids() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

static bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("RBM_NO_PDL");
    return !(e && e[0] == '1');
  }();
  return on;
}

// launch with programmatic stream serialisation allowed: the grid may start (and park in griddepcontrol.wait) while the
// previous kernel of the stream is still draining, which removes the launch gap between back-to-back batches
template <class... KArgs, class... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------------------------
// fast path, SoA
// ---------------------------------------------------------------------------------------------
// Rows of (q, qd, qdd) -- a = 0, 1, 2 -- that the fast SoA kernels load: never the gantry positions, the gantry velocities only when
// the twist is asked for (SequentialDesc::q_matters / qd_matters).
template <class D, bool OUT_TWIST>
struct SoaRows {
  static constexpr bool live(int a, int j) { return a == 0 ? D::q_matters(j) : a == 1 ? (OUT_TWIST || D::qd_matters(j)) : true; }
};

template <class T, class D, bool OUT_TWIST>
__global__ void __launch_bounds__(kBlock) k_rnea_fast_soa(const __grid_constant__ FastParams<T> P, const T* __restrict__ q,
                                                          const T* __restrict__ qd, const T* __restrict__ qdd, T* __restrict__ tau,
                                                          T* __restrict__ Vout, T* __restrict__ dVout, int64_t n, int64_t ld) {
  using Rows = SoaRows<D, OUT_TWIST>;
  // Programmatic dependent launch: let the next kernel in the stream be scheduled while this grid drains, and wait for
  // the previous grid's memory to be visible before the first global read (stream-order semantics are unchanged).
  pdl_launch_dependents();
  pdl_wait_prior_grids();
  const int64_t s = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (s >= n) return;
  T rq[6], rqd[6], rqdd[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    rq[j] = Rows::live(0, j) ? __ldg(q + j * ld + s) : T(0);
    rqd[j] = Rows::live(1, j) ? __ldg(qd + j * ld + s) : T(0);
    rqdd[j] = __ldg(qdd + j * ld + s);
  }
  FastResult<T> r;
  fast_rnea_tau<T, D, OUT_TWIST>(P, rq, rqd, rqdd, r);
#pragma unroll
  for (int j = 0; j < 6; ++j) tau[j * ld + s] = r.tau[j];
  if constexpr (OUT_TWIST) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Vout[j * ld + s] = r.v[j];
      Vout[(j + 3) * ld + s] = r.w[j];
      dVout[j * ld + s] = r.a[j];
      dVout[(j + 3) * ld + s] = r.l[j];
    }
  }
}

// fp32 variant with two consecutive samples per thread and 8-byte vector accesses: the fp32 kernel is issue-bound, and this
// halves the load / store / address instructions per sample while giving the scheduler two independent chains to interleave.
template <class D, bool OUT_TWIST>
__global__ void __launch_bounds__(kBlock) k_rnea_fast_soa_f32x2(const __grid_constant__ FastParams<float> P, const float* __restrict__ q,
                                                                const float* __restrict__ qd, const float* __restrict__ qdd, float* __restrict__ tau,
                                                                float* __restrict__ Vout, float* __restrict__ dVout, int64_t n, int64_t ld) {
  using Rows = SoaRows<D, OUT_TWIST>;
  pdl_launch_dependents();
  pdl_wait_prior_grids();
  const int64_t s = 2 * ((int64_t)blockIdx.x * kBlock + threadIdx.x);
  if (s >= n) return;
  float a_q[6], a_qd[6], a_qdd[6], b_q[6], b_qd[6], b_qdd[6];
  const bool pair = s + 1 < n;
  const float2 zero = make_float2(0.f, 0.f);
  if (pair) {
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const float2 v0 = Rows::live(0, j) ? __ldg(reinterpret_cast<const float2*>(q + j * ld + s)) : zero;
      const float2 v1 = Rows::live(1, j) ? __ldg(reinterpret_cast<const float2*>(qd + j * ld + s)) : zero;
      const float2 v2 = __ldg(reinterpret_cast<const float2*>(qdd + j * ld + s));
      a_q[j] = v0.x; b_q[j] = v0.y; a_qd[j] = v1.x; b_qd[j] = v1.y; a_qdd[j] = v2.x; b_qdd[j] = v2.y;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      a_q[j] = b_q[j] = Rows::live(0, j) ? __ldg(q + j * ld + s) : 0.f;
      a_qd[j] = b_qd[j] = Rows::live(1, j) ? __ldg(qd + j * ld + s) : 0.f;
      a_qdd[j] = b_qdd[j] = __ldg(qdd + j * ld + s);
    }
  }
  FastResult<float> ra, rb;
  fast_rnea_tau<float, D, OUT_TWIST>(P, a_q, a_qd, a_qdd, ra);
  fast_rnea_tau<float, D, OUT_TWIST>(P, b_q, b_qd, b_qdd, rb);
  if (pair) {
#pragma unroll
    for (int j = 0; j < 6; ++j) *reinterpret_cast<float2*>(tau + j * ld + s) = make_float2(ra.tau[j], rb.tau[j]);
    if constexpr (OUT_TWIST) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        *reinterpret_cast<float2*>(Vout + j * ld + s) = make_float2(ra.v[j], rb.v[j]);
        *reinterpret_cast<float2*>(Vout + (j + 3) * ld + s) = make_float2(ra.w[j], rb.w[j]);
        *reinterpret_cast<float2*>(dVout + j * ld + s) = make_float2(ra.a[j], rb.a[j]);
        *reinterpret_cast<float2*>(dVout + (j + 3) * ld + s) = make_float2(ra.l[j], rb.l[j]);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < 6; ++j) tau[j * ld + s] = ra.tau[j];
    if constexpr (OUT_TWIST) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        Vout[j * ld + s] = ra.v[j];
        Vout[(j + 3) * ld + s] = ra.w[j];
        dVout[j * ld + s] = ra.a[j];
        dVout[(j + 3) * ld + s] = ra.l[j];
      }
    }
  }
}

// Experiment log (round 1, B200): staging the SoA inputs through the TMA unit does NOT pay for this kernel.  fp32, G samples/s
// at 2^20 / 1e7 / 1e8 samples: plain coalesced loads (this kernel) 57.5 / 62.6 / 64.3; 18 one-row bulk copies per 256-sample tile
// 45.4 / 53.0 / 54.2 (the TMA unit is per-copy bound at 1 KB); three 2-D tensor-map copies (box 256 x 6) per tile 51.0 / 61.4 / 63.7;
// the same plus a tensor-map store of tau 51.5 / 59.9 / 62.0.  The AoS kernel below is different: there a tile is ONE contiguous
// span, one bulk load and one bulk store, and TMA wins clearly.

// ---------------------------------------------------------------------------------------------
// generic path, SoA.  Parameters are staged once per block into shared memory.
// ---------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ void stage_params(const T* __restrict__ gp, int count, T* sp) {
  for (int i = threadIdx.x; i < count; i += blockDim.x) sp[i] = gp[i];
  __syncthreads();
}

// NJ > 0: the parameter block is a by-value argument (constant bank), no staging; NJ == 0: run-time joint count, block staged in shared memory
template <class T, int NJ>
__global__ void __launch_bounds__(kBlock) k_rnea_generic_soa(const __grid_constant__ GenericBlock<T, (NJ > 0 ? NJ : 1)> P, const T* __restrict__ gp, int nj,
                                                             int nparams, const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd,
                                                             T* __restrict__ tau, T* __restrict__ Vout, T* __restrict__ dVout, int64_t n, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const T* sp;
  if constexpr (NJ > 0) {
    sp = P.v;
  } else {
    T* staged = reinterpret_cast<T*>(smem_raw);
    stage_params(gp, nparams, staged);
    sp = staged;
  }
  const int64_t s = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (s >= n) return;
  constexpr int MAXJ = NJ > 0 ? NJ : RBM_MAX_JOINTS;
  T rq[MAXJ], rqd[MAXJ], rqdd[MAXJ], rtau[MAXJ];
  const int njr = NJ > 0 ? NJ : nj;
#pragma unroll
  for (int j = 0; j < njr; ++j) {
    rq[j] = __ldg(q + j * ld + s);
    rqd[j] = __ldg(qd + j * ld + s);
    rqdd[j] = __ldg(qdd + j * ld + s);
  }
  T V[6], dV[6];
  generic_rnea<T, NJ>(sp, sp, nj, rq, rqd, rqdd, rtau, nullptr, nullptr, nullptr, V, dV);
#pragma unroll
  for (int j = 0; j < njr; ++j) tau[j * ld + s] = rtau[j];
  if (Vout) {
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      Vout[j * ld + s] = V[j];
      dVout[j * ld + s] = dV[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// AoS kernels: traj [n][3][nj] -> tau [n][nj].  A block's tile of kBlock samples is one contiguous span
// in both arrays; it is moved with coalesced accesses and transposed through shared memory.
// ---------------------------------------------------------------------------------------------
template <class T, class D>
__global__ void __launch_bounds__(kBlock) k_rnea_fast_aos(const __grid_constant__ FastParams<T> P, const T* __restrict__ traj,
                                                          T* __restrict__ tau, int64_t n) {
  __shared__ T tile[kBlock * 18];
  const int64_t s0 = (int64_t)blockIdx.x * kBlock;
  const int cnt = (int)min((int64_t)kBlock, n - s0);
  const T* src = traj + s0 * 18;
  for (int i = threadIdx.x; i < cnt * 18; i += kBlock) tile[i] = __ldg(src + i);
  __syncthreads();
  FastResult<T> r;
  if (threadIdx.x < cnt) {
    const T* my = tile + threadIdx.x * 18;
    T rq[6], rqd[6], rqdd[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) { rq[j] = my[j]; rqd[j] = my[6 + j]; rqdd[j] = my[12 + j]; }
    fast_rnea_tau<T, D, false>(P, rq, rqd, rqdd, r);
  }
  __syncthreads();
  if (threadIdx.x < cnt) {
#pragma unroll
    for (int j = 0; j < 6; ++j) tile[threadIdx.x * 6 + j] = r.tau[j];
  }
  __syncthreads();
  T* dst = tau + s0 * 6;
  for (int i = threadIdx.x; i < cnt * 6; i += kBlock) dst[i] = tile[i];
}

// TMA variant of the AoS kernel (fast paths): a tile of kBlock samples is ONE contiguous span in both arrays (18 KB in, 6 KB out in
// fp64), so each tile is one bulk load and one bulk store.  Persistent CTAs keep kAosStages loads in flight; results are staged
// in a double-buffered shared tile and leave through the async proxy while the next tile is being computed.
constexpr int kAosStages = 3;

template <class T, class D>
__global__ void __launch_bounds__(kBlock) k_rnea_fast_aos_tma(const __grid_constant__ FastParams<T> P, const T* __restrict__ traj, T* __restrict__ tau,
                                                              int64_t n) {
  constexpr int S = kAosStages;
  constexpr uint32_t kInBytes = kBlock * 18 * sizeof(T), kOutBytes = kBlock * 6 * sizeof(T);
  extern __shared__ __align__(128) unsigned char smem_tiles[];
  T* in_buf = reinterpret_cast<T*>(smem_tiles);                      // [S][kBlock * 18]
  T* out_buf = in_buf + (size_t)S * kBlock * 18;                   // [2][kBlock * 6]
  __shared__ __align__(8) uint64_t full[S];
  const int tid = threadIdx.x;
  const int64_t nfull = n / kBlock;  // full tiles go through the TMA pipeline; the ragged tail is handled with plain accesses
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) mbar_init(&full[s], 1);
    mbar_init_fence();
  }
  __syncthreads();
  auto issue = [&](int64_t it) {
    const int64_t tile = (int64_t)blockIdx.x + it * gridDim.x;
    if (tile >= nfull) return;
    const int st = (int)(it % S);
    mbar_arrive_expect_tx(&full[st], kInBytes);
    bulk_copy_g2s(in_buf + (size_t)st * kBlock * 18, traj + tile * (kBlock * 18), kInBytes, &full[st]);
  };
  if (tid == 0) {
    for (int it = 0; it < S; ++it) issue(it);
  }
  for (int64_t it = 0;; ++it) {
    const int64_t tile = (int64_t)blockIdx.x + it * gridDim.x;
    if (tile >= nfull) break;
    const int st = (int)(it % S);
    mbar_wait(&full[st], (uint32_t)((it / S) & 1));
    const T* my = in_buf + (size_t)st * kBlock * 18 + tid * 18;
    T rq[6], rqd[6], rqdd[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) { rq[j] = my[j]; rqd[j] = my[6 + j]; rqdd[j] = my[12 + j]; }
    if (tid == 0) bulk_wait_group_read<1>();  // the store that read out_buf[it & 1] two tiles ago has drained it
    __syncthreads();                          // inputs are in registers everywhere; out_buf[it & 1] is free
    if (tid == 0) issue(it + S);
    FastResult<T> r;
    fast_rnea_tau<T, D, false>(P, rq, rqd, rqdd, r);
    T* out = out_buf + (size_t)(it & 1) * kBlock * 6;
#pragma unroll
    for (int j = 0; j < 6; ++j) out[tid * 6 + j] = r.tau[j];
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      bulk_copy_s2g(tau + tile * (kBlock * 6), out, kOutBytes);
      bulk_commit_group();
    }
  }
  if (tid == 0) bulk_wait_group<0>();  // all stores complete before the CTA (and its shared memory) goes away
  // ragged tail: at most kBlock - 1 samples, owned by the CTA that would have received tile `nfull`
  if ((nfull % gridDim.x) == blockIdx.x) {
    const int64_t s = nfull * kBlock + tid;
    if (s < n) {
      const T* my = traj + s * 18;
      T rq[6], rqd[6], rqdd[6];
#pragma unroll
      for (int j = 0; j < 6; ++j) { rq[j] = __ldg(my + j); rqd[j] = __ldg(my + 6 + j); rqdd[j] = __ldg(my + 12 + j); }
      FastResult<T> r;
      fast_rnea_tau<T, D, false>(P, rq, rqd, rqdd, r);
#pragma unroll
      for (int j = 0; j < 6; ++j) tau[s * 6 + j] = r.tau[j];
    }
  }
}

template <class T>
__global__ void __launch_bounds__(kBlock) k_rnea_generic_aos(const T* __restrict__ gp, int nj, int nparams, const T* __restrict__ traj,
                                                             T* __restrict__ tau, T* __restrict__ poses, T* __restrict__ twists,
                                                             T* __restrict__ dtwists, int64_t n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  stage_params(gp, nparams, sp);
  const int64_t s = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (s >= n) return;
  T rq[RBM_MAX_JOINTS], rqd[RBM_MAX_JOINTS], rqdd[RBM_MAX_JOINTS], rtau[RBM_MAX_JOINTS];
  const T* my = traj + s * 3 * nj;
  for (int j = 0; j < nj; ++j) { rq[j] = my[j]; rqd[j] = my[nj + j]; rqdd[j] = my[2 * nj + j]; }
  generic_rnea<T, 0>(sp, sp, nj, rq, rqd, rqdd, rtau, poses ? poses + s * nj * 12 : nullptr, twists ? twists + s * (nj + 1) * 6 : nullptr,
                     dtwists ? dtwists + s * (nj + 1) * 6 : nullptr, nullptr, nullptr);
  for (int j = 0; j < nj; ++j) tau[s * nj + j] = rtau[j];
}

// ---------------------------------------------------------------------------------------------
// planner-driven kernels: the quintic rest-to-rest trajectory (reference planners/joint_position_planner.py:86-131)
// is evaluated in the kernel from its six coefficients, so a planned batch reads nothing from HBM and writes tau only.
// ---------------------------------------------------------------------------------------------
// The profile is always evaluated in double, also in fp32 mode: in the power basis of the integer step variable
// (k^5 up to ~1e16 against coefficients down to ~1e-16) single precision would lose every digit to cancellation.
// PlanArg / plan_profile live in rbm_rnea.cuh (shared with the closed-loop rollout of rbm_linearize.cu)
template <class T, class D>
__global__ void __launch_bounds__(kBlock) k_rnea_planned_fast(const __grid_constant__ FastParams<T> P, const __grid_constant__ PlanArg<T> pl,
                                                              T* __restrict__ tau, T* __restrict__ traj /* [3*6][ld] or null */, int64_t n, int64_t ld) {
  const int64_t s = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (s >= n) return;
  T sp, sv, sa;
  plan_profile(pl, s, sp, sv, sa);
  T rq[6], rqd[6], rqdd[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    rq[j] = pl.disp[j] * sp + pl.offset[j];
    rqd[j] = pl.disp[j] * sv;
    rqdd[j] = pl.disp[j] * sa;
  }
  FastResult<T> r;
  fast_rnea_tau<T, D, false>(P, rq, rqd, rqdd, r);
#pragma unroll
  for (int j = 0; j < 6; ++j) tau[j * ld + s] = r.tau[j];
  if (traj) {
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      traj[j * ld + s] = rq[j];
      traj[(6 + j) * ld + s] = rqd[j];
      traj[(12 + j) * ld + s] = rqdd[j];
    }
  }
}

template <class T>
__global__ void __launch_bounds__(kBlock) k_rnea_planned_generic(const T* __restrict__ gp, int nj, int nparams, const __grid_constant__ PlanArg<T> pl,
                                                                 T* __restrict__ tau, T* __restrict__ traj, int64_t n, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp_ = reinterpret_cast<T*>(smem_raw);
  stage_params(gp, nparams, sp_);
  const int64_t s = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (s >= n) return;
  T sp, sv, sa;
  plan_profile(pl, s, sp, sv, sa);
  T rq[RBM_MAX_JOINTS], rqd[RBM_MAX_JOINTS], rqdd[RBM_MAX_JOINTS], rtau[RBM_MAX_JOINTS];
  for (int j = 0; j < nj; ++j) {
    rq[j] = pl.disp[j] * sp + pl.offset[j];
    rqd[j] = pl.disp[j] * sv;
    rqdd[j] = pl.disp[j] * sa;
  }
  generic_rnea<T, 0>(sp_, sp_, nj, rq, rqd, rqdd, rtau, nullptr, nullptr, nullptr, nullptr, nullptr);
  for (int j = 0; j < nj; ++j) {
    tau[j * ld + s] = rtau[j];
    if (traj) {
      traj[j * ld + s] = rq[j];
      traj[(nj + j) * ld + s] = rqd[j];
      traj[(2 * nj + j) * ld + s] = rqdd[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static inline unsigned grid_for(int64_t n) { return (unsigned)((n + kBlock - 1) / kBlock); }

template <class T>
int launch_rnea_soa(const rbm_model* m, const T* q, const T* qd, const T* qdd, T* tau, T* V, T* dV, int64_t n, int64_t ld, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  const unsigned grid = grid_for(n);
  const bool tw = (V != nullptr);
  if constexpr (sizeof(T) == 4) {
    // two samples per thread with float2 accesses when every row is 8-byte aligned
    auto al8 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; };
    if (m->path != PATH_GENERIC && (ld % 2) == 0 && al8(q) && al8(qd) && al8(qdd) && al8(tau) && (!tw || (al8(V) && al8(dV)))) {
      const unsigned g2 = grid_for((n + 1) / 2);
      const FastParams<float>& P = ModelView<float>::fast(m);
      if (m->path == PATH_SEQ_ISO) {
        if (tw) RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa_f32x2<SeqIso, true>, g2, kBlock, 0, st, P, q, qd, qdd, tau, V, dV, n, ld));
        else RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa_f32x2<SeqIso, false>, g2, kBlock, 0, st, P, q, qd, qdd, tau, V, dV, n, ld));
      } else {
        if (tw) RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa_f32x2<SeqRigid, true>, g2, kBlock, 0, st, P, q, qd, qdd, tau, V, dV, n, ld));
        else RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa_f32x2<SeqRigid, false>, g2, kBlock, 0, st, P, q, qd, qdd, tau, V, dV, n, ld));
      }
      return RBM_OK;
    }
  }
  if (m->path == PATH_SEQ_ISO) {
    if (tw) RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa<T, SeqIso, true>, grid, kBlock, 0, st, ModelView<T>::fast(m), q, qd, qdd, tau, V, dV, n, ld));
    else RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa<T, SeqIso, false>, grid, kBlock, 0, st, ModelView<T>::fast(m), q, qd, qdd, tau, V, dV, n, ld));
  } else if (m->path == PATH_SEQ_RIGID) {
    if (tw) RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa<T, SeqRigid, true>, grid, kBlock, 0, st, ModelView<T>::fast(m), q, qd, qdd, tau, V, dV, n, ld));
    else RBM_CUDA_TRY(launch_pdl(k_rnea_fast_soa<T, SeqRigid, false>, grid, kBlock, 0, st, ModelView<T>::fast(m), q, qd, qdd, tau, V, dV, n, ld));
  } else {
    const int np = generic_param_count(m->nj);
    const size_t sm = sizeof(T) * np;
    if (m->nj == 6) {
      GenericBlock<T, 6> P;
      std::memcpy(P.v, ModelView<T>::generic_host(m), sizeof(P.v));
      k_rnea_generic_soa<T, 6><<<grid, kBlock, 0, st>>>(P, nullptr, 6, np, q, qd, qdd, tau, V, dV, n, ld);
    } else {
      k_rnea_generic_soa<T, 0><<<grid, kBlock, sm, st>>>(GenericBlock<T, 1>{}, ModelView<T>::generic(m), m->nj, np, q, qd, qdd, tau, V, dV, n, ld);
    }
  }
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_rnea_aos(const rbm_model* m, const T* traj, T* tau, int64_t n, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  const unsigned grid = grid_for(n);
  const bool aligned = ((reinterpret_cast<uintptr_t>(traj) | reinterpret_cast<uintptr_t>(tau)) & 15u) == 0;
  if (m->path != PATH_GENERIC && aligned && !m->no_tma && n >= kBlock) {
    constexpr size_t smem = ((size_t)kAosStages * 18 + 2 * 6) * kBlock * sizeof(T);
    static std::atomic<bool> attr_set[64];  // function attributes are per device; set once per device
    const int dev = (m->device >= 0 && m->device < 64) ? m->device : 0;
    if (!attr_set[dev].load(std::memory_order_acquire)) {
      RBM_CUDA_TRY(cudaFuncSetAttribute(k_rnea_fast_aos_tma<T, SeqIso>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      RBM_CUDA_TRY(cudaFuncSetAttribute(k_rnea_fast_aos_tma<T, SeqRigid>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_set[dev].store(true, std::memory_order_release);
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device);
    const int64_t tiles = n / kBlock;
    const unsigned pgrid = (unsigned)(tiles < (int64_t)sms * 3 ? tiles : (int64_t)sms * 3);  // ~68 KB of stages per CTA: three CTAs per SM
    if (m->path == PATH_SEQ_ISO) k_rnea_fast_aos_tma<T, SeqIso><<<pgrid, kBlock, smem, st>>>(ModelView<T>::fast(m), traj, tau, n);
    else k_rnea_fast_aos_tma<T, SeqRigid><<<pgrid, kBlock, smem, st>>>(ModelView<T>::fast(m), traj, tau, n);
  } else if (m->path == PATH_SEQ_ISO) {
    k_rnea_fast_aos<T, SeqIso><<<grid, kBlock, 0, st>>>(ModelView<T>::fast(m), traj, tau, n);
  } else if (m->path == PATH_SEQ_RIGID) {
    k_rnea_fast_aos<T, SeqRigid><<<grid, kBlock, 0, st>>>(ModelView<T>::fast(m), traj, tau, n);
  } else {
    const int np = generic_param_count(m->nj);
    k_rnea_generic_aos<T><<<grid, kBlock, sizeof(T) * np, st>>>(ModelView<T>::generic(m), m->nj, np, traj, tau, nullptr, nullptr, nullptr, n);
  }
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_rnea_full(const rbm_model* m, const T* traj, T* tau, T* poses, T* twists, T* dtwists, int64_t n, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  const int np = generic_param_count(m->nj);
  k_rnea_generic_aos<T><<<grid_for(n), kBlock, sizeof(T) * np, st>>>(ModelView<T>::generic(m), m->nj, np, traj, tau, poses, twists, dtwists, n);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_rnea_planned(const rbm_model* m, const double* coeffs, const double* disp, const double* offset, double timestep, double step0, double stride,
                        T* tau, T* traj, int64_t n, int64_t ld, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  PlanArg<T> pl;
  for (int k = 0; k < 6; ++k) pl.coeffs[k] = coeffs[k];
  for (int k = 0; k < RBM_MAX_JOINTS; ++k) {
    pl.disp[k] = k < m->nj ? (T)disp[k] : T(0);
    pl.offset[k] = k < m->nj ? (T)offset[k] : T(0);
  }
  pl.inv_dt = 1.0 / timestep;
  pl.inv_dt2 = 1.0 / (timestep * timestep);
  pl.step0 = step0;
  pl.stride = stride;
  const unsigned grid = grid_for(n);
  if (m->path == PATH_SEQ_ISO) {
    k_rnea_planned_fast<T, SeqIso><<<grid, kBlock, 0, st>>>(ModelView<T>::fast(m), pl, tau, traj, n, ld);
  } else if (m->path == PATH_SEQ_RIGID) {
    k_rnea_planned_fast<T, SeqRigid><<<grid, kBlock, 0, st>>>(ModelView<T>::fast(m), pl, tau, traj, n, ld);
  } else {
    const int np = generic_param_count(m->nj);
    k_rnea_planned_generic<T><<<grid, kBlock, sizeof(T) * np, st>>>(ModelView<T>::generic(m), m->nj, np, pl, tau, traj, n, ld);
  }
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template int launch_rnea_planned<double>(const rbm_model*, const double*, const double*, const double*, double, double, double, double*, double*, int64_t,
                                         int64_t, cudaStream_t);
template int launch_rnea_planned<float>(const rbm_model*, const double*, const double*, const double*, double, double, double, float*, float*, int64_t,
                                        int64_t, cudaStream_t);
template int launch_rnea_soa<double>(const rbm_model*, const double*, const double*, const double*, double*, double*, double*, int64_t, int64_t, cudaStream_t);
template int launch_rnea_soa<float>(const rbm_model*, const float*, const float*, const float*, float*, float*, float*, int64_t, int64_t, cudaStream_t);
template int launch_rnea_aos<double>(const rbm_model*, const double*, double*, int64_t, cudaStream_t);
template int launch_rnea_aos<float>(const rbm_model*, const float*, float*, int64_t, cudaStream_t);
template int launch_rnea_full<double>(const rbm_model*, const double*, double*, double*, double*, double*, int64_t, cudaStream_t);

}  // namespace rbm
