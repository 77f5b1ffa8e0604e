// Sensor-frame regressor and its Gram accumulation (inertial-parameter identification).
//
// Replaces, batched and fused:  core/simulate.py:202-209 (twists into the F/T sensor frame),
// dynamics/dynamics.py:215-249 (get_regressor_matrix, 6x10 per sample) and the stacking +
// np.linalg.lstsq of loggers/loggers.py:127-129, which is re-expressed as normal equations: the kernel
// accumulates  [Y f]^T [Y f]  (Y^T Y 10x10, Y^T f 10, f^T f) and never writes Y to HBM.
//
// Gram kernel: persistent grid, one sample per thread per iteration; each thread keeps the 70 distinct
// non-zero entries of the two diagonal blocks in registers, blocks reduce with warp shuffles + shared
// memory, and a second single-block kernel sums the per-block partials in a FIXED order (deterministic
// result for a given grid).  HBM traffic per sample: q, qd, qdd, f = 24 scalars read, nothing written.
#include <atomic>
#include <cstdlib>

#include "rbm_async.cuh"
#include "rbm_internal.h"
#include "rbm_gram.cuh"
#include "rbm_payload.cuh"
#include "rbm_rnea.cuh"

namespace rbm {

constexpr int kRowsBlock = 128;
constexpr int kGramBlock = 256;

// ---- last-link twist for one sample, any kernel path ------------------------------------------------
template <class T, int PATH>
__device__ __forceinline__ void last_link_twists(const FastParams<T>& P, const T* sp, int nj, const T* __restrict__ q, const T* __restrict__ qd,
                                                 const T* __restrict__ qdd, int64_t s, int64_t ld, T* V, T* dV) {
  if constexpr (PATH == PATH_GENERIC) {
    T rq[RBM_MAX_JOINTS], rqd[RBM_MAX_JOINTS], rqdd[RBM_MAX_JOINTS];
    for (int j = 0; j < nj; ++j) { rq[j] = __ldg(q + j * ld + s); rqd[j] = __ldg(qd + j * ld + s); rqdd[j] = __ldg(qdd + j * ld + s); }
    generic_rnea<T, 0>(sp, sp, nj, rq, rqd, rqdd, (T*)nullptr, nullptr, nullptr, nullptr, V, dV);
  } else {
    T rq[6], rqd[6], rqdd[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) { rq[j] = __ldg(q + j * ld + s); rqd[j] = __ldg(qd + j * ld + s); rqdd[j] = __ldg(qdd + j * ld + s); }
    FastResult<T> r;
    if constexpr (PATH == PATH_SEQ_ISO) fast_rnea<T, SeqIso, false>(P, rq, rqd, rqdd, r);
    else fast_rnea<T, SeqRigid, false>(P, rq, rqd, rqdd, r);
#pragma unroll
    for (int k = 0; k < 3; ++k) { V[k] = r.v[k]; V[3 + k] = r.w[k]; dV[k] = r.a[k]; dV[3 + k] = r.l[k]; }
  }
}

template <class T>
__device__ __forceinline__ const T* sensor_R(const FastParams<T>& P, const T* sp, bool generic) { return generic ? sp + GP_SENR : P.senR; }

// ---------------------------------------------------------------------------------------------
// regressor rows from given twists (get_regressor_matrix, dynamics.py:215-249), AoS
// ---------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ void store_rows(const T (&top)[3][4], const T (&bot)[3][9], T* __restrict__ Y) {
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int c = 0; c < 10; ++c) {
      Y[r * 10 + c] = c < 4 ? top[r][c] : T(0);
      Y[(3 + r) * 10 + c] = c == 0 ? T(0) : bot[r][c - 1];
    }
  }
}

template <class T>
__global__ void __launch_bounds__(kRowsBlock) k_regressor_rows(const T* __restrict__ tw, const T* __restrict__ dtw, T* __restrict__ Y, int64_t n) {
  const int64_t s = (int64_t)blockIdx.x * kRowsBlock + threadIdx.x;
  if (s >= n) return;
  T V[6], dV[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) { V[k] = tw[s * 6 + k]; dV[k] = dtw[s * 6 + k]; }
  T top[3][4], bot[3][9];
  regressor_blocks(V, dV, top, bot);
  store_rows(top, bot, Y + s * 60);
}

// sensor-frame twists from last-link twists, AoS (core/simulate.py:202-209)
template <class T>
struct PoseArg { T R[9]; T t[3]; };

template <class T>
__global__ void __launch_bounds__(kRowsBlock) k_sensor_twists(const __grid_constant__ PoseArg<T> pose, const T* __restrict__ tw, const T* __restrict__ dtw,
                                                              T* __restrict__ tws, T* __restrict__ dtws, int64_t n) {
  const int64_t s = (int64_t)blockIdx.x * kRowsBlock + threadIdx.x;
  if (s >= n) return;
  T V[6], dV[6], Vs[6], dVs[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) { V[k] = tw[s * 6 + k]; dV[k] = dtw[s * 6 + k]; }
  sensor_twists(pose.R, pose.t, V, dV, Vs, dVs);
#pragma unroll
  for (int k = 0; k < 6; ++k) { tws[s * 6 + k] = Vs[k]; dtws[s * 6 + k] = dVs[k]; }
}

// ---------------------------------------------------------------------------------------------
// fused: (q, qd, qdd) -> sensor-frame twists -> regressor rows / predicted wrench
// ---------------------------------------------------------------------------------------------
template <class T, int PATH>
__global__ void __launch_bounds__(kRowsBlock) k_regressor_from_traj(const __grid_constant__ FastParams<T> P, const T* __restrict__ gp, int nj, int nparams,
                                                                    const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd,
                                                                    T* __restrict__ Y /* [n][60] or null */, T* __restrict__ Vs_out /* [6][ld] or null */,
                                                                    T* __restrict__ dVs_out, const T* __restrict__ phi /* [10] device or null */,
                                                                    T* __restrict__ F_out /* [6][ld] or null */, int64_t n, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  if constexpr (PATH == PATH_GENERIC) {
    for (int i = threadIdx.x; i < nparams; i += blockDim.x) sp[i] = gp[i];
    __syncthreads();
  }
  const int64_t s = (int64_t)blockIdx.x * kRowsBlock + threadIdx.x;
  if (s >= n) return;
  T V[6], dV[6], Vs[6], dVs[6];
  last_link_twists<T, PATH>(P, sp, nj, q, qd, qdd, s, ld, V, dV);
  const T* R = sensor_R(P, sp, PATH == PATH_GENERIC);
  sensor_twists(R, R + 9, V, dV, Vs, dVs);
  if (Vs_out) {
#pragma unroll
    for (int k = 0; k < 6; ++k) { Vs_out[k * ld + s] = Vs[k]; dVs_out[k * ld + s] = dVs[k]; }
  }
  if (!Y && !F_out) return;
  T top[3][4], bot[3][9];
  regressor_blocks(Vs, dVs, top, bot);
  if (Y) store_rows(top, bot, Y + s * 60);
  if (F_out) {  // F = Y phi : the wrench a body with parameters phi would load the sensor with
    T ph[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) ph[k] = __ldg(phi + k);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      T f = T(0), m = T(0);
#pragma unroll
      for (int c = 0; c < 4; ++c) f += top[r][c] * ph[c];
#pragma unroll
      for (int c = 0; c < 9; ++c) m += bot[r][c] * ph[1 + c];
      F_out[r * ld + s] = f;
      F_out[(3 + r) * ld + s] = m;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Gram accumulation
// ---------------------------------------------------------------------------------------------
// bot_nz, gram_accumulate, gram_pack_entry: rbm_gram.cuh (shared with the host harness)

// fp32 only: warp-reduce the float partial sums and add them to the warp's double accumulators in shared memory
template <int N>
__device__ __forceinline__ void gram_flush_f32(float (&acc)[N], double* red_warp, int lane) {
#pragma unroll
  for (int k = 0; k < N; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == (k & 31)) red_warp[k] += (double)v;
    acc[k] = 0.f;
  }
}

// block epilogue: registers -> per-warp doubles in shared memory -> fixed-order sum over warps -> partials[blockIdx]
template <class T, int N>
__device__ __forceinline__ void gram_block_epilogue(T (&acc)[N], double (*red)[N], double* __restrict__ partials) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if constexpr (sizeof(T) == 4) {
    gram_flush_f32(acc, red[warp], lane);
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) {
      double v = acc[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == (k & 31)) red[warp][k] += v;
    }
  }
  __syncthreads();
  if (threadIdx.x < N) {
    double v = 0.0;
#pragma unroll
    for (int wq = 0; wq < kGramBlock / 32; ++wq) v += red[wq][threadIdx.x];  // fixed order
    partials[(int64_t)blockIdx.x * N + threadIdx.x] = v;
  }
}

constexpr int kFlush = 64;  // fp32: samples accumulated in float registers between flushes into double (rel. error ~64 * 2^-24)

// ---- simple variant: direct global loads (any kernel path, any alignment) ----------------------------------
template <class T, int PATH>
__global__ void __launch_bounds__(kGramBlock, 1) k_regressor_gram(const __grid_constant__ FastParams<T> P, const T* __restrict__ gp, int nj, int nparams,
                                                                  const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd,
                                                                  const T* __restrict__ f, double* __restrict__ partials /* [grid][kAcc] */,
                                                                  int64_t n, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  if constexpr (PATH == PATH_GENERIC) {
    for (int i = threadIdx.x; i < nparams; i += blockDim.x) sp[i] = gp[i];
  }
  __shared__ double red[kGramBlock / 32][kAcc];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = lane; k < kAcc; k += 32) red[warp][k] = 0.0;
  __syncthreads();
  T acc[kAcc];
#pragma unroll
  for (int k = 0; k < kAcc; ++k) acc[k] = T(0);
  const T* R = sensor_R(P, sp, PATH == PATH_GENERIC);
  const int64_t stride = (int64_t)gridDim.x * kGramBlock;
  // every lane of a warp runs the same number of iterations so the periodic warp reduction stays convergent
  const int64_t first = (int64_t)blockIdx.x * kGramBlock + warp * 32;
  int since_flush = 0;
  for (int64_t base = first; base < n; base += stride) {
    const int64_t s = base + lane;
    if (s < n) {
      T V[6], dV[6], Vs[6], dVs[6], fs[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) fs[k] = __ldg(f + k * ld + s);
      last_link_twists<T, PATH>(P, sp, nj, q, qd, qdd, s, ld, V, dV);
      sensor_twists(R, R + 9, V, dV, Vs, dVs);
      T top[3][4], bot[3][9];
      regressor_blocks(Vs, dVs, top, bot);
      gram_accumulate(acc, top, bot, fs);
    }
    if constexpr (sizeof(T) == 4) {
      if (++since_flush == kFlush) {
        since_flush = 0;
        gram_flush_f32(acc, red[warp], lane);
      }
    }
  }
  gram_block_epilogue<T>(acc, red, partials);
}

// ---- pipelined variant (fast paths): TMA bulk copies stage whole 512-sample tiles of the LIVE input streams (21 x 4 KB in fp64) into
// shared memory kPipeStages tiles ahead of the arithmetic, so the loads never wait on registers or occupancy.
// Only live streams are staged: V_6 and dV_6 of the sequential structure do not depend on the three gantry positions
// (SequentialDesc::q_matters), so q[0..2] are never read -- 21 bulk copies per tile instead of 24, 168 instead of 192 B of DRAM traffic per
// fp64 sample (ncu: 2.10 GB instead of 2.40 GB per 12.5 M samples).  The issue cost of a bulk copy is paid by the issuing warp, so the
// 21 copies are spread over the 8 warps with their source pointers formed once.
// What was measured on B200 on the way here (12.5 M samples, G samples/s fp64 / fp32, burst clocks; logs under profiles/):
//   round 1  direct global loads                                      23.6 / 25.0   (41 % of stall samples on the load scoreboard)
//            TMA, one elected thread issues all 24 copies             21.8 / 34.9   (the issuing warp pays ~24 x UBLKCP per tile)
//            same + "last warp to drain refills" instead of a barrier 20.8 / 34.6
//            per-warp pipelines with 256-byte copies                  17.6 / 26.5   (8x more copies: TMA-issue bound)
//            TMA, 24 copies spread over the 8 warps                   29.9 / 47.0   (round-1 production kernel)
//            per-stage empty mbarriers / warp-specialised split / FFMA2 accumulators: all slower (experiments/README.md)
//   round 2  live streams only, 256-sample tiles, 5 stages            31.3 / 47.6   (experiments/k_regressor_gram_tma_1spt.cu.inc)
//            + software-pipelined accumulation (sample i's 180 FMAs issued with sample i + 1's kinematic chain in one basic block)
//                                                                     28.2 / 44.2   (ptxas front-loads the FMAs; +14 % instructions)
//            warp-pair split of the 70 accumulators (12 warps / SM, 162 registers, 17 % more FP64 work)   29.9 / 43.2
//            dedicated TMA producer warpgroup, consumers without a CTA barrier                              30.1 /  --
//            fp32 on the tensor cores (tcgen05 tf32 hi/lo, experiments/k_regressor_gram_tc.cu.inc)           -- / 34.5
//            512-sample tiles, two samples per thread, 2 stages (THIS KERNEL)                              33.6 / 54.9
// ncu of the 256-sample kernel (profiles/r2_gram_v2_ncu_full.csv, r2_gram32_v2_ncu_full.csv): fp64 FP64 pipe 60 % active, issue slots 49 %,
// 19 % of the loop's stall samples in the per-tile hand-over; fp32 issue slots 75 % busy -- which is what the larger tile attacks.
constexpr int kLiveStreams = 21;  // q3..5 (3) | qd (6) | qdd (6) | f (6)
constexpr int kTmaTile = 2 * kGramBlock;  // samples per tile: two per thread
constexpr int kPipeStages = 2;

template <class T>
struct GramCarry {
  T x[3], w[3], l[3], f[6];
};

// accumulation half
template <class T>
__device__ __forceinline__ void gram_accumulate_carry(T (&acc)[kAcc], const GramCarry<T>& z) {
  T top[3][4], bot[3][9];
  regressor_blocks_xwl(z.x, z.w, z.l, top, bot);
  gram_accumulate(acc, top, bot, z.f);
}

// kinematics half: (q, qd, qdd) and the joint sines / cosines -> sensor-frame (x = dv + w x v, w, dw)
template <class T, int PATH, bool SEN_DIAG>
__device__ __forceinline__ void gram_kinematics_cs(const FastParams<T>& P, const T (&rq)[6], const T (&c)[6], const T (&s)[6], const T (&rqd)[6],
                                                   const T (&rqdd)[6], GramCarry<T>& z) {
  FastResult<T> r;
  if constexpr (PATH == PATH_SEQ_ISO) fast_rnea_cs<T, SeqIso, false>(P, rq, c, s, rqd, rqdd, r);
  else fast_rnea_cs<T, SeqRigid, false>(P, rq, c, s, rqd, rqdd, r);
  T V[6], dV[6], Vs[6], dVs[6];
#pragma unroll
  for (int k = 0; k < 3; ++k) { V[k] = r.v[k]; V[3 + k] = r.w[k]; dV[k] = r.a[k]; dV[3 + k] = r.l[k]; }
  if constexpr (SEN_DIAG) {  // Ad(T) is a component-wise sign pattern (the reference's F/T site: Rz(180 deg), no offset)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const T d = P.senR[4 * k];
      Vs[k] = d * V[k]; Vs[3 + k] = d * V[3 + k];
      dVs[k] = d * dV[k]; dVs[3 + k] = d * dV[3 + k];
    }
  } else {
    sensor_twists(P.senR, P.sent, V, dV, Vs, dVs);
  }
  regressor_x(Vs, dVs, z.x);
#pragma unroll
  for (int k = 0; k < 3; ++k) { z.w[k] = Vs[3 + k]; z.l[k] = dVs[3 + k]; }
}

template <class T>
__device__ __forceinline__ const T* live_stream(int k, const T* q, const T* qd, const T* qdd, const T* f, int64_t ld) {
  return k < 3 ? q + (int64_t)(3 + k) * ld : k < 9 ? qd + (int64_t)(k - 3) * ld : k < 15 ? qdd + (int64_t)(k - 9) * ld : f + (int64_t)(k - 15) * ld;
}

// Each thread takes TWO samples of a 512-sample tile (tid and tid + 256) and reads them straight from the stage, which is handed back
// after the arithmetic: the per-tile work every thread repeats (mbarrier wait, CTA barrier, copy issue, loop control: ~100 of the fp32
// kernel's 523 instructions per sample) is paid once per two samples, and there is no copy of the inputs to registers first.  Two
// stages of 21 x 512 values (fp64: 2 x 86 KB, one CTA per SM; fp32: 2 x 43 KB, two CTAs per SM).
template <class T, int PATH, bool SEN_DIAG>
__global__ void __launch_bounds__(kGramBlock, sizeof(T) == 4 ? 2 : 1) k_regressor_gram_tma(const __grid_constant__ FastParams<T> P, const T* __restrict__ q,
                                                                                              const T* __restrict__ qd, const T* __restrict__ qdd,
                                                                                              const T* __restrict__ f, double* __restrict__ partials,
                                                                                              int64_t n, int64_t ld) {
  constexpr int S = kPipeStages;
  constexpr int NW = kGramBlock / 32;
  constexpr uint32_t kRowBytes = kTmaTile * sizeof(T);
  extern __shared__ __align__(128) unsigned char smem_stages[];
  T* buf = reinterpret_cast<T*>(smem_stages);  // [S][kLiveStreams][512]
  __shared__ __align__(8) uint64_t full[S];
  __shared__ double red[NW][kAcc];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t nfull = n / kTmaTile;
  for (int k = lane; k < kAcc; k += 32) red[warp][k] = 0.0;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) mbar_init(&full[s], NW);
    mbar_init_fence();
  }
  __syncthreads();
  const int my_copies = (warp + 2 * NW < kLiveStreams) ? 3 : 2;
  const T* my_src[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) my_src[i] = live_stream(warp + NW * i < kLiveStreams ? warp + NW * i : warp, q, qd, qdd, f, ld);
  auto issue = [&](int64_t it) {
    const int64_t tile = (int64_t)blockIdx.x + it * gridDim.x;
    if (tile >= nfull) return;
    const int st = (int)(it % S);
    uint64_t* bar = &full[st];
    mbar_arrive_expect_tx(bar, my_copies * kRowBytes);
    T* dst = buf + ((size_t)st * kLiveStreams + warp) * kTmaTile;
    const int64_t s0 = tile * kTmaTile;
    bulk_copy_g2s(dst, my_src[0] + s0, kRowBytes, bar);
    bulk_copy_g2s(dst + NW * kTmaTile, my_src[1] + s0, kRowBytes, bar);
    if (my_copies == 3) bulk_copy_g2s(dst + 2 * NW * kTmaTile, my_src[2] + s0, kRowBytes, bar);
  };
  if (lane == 0) {
    for (int it = 0; it < S; ++it) issue(it);
  }
  T acc[kAcc];
#pragma unroll
  for (int k = 0; k < kAcc; ++k) acc[k] = T(0);
  auto sample = [&](const T* src, int stride) {  // one sample whose 21 values sit `stride` apart starting at src
    T rq[6], rqd[6], rqdd[6], c[6], sn[6];
    GramCarry<T> z;
    rq[0] = rq[1] = rq[2] = T(0);
#pragma unroll
    for (int k = 0; k < 3; ++k) rq[3 + k] = src[k * stride];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      rqd[k] = src[(3 + k) * stride];
      rqdd[k] = src[(9 + k) * stride];
      z.f[k] = src[(15 + k) * stride];
    }
    fast_sincos<T, SeqIso>(rq, c, sn);
    gram_kinematics_cs<T, PATH, SEN_DIAG>(P, rq, c, sn, rqd, rqdd, z);
    gram_accumulate_carry(acc, z);
  };
  int since_flush = 0;
  for (int64_t it = 0;; ++it) {
    const int64_t tile = (int64_t)blockIdx.x + it * gridDim.x;
    if (tile >= nfull) break;
    const int st = (int)(it % S);
    mbar_wait(&full[st], (uint32_t)((it / S) & 1));
    const T* src = buf + (size_t)st * kLiveStreams * kTmaTile + tid;
    sample(src, kTmaTile);
    sample(src + kGramBlock, kTmaTile);
    if constexpr (sizeof(T) == 4) {
      since_flush += 2;
      if (since_flush >= kFlush) {
        since_flush = 0;
        gram_flush_f32(acc, red[warp], lane);
      }
    }
    __syncthreads();               // everybody is done with the stage
    if (lane == 0) issue(it + S);  // refill it with the tile two ahead (the other stage is already loading / loaded)
  }
  // ragged tail (n % 512 samples): owned by the CTA that would have received tile `nfull`
  if ((nfull % gridDim.x) == blockIdx.x) {
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      const int64_t s = nfull * kTmaTile + h * kGramBlock + tid;
      if (s < n) {
        T rq[6], rqd[6], rqdd[6], c[6], sn[6];
        GramCarry<T> z;
        rq[0] = rq[1] = rq[2] = T(0);
#pragma unroll
        for (int k = 0; k < 3; ++k) rq[3 + k] = __ldg(q + (3 + k) * ld + s);
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          rqd[k] = __ldg(qd + k * ld + s);
          rqdd[k] = __ldg(qdd + k * ld + s);
          z.f[k] = __ldg(f + k * ld + s);
        }
        fast_sincos<T, SeqIso>(rq, c, sn);
        gram_kinematics_cs<T, PATH, SEN_DIAG>(P, rq, c, sn, rqd, rqdd, z);
        gram_accumulate_carry(acc, z);
      }
    }
  }
  gram_block_epilogue<T>(acc, red, partials);
}

// partials [nblocks][N] -> fixed-order totals -> pack [112] through `entry` (one thread per pack entry, 128 threads)
template <int N, class Entry>
__device__ __forceinline__ void gram_finalize(const double* __restrict__ partials, int nblocks, double n_samples, double* __restrict__ pack, Entry entry) {
  __shared__ double tot[N];
  if (threadIdx.x < N) {
    double v = 0.0;
    for (int b = 0; b < nblocks; ++b) v += partials[(int64_t)b * N + threadIdx.x];  // fixed order
    tot[threadIdx.x] = v;
  }
  __syncthreads();
  const int t = threadIdx.x;
  if (t < 111) pack[t] = entry(tot, t);
  else if (t == 111) pack[t] = n_samples;
}

// partials [nblocks][70] -> pack [112] = [Y^T Y (100, row-major) | Y^T f (10) | f^T f | n]
__global__ void __launch_bounds__(128) k_gram_finalize(const double* __restrict__ partials, int nblocks, double n_samples, double* __restrict__ pack) {
  gram_finalize<kAcc>(partials, nblocks, n_samples, pack, [](const double* tot, int t) { return gram_pack_entry(tot, t); });
}

// ---- grouped variant: one Gram pack per GROUP (environment / object), one group per thread ----------------------------------
// For logs laid out [frame][row][group] (the closed-loop rollout's frame log, rbm_linearize.cu): thread g walks its n_frames samples,
// keeps the 70 accumulators in registers and writes its own 112-double pack, value-major [112][ld_out] (coalesced).
template <class T, int PATH>
__global__ void __launch_bounds__(kRowsBlock) k_regressor_gram_grouped(const __grid_constant__ FastParams<T> P, const T* __restrict__ gp, int nj, int nparams,
                                                                       const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd,
                                                                       const T* __restrict__ f, int64_t frame_stride, int64_t f_frame_stride,
                                                                       int64_t n_frames, double* __restrict__ packs, int64_t n_groups, int64_t ld, int64_t ld_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  if constexpr (PATH == PATH_GENERIC) {
    for (int i = threadIdx.x; i < nparams; i += blockDim.x) sp[i] = gp[i];
    __syncthreads();
  }
  const int64_t g = (int64_t)blockIdx.x * kRowsBlock + threadIdx.x;
  if (g >= n_groups) return;
  const T* R = sensor_R(P, sp, PATH == PATH_GENERIC);
  double acc[kAcc];
#pragma unroll
  for (int k = 0; k < kAcc; ++k) acc[k] = 0.0;
#pragma unroll 1
  for (int64_t fr = 0; fr < n_frames; ++fr) {
    const int64_t off = fr * frame_stride;
    T V[6], dV[6], Vs[6], dVs[6], fs[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) fs[k] = __ldg(f + fr * f_frame_stride + k * ld + g);
    last_link_twists<T, PATH>(P, sp, nj, q + off, qd + off, qdd + off, g, ld, V, dV);
    sensor_twists(R, R + 9, V, dV, Vs, dVs);
    T top[3][4], bot[3][9];
    regressor_blocks(Vs, dVs, top, bot);
    gram_accumulate(acc, top, bot, fs);
  }
  double* out = packs + g;
#pragma unroll
  for (int t = 0; t < 111; ++t) out[(int64_t)t * ld_out] = gram_pack_entry(acc, t);
  out[(int64_t)111 * ld_out] = (double)n_frames;
}

// ---------------------------------------------------------------------------------------------
// joint-torque payload route (rbm_payload.cuh): tau = tau0 + Phi phi, Phi (nj x 10) per sample
// ---------------------------------------------------------------------------------------------
// Fast-path inputs of one sample: q[3..5], qd[3..5], qdd, and (Gram) tau -- q[0..2] and qd[0..2] are never read.
template <class T>
__device__ __forceinline__ void payload_load_fast(const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd, int64_t s, int64_t ld,
                                                  T (&rq)[6], T (&rqd)[6], T (&rqdd)[6]) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    rq[j] = T(0); rqd[j] = T(0);
    rq[3 + j] = __ldg(q + (3 + j) * ld + s); rqd[3 + j] = __ldg(qd + (3 + j) * ld + s);
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) rqdd[j] = __ldg(qdd + j * ld + s);
}

// one sample per thread: Phi [n][nj][10] and / or tau0 [nj][ld] (either may be null)
template <class T, int PATH>
__global__ void __launch_bounds__(kRowsBlock) k_payload_regressor(const __grid_constant__ FastParams<T> P, const T* __restrict__ gp, int nj, int nparams,
                                                                  const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd,
                                                                  T* __restrict__ Phi, T* __restrict__ tau0, int64_t n, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  if constexpr (PATH == PATH_GENERIC) {
    for (int i = threadIdx.x; i < nparams; i += blockDim.x) sp[i] = gp[i];
    __syncthreads();
  }
  const int64_t s = (int64_t)blockIdx.x * kRowsBlock + threadIdx.x;
  if (s >= n) return;
  if constexpr (PATH == PATH_GENERIC) {
    T rq[RBM_MAX_JOINTS], rqd[RBM_MAX_JOINTS], rqdd[RBM_MAX_JOINTS], t0[RBM_MAX_JOINTS];
    for (int j = 0; j < nj; ++j) { rq[j] = __ldg(q + j * ld + s); rqd[j] = __ldg(qd + j * ld + s); rqdd[j] = __ldg(qdd + j * ld + s); }
    payload_generic<T>(sp, nj, rq, rqd, rqdd, t0, [&](int i, const T (&phi)[10]) {
      if (Phi) {
#pragma unroll
        for (int c = 0; c < 10; ++c) Phi[(s * nj + i) * 10 + c] = phi[c];
      }
    });
    if (tau0)
      for (int j = 0; j < nj; ++j) tau0[j * ld + s] = t0[j];
  } else {
    using D = std::conditional_t<PATH == PATH_SEQ_ISO, SeqIso, SeqRigid>;
    T rq[6], rqd[6], rqdd[6], t0[6];
    payload_load_fast(q, qd, qdd, s, ld, rq, rqd, rqdd);
    auto store = [&](int j, const T (&phi)[10]) {
      if (Phi) {
#pragma unroll
        for (int c = 0; c < 10; ++c) Phi[(s * 6 + j) * 10 + c] = phi[c];
      }
    };
    if (P.sen_diag != T(0)) payload_fast<T, D, true>(P, rq, rqd, rqdd, t0, store);
    else payload_fast<T, D, false>(P, rq, rqd, rqdd, t0, store);
    if (tau0) {
#pragma unroll
      for (int j = 0; j < 6; ++j) tau0[j * ld + s] = t0[j];
    }
  }
}

// Normal equations of the payload route: the direct-load persistent form of k_regressor_gram with the 66 accumulators of
// [Phi r]^T [Phi r], r = tau - tau0 (payload_accumulate_row; the fast path's gantry rows add to the 15 entries of columns {0..3, r}).
template <class T, int PATH, bool SEN_DIAG>
__global__ void __launch_bounds__(kGramBlock, 1) k_payload_gram(const __grid_constant__ FastParams<T> P, const T* __restrict__ gp, int nj, int nparams,
                                                                const T* __restrict__ q, const T* __restrict__ qd, const T* __restrict__ qdd,
                                                                const T* __restrict__ tau, double* __restrict__ partials /* [grid][kPayAcc] */,
                                                                int64_t n, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* sp = reinterpret_cast<T*>(smem_raw);
  if constexpr (PATH == PATH_GENERIC) {
    for (int i = threadIdx.x; i < nparams; i += blockDim.x) sp[i] = gp[i];
  }
  __shared__ double red[kGramBlock / 32][kPayAcc];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = lane; k < kPayAcc; k += 32) red[warp][k] = 0.0;
  __syncthreads();
  T acc[kPayAcc];
#pragma unroll
  for (int k = 0; k < kPayAcc; ++k) acc[k] = T(0);
  const int64_t stride = (int64_t)gridDim.x * kGramBlock;
  const int64_t first = (int64_t)blockIdx.x * kGramBlock + warp * 32;  // warp-uniform trip count: the fp32 flush stays convergent
  int since_flush = 0;
  for (int64_t base = first; base < n; base += stride) {
    const int64_t s = base + lane;
    if (s < n) {
      if constexpr (PATH == PATH_GENERIC) {
        T rq[RBM_MAX_JOINTS], rqd[RBM_MAX_JOINTS], rqdd[RBM_MAX_JOINTS], rt[RBM_MAX_JOINTS], t0[RBM_MAX_JOINTS];
        for (int j = 0; j < nj; ++j) {
          rq[j] = __ldg(q + j * ld + s); rqd[j] = __ldg(qd + j * ld + s); rqdd[j] = __ldg(qdd + j * ld + s); rt[j] = __ldg(tau + j * ld + s);
        }
        payload_generic<T>(sp, nj, rq, rqd, rqdd, t0, [&](int i, const T (&phi)[10]) { payload_accumulate_row(acc, phi, rt[i] - t0[i], false); });
      } else {
        using D = std::conditional_t<PATH == PATH_SEQ_ISO, SeqIso, SeqRigid>;
        T rq[6], rqd[6], rqdd[6], rt[6], t0[6];
        payload_load_fast(q, qd, qdd, s, ld, rq, rqd, rqdd);
#pragma unroll
        for (int j = 0; j < 6; ++j) rt[j] = __ldg(tau + j * ld + s);
        payload_fast<T, D, SEN_DIAG>(P, rq, rqd, rqdd, t0,
                                     [&](int j, const T (&phi)[10]) { payload_accumulate_row(acc, phi, rt[j] - t0[j], fast_prismatic<D>(j)); });
      }
    }
    if constexpr (sizeof(T) == 4) {
      if (++since_flush == kFlush) {
        since_flush = 0;
        gram_flush_f32(acc, red[warp], lane);
      }
    }
  }
  gram_block_epilogue<T>(acc, red, partials);
}

// partials [nblocks][66] -> pack [112] = [Phi^T Phi (100, row-major) | Phi^T r (10) | r^T r | n]
__global__ void __launch_bounds__(128) k_payload_finalize(const double* __restrict__ partials, int nblocks, double n_samples, double* __restrict__ pack) {
  gram_finalize<kPayAcc>(partials, nblocks, n_samples, pack, [](const double* tot, int t) { return payload_pack_entry(tot, t); });
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static int sm_count(int device) {
  static int cached[64] = {0};
  if (device >= 0 && device < 64 && cached[device]) return cached[device];
  int v = 148;
  cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device);
  if (device >= 0 && device < 64) cached[device] = v;
  return v;
}

// persistent grid: `per_sm` 256-thread CTAs per SM (fp64: 1, register-limited; fp32: 2)
int gram_grid(const rbm_model* m, int64_t n, int per_sm) {
  int64_t need = (n + kGramBlock - 1) / kGramBlock;
  int64_t cap = (int64_t)sm_count(m->device) * per_sm;
  return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}

template <class T>
int launch_regressor_rows(const T* tw, const T* dtw, T* Y, int64_t n, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  k_regressor_rows<T><<<(unsigned)((n + kRowsBlock - 1) / kRowsBlock), kRowsBlock, 0, st>>>(tw, dtw, Y, n);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_sensor_twists(const double* pose_Rt, const T* tw, const T* dtw, T* tws, T* dtws, int64_t n, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  PoseArg<T> p;
  for (int k = 0; k < 9; ++k) p.R[k] = (T)pose_Rt[k];
  for (int k = 0; k < 3; ++k) p.t[k] = (T)pose_Rt[9 + k];
  k_sensor_twists<T><<<(unsigned)((n + kRowsBlock - 1) / kRowsBlock), kRowsBlock, 0, st>>>(p, tw, dtw, tws, dtws, n);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_regressor_from_traj(const rbm_model* m, const T* q, const T* qd, const T* qdd, T* Y, T* Vs, T* dVs, const T* phi, T* F, int64_t n, int64_t ld,
                               cudaStream_t st) {
  if (n == 0) return RBM_OK;
  const unsigned grid = (unsigned)((n + kRowsBlock - 1) / kRowsBlock);
  const int np = generic_param_count(m->nj);
  const FastParams<T>& P = ModelView<T>::fast(m);
  const T* gp = ModelView<T>::generic(m);
  if (m->path == PATH_SEQ_ISO) k_regressor_from_traj<T, PATH_SEQ_ISO><<<grid, kRowsBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, Y, Vs, dVs, phi, F, n, ld);
  else if (m->path == PATH_SEQ_RIGID) k_regressor_from_traj<T, PATH_SEQ_RIGID><<<grid, kRowsBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, Y, Vs, dVs, phi, F, n, ld);
  else k_regressor_from_traj<T, PATH_GENERIC><<<grid, kRowsBlock, sizeof(T) * np, st>>>(P, gp, m->nj, np, q, qd, qdd, Y, Vs, dVs, phi, F, n, ld);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_regressor_gram_grouped(const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* f, int64_t frame_stride, int64_t f_frame_stride,
                                  int64_t n_frames,
                                  double* packs, int64_t n_groups, int64_t ld, int64_t ld_out, cudaStream_t st) {
  if (n_groups == 0) return RBM_OK;
  const unsigned grid = (unsigned)((n_groups + kRowsBlock - 1) / kRowsBlock);
  const int np = generic_param_count(m->nj);
  const FastParams<T>& P = ModelView<T>::fast(m);
  const T* gp = ModelView<T>::generic(m);
  if (m->path == PATH_SEQ_ISO)
    k_regressor_gram_grouped<T, PATH_SEQ_ISO><<<grid, kRowsBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, f, frame_stride, f_frame_stride, n_frames, packs, n_groups, ld, ld_out);
  else if (m->path == PATH_SEQ_RIGID)
    k_regressor_gram_grouped<T, PATH_SEQ_RIGID><<<grid, kRowsBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, f, frame_stride, f_frame_stride, n_frames, packs, n_groups, ld, ld_out);
  else
    k_regressor_gram_grouped<T, PATH_GENERIC><<<grid, kRowsBlock, sizeof(T) * np, st>>>(P, gp, m->nj, np, q, qd, qdd, f, frame_stride, f_frame_stride, n_frames, packs, n_groups,
                                                                                      ld, ld_out);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}
template int launch_regressor_gram_grouped<double>(const rbm_model*, const double*, const double*, const double*, const double*, int64_t, int64_t, int64_t, double*,
                                                   int64_t, int64_t, int64_t, cudaStream_t);

template <class T>
int launch_regressor_gram(const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* f, double* pack, double* partials, int64_t n, int64_t ld,
                          cudaStream_t st) {
  int grid = gram_grid(m, n, 1);
  const int np = generic_param_count(m->nj);
  const FastParams<T>& P = ModelView<T>::fast(m);
  const T* gp = ModelView<T>::generic(m);
  if (n > 0) {
    // bulk copies need 16-byte aligned rows: base pointers and the row pitch
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const bool tma_ok = m->path != PATH_GENERIC && al16(q) && al16(qd) && al16(qdd) && al16(f) && ((ld * sizeof(T)) % 16 == 0) && n >= kTmaTile &&
                        !m->no_tma;
    const int dev = (m->device >= 0 && m->device < 64) ? m->device : 0;
    const bool diag = P.sen_diag != T(0);
    if (tma_ok) {
      const int64_t tiles = n / kTmaTile;  // the ragged tail rides with the CTA that would have received the next tile
      const int64_t cap = (int64_t)sm_count(m->device) * (sizeof(T) == 4 ? 2 : 1);  // fp64 254 registers: 1 CTA / SM; fp32 128: 2
      grid = (int)(tiles < cap ? tiles : cap);
      constexpr size_t smem = (size_t)kPipeStages * kLiveStreams * kTmaTile * sizeof(T);
      auto kfn = m->path == PATH_SEQ_ISO ? (diag ? k_regressor_gram_tma<T, PATH_SEQ_ISO, true> : k_regressor_gram_tma<T, PATH_SEQ_ISO, false>)
                                         : (diag ? k_regressor_gram_tma<T, PATH_SEQ_RIGID, true> : k_regressor_gram_tma<T, PATH_SEQ_RIGID, false>);
      static std::atomic<const void*> ready[64][4];  // the dynamic shared-memory limit is a per-device function attribute: raised once
      const int slot = (m->path == PATH_SEQ_ISO ? 0 : 2) + (diag ? 0 : 1);
      if (ready[dev][slot].load(std::memory_order_acquire) != (const void*)kfn) {
        RBM_CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ready[dev][slot].store((const void*)kfn, std::memory_order_release);
      }
      kfn<<<grid, kGramBlock, smem, st>>>(P, q, qd, qdd, f, partials, n, ld);
    } else if (m->path == PATH_SEQ_ISO) {
      k_regressor_gram<T, PATH_SEQ_ISO><<<grid, kGramBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, f, partials, n, ld);
    } else if (m->path == PATH_SEQ_RIGID) {
      k_regressor_gram<T, PATH_SEQ_RIGID><<<grid, kGramBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, f, partials, n, ld);
    } else {
      k_regressor_gram<T, PATH_GENERIC><<<grid, kGramBlock, sizeof(T) * np, st>>>(P, gp, m->nj, np, q, qd, qdd, f, partials, n, ld);
    }
    RBM_CUDA_TRY(cudaGetLastError());
  }
  k_gram_finalize<<<1, 128, 0, st>>>(partials, n > 0 ? grid : 0, (double)n, pack);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

template <class T>
int launch_payload_regressor(const rbm_model* m, const T* q, const T* qd, const T* qdd, T* Phi, T* tau0, int64_t n, int64_t ld, cudaStream_t st) {
  if (n == 0) return RBM_OK;
  const unsigned grid = (unsigned)((n + kRowsBlock - 1) / kRowsBlock);
  const int np = generic_param_count(m->nj);
  const FastParams<T>& P = ModelView<T>::fast(m);
  const T* gp = ModelView<T>::generic(m);
  if (m->path == PATH_SEQ_ISO) k_payload_regressor<T, PATH_SEQ_ISO><<<grid, kRowsBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, Phi, tau0, n, ld);
  else if (m->path == PATH_SEQ_RIGID) k_payload_regressor<T, PATH_SEQ_RIGID><<<grid, kRowsBlock, 0, st>>>(P, gp, m->nj, np, q, qd, qdd, Phi, tau0, n, ld);
  else k_payload_regressor<T, PATH_GENERIC><<<grid, kRowsBlock, sizeof(T) * np, st>>>(P, gp, m->nj, np, q, qd, qdd, Phi, tau0, n, ld);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

// one 256-thread CTA per SM (the 66 accumulators and the kinematics do not fit two): partials within rbm_gram_workspace_bytes
template <class T>
int launch_payload_gram(const rbm_model* m, const T* q, const T* qd, const T* qdd, const T* tau, double* pack, double* partials, int64_t n, int64_t ld,
                        cudaStream_t st) {
  const int grid = gram_grid(m, n, 1);
  if (n > 0) {
    const int np = generic_param_count(m->nj);
    const FastParams<T>& P = ModelView<T>::fast(m);
    const T* gp = ModelView<T>::generic(m);
    const bool diag = P.sen_diag != T(0);
#define RBM_PAYLOAD_GRAM(PATH, DIAG, SMEM) k_payload_gram<T, PATH, DIAG><<<grid, kGramBlock, SMEM, st>>>(P, gp, m->nj, np, q, qd, qdd, tau, partials, n, ld)
    if (m->path == PATH_SEQ_ISO) diag ? RBM_PAYLOAD_GRAM(PATH_SEQ_ISO, true, 0) : RBM_PAYLOAD_GRAM(PATH_SEQ_ISO, false, 0);
    else if (m->path == PATH_SEQ_RIGID) diag ? RBM_PAYLOAD_GRAM(PATH_SEQ_RIGID, true, 0) : RBM_PAYLOAD_GRAM(PATH_SEQ_RIGID, false, 0);
    else RBM_PAYLOAD_GRAM(PATH_GENERIC, false, sizeof(T) * np);
#undef RBM_PAYLOAD_GRAM
    RBM_CUDA_TRY(cudaGetLastError());
  }
  k_payload_finalize<<<1, 128, 0, st>>>(partials, n > 0 ? grid : 0, (double)n, pack);
  RBM_CUDA_TRY(cudaGetLastError());
  return RBM_OK;
}

#define RBM_INST(T)                                                                                                                        \
  template int launch_regressor_rows<T>(const T*, const T*, T*, int64_t, cudaStream_t);                                                    \
  template int launch_sensor_twists<T>(const double*, const T*, const T*, T*, T*, int64_t, cudaStream_t);                                  \
  template int launch_regressor_from_traj<T>(const rbm_model*, const T*, const T*, const T*, T*, T*, T*, const T*, T*, int64_t, int64_t, cudaStream_t); \
  template int launch_regressor_gram<T>(const rbm_model*, const T*, const T*, const T*, const T*, double*, double*, int64_t, int64_t, cudaStream_t); \
  template int launch_payload_regressor<T>(const rbm_model*, const T*, const T*, const T*, T*, T*, int64_t, int64_t, cudaStream_t);                  \
  template int launch_payload_gram<T>(const rbm_model*, const T*, const T*, const T*, const T*, double*, double*, int64_t, int64_t, cudaStream_t);
RBM_INST(double)
RBM_INST(float)

}  // namespace rbm
