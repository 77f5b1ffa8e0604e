// Gram accumulation shared by the Gram kernels of rbm_regressor.cu and the host harness (__host__ __device__).
#pragma once
#include "rbm_typed.cuh"

namespace rbm {

constexpr int kTop = 15;             // 5x5 symmetric: [x | X | f_force]
constexpr int kBot = 55;             // 10x10 symmetric: [-[x]x | Yb | f_torque]
constexpr int kAcc = kTop + kBot;    // 70

// structural zeros of the bottom block: -[x]x has a zero diagonal (rows 0..2 x cols 0..2)
__host__ __device__ constexpr bool bot_nz(int r, int c) { return !(c < 3 && c == r); }

// acc layout: [0,15) upper triangle of U^T U (5x5, row-major i<=j), [15,70) upper triangle of W^T W (10x10)
template <class TA, class T>
RBM_HD void gram_accumulate(TA (&acc)[kAcc], const T (&top)[3][4], const T (&bot)[3][9], const T (&f)[6]) {
  // U = [top | f_force] (3x5), W = [bot | f_torque] (3x10)
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    TA u[5], w[10];
#pragma unroll
    for (int c = 0; c < 4; ++c) u[c] = (TA)top[r][c];
    u[4] = (TA)f[r];
#pragma unroll
    for (int c = 0; c < 9; ++c) w[c] = (TA)bot[r][c];
    w[9] = (TA)f[3 + r];
    int k = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = i; j < 5; ++j) { acc[k] += u[i] * u[j]; ++k; }
#pragma unroll
    for (int i = 0; i < 10; ++i)
#pragma unroll
      for (int j = i; j < 10; ++j) {
        if (bot_nz(r, i) && bot_nz(r, j)) acc[k] += w[i] * w[j];
        ++k;
      }
  }
}

// Entry t (0..110) of the pack [Y^T Y (100, row-major) | Y^T f (10) | f^T f] from the 70 block accumulators: column 0 of Y lives
// only in the top block, columns 4..9 only in the bottom block, columns 1..3 in both.
template <class TA>
RBM_HD double gram_pack_entry(const TA* tot, int t) {
  auto tri = [](int n_, int i, int j) { if (i > j) { int k = i; i = j; j = k; } return i * n_ - i * (i - 1) / 2 + (j - i); };
  double v = 0.0;
  if (t < 100) {
    const int a = t / 10, b = t % 10;
    if (a <= 3 && b <= 3) v += (double)tot[tri(5, a, b)];
    if (a >= 1 && b >= 1) v += (double)tot[kTop + tri(10, a - 1, b - 1)];
  } else if (t < 110) {
    const int a = t - 100;
    if (a <= 3) v += (double)tot[tri(5, a, 4)];
    if (a >= 1) v += (double)tot[kTop + tri(10, a - 1, 9)];
  } else {
    v = (double)tot[tri(5, 4, 4)] + (double)tot[kTop + tri(10, 9, 9)];
  }
  return v;
}

// ---- joint-torque payload route (rbm_payload.cuh): [Phi r]^T [Phi r], Phi (nj x 10) and r = tau - tau0 per sample ----------------
constexpr int kPayAcc = 66;  // upper triangle of the 11 x 11 product, row-major i <= j

__host__ __device__ constexpr int tri11(int i, int j) { return i <= j ? i * 11 - i * (i - 1) / 2 + (j - i) : j * 11 - j * (j - 1) / 2 + (i - j); }

// One row [Phi_j | r_j].  A prismatic joint's row is zero in columns 4..9 and touches only the 15 entries among columns {0..3, r}.
template <class TA, class T>
RBM_HD void payload_accumulate_row(TA (&acc)[kPayAcc], const T (&phi)[10], T r, bool prismatic) {
  TA u[11];
#pragma unroll
  for (int c = 0; c < 10; ++c) u[c] = (TA)phi[c];
  u[10] = (TA)r;
#pragma unroll
  for (int i = 0; i < 11; ++i)
#pragma unroll
    for (int j = i; j < 11; ++j)
      if (!prismatic || ((i < 4 || i == 10) && (j < 4 || j == 10))) acc[tri11(i, j)] += u[i] * u[j];
}

// Entry t (0..110) of the pack [Phi^T Phi (100, row-major) | Phi^T r (10) | r^T r] from the 66 accumulators
template <class TA>
RBM_HD double payload_pack_entry(const TA* tot, int t) {
  if (t < 100) return (double)tot[tri11(t / 10, t % 10)];
  if (t < 110) return (double)tot[tri11(t - 100, 10)];
  return (double)tot[tri11(10, 10)];
}

}  // namespace rbm
