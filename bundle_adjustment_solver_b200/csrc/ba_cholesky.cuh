// ba_cholesky.cuh -- K5: dense FP64 Cholesky solve of the reduced camera system
// (replaces `Am_BCinvBt_mat.ldlt().solve(am_BCinv_b_mat)`, full...cpp:890-908).
//
// Storage: one buffer Saug of (n+1) x (n+1) doubles, leading dimension ld = n+1, viewed
// column-major with the LOWER triangle holding S (equivalently row-major upper, which is how the
// Schur kernel addresses it) and row n (elements c*ld + n) holding rhs^T.  Factorising the leading
// n x n block with the panel TRSM applied to every row below the diagonal block -- including row
// n -- turns that row into z^T = (L^-1 rhs)^T, so the forward substitution is free.  The backward
// substitution L^T x = z runs as a right-looking blocked sweep.
//
// v2: blocked right-looking, NB = 64, three kernels per panel: diagonal-block Cholesky + explicit
// triangular inverse in one CTA, panel TRSM as a tiled GEMM with that inverse, shared-memory tiled
// SYRK/GEMM trailing update on CUDA-core FP64.  The backward sweep reuses the block inverses.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "ba_cholesky_banded.cuh"
#include "ba_cholesky_cluster.cuh"
#include "ba_cholesky_nd.cuh"
#include "ba_device.cuh"

namespace ba {

constexpr int kNB = 64;
constexpr int kGroup = 4;   // panels per group of the two-level trailing update
constexpr size_t kCholDiagSmem = (3 * kNB * (kNB + 1) + 3 * kNB + 2) * sizeof(double);

// ---- diagonal block: Cholesky of an nb x nb block + its triangular inverse, one CTA of 1024 --------
// The 2080 lower-triangle entries live in registers (<= 3 per thread) for the whole elimination;
// only the current column travels through a double-buffered shared-memory vector, so each of the 64
// column steps costs one barrier:  a_rc -= a_rj a_cj / d_j  (columns stay unscaled until the end,
// then L = A D^-1/2).  L^-1 is then built by recursive doubling (X21 = -X22 L21 X11, block sizes
// 1,2,..,32: 12 barriers instead of 64 substitution steps).  Linv (row-major 64x64, lower) lets the
// panel TRSM and the backward substitution run as small GEMMs / GEMVs.
// reciprocal off the slow IEEE division path (it sits on the chain of all 64 column steps): hardware approximation
// + two Newton steps, full double precision up to the last bit
__device__ __forceinline__ double diag_rcp(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  double e = fma(-d, x, 1.0);
  x = fma(x, e, x);
  e = fma(-d, x, 1.0);
  x = fma(x, e, x);
  return x;
}

#ifndef BA_DIAG_THREADS
#define BA_DIAG_THREADS 1024
#endif
constexpr int kDiagThreads = BA_DIAG_THREADS;            // a barrier per column step: fewer threads, cheaper barrier
constexpr int kDiagNQ = (kNB * (kNB + 1) / 2 + kDiagThreads - 1) / kDiagThreads;   // lower-triangle entries per thread
__global__ void __launch_bounds__(kDiagThreads) k_chol_diag(double *__restrict__ A, int ld, int k0, int nb,
                                                    double *__restrict__ Linv_out, const LmState *st) {
  if (st->done) return;
  extern __shared__ double chol_smem[];  // kCholDiagSmem bytes (opt-in > 48 KB)
  double (*L)[kNB + 1] = reinterpret_cast<double (*)[kNB + 1]>(chol_smem);
  double (*X)[kNB + 1] = reinterpret_cast<double (*)[kNB + 1]>(chol_smem + kNB * (kNB + 1));
  double (*T)[kNB + 1] = reinterpret_cast<double (*)[kNB + 1]>(chol_smem + 2 * kNB * (kNB + 1));
  double *colbuf = chol_smem + 3 * kNB * (kNB + 1);  // [2][kNB + 1]: column j and 1/d_j
  double *dinv = colbuf + 2 * (kNB + 1);             // 1/sqrt(d)
  const int t = threadIdx.x;
  constexpr int NE = kNB * (kNB + 1) / 2;  // 2080
  int er[kDiagNQ], ec[kDiagNQ];
  double v[kDiagNQ];
#pragma unroll
  for (int q = 0; q < kDiagNQ; ++q) {
    const int e = t + kDiagThreads * q;
    int r = -1, c = -1;
    double val = 0.0;
    if (e < NE) {
      r = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
      while (r * (r + 1) / 2 > e) --r;
      while ((r + 1) * (r + 2) / 2 <= e) ++r;
      c = e - r * (r + 1) / 2;
      val = (r == c) ? 1.0 : 0.0;  // identity padding
      if (r < nb && c < nb) val = A[(size_t)(k0 + c) * ld + k0 + r];
    }
    er[q] = r; ec[q] = c; v[q] = val;
  }
  for (int j = 0; j < kNB; ++j) {
    double *cb = colbuf + (j & 1) * (kNB + 1);
#pragma unroll
    for (int q = 0; q < kDiagNQ; ++q)
      if (ec[q] == j) {
        cb[er[q]] = v[q];
        // the owner of the pivot alone pays for the FP64 reciprocal (32 warps doing it redundantly
        // made this kernel issue-bound).  Non-positive pivot (e.g. a pose without observations):
        // emulate LDLT's D^+ = 0.
        if (er[q] == j) cb[kNB] = (v[q] > 0.0) ? diag_rcp(v[q]) : 0.0;
      }
    __syncthreads();
    const double di = cb[kNB];
#pragma unroll
    for (int q = 0; q < kDiagNQ; ++q)
      if (ec[q] > j) v[q] -= cb[er[q]] * di * cb[ec[q]];
  }
#pragma unroll
  for (int q = 0; q < kDiagNQ; ++q)
    if (er[q] >= 0 && er[q] == ec[q]) dinv[er[q]] = (v[q] > 0.0) ? 1.0 / sqrt(v[q]) : 0.0;
  __syncthreads();
  const double kInf = __longlong_as_double(0x7ff0000000000000LL);
#pragma unroll
  for (int q = 0; q < kDiagNQ; ++q) {
    const int r = er[q], c = ec[q];
    if (r < 0) continue;
    const double l = (r == c) ? ((dinv[r] > 0.0) ? 1.0 / dinv[r] : kInf) : v[q] * dinv[c];
    L[r][c] = l;
    X[r][c] = (r == c) ? dinv[r] : 0.0;
    if (r < nb && c < nb) A[(size_t)(k0 + c) * ld + k0 + r] = l;
  }
  __syncthreads();
  // recursive doubling: block b of size 2m: rows R = b*2m+m.., cols C = b*2m..
  for (int m = 1; m < kNB; m <<= 1) {
    const int per_level = (kNB / (2 * m)) * m * m;  // outputs of this level (<= 1024)
    for (int tt = t; tt < per_level; tt += kDiagThreads) {
      const int bi = tt / (m * m), i = (tt / m) % m, k = tt % m;
      const int R0 = bi * 2 * m + m, C0 = bi * 2 * m;
      // T[i][k] = sum_q L[R0+i][C0+q] X[C0+q][C0+k], q >= k (X11 lower)
      double acc = 0.0;
      for (int q = k; q < m; ++q) acc += L[R0 + i][C0 + q] * X[C0 + q][C0 + k];
      T[R0 + i][C0 + k] = acc;
    }
    __syncthreads();
    for (int tt = t; tt < per_level; tt += kDiagThreads) {
      const int bi = tt / (m * m), i = (tt / m) % m, k = tt % m;
      const int R0 = bi * 2 * m + m, C0 = bi * 2 * m;
      // X21[i][k] = - sum_q X[R0+i][R0+q] T[q][k], q <= i (X22 lower)
      double acc = 0.0;
      for (int q = 0; q <= i; ++q) acc += X[R0 + i][R0 + q] * T[R0 + q][C0 + k];
      X[R0 + i][C0 + k] = -acc;
    }
    __syncthreads();
  }
  for (int e = t; e < kNB * kNB; e += kDiagThreads) {
    const int r = e / kNB, c = e % kNB;
    Linv_out[e] = (r >= c) ? X[r][c] : 0.0;
  }
}

// ---- FP64 tensor-core tile product (DMMA, mma.sync.m8n8k4.f64; measured 37.1 TFLOP/s on B200 against 34.2 for
// DFMA, at 1/8 of the issue slots and 1/5 of the shared-memory reads of a 4x4 register tile) ---------------
// C(64 x 64) += X^T Y for operands staged in shared memory as X[m][row], Y[m][col] (row stride kLdT = 68:
// stride = 4 mod 16 makes the 8 x 4 fragment reads conflict-free).  8 warps; warp w owns rows 16 (w % 4) + [0,16)
// and columns 32 (w / 4) + [0,32): 2 x 4 DMMA tiles, accumulators acc[i][j][2] in the m8n8 C layout
// (lane l: row l / 4, columns 2 (l % 4) + {0, 1}).
constexpr int kLdT = 68;
constexpr int kKH = 32;   // K staged per pass
__device__ __forceinline__ void dmma_884(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}
__device__ __forceinline__ void tile_mac_dmma(const double (*X)[kLdT], const double (*Y)[kLdT], double (&acc)[2][4][2]) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int rbase = 16 * (w & 3) + (lane >> 2), cbase = 32 * (w >> 2) + (lane >> 2), kq = lane & 3;
#pragma unroll
  for (int m0 = 0; m0 < kKH; m0 += 4) {
    double a[2], b[4];
#pragma unroll
    for (int i = 0; i < 2; ++i) a[i] = X[m0 + kq][rbase + 8 * i];
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = Y[m0 + kq][cbase + 8 * j];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma_884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
  }
}

// ---- panel: rows below the diagonal block: A[r, k0:k0+nb] <- A[r, k0:k0+nb] Linv^T (64-row tiles, DMMA)
__global__ void __launch_bounds__(256) k_chol_trsm(double *__restrict__ A, int ld, int n_rows, int k0, int nb,
                                                   const double *__restrict__ Linv,
                                                   const int *__restrict__ row_tiles, const LmState *st) {
  if (st->done) return;
  __shared__ double At[kKH][kLdT];   // [m][row]   panel entries A[row][k0+m]
  __shared__ double Lt[kKH][kLdT];   // [m][col]   Linv[col][m]
  const int r0 = row_tiles[blockIdx.x] * 64;  // tile rows inside the envelope of this panel
  double acc[2][4][2] = {};
  for (int mh = 0; mh < kNB; mh += kKH) {
    __syncthreads();
    for (int e = threadIdx.x; e < kKH * 64; e += 256) {
      const int i = e % 64, m = mh + e / 64;
      const int rr = r0 + i;
      At[e / 64][i] = (m < nb && rr < n_rows) ? A[(size_t)(k0 + m) * ld + rr] : 0.0;
    }
    for (int e = threadIdx.x; e < kKH * 64; e += 256) {
      const int m = mh + e % kKH, c = e / kKH;
      Lt[e % kKH][c] = Linv[c * kNB + m];  // X[c][m], zero for m > c
    }
    __syncthreads();
    tile_mac_dmma(At, Lt, acc);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int rr = r0 + 16 * (w & 3) + 8 * i + (lane >> 2);
        const int c = 32 * (w >> 2) + 8 * j + 2 * (lane & 3) + e;
        if (rr < n_rows && c < nb) A[(size_t)(k0 + c) * ld + rr] = acc[i][j][e];
      }
}

// ---- rhs row when it shares the (partial) last diagonal tile: z_k = rhs_k L_kk^-T for that tile ---
__global__ void __launch_bounds__(64) k_chol_trsm_tail(double *__restrict__ A, int ld, int n_rows, int k0, int nb,
                                                       const double *__restrict__ Linv, const LmState *st) {
  if (st->done) return;
  __shared__ double a[kNB];
  const int c = threadIdx.x, r = n_rows - 1;
  a[c] = (c < nb) ? A[(size_t)(k0 + c) * ld + r] : 0.0;
  __syncthreads();
  double acc = 0.0;
  for (int m = 0; m <= c; ++m) acc += a[m] * Linv[c * kNB + m];
  if (c < nb) A[(size_t)(k0 + c) * ld + r] = acc;
}

// ---- trailing update: A[r, c] -= sum_m P[r, m] P[c, m], r >= c, both in (k0+nb, n_rows) ------
// 64 x 64 output tile per CTA, 8 warps of DMMA (2 x 4 m8n8k4 tiles per warp), K = nb <= 64 staged in halves.
// n_cols == 0: blockIdx.x enumerates the pairs (ia >= ib) of row_tiles (triangular); n_cols > 0: rectangular,
// rows x the first n_cols entries of the same list (two-level blocking: the columns inside a panel group).
// K = nb may span several panels (k0 = first column of the group).
__global__ void __launch_bounds__(256) k_syrk_update(double *__restrict__ A, int ld, int n_rows, int k0,
                                                     int nb, const int *__restrict__ row_tiles, int n_cols,
                                                     const LmState *st) {
  if (st->done) return;
  int ia, ib;
  if (n_cols > 0) {
    ia = blockIdx.x / n_cols;
    ib = blockIdx.x - ia * n_cols;
    if (ia < ib) return;
  } else {
    ia = (int)((sqrt(8.0 * blockIdx.x + 1.0) - 1.0) * 0.5);
    while (ia * (ia + 1) / 2 > (int)blockIdx.x) --ia;
    while ((ia + 1) * (ia + 2) / 2 <= (int)blockIdx.x) ++ia;
    ib = blockIdx.x - ia * (ia + 1) / 2;
  }
  const int tr = row_tiles[ia], tc = row_tiles[ib];
  __shared__ double Pr[kKH][kLdT];     // [m][row]
  __shared__ double Pc[kKH][kLdT];     // [m][col]
  const int r0 = tr * 64, c0 = tc * 64;
  double acc[2][4][2] = {};
  for (int mh = 0; mh < nb; mh += kKH) {
    __syncthreads();
    for (int e = threadIdx.x; e < kKH * 64; e += 256) {
      const int i = e % 64, m = mh + e / 64;
      const int rr = r0 + i, cc = c0 + i;
      Pr[e / 64][i] = (m < nb && rr < n_rows) ? A[(size_t)(k0 + m) * ld + rr] : 0.0;
      Pc[e / 64][i] = (m < nb && cc < n_rows) ? A[(size_t)(k0 + m) * ld + cc] : 0.0;
    }
    __syncthreads();
    tile_mac_dmma(Pr, Pc, acc);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int rr = r0 + 16 * (w & 3) + 8 * i + (lane >> 2);
        const int cc = c0 + 32 * (w >> 2) + 8 * j + 2 * (lane & 3) + e;
        if (rr < n_rows && cc < n_rows - 1 && rr >= cc) A[(size_t)cc * ld + rr] -= acc[i][j][e];
      }
}

// ---- backward substitution L^T x = z, z = row n of the factor; single CTA, 1024 threads ---------
// Right-looking over 64-blocks from the bottom: x_k = Linv_k^T z_k, then z[0:k0] -= L[k0:k0+nb,0:k0]^T x_k.
__global__ void __launch_bounds__(1024) k_backward_solve(const double *__restrict__ A, int ld, int n,
                                                         const double *__restrict__ Linv_all,
                                                         const int *__restrict__ first_tile,
                                                         double *__restrict__ x_out, double *__restrict__ zbuf,
                                                         const LmState *st) {
  if (st->done) return;
  __shared__ double xk[kNB];
  __shared__ double zk[kNB];
  const int t = threadIdx.x;
  for (int i = t; i < n; i += blockDim.x) zbuf[i] = A[(size_t)i * ld + n];
  __syncthreads();
  const int nblk = (n + kNB - 1) / kNB;
  const int warp = t >> 5, lane = t & 31, nwarps = blockDim.x >> 5;
  for (int kb = nblk - 1; kb >= 0; --kb) {
    const int k0 = kb * kNB, nb = min(kNB, n - k0);
    const double *Xi = Linv_all + (size_t)kb * kNB * kNB;  // row-major X = L_kk^-1 (lower)
    if (t < kNB) zk[t] = (t < nb) ? zbuf[k0 + t] : 0.0;
    __syncthreads();
    // x_k[c] = sum_{r>=c} X[r][c] z_k[r]   (X^T z) ; warps over c, lanes over r
    for (int c = warp; c < kNB; c += nwarps) {
      double acc = 0.0;
      for (int r = c + lane; r < kNB; r += 32) acc += Xi[r * kNB + c] * zk[r];
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
      if (lane == 0) xk[c] = acc;
    }
    __syncthreads();
    if (t < nb) x_out[k0 + t] = xk[t];
    // z[c] -= sum_r L[k0+r, c] * x_k[r], c < k0 ; a warp takes 4 columns per trip (8 independent loads
    // per lane in flight), lanes over the 64 contiguous rows
    const double xa = xk[lane], xb = xk[lane + 32];
    const int cbeg = first_tile[kb] * kNB;  // columns left of the envelope hold zeros
    for (int c = cbeg + warp * 4; c < k0; c += nwarps * 4) {
      double acc[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int cc = c + u;
        double a0 = 0.0, a1 = 0.0;
        if (cc < k0) {
          const double *col = A + (size_t)cc * ld + k0;
          a0 = (lane < nb) ? col[lane] : 0.0;
          a1 = (lane + 32 < nb) ? col[lane + 32] : 0.0;
        }
        acc[u] = a0 * xa + a1 * xb;
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1)
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[u] += __shfl_down_sync(0xffffffffu, acc[u], d);
      if (lane == 0)
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (c + u < k0) zbuf[c + u] -= acc[u];
    }
    __syncthreads();
  }
}

// ---- backward substitution for LARGE systems: one launch per 64-block from the bottom, many CTAs ---------
// Every CTA recomputes x_k = Linv_k^T z_k (64 x 64 mat-vec, L2-resident operands) and then applies its share of
// z[c] -= sum_r L[k0 + r][c] x_k[r] for the columns c < k0 inside the envelope (a warp takes 4 columns per trip,
// lanes over the 64 contiguous rows of a column).  CTA 0 stores x_k.  z lives in zbuf (initialised from row n
// of the factor by k_backward_init).
constexpr int kBwdColsPerCta = 64;
__global__ void __launch_bounds__(256) k_backward_init(const double *__restrict__ A, int ld, int n,
                                                       double *__restrict__ zbuf, const LmState *st) {
  if (st->done) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) zbuf[i] = A[(size_t)i * ld + n];
}
__global__ void __launch_bounds__(256) k_backward_block(const double *__restrict__ A, int ld, int n, int kb,
                                                        const double *__restrict__ Linv_all, int cbeg,
                                                        double *__restrict__ x_out, double *zbuf,
                                                        const LmState *st) {
  if (st->done) return;
  __shared__ double zk[kNB];
  __shared__ double xk[kNB];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int k0 = kb * kNB, nb = min(kNB, n - k0);
  const double *Xi = Linv_all + (size_t)kb * kNB * kNB;  // row-major X = L_kk^-1 (lower)
  if (t < kNB) zk[t] = (t < nb) ? zbuf[k0 + t] : 0.0;
  __syncthreads();
  // x_k[c] = sum_{r >= c} X[r][c] z_k[r]; 8 warps x 8 columns, lanes over r
  for (int c = warp; c < kNB; c += 8) {
    double acc = 0.0;
    for (int r = c + lane; r < kNB; r += 32) acc += Xi[r * kNB + c] * zk[r];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
    if (lane == 0) xk[c] = acc;
  }
  __syncthreads();
  if (blockIdx.x == 0 && t < nb) x_out[k0 + t] = xk[t];
  const double xa = xk[lane], xb = xk[lane + 32];
  const int c_lo = cbeg + blockIdx.x * kBwdColsPerCta;
  const int c_hi = min(k0, c_lo + kBwdColsPerCta);
  for (int c = c_lo + warp * 4; c < c_hi; c += 8 * 4) {
    double acc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int cc = c + u;
      double a0 = 0.0, a1 = 0.0;
      if (cc < c_hi) {
        const double *col = A + (size_t)cc * ld + k0;
        a0 = (lane < nb) ? col[lane] : 0.0;
        a1 = (lane + 32 < nb) ? col[lane + 32] : 0.0;
      }
      acc[u] = a0 * xa + a1 * xb;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1)
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] += __shfl_down_sync(0xffffffffu, acc[u], d);
    if (lane == 0)
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (c + u < c_hi) zbuf[c + u] -= acc[u];
  }
}

// The reduced solve a plan runs.  Each path falls back to the next one when its launch fails (a partitioned solve
// whose cooperative launch is refused runs its per-level launches instead).
enum class SolvePath {
  NdPersistent,   // partitioned banded, one persistent launch (ba_cholesky_nd.cuh)
  NdLevels,       // partitioned banded, one launch per tree level
  Banded,         // serial window kernel (ba_cholesky_banded.cuh)
  Cluster,        // blocked Cholesky in one thread-block-cluster launch (ba_cholesky_cluster.cuh)
  Dense,          // blocked multi-kernel Cholesky (below)
};

// Tile-level row envelope (skyline) of S: Cholesky creates no fill left of a row's first non-zero, so
// tiles (r, c) with c < first_tile[r] stay zero and are skipped by TRSM / SYRK / the backward sweep.
// For a dense S (every pose co-visible with every other) first_tile is all zeros and nothing is skipped.
struct CholeskyPlan {
  int n = 0, T = 0;                 // matrix order, tile rows over n+1 rows (the last holds the rhs row)
  std::vector<int> first_tile;      // [T]
  std::vector<int> rows_ptr, rows;  // per panel k: tile rows r > k with first_tile[r] <= k
  int *d_first_tile = nullptr, *d_rows = nullptr, *d_rows_ptr = nullptr;
  double dense_fraction = 1.0;
  int max_rows = 0;       // largest number of envelope row tiles under any panel
  int cluster_size = 0;   // > 0: run the single-launch cluster kernel (small / narrow-envelope systems)
  // two-level blocking (large systems): panels are grouped by kGroup; inside a group the trailing update only
  // touches the group's own column tiles (narrow_cnt[k] = leading entries of panel k's row list that lie inside
  // the group); after the group one rank-(64 kGroup) update covers the rest (grp_off/grp_cnt index `rows`)
  std::vector<int> narrow_cnt, grp_off, grp_cnt;
  bool two_level = false;
  int bw = 0;             // scalar half-bandwidth of S: 6 (largest pose distance inside a track) + 5
  bool banded = false;    // banded reduced system: serial window kernel (ba_cholesky_banded.cuh) or the partition below
  NdPlan nd;              // partitioned banded solve (ba_cholesky_nd.cuh); nd.valid: preferred over the serial kernel
  NdDevice nd_dev;
  SolvePath path = SolvePath::Dense;   // chosen once the partition's device resources are known
};

// chol_mode: -1 auto (banded > cluster > multi-kernel), 0 forces the multi-kernel path, 1 the cluster path where the
// plan allows it.  force_depth / force_chunk (-1: chosen by the planner) force the partition's tree depth and chunk
// size in poses.
inline void cholesky_make_plan(CholeskyPlan &pl, int n, const std::vector<int> &first_pose /*per free pose: first co-visible pose*/,
                               int chol_mode, int force_depth, int force_chunk) {
  pl.n = n;
  pl.bw = 0;
  for (size_t j = 0; j < first_pose.size(); ++j) pl.bw = std::max(pl.bw, 6 * ((int)j - first_pose[j]) + 5);
  pl.bw = std::min(pl.bw, std::max(0, n - 1));
  pl.banded = cholesky_banded_supported(n, pl.bw) && n > kBandMaxW && chol_mode != 0 && chol_mode != 1;
  pl.nd = NdPlan();
  if (pl.banded && n % 6 == 0) nd_make_plan(pl.nd, n / 6, (pl.bw - 5) / 6, 128, force_depth, force_chunk);
  pl.T = (n + 1 + kNB - 1) / kNB;
  pl.first_tile.assign(pl.T, pl.T);
  for (size_t j = 0; j < first_pose.size(); ++j) {
    const int c_tile = (6 * first_pose[j]) / kNB;
    for (int r = (int)(6 * j) / kNB; r <= (int)(6 * j + 5) / kNB; ++r) pl.first_tile[r] = std::min(pl.first_tile[r], c_tile);
  }
  for (int r = 0; r < pl.T; ++r) pl.first_tile[r] = std::min(pl.first_tile[r], r);
  pl.first_tile[n / kNB] = 0;  // the tile row that holds the rhs row is dense
  pl.rows_ptr.assign(pl.T + 1, 0);
  pl.rows.clear();
  long long used = 0;
  for (int k = 0; k < pl.T; ++k) {
    pl.rows_ptr[k] = (int)pl.rows.size();
    for (int r = k + 1; r < pl.T; ++r)
      if (pl.first_tile[r] <= k) pl.rows.push_back(r);
    const long long m = (long long)pl.rows.size() - pl.rows_ptr[k];
    used += m * (m + 1) / 2;
  }
  pl.rows_ptr[pl.T] = (int)pl.rows.size();
  // two-level plan
  pl.two_level = n > 2048;
  pl.narrow_cnt.assign(pl.T, 0);
  pl.grp_off.clear(); pl.grp_cnt.clear();
  if (pl.two_level) {
    for (int g0 = 0; g0 < pl.T; g0 += kGroup) {
      const int g1 = std::min(pl.T, g0 + kGroup);
      for (int k = g0; k < g1; ++k) {
        int c = 0;
        for (int q = pl.rows_ptr[k]; q < pl.rows_ptr[k + 1] && pl.rows[q] < g1; ++q) ++c;
        pl.narrow_cnt[k] = c;
      }
      pl.grp_off.push_back((int)pl.rows.size());
      int cnt = 0;
      for (int r = g1; r < pl.T; ++r)
        if (pl.first_tile[r] < g1) { pl.rows.push_back(r); ++cnt; }
      pl.grp_cnt.push_back(cnt);
    }
  }
  pl.max_rows = 0;
  for (int k = 0; k < pl.T; ++k) pl.max_rows = std::max(pl.max_rows, pl.rows_ptr[k + 1] - pl.rows_ptr[k]);
  // cluster path: every panel's tile jobs fit a few rounds of a <=16-CTA cluster
  pl.cluster_size = 0;
  if (n > 0 && n <= kClusterMaxN && pl.max_rows <= 12 && chol_mode != 0) {
    const int jobs = pl.max_rows * (pl.max_rows + 1) / 2;
    pl.cluster_size = jobs <= 1 ? 1 : jobs <= 2 ? 2 : jobs <= 4 ? 4 : jobs <= 8 ? 8 : 16;
  }
  long long dense = 0;
  for (int k = 0; k < pl.T; ++k) { const long long m = pl.T - 1 - k; dense += m * (m + 1) / 2; }
  pl.dense_fraction = dense > 0 ? (double)used / (double)dense : 1.0;
}

inline size_t cholesky_linv_doubles(int n) { return (size_t)((n + kNB - 1) / kNB) * kNB * kNB; }

// Enqueue factor + solve on `stream`.  Saug: (n+1)^2 doubles, ld = n+1.  x: n doubles.  zbuf: n.
// linv: ceil(n/64) * 64*64 doubles (inverses of the diagonal blocks).
// parts: bit 0 diag, 1 trsm, 2 syrk, 3 backward (all by default: the plan's path; a subset runs those parts of the
// multi-kernel path, for in-situ timing only).  verbose: print the plan and time the single-launch kernels.
inline void cholesky_solve_enqueue(const CholeskyPlan &pl, double *Saug, double *x, double *zbuf, double *linv,
                                   const LmState *st, cudaStream_t stream, long long *launches, bool verbose,
                                   int parts = 15) {
  const int n = pl.n, ld = n + 1, n_rows = n + 1;
  if (verbose) fprintf(stderr, "[ba_b200] cholesky n=%d T=%d max_rows=%d cluster_size=%d dense_fraction=%.3f bw=%d banded=%d path=%d parts=%d\n", n, pl.T, pl.max_rows, pl.cluster_size, pl.dense_fraction, pl.bw, (int)pl.banded, (int)pl.path, parts);
  if (parts == 15) {
    switch (pl.path) {
      case SolvePath::NdPersistent:
      case SolvePath::NdLevels: {
        if (nd_enqueue(pl.nd, pl.nd_dev, Saug, x, pl.path == SolvePath::NdPersistent, verbose ? 1 : 0, st, stream, launches)) return;
        const cudaError_t ce = cudaGetLastError();
        if (verbose) fprintf(stderr, "[ba_b200] partitioned banded launch failed: %s\n", cudaGetErrorString(ce));
      }
        [[fallthrough]];
      case SolvePath::Banded:
        if (cholesky_banded_enqueue(Saug, n, pl.bw, x, linv, verbose ? 1 : 0, st, stream)) {
          if (launches) *launches += 1;
          return;
        }
        [[fallthrough]];
      case SolvePath::Cluster:
        if (pl.cluster_size > 0) {
          if (cholesky_cluster_enqueue(Saug, n, pl.d_rows_ptr, pl.d_rows, pl.d_first_tile, x, verbose ? 1 : 0, st, stream, pl.cluster_size)) {
            if (launches) *launches += 1;
            return;
          }
          const cudaError_t ce = cudaGetLastError();  // cluster launch unavailable: fall through to the multi-kernel path
          if (verbose) fprintf(stderr, "[ba_b200] cluster launch failed: %s\n", cudaGetErrorString(ce));
        }
        break;
      case SolvePath::Dense:
        break;
    }
  }
  static PerDeviceOnce once;
  if (once.first()) cudaFuncSetAttribute(k_chol_diag, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCholDiagSmem);
  for (int k0 = 0, kb = 0; k0 < n; k0 += kNB, ++kb) {
    const int nb = (n - k0 < kNB) ? (n - k0) : kNB;
    double *Li = linv + (size_t)kb * kNB * kNB;
    if (parts & 1) {
      k_chol_diag<<<1, kDiagThreads, kCholDiagSmem, stream>>>(Saug, ld, k0, nb, Li, st);
      if (launches) *launches += 1;
    }
    // rows of the same tile below a partial last diagonal block (only the rhs row can be there)
    const int m = pl.rows_ptr[kb + 1] - pl.rows_ptr[kb];
    const bool tail_in_tile = (k0 + nb < n_rows) && (k0 + nb < k0 + kNB);
    if (tail_in_tile && (parts & 2)) {
      // the diagonal tile itself carries the rhs row: treat tile kb as one more row tile
      k_chol_trsm_tail<<<1, 64, 0, stream>>>(Saug, ld, n_rows, k0, nb, Li, st);
      if (launches) *launches += 1;
    }
    if (m > 0) {
      const int *rows = pl.d_rows + pl.rows_ptr[kb];
      if (parts & 2) k_chol_trsm<<<m, 256, 0, stream>>>(Saug, ld, n_rows, k0, nb, Li, rows, st);
      if (parts & 4) {
        if (!pl.two_level) {
          k_syrk_update<<<m * (m + 1) / 2, 256, 0, stream>>>(Saug, ld, n_rows, k0, nb, rows, 0, st);
        } else if (pl.narrow_cnt[kb] > 0) {
          k_syrk_update<<<m * pl.narrow_cnt[kb], 256, 0, stream>>>(Saug, ld, n_rows, k0, nb, rows, pl.narrow_cnt[kb], st);
        }
      }
      if (launches) *launches += ((parts >> 1) & 1) + ((parts >> 2) & 1);
    }
    if (pl.two_level && (parts & 4) && ((kb + 1) % kGroup == 0 || k0 + kNB >= n)) {
      const int g = kb / kGroup, mg = pl.grp_cnt[g];
      if (mg > 0) {
        const int kg0 = g * kGroup * kNB, kw = std::min(n, (kb + 1) * kNB) - kg0;
        k_syrk_update<<<mg * (mg + 1) / 2, 256, 0, stream>>>(Saug, ld, n_rows, kg0, kw, pl.d_rows + pl.grp_off[g], 0, st);
        if (launches) *launches += 1;
      }
    }
  }
  if (parts & 8) {
    if (n <= 2048) {
      k_backward_solve<<<1, 1024, 0, stream>>>(Saug, ld, n, linv, pl.d_first_tile, x, zbuf, st);
      if (launches) *launches += 1;
    } else {
      k_backward_init<<<(n + 255) / 256, 256, 0, stream>>>(Saug, ld, n, zbuf, st);
      const int nblk = (n + kNB - 1) / kNB;
      for (int kb = nblk - 1; kb >= 0; --kb) {
        const int k0 = kb * kNB, cbeg = std::min(k0, pl.first_tile[kb] * kNB);
        const int grid = std::max(1, (k0 - cbeg + kBwdColsPerCta - 1) / kBwdColsPerCta);
        k_backward_block<<<grid, 256, 0, stream>>>(Saug, ld, n, kb, linv, cbeg, x, zbuf, st);
      }
      if (launches) *launches += 1 + nblk;
    }
  }
}

}  // namespace ba
