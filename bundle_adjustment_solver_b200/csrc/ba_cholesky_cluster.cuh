// ba_cholesky_cluster.cuh -- K5 for small / narrow-envelope reduced systems: the whole blocked Cholesky
// (diagonal block + inverse, panel TRSM, trailing SYRK, backward sweep) in ONE kernel launched as a single
// thread-block cluster.  The per-panel dependencies are resolved with the hardware cluster barrier
// (~0.2 us) instead of kernel boundaries (3 launches x ~3 us per panel), which is what bounds the
// multi-kernel path when a panel touches only a handful of 64x64 tiles (C1: n = 330; C3: 3 row tiles per
// panel inside the co-visibility envelope).
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <mutex>

#include <cstdlib>

#include "ba_device.cuh"

namespace ba {
namespace cg = cooperative_groups;

constexpr int kCB = 64;          // block size (== kNB)
constexpr int kCLD = kCB + 1;
constexpr int kClusterThreads = 256;
// shared memory (doubles): two staged operands [64][65] | scratch: column buffers [2][4][64], di [2], dval/dinv/invd [3][64]
constexpr int kScratch = 16 * kCB;
constexpr size_t kClusterSmem = (2 * kCB * kCLD + kScratch) * sizeof(double);
constexpr int kClusterMaxN = kCB * kCLD;  // x is staged in the second operand buffer during the backward sweep

// reciprocal off the slow division path (it sits on the per-column critical path of the sweep): hardware
// approximation (~20 bits) refined by two Newton steps (-> ~1e-24 relative, i.e. limited by rounding); no
// branches, no conversions.
// cudaFuncSetAttribute applies to the current device only: one opt-in per (kernel set, device), thread-safe
struct PerDeviceOnce {
  std::mutex mu;
  bool done[64] = {};
  bool first() {
    int d = 0;
    cudaGetDevice(&d);
    if (d < 0 || d >= 64) return true;
    std::lock_guard<std::mutex> lk(mu);
    if (done[d]) return false;
    done[d] = true;
    return true;
  }
};

__device__ __forceinline__ double fast_rcp(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  double e = fma(-d, x, 1.0);
  x = fma(x, e, x);
  e = fma(-d, x, 1.0);
  x = fma(x, e, x);
  return x;
}

// NOTE: no __restrict__ on the matrix / shared-memory pointers in this file: other threads (and other CTAs of
// the cluster) write the same locations between barriers, and a restrict-qualified pointer lets the compiler
// reuse a value loaded two column steps earlier from the double-buffered column vector.

// ---- tall panel (256 threads as a 16 x 16 grid, 2-D cyclic 4 x 4 register slots per 64 x 64 tile) --------
// Factorises the diagonal block AND up to NT row tiles below it in the same column sweep: thread (ty, tx)
// owns elements (r = ty + 16a, c = tx + 16b) of every tile.  Column step j (fully unrolled, dead slot groups
// pruned at compile time): the owners of column j publish it for all tiles (plus the pivot reciprocal)
// through a double-buffered shared vector, one barrier, then every thread applies the rank-1 update as 4 x 4
// outer products.  a_rc -= a_rj a_cj / d_j ; columns stay unscaled in registers and are scaled once at the
// end: L = A D^-1/2.  The panel rows thus cost no extra latency (no separate TRSM phase, no inverse).
// Non-positive pivots (pose without observations) emulate LDLT's D^+ = 0.
template <int NT>
__device__ __forceinline__ void chol_panel_tall(double *A, int ld, int n_rows, int k0, int nb, const int *rw,
                                                double *sm) {
  const int t = threadIdx.x, ty = t >> 4, tx = t & 15;
  double (*Ls)[kCLD] = reinterpret_cast<double (*)[kCLD]>(sm);  // scaled diagonal block (for the rhs tail)
  double *cb = sm + 2 * kCB * kCLD;   // [2][4][64]
  double *dib = cb + 8 * kCB;         // [2]
  double *dval = cb + 9 * kCB;        // [64] d_j, then sqrt(d_j)
  double *dinv = cb + 10 * kCB;       // [64] 1/sqrt(d_j)
  double v[4][4];
  double p[NT > 0 ? NT : 1][4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int r = ty + 16 * a, c = tx + 16 * b;
      double val = (r == c) ? 1.0 : 0.0;  // identity padding
      if (c <= r && r < nb) val = __ldcg(&A[(size_t)(k0 + c) * ld + k0 + r]);
      v[a][b] = val;
    }
#pragma unroll
  for (int q = 0; q < NT; ++q) {
    const int r0 = rw[q] * kCB;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int r = r0 + ty + 16 * a, c = tx + 16 * b;
        p[q][a][b] = (r < n_rows && c < nb) ? __ldcg(&A[(size_t)(k0 + c) * ld + r]) : 0.0;
      }
  }
#ifdef BA_DIAG_TIMING
  __syncthreads();
  long long tt1 = clock64();
#endif
#pragma unroll
  for (int j = 0; j < kCB; ++j) {
    const int par = (j & 1) * 4 * kCB, g = j >> 4, jm = j & 15;
    if (tx == jm) {
#pragma unroll
      for (int a = g; a < 4; ++a) cb[par + ty + 16 * a] = v[a][g];   // rows < j are stale but never read live
#pragma unroll
      for (int q = 0; q < NT; ++q)
#pragma unroll
        for (int a = 0; a < 4; ++a) cb[par + (1 + q) * kCB + ty + 16 * a] = p[q][a][g];
      if (ty == jm) {
        const double d = v[g][g];
        const double r = fast_rcp(d);
        dib[j & 1] = (d > 0.0) ? r : 0.0;
        dval[j] = d;
      }
    }
    __syncthreads();
    const double di = dib[j & 1];
    const bool own_live = tx > jm;  // in column group g only columns right of j are still live
    double lc[4];
#pragma unroll
    for (int b = g; b < 4; ++b) lc[b] = cb[par + tx + 16 * b];
    {
      double lr[4];
#pragma unroll
      for (int a = g; a < 4; ++a) lr[a] = cb[par + ty + 16 * a] * di;
#pragma unroll
      for (int a = g; a < 4; ++a) {
        if (own_live && g <= a) v[a][g] -= lr[a] * lc[g];
#pragma unroll
        for (int b = g + 1; b <= a; ++b) v[a][b] -= lr[a] * lc[b];
      }
    }
#pragma unroll
    for (int q = 0; q < NT; ++q) {
      double lr[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) lr[a] = cb[par + (1 + q) * kCB + ty + 16 * a] * di;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        if (own_live) p[q][a][g] -= lr[a] * lc[g];
#pragma unroll
        for (int b = g + 1; b < 4; ++b) p[q][a][b] -= lr[a] * lc[b];
      }
    }
  }
#ifdef BA_DIAG_TIMING
  long long tt2 = clock64();
#endif
  __syncthreads();
  if (t < kCB) {
    const double d = dval[t];
    const double s = (d > 0.0) ? rsqrt(d) : 0.0;  // 1/sqrt(d)
    dinv[t] = s;
    dval[t] = (s > 0.0) ? d * s : __longlong_as_double(0x7ff0000000000000LL);  // sqrt(d) or +inf
  }
  __syncthreads();
#ifdef BA_DIAG_TIMING
  long long tt3 = clock64();
#endif
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int r = ty + 16 * a, c = tx + 16 * b;
      double l = 0.0;
      if (r >= c) {
        l = (r == c) ? dval[c] : v[a][b] * dinv[c];
        if (r < nb) A[(size_t)(k0 + c) * ld + k0 + r] = l;
      }
      Ls[r][c] = l;
    }
#pragma unroll
  for (int q = 0; q < NT; ++q) {
    const int r0 = rw[q] * kCB;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int r = r0 + ty + 16 * a, c = tx + 16 * b;
        if (r < n_rows && c < nb) A[(size_t)(k0 + c) * ld + r] = p[q][a][b] * dinv[c];
      }
  }
  __syncthreads();
#ifdef BA_DIAG_TIMING
  if (t == 0) { g_t[1] = tt2 - tt1; g_t[2] = tt3 - tt2; g_t[3] = clock64() - tt3; }
#endif
}

// ---- panel tile by substitution: X L_kk^T = A_tile.  4 threads per row (q = t%4 owns columns m = q + 4i in
// registers); step c: the owner scales x_c = a_c / L_cc, broadcasts it inside the quad by shuffle, and the
// quad updates its remaining columns.  Warp-local (8 rows per warp): no barriers in the sweep.
__device__ __forceinline__ void job_trsm_subst(double *A, int ld, int n_rows, int k0, int nb, int r0,
                                               bool L_in_smem, double *sm) {
  double (*Ls)[kCLD] = reinterpret_cast<double (*)[kCLD]>(sm);
  double *invd = sm + 2 * kCB * kCLD + 11 * kCB;
  const int t = threadIdx.x;
  if (!L_in_smem) {
    __syncthreads();
    double tmp[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int e = t + kClusterThreads * u, r = e % kCB, c = e / kCB;
      tmp[u] = (r >= c && r < nb) ? __ldcg(&A[(size_t)(k0 + c) * ld + k0 + r]) : ((r == c) ? 1.0 : 0.0);
    }
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int e = t + kClusterThreads * u;
      Ls[e % kCB][e / kCB] = tmp[u];
    }
  }
  __syncthreads();
  if (t < kCB) invd[t] = 1.0 / Ls[t][t];   // +inf diagonal (zero pivot) -> 0
  __syncthreads();
  const int row = t >> 2, q = t & 3, lane = t & 31;
  const int rr = r0 + row;
  const bool live = rr < n_rows;
  double a[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int m = q + 4 * i;
    a[i] = (live && m < nb) ? __ldcg(&A[(size_t)(k0 + m) * ld + rr]) : 0.0;
  }
#pragma unroll
  for (int c = 0; c < kCB; ++c) {
    const int ci = c >> 2, cq = c & 3;
    double xc = a[ci] * invd[c];
    xc = __shfl_sync(0xffffffffu, xc, (lane & ~3) | cq);
    if (q == cq) a[ci] = xc;
#pragma unroll
    for (int i = ci; i < 16; ++i) {
      const int m = q + 4 * i;
      if (m > c) a[i] -= xc * Ls[m][c];
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int m = q + 4 * i;
    if (live && m < nb) A[(size_t)(k0 + m) * ld + rr] = a[i];
  }
}

// ---- 64x64 trailing tile (256 threads, 4x4 outputs per thread, K = 64 staged in shared memory) --------
__device__ __forceinline__ void tile_mac(const double (*P)[kCLD], const double (*Q)[kCLD], double (&acc)[4][4]) {
  const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
#pragma unroll 8
  for (int m = 0; m < kCB; ++m) {
    double a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = P[m][tx + 16 * i];
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = Q[m][ty + 16 * j];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] += a[i] * b[j];
  }
}

// trailing tile: A[r0.., c0..] -= P_r P_c^T (lower part only), P = panel k
__device__ __forceinline__ void job_syrk(double *A, int ld, int n_rows, int k0, int nb, int r0, int c0,
                                         double *sm) {
  double (*P)[kCLD] = reinterpret_cast<double (*)[kCLD]>(sm);
  double (*Q)[kCLD] = reinterpret_cast<double (*)[kCLD]>(sm + kCB * kCLD);
  const int t = threadIdx.x;
  const int ty = t / 16, tx = t % 16;
  // all global loads are issued before the first shared store (one exposed L2 latency, not sixteen)
  double tp[16], tq[16], tcur[16];
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int e = t + kClusterThreads * u, i = e % kCB, m = e / kCB;
    const int rr = r0 + i, cc = c0 + i;
    tp[u] = (m < nb && rr < n_rows) ? __ldcg(&A[(size_t)(k0 + m) * ld + rr]) : 0.0;
    tq[u] = (m < nb && cc < n_rows) ? __ldcg(&A[(size_t)(k0 + m) * ld + cc]) : 0.0;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int cc = c0 + ty + 16 * j, rr = r0 + tx + 16 * i;
      tcur[j * 4 + i] = (rr < n_rows && cc < n_rows - 1 && rr >= cc) ? __ldcg(&A[(size_t)cc * ld + rr]) : 0.0;
    }
  __syncthreads();
#pragma unroll
  for (int u = 0; u < 16; ++u) {
    const int e = t + kClusterThreads * u;
    P[e / kCB][e % kCB] = tp[u];
    Q[e / kCB][e % kCB] = tq[u];
  }
  __syncthreads();
  double acc[4][4] = {};
  tile_mac(P, Q, acc);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int cc = c0 + ty + 16 * j;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int rr = r0 + tx + 16 * i;
      if (rr < n_rows && cc < n_rows - 1 && rr >= cc) A[(size_t)cc * ld + rr] = tcur[j * 4 + i] - acc[i][j];
    }
  }
}

__device__ unsigned long long g_cl_dbg[8];
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ---- the cluster kernel -------------------------------------------------------------------------
__global__ void __launch_bounds__(kClusterThreads)
k_chol_cluster(double *A, int n, const int *__restrict__ rows_ptr, const int *__restrict__ rows,
               const int *__restrict__ first_tile, double *x_out, int timing,
               const LmState *st) {
  if (st->done) return;  // uniform across the cluster
  extern __shared__ double csm[];
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), ncta = (int)cluster.num_blocks();
  const int ld = n + 1, n_rows = n + 1;
  const int nblk = (n + kCB - 1) / kCB;
  const int t = threadIdx.x;
  unsigned long long tacc[6] = {0, 0, 0, 0, 0, 0};
  for (int kb = 0; kb < nblk; ++kb) {
    const int k0 = kb * kCB, nb = min(kCB, n - k0);
    const int m = rows_ptr[kb + 1] - rows_ptr[kb];
    const int *rw = rows + rows_ptr[kb];
    unsigned long long t0 = timing ? gtime() : 0;
    // Row tiles factorised together with the diagonal block.  Measured on B200: the extra FP64 work runs on
    // ONE SM inside a barrier-per-column sweep (963 vs 294 cycles per column for 3 extra tiles), slower than
    // handing the tiles to the other CTAs of the cluster, so the tall variant is kept for cluster size 1 only.
    const int NTk = (ncta == 1) ? (m < 3 ? m : 3) : 0;
    if (rank == 0) {
      switch (NTk) {
        case 0: chol_panel_tall<0>(A, ld, n_rows, k0, nb, rw, csm); break;
        case 1: chol_panel_tall<1>(A, ld, n_rows, k0, nb, rw, csm); break;
        case 2: chol_panel_tall<2>(A, ld, n_rows, k0, nb, rw, csm); break;
        default: chol_panel_tall<3>(A, ld, n_rows, k0, nb, rw, csm); break;
      }
      if (nb < kCB) {
        // rhs row inside the partial last diagonal tile: z_k L_kk^T = rhs_k by substitution (thread 0..)
        double (*Ls)[kCLD] = reinterpret_cast<double (*)[kCLD]>(csm);
        double *zz = csm + kCB * kCLD;
        if (t < kCB) zz[t] = (t < nb) ? A[(size_t)(k0 + t) * ld + n] : 0.0;
        __syncthreads();
        if (t == 0) {
          for (int c = 0; c < nb; ++c) {
            double acc = zz[c];
            for (int mm = 0; mm < c; ++mm) acc -= zz[mm] * Ls[c][mm];
            zz[c] = acc / Ls[c][c];
          }
        }
        __syncthreads();
        if (t < nb) A[(size_t)(k0 + t) * ld + n] = zz[t];
      }
    }
    if (m == 0) continue;  // uniform
    unsigned long long t1 = timing ? gtime() : 0;
    cluster.sync();
    unsigned long long t2 = timing ? gtime() : 0;
    // row tiles beyond the tall panel (wide envelopes only): substitution jobs on all ranks
    for (int job = NTk + rank; job < m; job += ncta) job_trsm_subst(A, ld, n_rows, k0, nb, rw[job] * kCB, false, csm);
    unsigned long long t3 = timing ? gtime() : 0;
    if (m > NTk) cluster.sync();  // uniform
    unsigned long long t4 = timing ? gtime() : 0;
    const int npairs = m * (m + 1) / 2;
    for (int job = rank; job < npairs; job += ncta) {
      int ia = (int)((sqrt(8.0 * job + 1.0) - 1.0) * 0.5);
      while (ia * (ia + 1) / 2 > job) --ia;
      while ((ia + 1) * (ia + 2) / 2 <= job) ++ia;
      const int ib = job - ia * (ia + 1) / 2;
      job_syrk(A, ld, n_rows, k0, nb, rw[ia] * kCB, rw[ib] * kCB, csm);
    }
    unsigned long long t5 = timing ? gtime() : 0;
    cluster.sync();
    if (timing) {
      unsigned long long t6 = gtime();
      tacc[0] += t1 - t0; tacc[1] += t2 - t1; tacc[2] += t3 - t2; tacc[3] += t4 - t3; tacc[4] += t5 - t4; tacc[5] += t6 - t5;
    }
  }
  unsigned long long tb0 = timing ? gtime() : 0;
  // ---- backward sweep L^T x = z by rank 0 (left-looking over the envelope tiles)
  if (rank != 0) return;
  __syncthreads();
  double *xs = csm + kCB * kCLD;             // x for all blocks (second operand buffer onwards is free here)
  double (*Ls)[kCLD] = reinterpret_cast<double (*)[kCLD]>(csm);
  double *acc_s = csm + 2 * kCB * kCLD + 12 * kCB;       // [64]
  const int warp = t >> 5, lane = t & 31;
  for (int kb = nblk - 1; kb >= 0; --kb) {
    const int k0 = kb * kCB, nb = min(kCB, n - k0);
    // diagonal block to shared memory (coalesced by columns)
    {
      double tmp[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int e = t + kClusterThreads * u, r = e % kCB, c = e / kCB;
        tmp[u] = (r >= c && r < nb) ? __ldcg(&A[(size_t)(k0 + c) * ld + k0 + r]) : ((r == c) ? 1.0 : 0.0);
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int e = t + kClusterThreads * u;
        Ls[e % kCB][e / kCB] = tmp[u];
      }
    }
    __syncthreads();
    double *invd = csm + 2 * kCB * kCLD + 11 * kCB;
    if (t < kCB) invd[t] = 1.0 / Ls[t][t];
    {
      // acc[c] = z[k0+c] - sum over envelope rows r >= k0+64 of L[r][k0+c] x[r];
      // warp w owns columns c = w + 8u (u = 0..7); all their loads are issued together per envelope tile
      double s[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) s[u] = 0.0;
      for (int mt = kb + 1; mt < nblk; ++mt) {
        if (first_tile[mt] > kb) continue;
        const int r1 = mt * kCB + lane, r2 = r1 + 32;
        const double x1 = (r1 < n) ? xs[r1] : 0.0, x2 = (r2 < n) ? xs[r2] : 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int c = warp + 8 * u;
          if (c < nb) {
            const double *col = A + (size_t)(k0 + c) * ld;
            const double a1 = (r1 < n) ? __ldcg(col + r1) : 0.0;
            const double a2 = (r2 < n) ? __ldcg(col + r2) : 0.0;
            s[u] += a1 * x1 + a2 * x2;
          }
        }
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1)
#pragma unroll
        for (int u = 0; u < 8; ++u) s[u] += __shfl_down_sync(0xffffffffu, s[u], d);
      if (lane == 0) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int c = warp + 8 * u;
          acc_s[c] = (c < nb) ? (__ldcg(&A[(size_t)(k0 + c) * ld + n]) - s[u]) : 0.0;
        }
      }
    }
    __syncthreads();
    // L_kk^T x_k = acc by backward substitution in warp 0: lane owns entries lane and lane+32
    if (warp == 0) {
      double a0 = acc_s[lane], a1 = acc_s[lane + 32];
      for (int c = kCB - 1; c >= 0; --c) {
        const double owner = (c >= 32) ? a1 : a0;
        const double xc = __shfl_sync(0xffffffffu, owner, c & 31) * invd[c];
        if (lane == (c & 31)) { if (c >= 32) a1 = xc; else a0 = xc; }
        // acc_m -= L[c][m] x_c for m < c
        if (lane < c) a0 -= Ls[c][lane] * xc;
        if (lane + 32 < c) a1 -= Ls[c][lane + 32] * xc;
      }
      if (lane < nb) { xs[k0 + lane] = a0; x_out[k0 + lane] = a0; }
      if (lane + 32 < nb) { xs[k0 + lane + 32] = a1; x_out[k0 + lane + 32] = a1; }
    }
    __syncthreads();
  }
  if (timing && t == 0) { for (int i = 0; i < 6; ++i) g_cl_dbg[i] = tacc[i]; g_cl_dbg[6] = gtime() - tb0; }
}

// timing: the kernel records its phase times in g_cl_dbg
inline bool cholesky_cluster_enqueue(double *Saug, int n, const int *d_rows_ptr, const int *d_rows,
                                     const int *d_first_tile, double *x, int timing, const LmState *st,
                                     cudaStream_t stream, int cluster_size) {
  static PerDeviceOnce once;
  if (once.first()) {
    cudaFuncSetAttribute(k_chol_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kClusterSmem);
    cudaFuncSetAttribute(k_chol_cluster, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cluster_size);
  cfg.blockDim = dim3(kClusterThreads);
  cfg.dynamicSmemBytes = kClusterSmem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = cluster_size;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_chol_cluster, Saug, n, d_rows_ptr, d_rows, d_first_tile, x, timing, st) ==
         cudaSuccess;
}

}  // namespace ba
