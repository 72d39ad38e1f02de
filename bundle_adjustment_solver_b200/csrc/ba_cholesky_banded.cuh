// ba_cholesky_banded.cuh -- K5 for BANDED reduced camera systems (sequential trajectories: every landmark
// is seen by a short run of consecutive poses, so S has scalar half-bandwidth bw = 6 (track span) + 5).
// Replaces `Am_BCinvBt_mat.ldlt().solve(am_BCinv_b_mat)` (core/full_bundle_adjustment_solver.cpp:890-908).
//
// The dependency chain of a Cholesky factorisation is n column steps long no matter how it is blocked; for a
// band the work per step is only bw^2/2 FMAs, so the solve is bound by the LATENCY of the chain.  This file holds
// the SERIAL banded kernel k_chol_banded_smem: one CTA, 8-column block steps, the W x W window (W >= bw + 16) in
// shared memory as 8 x 8 tiles in ring slots, nine consumer warps apply the rank-8 update with DMMAs, one producer
// warp factors the 8 x 8 diagonal block and applies the triangular solve.  Since round 2 it is the FALLBACK of the
// partitioned (nested-dissection) solve in ba_cholesky_nd.cuh -- used when no partition is valid -- and its
// yardstick (BA_B200_BAND_MODE=4).  The two earlier variants (scalar register window, DMMA register tiles) were
// removed from the build.
//   * the rhs travels as one more window row, so z = L^-1 rhs falls out of the factorisation;
//   * non-positive pivots (pose without observations) emulate Eigen LDLT's D^+ = 0.
//
// The backward sweep L^T x = z runs in the same launch: 16-column blocks from the bottom; the block's
// off-diagonal part is a set of 16 dot products over <= bw rows (8 warps, shuffle reductions, L prefetched one
// block ahead), the 16 x 16 triangle is solved inside one warp with shuffles.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <type_traits>

#include "ba_cholesky_cluster.cuh"  // fast_rcp, gtime
#include "ba_device.cuh"

namespace ba {

constexpr int kBandThreads = 256;
constexpr int kBandMaxW = 112;

template <int W>
struct BandSmem {
  union {
    // factorisation: published columns of the current 16-step group (double-buffered by group parity):
    // [pos < W] column entries by frame position, [W] rhs entry z_j (unscaled), [W + 1] 1 / d_j
    double cb[2][16][W + 2];
    // inverse pre-pass: per half-warp staging of a 16 x 16 diagonal block of L and its diagonal reciprocals
    struct {
      double lst[8][2][16][17];
      double linvd[8][2][16];
    } pre;
  };
  double xr[W + 32];     // ring of solved x entries (backward sweep), index r mod (W+32)
  double acc[2][16];     // backward sweep: block right-hand side (double-buffered by block parity)
  unsigned long long mbar;   // column-published barrier (one phase per column step, 8 warp arrivals)
};

// mbarrier wrappers (shared::cta): split arrive / wait so that the bulk of a column step's update is issued
// between publishing the next column and waiting for everybody else's part of it
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "BA_MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra BA_MBAR_DONE;\n"
      "bra BA_MBAR_WAIT;\n"
      "BA_MBAR_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}

__device__ unsigned long long g_band_dbg[16];

__device__ __forceinline__ void dmma_884b(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// value of S(r, c) (r >= c) for the window, or the identity padding outside the matrix / zero outside the band
__device__ __forceinline__ double band_load(const double *A, int ld, int n, int bw, int r, int c) {
  if (r >= n) return (r == c) ? 1.0 : 0.0;
  if (r - c > bw) return 0.0;
  return __ldcg(A + (size_t)c * ld + r);
}
__device__ __forceinline__ double band_load_sym(const double *A, int ld, int n, int bw, int r, int c) {
  return r >= c ? band_load(A, ld, n, bw, r, c) : band_load(A, ld, n, bw, c, r);
}

// ---- backward sweep (shared by the banded kernels); runs on the first 256 threads of the CTA, named barrier 1
template <int W, typename SM>
__device__ __forceinline__ void band_backward(double *A, int n, int bw, double *x_out, double *linv, SM &sm) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int ld = n + 1;
  // ---- inverse pre-pass: X_k = L_kk^-1 for every 16 x 16 diagonal block (independent: all half-warps) ------
  const int nblk = (n + 15) / 16;
  {
    const int h = lane >> 4, m = lane & 15;
    double (*Ls)[17] = sm.pre.lst[warp][h];
    double *idg = sm.pre.linvd[warp][h];
#pragma unroll 1
    for (int it = 0; it < (nblk + 15) / 16; ++it) {   // uniform trip count
      const int kb = 16 * it + 2 * warp + h;
      const bool live = kb < nblk;
      const int j0 = kb * 16;
      __syncwarp();
      if (live) {
        // lane m stages column m (rows m..15) of the block
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          double val = (r == m) ? 1.0 : 0.0;
          if (r >= m && j0 + r < n) val = __ldcg(A + (size_t)(j0 + m) * ld + j0 + r);
          Ls[r][m] = val;
          if (r == m) idg[m] = 1.0 / val;   // +inf diagonal (zero pivot) -> 0
        }
      }
      __syncwarp();
      if (live) {
        // lane c solves L x = e_c by right-looking substitution in registers
        double xs[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) xs[r] = (r == m) ? 1.0 : 0.0;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
          xs[r] *= idg[r];
#pragma unroll
          for (int q = r + 1; q < 16; ++q) xs[q] -= Ls[q][r] * xs[r];
        }
        double *out = linv + (size_t)kb * 256;
#pragma unroll
        for (int r = 0; r < 16; ++r) out[r * 16 + m] = (r >= m) ? xs[r] : 0.0;   // X[r][c = m]
      }
    }
  }
  asm volatile("bar.sync 1, 256;" ::: "memory");

  // ---- backward sweep L^T x = z ------------------------------------------------------------------
  // blocks of 16 columns from the bottom.  Block [j0, j0+16):
  //   acc_c = z_c - sum_{r >= j0+16, r <= c+bw} L_rc x_r      (8 warps x 2 columns, shuffle reductions)
  //   x_c   = sum_{m >= c} X[m][c] acc_m  (X = L_kk^-1)       (every warp redundantly: one barrier per block)
  constexpr int XR = W + 32;
  constexpr int NSEG = (W + 31) / 32;
  constexpr int D = 3;  // register prefetch distance (blocks)
  double lo0[D][NSEG], lo1[D][NSEG], zc0[D], zc1[D], li[D][8];
  auto load_block = [&](int kb, double (&l0)[NSEG], double (&l1)[NSEG], double &z0, double &z1, double (&lv)[8]) {
    const int j0 = kb * 16;
    const int c0 = j0 + warp, c1 = j0 + warp + 8;
    const bool ok = kb >= 0;
#pragma unroll
    for (int k = 0; k < NSEG; ++k) {
      const int r = j0 + 16 + lane + 32 * k;
      l0[k] = (ok && c0 < n && r < n && r - c0 <= bw) ? __ldcg(A + (size_t)c0 * ld + r) : 0.0;
      l1[k] = (ok && c1 < n && r < n && r - c1 <= bw) ? __ldcg(A + (size_t)c1 * ld + r) : 0.0;
    }
    z0 = (ok && lane == 0 && c0 < n) ? __ldcg(A + (size_t)c0 * ld + n) : 0.0;
    z1 = (ok && lane == 0 && c1 < n) ? __ldcg(A + (size_t)c1 * ld + n) : 0.0;
    // lane (h, c): X[m][c] for m = 8h .. 8h+7
    const int h = lane >> 4, c = lane & 15;
#pragma unroll
    for (int q = 0; q < 8; ++q) lv[q] = ok ? __ldcg(linv + (size_t)kb * 256 + (8 * h + q) * 16 + c) : 0.0;
  };
#pragma unroll
  for (int u = 0; u < D; ++u) load_block(nblk - 1 - u, lo0[u], lo1[u], zc0[u], zc1[u], li[u]);
#pragma unroll 1
  for (int kb0 = nblk - 1; kb0 >= 0; kb0 -= D) {
#pragma unroll
    for (int u = 0; u < D; ++u) {
      const int kb = kb0 - u;
      if (kb < 0) break;  // uniform
      const int j0 = kb * 16, bp = kb & 1;
      double s0 = 0.0, s1 = 0.0;
#pragma unroll
      for (int k = 0; k < NSEG; ++k) {
        const int r = j0 + 16 + lane + 32 * k;
        const double xv = (r < n) ? sm.xr[r % XR] : 0.0;
        s0 += lo0[u][k] * xv;
        s1 += lo1[u][k] * xv;
      }
#pragma unroll
      for (int d = 16; d > 0; d >>= 1) {
        s0 += __shfl_down_sync(0xffffffffu, s0, d);
        s1 += __shfl_down_sync(0xffffffffu, s1, d);
      }
      if (lane == 0) {
        sm.acc[bp][warp] = zc0[u] - s0;
        sm.acc[bp][warp + 8] = zc1[u] - s1;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      {
        const int h = lane >> 4, c = lane & 15;
        double xa = 0.0, xb = 0.0;
#pragma unroll
        for (int q = 0; q < 8; q += 2) {
          xa += li[u][q] * sm.acc[bp][8 * h + q];
          xb += li[u][q + 1] * sm.acc[bp][8 * h + q + 1];
        }
        double xc = xa + xb;
        xc += __shfl_down_sync(0xffffffffu, xc, 16);
        if (lane < 16 && j0 + c < n) {
          sm.xr[(j0 + c) % XR] = xc;          // every warp writes the same value
          if (warp == 0) x_out[j0 + c] = xc;
        }
      }
      __syncwarp();
      load_block(kb - D, lo0[u], lo1[u], zc0[u], zc1[u], li[u]);
    }
  }
}

// Frame of group G (steps j = 16G .. 16G+15): slot (a, b) of thread (ty, tx) holds the window element
// (16(G+a) + ty, 16(G+b) + tx); once step jm has retired index 16G + jm, the a == 0 slots of the threads
// ty == jm (and the b == 0 slots of tx == jm) hold index 16G + jm + W instead.  After the group the slot
// arrays are rotated by one so that the next group is again at a == b == 0: the 16-step body is the same code
// for every group (it stays resident in the instruction cache).
// reciprocal square root off the slow libm path: hardware approximation (2^-22) + two Newton steps
__device__ __forceinline__ double fast_rsqrt(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double h = 0.5 * d;
  double e = fma(-h * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-h * y, y, 0.5);
  y = fma(y, e, y);
  return y;
}

constexpr int kBand4Cons = 9;                        // consumer warps (sub-partitions 0-2)
constexpr int kBand4Threads = 384;                   // 12 warps: 9 consumers, 1 producer (warp 3), 2 idle
constexpr int kBand4Active = 32 * (kBand4Cons + 1);  // threads that take part in the hand-off barriers

template <int W>
struct Band4Smem {
  union {
    struct {
      double win[(W / 8) * (W / 8)][64];   // tile (row slot, col slot), row-major 8 x 8
      double Lp[2][W + 1][12];             // factored panel (row stride 12: conflict-free 8 x 4 fragment reads)
      double zwin[W];                      // rhs entries of the window columns (ring position)
    } f;
    struct {
      double lst[8][2][16][17];
      double linvd[8][2][16];
    } pre;
  };
  double xr[W + 32];
  double acc[2][16];
  unsigned long long bar_raw[2], bar_L[2];
};

template <int W>
__global__ void __launch_bounds__(kBand4Threads, 1)
k_chol_banded_smem(double *A, int n, int bw, double *x_out, double *linv, int timing, const LmState *st) {
  if (st->done) return;
  constexpr int NT = W / 8;
  constexpr int T2 = (NT - 2) * (NT - 1) / 2;   // tiles outside the next panel: 2 <= rb <= ra <= NT - 1
  constexpr int TP2 = (T2 + kBand4Cons - 1) / kBand4Cons;
  constexpr int NSL = (W + 1 + 31) / 32;        // panel rows per producer lane
  // Roles by scheduler: warp w runs on SM sub-partition w % 4.  DMMA and DFMA share the FP64 pipe of a
  // sub-partition and a DMMA holds it for 16 cycles, so the latency-critical pivot chain of the panel warp
  // gets a sub-partition without DMMA traffic: warp 3 is the producer, warps 7 and 11 stay idle, the nine
  // warps on sub-partitions 0-2 are the consumers.
  const bool is_producer = (threadIdx.x >> 5) == 3;
  const bool is_idle = ((threadIdx.x >> 5) & 3) == 3 && !is_producer;
  const int cwi = (threadIdx.x >> 5) - ((threadIdx.x >> 5) >> 2);   // consumer index 0..8 (warps 0,1,2,4,5,6,8,9,10)
  const int ct = cwi * 32 + (threadIdx.x & 31);                     // consumer thread index 0..287
  extern __shared__ unsigned char band4_raw[];
  Band4Smem<W> &sm = *reinterpret_cast<Band4Smem<W> *>(band4_raw);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int ld = n + 1;
  const int nsteps = (n + 7) / 8;
  unsigned long long t_begin = 0;
  if (timing) t_begin = gtime();
  if (t == 0) {
    mbar_init(&sm.bar_raw[0], 8); mbar_init(&sm.bar_raw[1], 8);
    mbar_init(&sm.bar_L[0], 1);   mbar_init(&sm.bar_L[1], 1);
  }
  // initial window: tiles (I, J), I >= J (the upper ones are never read)
  for (int e = t; e < NT * NT * 64; e += kBand4Threads) {
    const int tile = e >> 6, i = (e >> 3) & 7, j = e & 7;
    const int I = tile / NT, J = tile - I * NT;
    sm.f.win[tile][8 * i + j] = (I >= J) ? band_load_sym(A, ld, n, bw, 8 * I + i, 8 * J + j) : 0.0;
  }
  for (int e = t; e < W; e += kBand4Threads) sm.f.zwin[e] = (e < n) ? __ldcg(A + (size_t)e * ld + n) : 0.0;
  __syncthreads();

  if (is_idle) {
    // nothing: joins the block-wide barrier below
  } else if (is_producer) {
    // ------------------------------------------------ producer: panel factorisation ----------------
    int P = 0;
    long long tw = 0, tk = 0;
#pragma unroll 1
    for (int s = 0; s < nsteps; ++s) {
      const int par = s & 1;
      const long long c0 = timing ? clock64() : 0;
      if (s > 0) asm volatile("bar.sync %0, %1;" ::"r"(5 + par), "n"(kBand4Active) : "memory");   // panel carries every earlier update
      const long long c1 = timing ? clock64() : 0;
      double a[NSL][8];
#pragma unroll
      for (int sl = 0; sl < NSL; ++sl) {
        const int pos = lane + 32 * sl;
        if (pos < W) {
          const double4 *src = reinterpret_cast<const double4 *>(&sm.f.win[(pos >> 3) * NT + P][8 * (pos & 7)]);
          const double4 v0 = src[0], v1 = src[1];
          a[sl][0] = v0.x; a[sl][1] = v0.y; a[sl][2] = v0.z; a[sl][3] = v0.w;
          a[sl][4] = v1.x; a[sl][5] = v1.y; a[sl][6] = v1.z; a[sl][7] = v1.w;
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k) a[sl][k] = (pos == W) ? sm.f.zwin[8 * P + k] : 0.0;
        }
      }
      double D[8][8], rs[8];
      {
        const double4 *dsrc = reinterpret_cast<const double4 *>(&sm.f.win[P * NT + P][0]);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const double4 v0 = dsrc[2 * i], v1 = dsrc[2 * i + 1];
          D[i][0] = v0.x; D[i][1] = v0.y; D[i][2] = v0.z; D[i][3] = v0.w;
          D[i][4] = v1.x; D[i][5] = v1.y; D[i][6] = v1.z; D[i][7] = v1.w;
        }
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const double d = D[k][k];
        const bool pos_def = d > 0.0;
        const double rc = pos_def ? fast_rcp(d) : 0.0;       // non-positive pivot: LDLT's D^+ = 0
        rs[k] = pos_def ? fast_rsqrt(d) : 0.0;
#pragma unroll
        for (int i = k + 1; i < 8; ++i) {
          const double ti = D[i][k] * rc;
#pragma unroll
          for (int j = k + 1; j <= i; ++j) D[i][j] -= ti * D[j][k];
        }
#pragma unroll
        for (int sl = 0; sl < NSL; ++sl) {
          const double u = a[sl][k] * rc;
#pragma unroll
          for (int m = k + 1; m < 8; ++m) a[sl][m] -= u * D[m][k];
        }
      }
#pragma unroll
      for (int sl = 0; sl < NSL; ++sl) {
        const int pos = lane + 32 * sl;
        if (pos <= W) {
          double4 *dst = reinterpret_cast<double4 *>(&sm.f.Lp[par][pos][0]);
          dst[0] = make_double4(a[sl][0] * rs[0], a[sl][1] * rs[1], a[sl][2] * rs[2], a[sl][3] * rs[3]);
          dst[1] = make_double4(a[sl][4] * rs[4], a[sl][5] * rs[5], a[sl][6] * rs[6], a[sl][7] * rs[7]);
        }
      }
      asm volatile("bar.arrive %0, %1;" ::"r"(3 + par), "n"(kBand4Active) : "memory");
      if (timing) { tw += c1 - c0; tk += clock64() - c1; }
      P = (P + 1 == NT) ? 0 : P + 1;
    }
    if (timing && lane == 0) { g_band_dbg[2] = tw; g_band_dbg[3] = tk; }
  } else {
    // ------------------------------------------------ consumers -------------------------------------
    const int fr = lane >> 2, fc = 2 * (lane & 3), kq = lane & 3;
    const int laneL = fr * 12 + kq, laneC = fr * 8 + fc;
    // relative coordinates of this warp's bulk tiles (the same at every step)
    int ra2[TP2], rb2[TP2];
#pragma unroll
    for (int i = 0; i < TP2; ++i) {
      int e = cwi + kBand4Cons * i, ra = 2, len = 1;    // row ra holds rb = 2 .. ra: (ra - 1) tiles
      const bool live = e < T2;
      if (live) {
        while (e >= len) { e -= len; ++ra; ++len; }
      }
      ra2[i] = live ? ra : -1;
      rb2[i] = live ? 2 + e : 0;
    }
    auto tile_update = [&](const double *Lp, int sa, int sb) {
      double *c = &sm.f.win[sa * NT + sb][laneC];
      double2 v = *reinterpret_cast<double2 *>(c);
#pragma unroll
      for (int h = 0; h < 2; ++h) dmma_884b(v.x, v.y, -Lp[sa * 96 + laneL + 4 * h], Lp[sb * 96 + laneL + 4 * h]);
      *reinterpret_cast<double2 *>(c) = v;
    };
    // streams of the elements this thread reloads when ring slot P is recycled for tile row s + NT: element
    // e = t + 256 q -> relative column tile rc = 1 + e / 64, (i, j) inside the tile; every step moves it by
    // 8 rows and 8 columns.  In-band is a static property of (rc, i, j); only the matrix bound moves.
    constexpr int NV = (NT * 64 + 32 * kBand4Cons - 1) / (32 * kBand4Cons);
    const double *nvp[NV];
    int nvhi[NV];
    unsigned nvok = 0;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
      const int e = ct + 32 * kBand4Cons * q;
      const int rc = 1 + (e >> 6), i = (e >> 3) & 7, j = e & 7;
      const int r = 8 * NT + i, c = 8 * rc + j;          // step 0
      const int lo = min(r, c), hi = max(r, c);
      nvp[q] = A + (size_t)lo * ld + hi;
      nvhi[q] = hi;
      if (e < NT * 64 && rc >= 2 && hi - lo <= bw) nvok |= 1u << q;
    }
    const size_t nvstride = (size_t)8 * (ld + 1);
    long long ctm[5] = {0, 0, 0, 0, 0};
    int zc = 8 * NT + (ct & 7);      // column whose rhs entry the threads of the retiring slot load (t / 8 == P)
    int P = 0;
#pragma unroll 1
    for (int s = 0; s < nsteps; ++s) {
      const int par = s & 1;
      const int Pn = (P + 1 == NT) ? 0 : P + 1;
      const double *Lp = &sm.f.Lp[par][0][0];
      const long long c0 = timing ? clock64() : 0;
      // new tile row (8 s + W ..): loads issued now, stored after the bulk update
      double nv[NV];
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        nv[q] = (((nvok >> q) & 1u) && nvhi[q] < n) ? __ldcg(nvp[q]) : 0.0;
        nvp[q] += nvstride;
        nvhi[q] += 8;
      }
      const bool z_retire = (ct >> 3) == P && ct < W;
      double znew = 0.0;
      if (z_retire) znew = (zc < n) ? __ldcg(A + (size_t)zc * ld + n) : 0.0;
      zc += 8;
      const long long c1 = timing ? clock64() : 0;
      asm volatile("bar.sync %0, %1;" ::"r"(3 + par), "n"(kBand4Active) : "memory");
      const long long c2 = timing ? clock64() : 0;
      // ---- priority: the next panel = relative column 1
      for (int ra = 1 + cwi; ra < NT; ra += kBand4Cons) {
        int sa = P + ra;
        if (sa >= NT) sa -= NT;
        tile_update(Lp, sa, Pn);
      }
      if (cwi == 0) {   // tile (new row, next panel) lies outside the band (W >= bw + 16): zeros
        *reinterpret_cast<double2 *>(&sm.f.win[P * NT + Pn][2 * lane]) = make_double2(0.0, 0.0);
      }
      const bool z_next = (ct >> 3) == Pn && ct < W;
      auto z_update = [&]() {
        const double4 *lz = reinterpret_cast<const double4 *>(Lp + W * 12);
        const double4 *lt = reinterpret_cast<const double4 *>(Lp + ct * 12);
        const double4 z0 = lz[0], z1 = lz[1], l0 = lt[0], l1 = lt[1];
        sm.f.zwin[ct] -= z0.x * l0.x + z0.y * l0.y + z0.z * l0.z + z0.w * l0.w + z1.x * l1.x + z1.y * l1.y + z1.z * l1.z + z1.w * l1.w;
      };
      if (z_next) z_update();
      asm volatile("bar.arrive %0, %1;" ::"r"(5 + (par ^ 1)), "n"(kBand4Active) : "memory");
      const long long c3 = timing ? clock64() : 0;
      // ---- bulk: operands of all tiles first, then the DMMAs (two dependent ones per tile), then the stores
      if (ct < W && !z_retire && !z_next) z_update();
      {
        double2 cv[TP2];
        double af[TP2][2], bf[TP2][2];
        double *cp[TP2];
#pragma unroll
        for (int i = 0; i < TP2; ++i) {
          int sa = P + max(ra2[i], 0), sb = P + rb2[i];
          if (sa >= NT) sa -= NT;
          if (sb >= NT) sb -= NT;
          cp[i] = &sm.f.win[sa * NT + sb][laneC];
          cv[i] = *reinterpret_cast<double2 *>(cp[i]);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            af[i][h] = -Lp[sa * 96 + laneL + 4 * h];
            bf[i][h] = Lp[sb * 96 + laneL + 4 * h];
          }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int i = 0; i < TP2; ++i) dmma_884b(cv[i].x, cv[i].y, af[i][h], bf[i][h]);
#pragma unroll
        for (int i = 0; i < TP2; ++i)
          if (ra2[i] >= 0) *reinterpret_cast<double2 *>(cp[i]) = cv[i];
      }
      // ---- finished panel to global memory: warp w writes column w (coalesced over rows)
      {
        const int c = 8 * s + cwi;
        if (cwi < 8 && c < n) {
          double *col = A + (size_t)c * ld + 8 * s;
#pragma unroll
          for (int q = 0; q < (W + 31) / 32; ++q) {
            const int pos = lane + 32 * q;
            int rel = pos - 8 * P;
            if (rel < 0) rel += W;
            if (pos < W && rel >= cwi && rel - cwi <= bw && 8 * s + rel < n) {
              double l = Lp[pos * 12 + cwi];
              if (rel == cwi && !(l > 0.0)) l = __longlong_as_double(0x7ff0000000000000LL);
              col[rel] = l;
            }
          }
          if (lane == 0) A[(size_t)c * ld + n] = Lp[W * 12 + cwi];
        }
      }
      // ---- recycle ring slot P for tile row s + NT (columns s + 2 .. s + NT; s + 1 was zeroed above)
#pragma unroll
      for (int q = 0; q < NV; ++q) {
        const int e = ct + 32 * kBand4Cons * q;
        const int rc = 1 + (e >> 6);
        if (e < NT * 64 && rc >= 2) {
          int sb = P + rc;
          if (sb >= NT) sb -= NT;
          sm.f.win[P * NT + sb][e & 63] = nv[q];
        }
      }
      if (z_retire) sm.f.zwin[ct] = znew;
      const long long c4 = timing ? clock64() : 0;
      asm volatile("bar.sync 2, %0;" ::"n"(32 * kBand4Cons) : "memory");   // tiles change hands between steps
      if (timing) { ctm[0] += c1 - c0; ctm[1] += c2 - c1; ctm[2] += c3 - c2; ctm[3] += c4 - c3; ctm[4] += clock64() - c4; }
      P = Pn;
    }
    if (timing && t == 0) { for (int i = 0; i < 5; ++i) g_band_dbg[4 + i] = ctm[i]; }
  }
  __syncthreads();
  unsigned long long t_factor = 0;
  if (timing) t_factor = gtime();
  if (warp < 8) band_backward<W>(A, n, bw, x_out, linv, sm);
  if (timing && t == 0) {
    g_band_dbg[0] = t_factor - t_begin;
    g_band_dbg[1] = gtime() - t_factor;
  }
}

template <int W>
inline bool launch_band4(double *Saug, int n, int bw, double *x, double *linv, int timing, const LmState *st,
                         cudaStream_t stream) {
  static PerDeviceOnce once;
  if (once.first())
    cudaFuncSetAttribute(k_chol_banded_smem<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Band4Smem<W>));
  k_chol_banded_smem<W><<<1, kBand4Threads, sizeof(Band4Smem<W>), stream>>>(Saug, n, bw, x, linv, timing, st);
  return cudaGetLastError() == cudaSuccess;
}

inline bool cholesky_banded_supported(int n, int bw) { return n > 0 && bw + 8 <= kBandMaxW; }

// timing: the kernel records its phase times in g_band_dbg
inline bool cholesky_banded_enqueue(double *Saug, int n, int bw, double *x, double *linv, int timing, const LmState *st,
                                    cudaStream_t stream) {
  // DMMA block steps, window in shared memory (needs W >= bw + 16; cholesky_banded_supported guarantees bw <= 104)
  if (bw + 16 <= 56) return launch_band4<56>(Saug, n, bw, x, linv, timing, st, stream);
  if (bw + 16 <= 88) return launch_band4<88>(Saug, n, bw, x, linv, timing, st, stream);
  if (bw + 16 <= 120) return launch_band4<120>(Saug, n, bw, x, linv, timing, st, stream);
  return false;
}

}  // namespace ba
