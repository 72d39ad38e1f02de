// ba_cholesky_nd.cuh -- K5 for banded reduced camera systems, PARTITIONED: nested dissection of the pose chain
// into independent dense fronts (plan: ba_nd_plan.h), one CTA per front, FP64 tensor-core (DMMA) panel solves and
// trailing updates.  Replaces `Am_BCinvBt_mat.ldlt().solve(am_BCinv_b_mat)`
// (core/full_bundle_adjustment_solver.cpp:890-908).
//
// The serial banded kernel (ba_cholesky_banded.cuh) walks n/8 dependent panel steps on ONE SM.  Here the pose
// chain is cut by separators into 2^L leaves that are eliminated concurrently on 2^L SMs; the separators are
// eliminated level by level (L levels).  The dependent chain is 6 (N / 2^L) / 8 + L (6 b / 8) panel steps.
//
// One front = [own | Rb | Lb | rhs] (ba_nd_plan.h).  Per front, one CTA of 12 warps:
//   * assembly: the own columns (own x own lower trapezoid and boundary x own) are gathered into shared memory as
//     8 x 8 tiles (swizzled so that DMMA fragment reads are conflict-free): entries of S (global, column-major
//     lower + rhs row) plus the contribution blocks U of the children (extend-add through per-child index maps),
//     a batch of tiles per warp with every load of the batch in flight at once; the boundary x boundary part
//     never enters shared memory: it lives in the DMMA accumulator registers of the consumer warps.
//   * factor: panel steps of 8 columns.  The diagonal warp (warp 3, alone on its SM sub-partition) only factors
//     the 8 x 8 diagonal block and inverts the factor (W = L_ss^-1, redundantly in every lane: no shuffles on the
//     chain).  The nine consumer warps turn the panel solve into tensor-core work, L_Is = A_Is W^T (two DMMAs per
//     tile, in place), and after one consumer-wide barrier apply the rank-8 update to the tiles they own (two
//     DMMAs per tile) and to their boundary x boundary accumulators.  LOOK-AHEAD: the owner of the next diagonal
//     tile solves row tile s+1 itself and updates tile (s+1, s+1) before that barrier, so the dependent chain per
//     step is  diagonal factor -> 4 DMMAs -> diagonal factor.
//   * L (tiles, as they stand in shared memory) and W go to global memory for backward passes that run after the
//     front has left shared memory; the accumulators are written out as the contribution block U.
// Backward (root first): x_own = -L11^-T (L21^T x_boundary - z): boundary part in parallel over the warps from the
// tiles in shared memory, then an 8-column block chain inside one warp with the W blocks.
//
// Two drivers over the same per-front code: one launch per tree level (`k_nd_forward_level` / `k_nd_backward_level`)
// and a single persistent launch (`k_nd_persistent`): every CTA walks its list of fronts, hand-overs between CTAs go
// through acquire / release flags in global memory; the last front of a list is still resident in shared memory
// when its backward pass starts.
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "ba_cholesky_banded.cuh"   // dmma_884b, fast_rcp, fast_rsqrt
#include "ba_nd_plan.h"

namespace ba {

constexpr int kNdThreads = 384;
constexpr int kNdWarps = kNdThreads / 32;
// NC consumer warps (template parameter): 9 = warps 0,1,2,4,5,6,8,9,10, the diagonal warp alone on its SM
// sub-partition (small fronts: the chain of diagonal blocks bounds the step); 11 = every warp but the diagonal warp
// (large fronts: the DMMA updates bound the step)
constexpr int kNdBarA = 3;                           // diagonal warp -> consumers: W(s) published
constexpr int kNdBarB = 4;                           // consumers: panel s solved
constexpr int kNdBarC = 5;                           // look-ahead warp -> diagonal warp: tile (s+1, s+1) final
constexpr int kNdCntC = 64;
constexpr int kNdSpinLimit = 1 << 22;

struct NdArgs {
  const NdNode *nodes;
  const int *list;        // level driver: node ids by level; persistent driver: per-CTA lists
  const int *list_ptr;    // persistent driver: [n_ctas + 1]
  const double *S;        // (n+1)^2, entry (r, c), r >= c, at S[c * ld + r]; rhs in row n
  int n, ld, bw;
  double *Lws, *Uws, *x;
  int *flags;             // persistent driver: [n_nodes] forward done, [n_nodes] backward done, [n_step_flags] panel
                          // steps of the helped fronts, abort, sticky error
  int n_nodes;
  int abort_idx;          // index of the abort word (the sticky error word follows it)
  int step_base;          // index of the first per-step flag
  int n_main;             // CTAs that walk front lists; CTA n_main + h is helper h
  const int *helper_list; // front of every helper CTA
  int use_helpers;        // 0 in the one-launch-per-level driver
  int max_R8, max_tiles, max_KT;  // shared-memory carve-up
};

__device__ unsigned long long g_nd_dbg[16];

__device__ __forceinline__ int nd_tidx(int I, int J) { return I * (I + 1) / 2 + J; }   // lower-triangular tile index
// element (r, c) of a swizzled 8 x 8 tile: the two column halves of rows 2, 3, 6, 7 are exchanged, which makes the
// DMMA operand fragment (row lane / 4, column lane % 4 [+ 4]) hit 16 distinct bank pairs per half-warp
__device__ __forceinline__ int nd_sw(int r, int c) { return r * 8 + (c ^ ((r & 2) << 1)); }

struct NdSmem {
  double *win;    // own trapezoid tiles [max_tiles][64], column by column
  double *winv;   // inverses of the diagonal blocks [max_KT][64]
  double *xs;     // backward: x by front-local index [max_R8]
  double *tb;     // backward: right-hand side of the block chain [max_R8]
  int *pm;        // my boundary index -> front-local index of my parent [max_R8] (second half unused)
  int *grow;      // global index of a front-local row / column in S (n: rhs row, -1: padding) [max_R8]
  int *tt;        // tile table: (I << 16) | J by storage position
  NdNode *node;   // current node
  NdNode *cn;     // its two children [2]
  NdNode *par;    // its parent
};

__device__ __forceinline__ NdSmem nd_carve(unsigned char *raw, const NdArgs &g) {
  NdSmem sm;
  sm.win = reinterpret_cast<double *>(raw);
  sm.winv = sm.win + (size_t)g.max_tiles * 64;
  sm.xs = sm.winv + (size_t)g.max_KT * 64;
  sm.tb = sm.xs + g.max_R8;
  sm.pm = reinterpret_cast<int *>(sm.tb + g.max_R8);
  sm.grow = sm.pm + 2 * g.max_R8;
  sm.tt = sm.grow + g.max_R8;
  sm.node = reinterpret_cast<NdNode *>(sm.tt + ((g.max_tiles + 1) & ~1));
  sm.cn = sm.node + 1;
  sm.par = sm.node + 3;
  return sm;
}
inline size_t nd_smem_bytes(const NdPlan &pl) {
  return ((size_t)pl.max_tiles + pl.max_KT) * 64 * sizeof(double) + (size_t)2 * pl.max_R8 * sizeof(double) +
         (size_t)3 * pl.max_R8 * sizeof(int) + (size_t)((pl.max_tiles + 1) & ~1) * sizeof(int) + 4 * sizeof(NdNode) + 64;
}

// Sources of the initial value of front entry (i, j), i >= j (front-local indices): an entry of S (own columns only),
// one entry of each child's contribution block, or a constant (identity padding).  Addresses first, loads later, so
// that a batch of entries has all its loads in flight together.
// Initial value of front entry (i, j), i >= j, j an own column, as far as S is concerned: the offset of the entry in
// S, kNdNone (nothing), or kNdOne (identity padding).  The children's contributions arrive as whole tiles.
constexpr unsigned kNdNone = 0xffffffffu, kNdOne = 0xfffffffeu;
struct NdGather {
  const double *S, *U0, *U1;     // U0 / U1: the children's contribution blocks in THIS front's layout (nullptr: no child)
  int ld, n, bw;
};
__device__ __forceinline__ unsigned nd_front_src(const NdGather &q, const NdSmem &sm, int i, int j, bool on) {
  if (!on) return kNdNone;
  const int gi = sm.grow[i], gj = sm.grow[j];
  if (gj < 0) return (i == j) ? kNdOne : kNdNone;    // identity padding of the own block
  if (gi < 0) return kNdNone;
  const int lo = min(gi, gj), hi = max(gi, gj);
  if (hi == q.n || hi - lo <= q.bw) return (unsigned)lo * (unsigned)q.ld + (unsigned)hi;
  return kNdNone;
}
__device__ __forceinline__ double nd_src_value(const NdGather &q, unsigned os) {
  return os < kNdOne ? __ldcg(q.S + os) : (os == kNdOne ? 1.0 : 0.0);
}

// stage the node record (and its children's) in shared memory; ends with a CTA barrier
__device__ __forceinline__ void nd_stage_node(const NdArgs &g, const NdSmem &sm, int node_id, bool children) {
  const int t = threadIdx.x;
  constexpr int NW = (int)(sizeof(NdNode) / sizeof(int));
  if (t < NW) reinterpret_cast<int *>(sm.node)[t] = reinterpret_cast<const int *>(g.nodes + node_id)[t];
  __syncthreads();
  if (children) {
    const NdNode &nd = *sm.node;
    for (int c = 0; c < 2; ++c)
      if (nd.child[c] >= 0 && t >= 32 * (1 + c) && t < 32 * (1 + c) + NW)
        reinterpret_cast<int *>(sm.cn + c)[t - 32 * (1 + c)] = reinterpret_cast<const int *>(g.nodes + nd.child[c])[t - 32 * (1 + c)];
    if (nd.parent >= 0 && t >= 96 && t < 96 + NW)
      reinterpret_cast<int *>(sm.par)[t - 96] = reinterpret_cast<const int *>(g.nodes + nd.parent)[t - 96];
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------------------
// forward elimination of one front.  TPW: boundary x boundary tiles per consumer warp (register accumulators)
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int nd_ld_acquire(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void nd_st_release(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Everything of a front that does not depend on its children's results: node records and index tables in shared
// memory.  The persistent driver runs it BEFORE it waits for the children's flags (off the critical path).
__device__ void nd_forward_prepare(const NdArgs &g, const NdSmem &sm, int node_id, bool with_S = true) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  nd_stage_node(g, sm, node_id, true);
  const NdNode &nd = *sm.node;
  const int KT = nd.k8 >> 3, BT = nd.b8 >> 3, NT = KT + BT;
  auto colbase = [&](int J) { return J * NT - (J * (J - 1)) / 2; };   // tile (I, J), I >= J, at colbase(J) + I - J
  // pm: my boundary index -> front-local index of my PARENT (where my Schur complement goes); -1: padding
  for (int i = t; i < nd.b8; i += kNdThreads) {
    int m = -1;
    if (nd.parent >= 0) {
      if (i < nd.wr) m = nd.rb_off + i;
      else if (i < nd.wr + nd.wl) m = nd.lb_off + (i - nd.wr);
      else if (i == nd.wr + nd.wl) m = nd.rhs_off;
    }
    sm.pm[i] = m;
  }
  for (int i = t; i < 64 * KT; i += kNdThreads) sm.winv[i] = 0.0;
  for (int i = t; i < 8 * NT; i += kNdThreads) {
    const int bi = i - nd.k8;
    int gi = -1;
    if (i < nd.k) gi = nd.own0 + i;
    else if (bi >= 0 && bi < nd.wr) gi = nd.rb0 + bi;
    else if (bi >= 0 && bi < nd.wr + nd.wl) gi = nd.lb0 + (bi - nd.wr);
    else if (bi == nd.wr + nd.wl) gi = g.n;
    sm.grow[i] = gi;
  }
  for (int J = warp; J < KT; J += kNdWarps) {
    const int base = colbase(J) - J;
    for (int I = J + lane; I < NT; I += 32) sm.tt[base + I] = (I << 16) | J;
  }
  __syncthreads();
  if (!with_S) return;
  // the band of S for the own columns (does not depend on the children either): a warp takes UN tiles per round, lane
  // (fr, fc) two adjacent entries of each; gathered through the row table with every load of the round in flight
  {
    const int fr = lane >> 2, fc = 2 * (lane & 3);
    const int offC = fr * 8 + (fc ^ ((fr & 2) << 1));
    const int n_tiles = colbase(KT);
    NdGather gq;
    gq.S = g.S; gq.ld = g.ld; gq.n = g.n; gq.bw = g.bw; gq.U0 = gq.U1 = nullptr;
    constexpr int UN = 8;
    for (int tb0 = warp; tb0 < n_tiles; tb0 += kNdWarps * UN) {
      unsigned src[UN][2];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int tile = tb0 + kNdWarps * u;
        const bool live = tile < n_tiles;
        const int ij = sm.tt[live ? tile : tb0];
        const int I = ij >> 16, J = ij & 0xffff;
        const int i = 8 * I + fr, j = 8 * J + fc;
        bool in_band = true;            // tiles entirely outside the band of S hold no entry of S
        if (I > J) {
          const int gr = sm.grow[8 * I], gr7 = sm.grow[8 * I + 7], gc = sm.grow[8 * J], gc7 = sm.grow[8 * J + 7];
          const bool rows_ok = gr >= 0 && gr7 - gr == 7 && gr7 != g.n;     // eight consecutive rows of S
          in_band = !(rows_ok && ((gc7 >= 0 && gr - gc7 > g.bw) || gc - gr7 > g.bw));
        }
        src[u][0] = nd_front_src(gq, sm, i, j, live && in_band && i >= j);
        src[u][1] = nd_front_src(gq, sm, i, j + 1, live && in_band && i >= j + 1);
      }
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int tile = tb0 + kNdWarps * u;
        if (tile < n_tiles)
          *reinterpret_cast<double2 *>(sm.win + (size_t)tile * 64 + offC) = make_double2(nd_src_value(gq, src[u][0]), nd_src_value(gq, src[u][1]));
      }
    }
  }
  __syncthreads();
}

template <int TPW, int NC>
__device__ void nd_forward_node(const NdArgs &g, const NdSmem &sm, int node_id, int timing) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const bool is_diag = warp == 3;
  static_assert(NC == 9 || NC == 11, "consumer warps");
  constexpr int kNdCons = NC, kNdCntA = 32 * (NC + 1), kNdCntB = 32 * NC;
  const bool is_idle = NC == 9 && (warp & 3) == 3 && !is_diag;
  const int cwi = NC == 9 ? warp - (warp >> 2) : warp - (warp > 3 ? 1 : 0);   // consumer index
  unsigned long long t_in = 0;
  if (timing && t == 0) t_in = gtime();
  const NdNode &nd = *sm.node;                  // staged by nd_forward_prepare
  const int KT = nd.k8 >> 3, BT = nd.b8 >> 3, NT = KT + BT;
  auto colbase = [&](int J) { return J * NT - (J * (J - 1)) / 2; };   // tile (I, J), I >= J, at colbase(J) + I - J
  const int n_tiles = colbase(KT);
  const int LbT0 = (nd.k8 + nd.wr) >> 3;        // first row tile of [Lb | rhs]
  const int fr = lane >> 2, fc = 2 * (lane & 3), kq = lane & 3;
  const int swz = (fr & 2) << 1;
  const int offC = fr * 8 + (fc ^ swz);                          // accumulator fragment (double2) inside a tile
  const int offA0 = fr * 8 + (kq ^ swz), offA1 = offA0 ^ 4;      // operand fragments: columns kq and kq + 4
  NdGather gq;
  gq.S = g.S; gq.ld = g.ld; gq.n = g.n; gq.bw = g.bw;
  gq.U0 = nd.child[0] >= 0 ? g.Uws + sm.cn[0].U_off : nullptr;
  gq.U1 = nd.child[1] >= 0 ? g.Uws + sm.cn[1].U_off : nullptr;
  const bool has_children = gq.U0 || gq.U1;
  const bool helped = g.use_helpers && nd.helper >= 0;     // a helper CTA holds the boundary x boundary accumulators
  // ---- boundary x boundary accumulators (consumers): children's contributions passed through (loads issued first:
  //      they are in flight while the own columns are assembled)
  const int n_utiles = BT * (BT + 1) / 2;
  double2 acc[TPW];
  int ub[TPW];                                   // (row tile << 8) | column tile of the boundary block, -1: none
#pragma unroll
  for (int q = 0; q < TPW; ++q) {
    acc[q] = make_double2(0.0, 0.0);
    ub[q] = -1;
  }
  if (!is_diag && !is_idle && !helped) {
#pragma unroll
    for (int q = 0; q < TPW; ++q) {
      const int e = cwi + kNdCons * q;
      if (e < n_utiles) {
        int I = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
        while (I * (I + 1) / 2 > e) --I;
        while ((I + 1) * (I + 2) / 2 <= e) ++I;
        ub[q] = (I << 8) | (e - I * (I + 1) / 2);
      }
    }
    if (has_children) {
      const int offU = fr * 8 + fc;
#pragma unroll
      for (int q = 0; q < TPW; ++q) {
        if (ub[q] >= 0) {
          const size_t off = ((size_t)n_tiles + nd_tidx(ub[q] >> 8, ub[q] & 0xff)) * 64 + offU;
          const double2 a = gq.U0 ? __ldcg(reinterpret_cast<const double2 *>(gq.U0 + off)) : make_double2(0.0, 0.0);
          const double2 b = gq.U1 ? __ldcg(reinterpret_cast<const double2 *>(gq.U1 + off)) : make_double2(0.0, 0.0);
          acc[q] = make_double2(a.x + b.x, a.y + b.y);
        }
      }
    }
  }
  // ---- assembly of the own columns: the band of S is already in the window (nd_forward_prepare); the children's
  //      contribution tiles arrive in this front's layout and are added as whole tiles (coalesced double2 loads)
  if (has_children) {
    constexpr int UN = 8;
    for (int tb0 = warp; tb0 < n_tiles; tb0 += kNdWarps * UN) {
      double2 c0[UN], c1[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int tile = tb0 + kNdWarps * u;
        const bool live = tile < n_tiles;
        c0[u] = (live && gq.U0) ? __ldcg(reinterpret_cast<const double2 *>(gq.U0 + (size_t)tile * 64 + offC)) : make_double2(0.0, 0.0);
        c1[u] = (live && gq.U1) ? __ldcg(reinterpret_cast<const double2 *>(gq.U1 + (size_t)tile * 64 + offC)) : make_double2(0.0, 0.0);
      }
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int tile = tb0 + kNdWarps * u;
        if (tile < n_tiles) {
          double2 *w = reinterpret_cast<double2 *>(sm.win + (size_t)tile * 64 + offC);
          const double2 v = *w;
          *w = make_double2(v.x + (c0[u].x + c1[u].x), v.y + (c0[u].y + c1[u].y));
        }
      }
    }
  }
  if (timing && t == 0 && blockIdx.x == 0) g_nd_dbg[14] += gtime() - t_in;   // + own columns (warp 0's share)
  __syncthreads();
  unsigned long long t0 = 0;
  if (timing && t == 0) {
    t0 = gtime();
    if (blockIdx.x == 0) g_nd_dbg[10] += t0 - t_in;     // staging + assembly (CTA 0 / first front of a level)
  }

  // ---- factorisation of the own columns
  double *Lg = g.Lws + nd.L_off;
  double *Wg = Lg + (size_t)n_tiles * 64;
  if (is_idle) {
    // nothing
  } else if (is_diag) {
#pragma unroll 1
    for (int s = 0; s < KT; ++s) {
      long long c0 = 0;
      if (timing) c0 = clock64();
      if (s > 0) asm volatile("bar.sync %0, %1;" ::"n"(kNdBarC), "n"(kNdCntC) : "memory");
      long long c1 = 0;
      if (timing) c1 = clock64();
      double *dt = sm.win + (size_t)colbase(s) * 64;          // tile (s, s)
      double D[8][8], rs[8];
      {
        const double4 *dsrc = reinterpret_cast<const double4 *>(dt);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const double4 lo = dsrc[2 * i + ((i & 2) ? 1 : 0)], hi = dsrc[2 * i + ((i & 2) ? 0 : 1)];
          D[i][0] = lo.x; D[i][1] = lo.y; D[i][2] = lo.z; D[i][3] = lo.w;
          D[i][4] = hi.x; D[i][5] = hi.y; D[i][6] = hi.z; D[i][7] = hi.w;
        }
      }
      // Cholesky with the reciprocal square root on the chain: the columns come out scaled (D becomes L), which
      // measured shorter than a reciprocal chain plus square roots off it (profiles/micro/diag8_bench.cu)
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const double d = D[k][k];
        rs[k] = (d > 0.0) ? fast_rsqrt(d) : 0.0;       // non-positive pivot: zero column, like LDLT's D^+ = 0
#pragma unroll
        for (int i = k; i < 8; ++i) D[i][k] *= rs[k];
#pragma unroll
        for (int i = k + 1; i < 8; ++i) {
#pragma unroll
          for (int j = k + 1; j <= i; ++j) D[i][j] -= D[i][k] * D[j][k];
        }
      }
      // W = L^-1 by forward substitution on the identity, column by column
      double W[8][8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        W[j][j] = rs[j];
#pragma unroll
        for (int i = j + 1; i < 8; ++i) {
          double sacc = 0.0;
#pragma unroll
          for (int m = j; m < i; ++m) sacc += D[i][m] * W[m][j];
          W[i][j] = -sacc * rs[i];
        }
      }
      // publish W (lower part; the upper part was cleared during assembly): every lane holds every entry, so the
      // stores are warp-uniform with compile-time addresses (a lane-dependent selection of registers costs 1,400 cycles)
      double *wt = sm.winv + (size_t)s * 64;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
#pragma unroll
        for (int c = 0; c <= r; c += 2)
          *reinterpret_cast<double2 *>(wt + r * 8 + (c ^ ((r & 2) << 1))) = make_double2(W[r][c], (c + 1 <= r) ? W[r][c + 1] : 0.0);
      }
      asm volatile("bar.arrive %0, %1;" ::"n"(kNdBarA), "n"(kNdCntA) : "memory");
      if (timing && lane == 0 && nd.parent < 0) {    // root front: cycles waiting for the look-ahead warp / working
        g_nd_dbg[8] += (unsigned long long)(c1 - c0);
        g_nd_dbg[15] += (unsigned long long)(clock64() - c1);
      }
    }
  } else {
    // ---------------------------------------------- consumers ----------------------------------------------
    // L_Is = A_Is W^T in place (tile (I, s) at `tile`), also to global memory
    auto solve_tile = [&](double *tile, const double *wt, size_t goff) {
      const double a0 = tile[offA0], a1 = tile[offA1];
      const double b0 = wt[offA0], b1 = wt[offA1];
      double2 c = make_double2(0.0, 0.0);
      dmma_884b(c.x, c.y, a0, b0);
      dmma_884b(c.x, c.y, a1, b1);
      __syncwarp();
      *reinterpret_cast<double2 *>(tile + offC) = c;
      *reinterpret_cast<double2 *>(Lg + goff + offC) = c;
    };
    // Row tile I of the trapezoid (tiles (I, J), J <= min(I, KT - 1)) belongs to consumer I mod 9: the panel solve of
    // tile (I, s) and every update of the row stay inside one warp, the operand of the row is loaded once per step
#pragma unroll 1
    for (int s = 0; s < KT; ++s) {
      const double *wt = sm.winv + (size_t)s * 64;
      double *ps = sm.win + (size_t)(colbase(s) - s) * 64;           // tile (I, s) at ps + 64 I
      const size_t gs = (size_t)(colbase(s) - s) * 64;
      asm volatile("bar.sync %0, %1;" ::"n"(kNdBarA), "n"(kNdCntA) : "memory");
      if ((s + 5) % kNdCons == cwi)      // W(s) to global memory (backward passes after the front left shared memory)
        *reinterpret_cast<double2 *>(Wg + (size_t)s * 64 + 2 * lane) = *reinterpret_cast<const double2 *>(wt + 2 * lane);
      // look-ahead: the owner of row s + 1 solves tile (s + 1, s) and finishes the next diagonal tile
      const bool la = (s + 1 < KT) && ((s + 1) % kNdCons == cwi);
      int I0 = s + 1 + ((cwi - (s + 1)) % kNdCons + kNdCons) % kNdCons;   // my first row below the diagonal tile
      if (la) {
        solve_tile(ps + (size_t)(s + 1) * 64, wt, gs + (size_t)(s + 1) * 64);
        __syncwarp();
        double *dn = sm.win + (size_t)colbase(s + 1) * 64 + offC;
        double2 cv = *reinterpret_cast<const double2 *>(dn);
        const double a0 = ps[(size_t)(s + 1) * 64 + offA0], a1 = ps[(size_t)(s + 1) * 64 + offA1];
        dmma_884b(cv.x, cv.y, -a0, a0);
        dmma_884b(cv.x, cv.y, -a1, a1);
        *reinterpret_cast<double2 *>(dn) = cv;
        __syncwarp();
        asm volatile("bar.arrive %0, %1;" ::"n"(kNdBarC), "n"(kNdCntC) : "memory");
        I0 += kNdCons;                                               // row s + 1 is complete
      }
      // rows of [own | Rb] beyond the band of column s hold zeros (no fill reaches them): skipped, zero in global L
      const int rmax = min(NT - 1, s + nd.bandT);
      auto row_live = [&](int I) { return I <= rmax || I >= LbT0; };
      for (int I = I0; I < NT; I += kNdCons) {
        if (row_live(I)) solve_tile(ps + (size_t)I * 64, wt, gs + (size_t)I * 64);
        else *reinterpret_cast<double2 *>(Lg + gs + (size_t)I * 64 + offC) = make_double2(0.0, 0.0);
      }
      asm volatile("bar.sync %0, %1;" ::"n"(kNdBarB), "n"(kNdCntB) : "memory");
      if (helped && cwi == 0 && lane == 0) {      // panel s is solved and in global memory: the helper may take it
        __threadfence();
        nd_st_release(g.flags + g.step_base + nd.step_flag0 + s, 1);
      }
      // trailing update, two rows at a time (they share the column operands), two columns per round
      const int Jlim = min(KT - 1, rmax);                            // live column tiles of the trailing block
      for (int I1 = I0; I1 < NT; I1 += 2 * kNdCons) {
        const int I2 = I1 + kNdCons;
        const bool two = I2 < NT && row_live(I2);
        const int I2c = two ? I2 : I1;
        const int Jm1 = row_live(I1) ? min(I1, Jlim) : -1, Jm2 = two ? min(I2, Jlim) : -1;
        const double a10 = -ps[(size_t)I1 * 64 + offA0], a11 = -ps[(size_t)I1 * 64 + offA1];
        const double a20 = -ps[(size_t)I2c * 64 + offA0], a21 = -ps[(size_t)I2c * 64 + offA1];
        const int Jend = max(Jm1, Jm2);
        for (int J = s + 1; J <= Jend; J += 2) {
          double2 c1[2], c2[2];
          double b0[2], b1[2];
          bool v1[2], v2[2];
          double *p1[2], *p2[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int Ju = min(J + u, KT - 1);
            v1[u] = J + u <= Jm1;
            v2[u] = J + u <= Jm2;
            double *cb = sm.win + (size_t)(colbase(Ju) - Ju) * 64 + offC;
            p1[u] = cb + (size_t)(v1[u] ? I1 : Ju) * 64;
            p2[u] = cb + (size_t)(v2[u] ? I2c : Ju) * 64;
            b0[u] = ps[(size_t)Ju * 64 + offA0];
            b1[u] = ps[(size_t)Ju * 64 + offA1];
            c1[u] = *reinterpret_cast<const double2 *>(p1[u]);
            c2[u] = *reinterpret_cast<const double2 *>(p2[u]);
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            dmma_884b(c1[u].x, c1[u].y, a10, b0[u]);
            dmma_884b(c2[u].x, c2[u].y, a20, b0[u]);
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            dmma_884b(c1[u].x, c1[u].y, a11, b1[u]);
            dmma_884b(c2[u].x, c2[u].y, a21, b1[u]);
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            if (v1[u]) *reinterpret_cast<double2 *>(p1[u]) = c1[u];
            if (v2[u]) *reinterpret_cast<double2 *>(p2[u]) = c2[u];
          }
        }
      }
      // boundary x boundary tiles (registers)
      const double *pB = ps + (size_t)KT * 64;
#pragma unroll
      for (int q = 0; q < TPW; ++q) {
        if (ub[q] >= 0 && row_live(KT + (ub[q] >> 8)) && row_live(KT + (ub[q] & 0xff))) {
          const double *pa = pB + (size_t)(ub[q] >> 8) * 64, *pb = pB + (size_t)(ub[q] & 0xff) * 64;
          const double a0 = -pa[offA0], a1 = -pa[offA1], b0 = pb[offA0], b1 = pb[offA1];
          dmma_884b(acc[q].x, acc[q].y, a0, b0);
          dmma_884b(acc[q].x, acc[q].y, a1, b1);
        }
      }
    }
    // ---- contribution block: my Schur complement, scattered into the layout of my parent's front (own-column tiles
    //      swizzled like its shared-memory window, then its boundary x boundary tiles)
    if (nd.parent >= 0 && !helped) {
      double *Ug = g.Uws + nd.U_off;
      const int KTp = sm.par->k8 >> 3, NTp = (sm.par->k8 + sm.par->b8) >> 3, k8p = sm.par->k8;
      const int ntp = KTp * NTp - (KTp * (KTp - 1)) / 2;
#pragma unroll
      for (int q = 0; q < TPW; ++q) {
        if (ub[q] < 0) continue;
        const int bi = 8 * (ub[q] >> 8) + fr, bj0 = 8 * (ub[q] & 0xff) + fc;
        const int pi = sm.pm[bi];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int bj = bj0 + e;
          if (bj > bi || pi < 0) continue;                  // upper half of a diagonal tile / padding rows
          const int pj = sm.pm[bj];
          if (pj < 0) continue;
          const int a = max(pi, pj), b = min(pi, pj);
          const double v = e ? acc[q].y : acc[q].x;
          if (b < k8p) {
            const int I = a >> 3, J = b >> 3;
            Ug[(size_t)(J * NTp - (J * (J - 1)) / 2 + I - J) * 64 + nd_sw(a & 7, b & 7)] = v;
          } else {
            Ug[((size_t)ntp + nd_tidx((a - k8p) >> 3, (b - k8p) >> 3)) * 64 + ((a - k8p) & 7) * 8 + ((b - k8p) & 7)] = v;
          }
        }
      }
    }
  }
  __syncthreads();
  if (timing && t == 0) {
    const unsigned long long t1 = gtime();
    atomicAdd(&g_nd_dbg[2 + min(nd.level, 6)], t1 - t0);
    if (blockIdx.x == 0) g_nd_dbg[11] += t1 - t0;
  }
}

// ------------------------------------------------------------------------------------------------------------
// backward substitution of one front: x_own from x_boundary
// ------------------------------------------------------------------------------------------------------------
// factor of a front that has left shared memory: node record, tiles and W blocks from global memory
__device__ void nd_backward_load(const NdArgs &g, const NdSmem &sm, int node_id) {
  const int t = threadIdx.x;
  __syncthreads();
  nd_stage_node(g, sm, node_id, false);
  const NdNode &nd = *sm.node;
  const int KT = nd.k8 >> 3, BT = nd.b8 >> 3, NT = KT + BT;
  const int n_tiles = KT * NT - (KT * (KT - 1)) / 2;
  const double2 *src = reinterpret_cast<const double2 *>(g.Lws + nd.L_off);
  double2 *dw = reinterpret_cast<double2 *>(sm.win), *di = reinterpret_cast<double2 *>(sm.winv);
  const int nw = n_tiles * 32, ni = KT * 32;
  for (int e = t; e < nw; e += kNdThreads) dw[e] = __ldcg(src + e);
  for (int e = t; e < ni; e += kNdThreads) di[e] = __ldcg(src + nw + e);
  __syncthreads();
}

// sm.node, sm.win and sm.winv hold the front
__device__ void nd_backward_solve(const NdArgs &g, const NdSmem &sm) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const NdNode &nd = *sm.node;
  const int KT = nd.k8 >> 3, BT = nd.b8 >> 3, NT = KT + BT, R8 = 8 * NT, k8 = nd.k8;
  auto colbase = [&](int J) { return J * NT - (J * (J - 1)) / 2; };
  for (int i = t; i < R8; i += kNdThreads) {
    double v = 0.0;
    const int bi = i - k8;
    if (bi >= 0) {
      if (bi < nd.wr) v = __ldcg(g.x + nd.rb0 + bi);
      else if (bi < nd.wr + nd.wl) v = __ldcg(g.x + nd.lb0 + (bi - nd.wr));
      else if (bi == nd.wr + nd.wl) v = -1.0;
    }
    sm.xs[i] = v;
  }
  __syncthreads();
  // boundary part: tb[c] = sum_{r >= k8} L[r][c] xs[r]   (warp per column tile; lane = column + 8 (row mod 4))
  {
    const int cc = lane & 7, rg = lane >> 3;
    const int o0 = nd_sw(rg, cc), o1 = nd_sw(rg + 4, cc);
    for (int J = warp; J < KT; J += kNdWarps) {
      const double *col = sm.win + (size_t)(colbase(J) - J) * 64;   // tile (I, J) at col + 64 I
      double p0 = 0.0, p1 = 0.0;
      for (int I = KT; I < NT; ++I) {
        p0 += col[(size_t)I * 64 + o0] * sm.xs[8 * I + rg];
        p1 += col[(size_t)I * 64 + o1] * sm.xs[8 * I + rg + 4];
      }
      double p = p0 + p1;
      p += __shfl_xor_sync(0xffffffffu, p, 8);
      p += __shfl_xor_sync(0xffffffffu, p, 16);
      if (rg == 0) sm.tb[8 * J + cc] = p;
    }
  }
  __syncthreads();
  // block chain inside warp 0: x_s = -W_s^T tb_s, then tb[c] += L[8 s + q][c] x_q for the columns left of it
  if (warp == 0) {
    for (int s = KT - 1; s >= 0; --s) {
      const double *wt = sm.winv + (size_t)s * 64;
      if (lane < 8) {
        double xa = 0.0, xb = 0.0;
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
          xa += (i >= lane) ? wt[nd_sw(i, lane)] * sm.tb[8 * s + i] : 0.0;
          xb += (i + 1 >= lane) ? wt[nd_sw(i + 1, lane)] * sm.tb[8 * s + i + 1] : 0.0;
        }
        sm.xs[8 * s + lane] = -(xa + xb);
      }
      __syncwarp();
      double xq[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) xq[q] = sm.xs[8 * s + q];
      for (int c = lane; c < 8 * s; c += 32) {
        const int J = c >> 3, cj = c & 7;
        const double *Lt = sm.win + (size_t)(colbase(J) + s - J) * 64;   // tile (s, J)
        double u = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) u += Lt[nd_sw(q, cj)] * xq[q];
        sm.tb[c] += u;
      }
      __syncwarp();
    }
  }
  __syncthreads();
  for (int j = t; j < nd.k; j += kNdThreads) g.x[nd.own0 + j] = sm.xs[j];
}

// ------------------------------------------------------------------------------------------------------------
// drivers
// ------------------------------------------------------------------------------------------------------------
template <int TPW, int NC>
__global__ void __launch_bounds__(kNdThreads, 1)
k_nd_forward_level(NdArgs g, int list_begin, int timing, const LmState *st) {
  if (st->done) return;
  extern __shared__ __align__(16) unsigned char nd_raw[];
  const NdSmem sm = nd_carve(nd_raw, g);
  nd_forward_prepare(g, sm, g.list[list_begin + blockIdx.x]);
  nd_forward_node<TPW, NC>(g, sm, g.list[list_begin + blockIdx.x], timing);
}

__global__ void __launch_bounds__(kNdThreads, 1)
k_nd_backward_level(NdArgs g, int list_begin, const LmState *st) {
  if (st->done) return;
  extern __shared__ __align__(16) unsigned char nd_raw[];
  const NdSmem sm = nd_carve(nd_raw, g);
  nd_backward_load(g, sm, g.list[list_begin + blockIdx.x]);
  nd_backward_solve(g, sm);
}

// thread 0 spins (bounded: a lost hand-over must not hang the device), everybody follows through the barrier
__device__ __forceinline__ void nd_wait_flag(const NdArgs &g, int idx) {
  if (threadIdx.x == 0) {
    int it = 0;
    while (nd_ld_acquire(g.flags + idx) == 0) {
      if (++it > kNdSpinLimit || nd_ld_acquire(g.flags + g.abort_idx) != 0) {
        atomicExch(g.flags + g.abort_idx, 1);         // abort this launch
        atomicExch(g.flags + g.abort_idx + 1, 1);     // sticky: reported by the host (never cleared by the launch)
        break;
      }
      __nanosleep(20);
    }
  }
  __syncthreads();
}
__device__ __forceinline__ void nd_set_flag(const NdArgs &g, int idx) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    nd_st_release(g.flags + idx, 1);
  }
}

// Helper CTA of a large front: holds the boundary x boundary accumulators (12 warps x TPW tiles), follows the main
// CTA panel by panel (per-step flags), reads the solved boundary tiles of every panel from the factor in global memory
// and scatters the finished Schur complement into the parent's layout.  It -- not the main CTA -- sets the front's
// forward flag.
template <int TPW>
__device__ void nd_helper_node(const NdArgs &g, const NdSmem &sm, int node_id) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  nd_forward_prepare(g, sm, node_id, false);
  const NdNode &nd = *sm.node;
  for (int c = 0; c < 2; ++c)
    if (nd.child[c] >= 0) nd_wait_flag(g, nd.child[c]);
  const int KT = nd.k8 >> 3, BT = nd.b8 >> 3, NT = KT + BT;
  auto colbase = [&](int J) { return J * NT - (J * (J - 1)) / 2; };
  const int n_tiles = colbase(KT);
  const int LbT0 = (nd.k8 + nd.wr) >> 3;
  const int fr = lane >> 2, fc = 2 * (lane & 3), kq = lane & 3;
  const int swz = (fr & 2) << 1;
  const int offA0 = fr * 8 + (kq ^ swz), offA1 = offA0 ^ 4, offU = fr * 8 + fc;
  const double *U0 = nd.child[0] >= 0 ? g.Uws + sm.cn[0].U_off : nullptr;
  const double *U1 = nd.child[1] >= 0 ? g.Uws + sm.cn[1].U_off : nullptr;
  const int n_utiles = BT * (BT + 1) / 2;
  double2 acc[TPW];
  int ub[TPW];
#pragma unroll
  for (int q = 0; q < TPW; ++q) {
    acc[q] = make_double2(0.0, 0.0);
    ub[q] = -1;
    const int e = warp + kNdWarps * q;
    if (e < n_utiles) {
      int I = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
      while (I * (I + 1) / 2 > e) --I;
      while ((I + 1) * (I + 2) / 2 <= e) ++I;
      ub[q] = (I << 8) | (e - I * (I + 1) / 2);
      const size_t off = ((size_t)n_tiles + e) * 64 + offU;
      const double2 a = U0 ? __ldcg(reinterpret_cast<const double2 *>(U0 + off)) : make_double2(0.0, 0.0);
      const double2 b = U1 ? __ldcg(reinterpret_cast<const double2 *>(U1 + off)) : make_double2(0.0, 0.0);
      acc[q] = make_double2(a.x + b.x, a.y + b.y);
    }
  }
  const double *Lg = g.Lws + nd.L_off;
  double *panel = sm.win;                       // [2][BT][64]
#pragma unroll 1
  for (int s = 0; s < KT; ++s) {
    nd_wait_flag(g, g.step_base + nd.step_flag0 + s);
    double *pb = panel + (size_t)(s & 1) * BT * 64;
    const double2 *src = reinterpret_cast<const double2 *>(Lg + (size_t)(colbase(s) - s + KT) * 64);   // tiles (KT .. NT-1, s)
    for (int e = t; e < BT * 32; e += kNdThreads) reinterpret_cast<double2 *>(pb)[e] = __ldcg(src + e);
    __syncthreads();
    const int rmax = min(NT - 1, s + nd.bandT);
#pragma unroll
    for (int q = 0; q < TPW; ++q) {
      if (ub[q] < 0) continue;
      const int ra = KT + (ub[q] >> 8), rb = KT + (ub[q] & 0xff);
      if (!((ra <= rmax || ra >= LbT0) && (rb <= rmax || rb >= LbT0))) continue;
      const double *pa = pb + (size_t)(ub[q] >> 8) * 64, *pc = pb + (size_t)(ub[q] & 0xff) * 64;
      const double a0 = -pa[offA0], a1 = -pa[offA1], b0 = pc[offA0], b1 = pc[offA1];
      dmma_884b(acc[q].x, acc[q].y, a0, b0);
      dmma_884b(acc[q].x, acc[q].y, a1, b1);
    }
  }
  // Schur complement into the parent's layout (same scatter as nd_forward_node)
  {
    double *Ug = g.Uws + nd.U_off;
    const int KTp = sm.par->k8 >> 3, NTp = (sm.par->k8 + sm.par->b8) >> 3, k8p = sm.par->k8;
    const int ntp = KTp * NTp - (KTp * (KTp - 1)) / 2;
#pragma unroll
    for (int q = 0; q < TPW; ++q) {
      if (ub[q] < 0) continue;
      const int bi = 8 * (ub[q] >> 8) + fr, bj0 = 8 * (ub[q] & 0xff) + fc;
      const int pi = sm.pm[bi];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int bj = bj0 + e;
        if (bj > bi || pi < 0) continue;
        const int pj = sm.pm[bj];
        if (pj < 0) continue;
        const int a = max(pi, pj), b = min(pi, pj);
        const double v = e ? acc[q].y : acc[q].x;
        if (b < k8p) {
          const int I = a >> 3, J = b >> 3;
          Ug[(size_t)(J * NTp - (J * (J - 1)) / 2 + I - J) * 64 + nd_sw(a & 7, b & 7)] = v;
        } else {
          Ug[((size_t)ntp + nd_tidx((a - k8p) >> 3, (b - k8p) >> 3)) * 64 + ((a - k8p) & 7) * 8 + ((b - k8p) & 7)] = v;
        }
      }
    }
  }
  nd_set_flag(g, node_id);
}

// One launch: every CTA walks its list of fronts forward (children first) and then backward; a front whose child
// (forward) or parent (backward) belongs to another CTA waits for that CTA's flag.  The flags are cleared by a
// memset node that precedes the launch.  Requires all CTAs to be co-resident (grid <= SM count, one CTA per SM).
template <int TPW, int NC>
__global__ void __launch_bounds__(kNdThreads, 1)
k_nd_persistent(NdArgs g, int timing, const LmState *st) {
  if (st->done) return;
  extern __shared__ __align__(16) unsigned char nd_raw[];
  const NdSmem sm = nd_carve(nd_raw, g);
  if ((int)blockIdx.x >= g.n_main) {      // helper CTA: one front's boundary x boundary block, forward pass only
    nd_helper_node<TPW>(g, sm, g.helper_list[blockIdx.x - g.n_main]);
    return;
  }
  const int lb = g.list_ptr[blockIdx.x], le = g.list_ptr[blockIdx.x + 1];
  const int me = blockIdx.x;
  unsigned long long t0 = 0;
  if (timing && threadIdx.x == 0) t0 = gtime();
  for (int q = lb; q < le; ++q) {
    const int id = g.list[q];
    unsigned long long tw = 0;
    nd_forward_prepare(g, sm, id);       // records and tables while the children are still working
    if (timing && threadIdx.x == 0) tw = gtime();
    for (int c = 0; c < 2; ++c) {
      const int ch = sm.node->child[c];
      if (ch >= 0 && (sm.cn[c].cta != me || sm.cn[c].helper >= 0)) nd_wait_flag(g, ch);   // another CTA or a helper finishes it
    }
    if (timing && threadIdx.x == 0 && blockIdx.x == 0) g_nd_dbg[9] += gtime() - tw;
    nd_forward_node<TPW, NC>(g, sm, id, timing);
    if (timing && threadIdx.x == 0) tw = gtime();
    if (sm.node->helper < 0) nd_set_flag(g, id);        // a helped front is complete when its helper says so
    if (timing && threadIdx.x == 0 && blockIdx.x == 0) g_nd_dbg[12] += gtime() - tw;
  }
  if (timing && threadIdx.x == 0 && blockIdx.x == 0) g_nd_dbg[0] = gtime() - t0;
  for (int q = le - 1; q >= lb; --q) {
    const int id = g.list[q];
    if (q != le - 1) nd_backward_load(g, sm, id);     // the last front of the list is still resident
    const int parent = g.nodes[id].parent;
    if (parent >= 0 && g.nodes[parent].cta != me) nd_wait_flag(g, g.n_nodes + parent);
    nd_backward_solve(g, sm);
    nd_set_flag(g, g.n_nodes + id);
  }
  if (timing && threadIdx.x == 0 && blockIdx.x == 0) g_nd_dbg[1] = gtime() - t0;
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
struct NdDevice {
  NdArgs level_args{}, cta_args{};
  size_t smem = 0;
  int tpw = 0;
};

// consumer warps and accumulator tiles per consumer warp for fronts with up to BT boundary row tiles
inline int nd_cons_for(int BT) { return BT >= 12 ? 11 : 9; }
inline int nd_tpw_for(int BT) {
  const int nc = nd_cons_for(BT);
  const int need = (BT * (BT + 1) / 2 + nc - 1) / nc;
  const int opts9[] = {4, 8}, opts11[] = {8, 12, 14, 19, 24};
  if (nc == 9) {
    for (int o : opts9)
      if (need <= o) return o;
  } else {
    for (int o : opts11)
      if (need <= o) return o;
  }
  return -1;
}

template <int TPW, int NC>
inline bool nd_enqueue_t(const NdPlan &pl, const NdDevice &dv, const double *Saug, double *x, bool persistent, int timing,
                         const LmState *st, cudaStream_t stream, long long *launches) {
  static PerDeviceOnce once;
  if (once.first()) {
    cudaFuncSetAttribute(k_nd_forward_level<TPW, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNdSmemLimit);
    cudaFuncSetAttribute(k_nd_persistent<TPW, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNdSmemLimit);
    cudaFuncSetAttribute(k_nd_backward_level, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNdSmemLimit);
  }
  if (persistent) {
    cudaMemsetAsync(dv.cta_args.flags, 0, (size_t)(dv.cta_args.abort_idx + 1) * sizeof(int), stream);
    NdArgs a = dv.cta_args;
    a.S = Saug; a.x = x;
    void *args[] = {(void *)&a, (void *)&timing, (void *)&st};
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(pl.n_ctas + pl.n_helpers);
    cfg.blockDim = dim3(kNdThreads);
    cfg.dynamicSmemBytes = dv.smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelExC(&cfg, (const void *)k_nd_persistent<TPW, NC>, args);
    if (e == cudaSuccess) {
      if (launches) *launches += 1;
      return true;
    }
    // The cooperative launch guarantees that all CTAs are co-resident (the hand-over flags need it).  When it is
    // refused (device shared with another process, fewer SMs than the plan's CTAs) the per-level launches below do
    // the same work without any cross-CTA waiting.
    cudaGetLastError();
  }
  NdArgs la = dv.level_args;
  la.S = Saug; la.x = x;
  for (int l = 0; l < pl.n_levels; ++l) {
    const int cnt = pl.level_ptr[l + 1] - pl.level_ptr[l];
    k_nd_forward_level<TPW, NC><<<cnt, kNdThreads, dv.smem, stream>>>(la, pl.level_ptr[l], timing, st);
  }
  for (int l = pl.n_levels - 1; l >= 0; --l) {
    const int cnt = pl.level_ptr[l + 1] - pl.level_ptr[l];
    k_nd_backward_level<<<cnt, kNdThreads, dv.smem, stream>>>(la, pl.level_ptr[l], st);
  }
  if (launches) *launches += 2 * pl.n_levels;
  return cudaGetLastError() == cudaSuccess;
}

// persistent: one cooperative launch over all fronts (the per-level launches if it is refused); else one launch per level
inline bool nd_enqueue(const NdPlan &pl, const NdDevice &dv, const double *Saug, double *x, bool persistent, int timing,
                       const LmState *st, cudaStream_t stream, long long *launches) {
  if (nd_cons_for(pl.max_BT) == 9) {
    switch (dv.tpw) {
      case 4: return nd_enqueue_t<4, 9>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
      case 8: return nd_enqueue_t<8, 9>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
      default: return false;
    }
  }
  switch (dv.tpw) {
    case 8: return nd_enqueue_t<8, 11>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
    case 12: return nd_enqueue_t<12, 11>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
    case 14: return nd_enqueue_t<14, 11>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
    case 19: return nd_enqueue_t<19, 11>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
    case 24: return nd_enqueue_t<24, 11>(pl, dv, Saug, x, persistent, timing, st, stream, launches);
    default: return false;
  }
}

}  // namespace ba
