// ba_engine.cu -- B200 (sm_100a) full bundle-adjustment engine behind the C-ABI of include/ba_b200.h.
//
// Device pipeline of one LM iteration (reference: core/full_bundle_adjustment_solver.cpp:709-1008); six launches on
// one GPU for a sequential trajectory (C3 / C4), replayed as a CUDA graph:
//   K2 pose side            : the sums A (21) / a (6) per pose come from the trial-cost pass of the previous iteration
//                             (K7; speculative, Au[parameter buffer]; per-observation Jacobians in pose order, per-chunk
//                             partials, ordered per-pose sum in the pose's last chunk, :795-810, :833-844, :878-888);
//                             damped and stored at the start of the iteration by the storing form of k_tile_reduce
//                             (banded plans) or k_pose_diag.  ba_solve's initial cost and ba_build_only run the same
//                             pass at the accepted parameters first
//   K1b+K3+K4 k_build_tiles : landmarks whose poses fit a 16-pose window (ba_build_tiles.cuh): linearisation, C, b,
//      + k_tile_reduce        B (last-writer rule), damping + pivoted 3x3 LDLT inverse, E = B C^-1 and the Schur
//                             products S -= E B^T as an FP64 tensor-core GEMM, fused (:716-831, :846-856, :858-888);
//                             windows flushed into private staging segments and added into S in segment order
//   K1a/K3/K4 by-point path : everything else -- k_linearize_by_point (C, b), k_pair_blocks (B), k_finish_points
//                             (C^-1), then k_schur_dense_gemm (small reduced systems: dense DMMA GEMM) or
//                             k_schur_pairs_list (FP64 reds)
//   K5 cholesky_solve       : FP64 Cholesky of S with the rhs carried along (:890-908): partitioned banded
//                             (k_nd_persistent, nested-dissection fronts over many CTAs, ba_cholesky_nd.cuh), cluster
//                             (small dense, ba_cholesky_cluster.cuh), multi-kernel blocked DMMA (large dense,
//                             ba_cholesky.cuh); the serial window kernel of ba_cholesky_banded.cuh is the fallback
//   K6 k_backsub_tiles / k_backsub_pairs, k_backsub_points_update_poses : y = C^-1 b - C^-1 sum_j B^T x_j (tile
//                             landmarks: B formed again from their observations, ba_build_tiles.cuh; by-point landmarks:
//                             the stored B), model change, trial points
//                             (:910-917,:435-455) and, in the same launch, the se3Exp pose update (:922-927);
//                             gradient-descent variant for FullBundleAdjustmentSolverRefactor::SolveByGradientDescent
//   K7 k_cost_linearize_by_pose : trial cost in pose order + the pose-side sums at the trial parameters; the last CTA
//                             sums the partials in order and takes the rho / accept / lambda / convergence decision
//                             on the device (:930-1007)
// Outside the loop, k_obs_residuals (ba_observation_residuals) reports the residual and an inlier / outlier / behind-
// camera status of every observation row at the accepted parameters, for callers that reject outliers between solves.
// Multi-GPU: landmarks sharded; the band of [S | rhs] is exchanged through peer memory (one-shot pushes + epoch flags,
// summed in rank order; NCCL all-reduce as the fallback), the five LM scalars by k_exchange_decide.
// There is no CPU fallback: every entry point that computes requires a CUDA device.
// The A/B and diagnostic switches (BA_B200_*, DESIGN §4.0) are read from the environment once per solver, by ba_create
// (read_switches); the reduced solve a plan runs is chosen once, in upload_cholesky_plan (CholeskyPlan::path).
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <stdint.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <condition_variable>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/ba_b200.h"
#include "ba_cholesky.cuh"
#include "ba_device.cuh"

namespace ba {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kPtBlk = 18;  // per-point SoA rows: b(3) Cd(6) Cinv(6) Cinv_b(3)
constexpr int PB_b = 0, PB_Cd = 3, PB_Cinv = 9, PB_Cinvb = 15;

struct ChunkA {  // by-pose chunk: one free pose per chunk
  int obs_start;
  int obs_count;
  int j_opt;
  int _pad;
};

// parameter double buffer
struct Params {
  const double *poses[2];  // [N_total*12]
  const double *points[2]; // [M_total*3]
};
struct ParamsW {
  double *poses[2];
  double *points[2];
};

// ---------------------------------------------------------------------------
// K1: linearise in point order.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void finish_point(const double *Craw, const double *braw, double lambda,
                                             double *__restrict__ ptblk, size_t Mp, int pt) {
  // fill-lower is implicit (symmetric 6-pack); damping (:850-852); Cinv = ldlt().solve(I) (:854)
  const double lp1 = 1.0 + lambda;
  double cd[6] = {Craw[0] * lp1, Craw[1], Craw[2], Craw[3] * lp1, Craw[4], Craw[5] * lp1};
  double inv[9];
  ldlt3_inverse(cd, inv);
  const double cb0 = inv[0] * braw[0] + inv[1] * braw[1] + inv[2] * braw[2];
  const double cb1 = inv[3] * braw[0] + inv[4] * braw[1] + inv[5] * braw[2];
  const double cb2 = inv[6] * braw[0] + inv[7] * braw[1] + inv[8] * braw[2];
  ptblk[(PB_b + 0) * Mp + pt] = braw[0];
  ptblk[(PB_b + 1) * Mp + pt] = braw[1];
  ptblk[(PB_b + 2) * Mp + pt] = braw[2];
#pragma unroll
  for (int k = 0; k < 6; ++k) ptblk[(PB_Cd + k) * Mp + pt] = cd[k];
  // the LDLT inverse is symmetric up to rounding; keep the upper triangle (r<=c) of the row-major result
  ptblk[(PB_Cinv + 0) * Mp + pt] = inv[0];
  ptblk[(PB_Cinv + 1) * Mp + pt] = inv[1];
  ptblk[(PB_Cinv + 2) * Mp + pt] = inv[2];
  ptblk[(PB_Cinv + 3) * Mp + pt] = inv[4];
  ptblk[(PB_Cinv + 4) * Mp + pt] = inv[5];
  ptblk[(PB_Cinv + 5) * Mp + pt] = inv[8];
  ptblk[(PB_Cinvb + 0) * Mp + pt] = cb0;
  ptblk[(PB_Cinvb + 1) * Mp + pt] = cb1;
  ptblk[(PB_Cinvb + 2) * Mp + pt] = cb2;
}

struct ChunkPoint {  // one landmark inside a point-order chunk
  int point;        // original landmark id
  int local_start;  // first observation slot inside the chunk
  int len;          // observations of the landmark inside the chunk
  int free;         // landmark is optimised
};

constexpr int kValsLd = kThreads + 1;  // padded row of the per-observation staging in shared memory

// 96-byte pose gather as six 16-byte loads
__device__ __forceinline__ void load_pose(const double *__restrict__ Tp, double *T) {
  const double2 *p2 = reinterpret_cast<const double2 *>(Tp);
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const double2 v = __ldg(p2 + i);
    T[2 * i] = v.x;
    T[2 * i + 1] = v.y;
  }
}

// K1a: landmark side (C, b, then damping + inverse).  One thread per observation of a chunk of whole
// landmarks; the 9 per-observation terms are staged in shared memory and summed per landmark by 9 threads
// (one per component) walking the landmark's contiguous run.
__global__ void __launch_bounds__(kThreads, 3)
k_linearize_by_point(const Chunk *__restrict__ chunks, const int2 *__restrict__ chunk_pts /*first, count*/,
                     const ChunkPoint *__restrict__ cpts, const double2 *__restrict__ obs_uv,
                     const int *__restrict__ obs_pose, const int *__restrict__ obs_point,
                     const int *__restrict__ obs_camflags, Params prm, const double *__restrict__ cams,
                     double thres_huber, double *__restrict__ ptblk, size_t Mp,
                     const LmState *__restrict__ st) {
  if (st->done) return;
  __shared__ double vals[9][kValsLd];
  __shared__ double sums[kThreads][9];  // a chunk holds at most kThreads landmarks
  const Chunk ch = chunks[blockIdx.x];
  const int2 cp = chunk_pts[blockIdx.x];
  const int t = threadIdx.x;
  const int k = ch.obs_start + t;
  const double *poses = prm.poses[st->cur];
  const double *points = prm.points[st->cur];
  double v[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) v[i] = 0.0;
  if (t < ch.obs_count) {
    const int cf = obs_camflags[k];
    if (cf & kFlagPointFree) {
      const int pt = obs_point[k];
      const double2 uv = obs_uv[k];
      double T[12], X[3];
      load_pose(poses + (size_t)obs_pose[k] * 12, T);
      X[0] = __ldg(points + (size_t)pt * 3);
      X[1] = __ldg(points + (size_t)pt * 3 + 1);
      X[2] = __ldg(points + (size_t)pt * 3 + 2);
      const double *cam = cams + (cf & kCamMask) * kCamStride;
      Proj p;
      project(T, X, cam, uv.x, uv.y, p);
      const double w = huber_weight(p.r0, p.r1, thres_huber);
      const double wr0 = w * p.r0, wr1 = w * p.r1;
      double G[6], Rm[6];
      jac_G(p, cam, G);
      jac_R(G, T, Rm);
      // C_i(upper) += w Rm^T Rm (:503-517,821) ; b_i -= Rm^T (w r) (:823)
      v[0] = w * (Rm[0] * Rm[0] + Rm[3] * Rm[3]);
      v[1] = w * (Rm[0] * Rm[1] + Rm[3] * Rm[4]);
      v[2] = w * (Rm[0] * Rm[2] + Rm[3] * Rm[5]);
      v[3] = w * (Rm[1] * Rm[1] + Rm[4] * Rm[4]);
      v[4] = w * (Rm[1] * Rm[2] + Rm[4] * Rm[5]);
      v[5] = w * (Rm[2] * Rm[2] + Rm[5] * Rm[5]);
      v[6] = -(Rm[0] * wr0 + Rm[3] * wr1);
      v[7] = -(Rm[1] * wr0 + Rm[4] * wr1);
      v[8] = -(Rm[2] * wr0 + Rm[5] * wr1);
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) vals[i][t] = v[i];
  __syncthreads();
  // component sums: thread u -> (landmark p = u / 9, component c = u % 9)
  for (int u = t; u < 9 * cp.y; u += kThreads) {
    const int pidx = u / 9, c = u - 9 * pidx;
    const ChunkPoint q = cpts[cp.x + pidx];
    const double *row = &vals[c][q.local_start];
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int i = 0;
    for (; i + 4 <= q.len; i += 4) { a0 += row[i]; a1 += row[i + 1]; a2 += row[i + 2]; a3 += row[i + 3]; }
    for (; i < q.len; ++i) a0 += row[i];
    sums[pidx][c] = (a0 + a1) + (a2 + a3);
  }
  __syncthreads();
  // raw sums -> ptblk (Cd slots hold the un-damped C until k_finish_points runs); 9 consecutive threads
  // write one landmark
  for (int u = t; u < 9 * cp.y; u += kThreads) {
    const int pidx = u / 9, c = u - 9 * pidx;
    const ChunkPoint q = cpts[cp.x + pidx];
    if (!q.free) continue;
    const int slot = c < 6 ? PB_Cd + c : PB_b + (c - 6);
    if (ch.flags & kChunkSplit) atomicAdd(&ptblk[(size_t)slot * Mp + q.point], sums[pidx][c]);
    else ptblk[(size_t)slot * Mp + q.point] = sums[pidx][c];
  }
}

// K1b: off-diagonal blocks.  One thread per (pose, point) pair: B_ji = w Q^T Rm of the pair's LAST inserted
// observation (reference-exact, full...cpp:826) or the sum over the pair's observations (corrected mode).
// Every lane does useful work and consecutive pairs write consecutive slots of the component-major Bsoa.
// Launched over the by-point pairs, or over every pair (list = null) when the blocks are kept for ba_debug_dump.
template <bool ACCUM_B>
__global__ void __launch_bounds__(kThreads, ACCUM_B ? 2 : 3)
k_pair_blocks(int n_list, const int *__restrict__ list /*pair indices, or null = identity*/,
              const int2 *__restrict__ pair_obs /*first, last observation (point order)*/,
              const double2 *__restrict__ obs_uv, const int *__restrict__ obs_pose,
              const int *__restrict__ obs_point, const int *__restrict__ obs_camflags, Params prm,
              const double *__restrict__ cams, double thres_huber, double *__restrict__ Bsoa, size_t Pp,
              const LmState *__restrict__ st) {
  if (st->done) return;
  const int li = blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= n_list) return;
  const int p = list ? list[li] : li;
  const double *poses = prm.poses[st->cur];
  const double *points = prm.points[st->cur];
  const int2 po = pair_obs[p];
  double Bv[18];
#pragma unroll
  for (int i = 0; i < 18; ++i) Bv[i] = 0.0;
  double T[12], X[3];
  load_pose(poses + (size_t)obs_pose[po.y] * 12, T);
  const int pt = obs_point[po.y];
  X[0] = __ldg(points + (size_t)pt * 3);
  X[1] = __ldg(points + (size_t)pt * 3 + 1);
  X[2] = __ldg(points + (size_t)pt * 3 + 2);
  for (int k = ACCUM_B ? po.x : po.y; k <= po.y; ++k) {
    const double2 uv = obs_uv[k];
    ObsLin o;
    linearize_obs(T, X, cams + (obs_camflags[k] & kCamMask) * kCamStride, uv.x, uv.y, thres_huber, o);
    add_B(o, Bv);
  }
#pragma unroll
  for (int i = 0; i < 18; ++i) Bsoa[(size_t)i * Pp + p] = Bv[i];
}

__global__ void k_zero_split(const int *__restrict__ split_points, int n_split, double *__restrict__ ptblk,
                             size_t Mp, const LmState *st) {
  if (st->done) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_split) {
    const int pt = split_points[i];
    for (int k = 0; k < 9; ++k) ptblk[(size_t)k * Mp + pt] = 0.0;
  }
}

// K3: damping + 3x3 LDLT inverse + C^-1 b for every free landmark (one thread each, coalesced SoA rows)
__global__ void __launch_bounds__(128)
k_finish_points(int M_total, const uint8_t *__restrict__ point_fb /*free landmark on the by-point path*/,
                double *__restrict__ ptblk, size_t Mp, const LmState *st) {
  if (st->done) return;
  const int pt = blockIdx.x * blockDim.x + threadIdx.x;
  if (pt >= M_total || !point_fb[pt]) return;
  double c[6], b[3];
  for (int k = 0; k < 6; ++k) c[k] = ptblk[(PB_Cd + k) * Mp + pt];
  for (int k = 0; k < 3; ++k) b[k] = ptblk[(PB_b + k) * Mp + pt];
  finish_point(c, b, st->lambda, ptblk, Mp, pt);
}

// ---------------------------------------------------------------------------
// K2: the pose side.  The pose-order pass of the trial cost (k_cost_linearize_by_pose, K7) leaves per-chunk partial
// A (upper 21) and a (6); the LAST chunk of a pose to finish (ticket per pose) sums the pose's partials in chunk order
// into Au (a pose without observations keeps its zeros).
// ---------------------------------------------------------------------------
// one warp per free pose.  pose_partial_sum: ordered sum of the pose's chunk partials (lane e < 21: packed upper element
// e of A, lanes 21..26: a).  pose_diag_store: fill-lower, damping, A / a store, S diagonal block and rhs initialisation.
__device__ __forceinline__ double pose_partial_sum(int j, int lane, const int *__restrict__ pose_chunk_ptr,
                                                   const double *partials) {
  double s = 0.0;
  if (lane < 27)
    for (int c = pose_chunk_ptr[j]; c < pose_chunk_ptr[j + 1]; ++c) s += __ldcg(partials + (size_t)c * 27 + lane);
  return s;
}
__device__ __forceinline__ void pose_diag_store(int j, int lane, double s, double *__restrict__ A /*[N][36]*/,
                                                double *__restrict__ a /*[N][6]*/, double *__restrict__ Saug, int ld,
                                                const LmState *st) {
  const double lp1 = 1.0 + st->lambda;
  // lane e<21 holds packed upper element e ; lanes 21..26 hold a.  Scatter to the full 6x6 in two
  // warp-wide rounds (36 entries > 32 lanes); every lane takes part in both shuffles.
#pragma unroll
  for (int round = 0; round < 2; ++round) {
    const int e = lane + 32 * round;
    const int ee = e < 36 ? e : 35;
    const int r = ee / 6, c = ee % 6;
    const int rr = r < c ? r : c, cc = r < c ? c : r;
    const int idx = rr * 6 - rr * (rr - 1) / 2 + (cc - rr);  // packed upper index
    double val = __shfl_sync(0xffffffffu, s, idx);
    if (r == c) val *= lp1;
    if (e < 36) {
      A[(size_t)j * 36 + e] = val;
      Saug[(size_t)(6 * j + r) * ld + 6 * j + c] = val;  // row-major (6j+r, 6j+c)
    }
  }
  if (lane >= 21 && lane < 27) {
    a[(size_t)j * 6 + (lane - 21)] = s;
    Saug[(size_t)(6 * j + (lane - 21)) * ld + (ld - 1)] = s;  // rhs column
  }
}
// Speculative pose side (single launch with the trial cost, k_cost_linearize_by_pose below): the undamped sums of a
// pose (27 values) live in Au[parameter buffer]; at the start of an iteration one warp per free pose damps the sums of
// the ACCEPTED buffer with the current lambda and stores A, a, the S diagonal block and the rhs.
__global__ void k_pose_diag(int N, const double *__restrict__ Au0, const double *__restrict__ Au1,
                            double *__restrict__ A, double *__restrict__ a, double *__restrict__ Saug, int ld,
                            const LmState *__restrict__ st) {
  if (st->done) return;
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= N) return;
  const double *Au = st->cur ? Au1 : Au0;
  const double s = lane < 27 ? Au[(size_t)j * 27 + lane] : 0.0;
  pose_diag_store(j, lane, s, A, a, Saug, ld, st);
}


// ---------------------------------------------------------------------------
// K4: Schur complement  S -= sum_i E_ji B_ki^T (j<=k), rhs_j -= E_ji b_i, E_ji = B_ji Cinv_i  (:858-888).
//
// k_build_tiles (below): landmarks whose observing poses fall inside one window of 16 consecutive free poses:
// linearisation, C^-1 and the Schur products fused, the products as a DMMA GEMM over landmark batches.
// k_schur_pairs_list: landmarks whose poses do not fit a window (wide baselines, loop closures, dense
// co-visibility): one thread per pair, direct FP64 reds.
// ---------------------------------------------------------------------------
struct SchurChunk {
  int pt_start;   // first index into the tile-eligible landmark list
  int pt_count;
  int jmin;       // first free pose (j_opt) of the window
  int width;      // poses actually spanned by the chunk (<= kSchurW): tasks are the width(width+1)/2 pairs
};

constexpr int kTileW = 16;          // widest window (free poses) a tile landmark may span
constexpr int kTileMaxInc = 20;     // incidences per tile landmark (free and fixed poses)

__device__ __forceinline__ void bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// 3x3 symmetric inverse (Eigen LDLT semantics) of the damped block, results in registers
__device__ __forceinline__ void damp_invert(const double *Craw, double lambda, double *cd, double *ci /*6 upper*/) {
  const double lp1 = 1.0 + lambda;
  cd[0] = Craw[0] * lp1; cd[1] = Craw[1]; cd[2] = Craw[2]; cd[3] = Craw[3] * lp1; cd[4] = Craw[4]; cd[5] = Craw[5] * lp1;
  double inv[9];
  ldlt3_inverse(cd, inv);
  ci[0] = inv[0]; ci[1] = inv[1]; ci[2] = inv[2]; ci[3] = inv[4]; ci[4] = inv[5]; ci[5] = inv[8];
}

#include "ba_build_tiles.cuh"

__global__ void __launch_bounds__(128)
k_schur_pairs_list(int n_list, const int *__restrict__ list /*pair indices p1*/,
                   const int *__restrict__ pair_pose, const int *__restrict__ pair_point,
                   const int *__restrict__ pair_end /*index one past the last pair of this pair's point*/,
                   const double *__restrict__ Bsoa, size_t Pp, const double *__restrict__ ptblk, size_t Mp,
                   double *__restrict__ Saug, int ld, const LmState *__restrict__ st) {
  if (st->done) return;
  const int li = blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= n_list) return;
  const int p1 = list[li];
  const int pt = pair_point[p1];
  const int j1 = pair_pose[p1];
  double B1[18];
#pragma unroll
  for (int i = 0; i < 18; ++i) B1[i] = Bsoa[(size_t)i * Pp + p1];
  double ci[6], cb[3];
#pragma unroll
  for (int i = 0; i < 6; ++i) ci[i] = ptblk[(PB_Cinv + i) * Mp + pt];
#pragma unroll
  for (int i = 0; i < 3; ++i) cb[i] = ptblk[(PB_Cinvb + i) * Mp + pt];
  double E[18];
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    const double b0 = B1[r * 3], b1 = B1[r * 3 + 1], b2 = B1[r * 3 + 2];
    E[r * 3 + 0] = b0 * ci[0] + b1 * ci[1] + b2 * ci[2];
    E[r * 3 + 1] = b0 * ci[1] + b1 * ci[3] + b2 * ci[4];
    E[r * 3 + 2] = b0 * ci[2] + b1 * ci[4] + b2 * ci[5];
  }
  // rhs_j -= BCinv b = B (Cinv b) (:864,888)
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    const double g = B1[r * 3] * cb[0] + B1[r * 3 + 1] * cb[1] + B1[r * 3 + 2] * cb[2];
    atomicAdd(&Saug[(size_t)(6 * j1 + r) * ld + (ld - 1)], -g);
  }
  const int pend = pair_end[p1];
  for (int p2 = p1; p2 < pend; ++p2) {
    const int j2 = pair_pose[p2];
    double B2[18];
#pragma unroll
    for (int i = 0; i < 18; ++i) B2[i] = Bsoa[(size_t)i * Pp + p2];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        if (p2 == p1 && c < r) continue;
        const double val = E[r * 3] * B2[c * 3] + E[r * 3 + 1] * B2[c * 3 + 1] + E[r * 3 + 2] * B2[c * 3 + 2];
        atomicAdd(&Saug[(size_t)(6 * j1 + r) * ld + 6 * j2 + c], -val);
      }
  }
}

// ---------------------------------------------------------------------------
// K6: back-substitution.
// ---------------------------------------------------------------------------
// by-point landmarks (the tile landmarks: k_backsub_tiles), per pair: w = B^T x_j ; segmented sum by point -> Btx[pt]
__global__ void __launch_bounds__(kThreads)
k_backsub_pairs(const Chunk *__restrict__ chunks, const int *__restrict__ chunk_pair_count,
                const int *__restrict__ pair_pose, const int *__restrict__ pair_point,
                const double *__restrict__ Bsoa, size_t Pp, const double *__restrict__ x,
                double *__restrict__ Btx /*[3][Mp]*/, size_t Mp, const LmState *__restrict__ st) {
  if (st->done) return;
  __shared__ SegSmem<3, kWarps> sm3;
  const Chunk ch = chunks[blockIdx.x];
  const int cnt = chunk_pair_count[blockIdx.x];
  const int t = threadIdx.x;
  const bool active = t < cnt;
  const int p = ch.pair_start + t;
  double v[3] = {0.0, 0.0, 0.0};
  int pt = -1 - t;
  if (active) {
    pt = pair_point[p];
    const double *xj = x + (size_t)pair_pose[p] * 6;
    double xv[6];
#pragma unroll
    for (int r = 0; r < 6; ++r) xv[r] = __ldg(xj + r);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      double s = 0.0;
#pragma unroll
      for (int r = 0; r < 6; ++r) s += Bsoa[(size_t)(r * 3 + c) * Pp + p] * xv[r];
      v[c] = s;
    }
  }
  const bool head = !active || t == 0 || pair_point[p - 1] != pt;
  const bool tail = active && (t == cnt - 1 || pair_point[p + 1] != pt);
  block_segmented_sum<3, kWarps>(v, head, tail, sm3);
  if (tail) {
    if (ch.flags & kChunkSplit) {
      for (int c = 0; c < 3; ++c) atomicAdd(&Btx[(size_t)c * Mp + pt], v[c]);
    } else {
      for (int c = 0; c < 3; ++c) Btx[(size_t)c * Mp + pt] = v[c];
    }
  }
}

// per point: y = Cinv_b - Cinv Btx (:916) ; model terms b.y + y^T C y + 2 y.Btx (:443-452) ;
// |y| ; trial point X + y (:498).  Partials per block: {model, step}.
__device__ __forceinline__ void backsub_points_body(int blk, int M_total, const int *__restrict__ point_has_pairs,
                                                    const uint8_t *__restrict__ point_free, const double *__restrict__ ptblk,
                                                    size_t Mp, const double *__restrict__ Btx, double *__restrict__ y,
                                                    const Params &prm, const ParamsW &prw, double *__restrict__ partials,
                                                    int method, const LmState *__restrict__ st) {
  __shared__ double sm[kWarps][2];
  const int i = blk * blockDim.x + threadIdx.x;
  double acc[2] = {0.0, 0.0};
  if (i < M_total) {
    const double *Xc = prm.points[st->cur] + (size_t)i * 3;
    double *Xt = prw.points[st->cur ^ 1] + (size_t)i * 3;
    double yv[3] = {0.0, 0.0, 0.0};
    if (point_free[i] && method == BA_METHOD_GRADIENT_DESCENT) {
      // SolveByGradientDescent (full_bundle_adjustment_solver_refactor.cpp:1277-1283): the step is the gradient
      // block b_i itself, clipped to max_point_step = 0.001
#pragma unroll
      for (int k = 0; k < 3; ++k) yv[k] = ptblk[(PB_b + k) * Mp + i];
      const double nrm = sqrt(yv[0] * yv[0] + yv[1] * yv[1] + yv[2] * yv[2]);
      if (nrm > 0.001) {
        const double sc = 0.001 / nrm;
#pragma unroll
        for (int k = 0; k < 3; ++k) yv[k] = yv[k] * sc;
      }
      acc[1] = sqrt(yv[0] * yv[0] + yv[1] * yv[1] + yv[2] * yv[2]);
    } else if (point_free[i]) {
      double b[3], cd[6], ci[6], cb[3], bx[3] = {0.0, 0.0, 0.0};
#pragma unroll
      for (int k = 0; k < 3; ++k) b[k] = ptblk[(PB_b + k) * Mp + i];
#pragma unroll
      for (int k = 0; k < 6; ++k) cd[k] = ptblk[(PB_Cd + k) * Mp + i];
#pragma unroll
      for (int k = 0; k < 6; ++k) ci[k] = ptblk[(PB_Cinv + k) * Mp + i];
#pragma unroll
      for (int k = 0; k < 3; ++k) cb[k] = ptblk[(PB_Cinvb + k) * Mp + i];
      if (point_has_pairs[i]) {
#pragma unroll
        for (int k = 0; k < 3; ++k) bx[k] = Btx[(size_t)k * Mp + i];
      }
      yv[0] = cb[0] - (ci[0] * bx[0] + ci[1] * bx[1] + ci[2] * bx[2]);
      yv[1] = cb[1] - (ci[1] * bx[0] + ci[3] * bx[1] + ci[4] * bx[2]);
      yv[2] = cb[2] - (ci[2] * bx[0] + ci[4] * bx[1] + ci[5] * bx[2]);
      const double by = b[0] * yv[0] + b[1] * yv[1] + b[2] * yv[2];
      const double c0 = cd[0] * yv[0] + cd[1] * yv[1] + cd[2] * yv[2];
      const double c1 = cd[1] * yv[0] + cd[3] * yv[1] + cd[4] * yv[2];
      const double c2 = cd[2] * yv[0] + cd[4] * yv[1] + cd[5] * yv[2];
      const double ycy = yv[0] * c0 + yv[1] * c1 + yv[2] * c2;
      const double ybx = yv[0] * bx[0] + yv[1] * bx[1] + yv[2] * bx[2];
      acc[0] = by + ycy + 2.0 * ybx;
      acc[1] = sqrt(yv[0] * yv[0] + yv[1] * yv[1] + yv[2] * yv[2]);
    }
    y[(size_t)i * 3] = yv[0];
    y[(size_t)i * 3 + 1] = yv[1];
    y[(size_t)i * 3 + 2] = yv[2];
    Xt[0] = Xc[0] + yv[0];
    Xt[1] = Xc[1] + yv[1];
    Xt[2] = Xc[2] + yv[2];
  }
  block_sum<2, kWarps>(acc, sm);
  if (threadIdx.x == 0) {
    partials[(size_t)blk * 2] = acc[0];
    partials[(size_t)blk * 2 + 1] = acc[1];
  }
}

// SolveByGradientDescent, pose side (full_bundle_adjustment_solver_refactor.cpp:1274-1276): x_j = a_j clipped to
// max_pose_step = 0.001
__global__ void k_gd_poses(int N, const double *__restrict__ a, double *__restrict__ x, const LmState *__restrict__ st) {
  if (st->done) return;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  double v[6], s2 = 0.0;
#pragma unroll
  for (int k = 0; k < 6; ++k) { v[k] = a[(size_t)j * 6 + k]; s2 += v[k] * v[k]; }
  const double nrm = sqrt(s2);
  const double sc = (nrm > 0.001) ? 0.001 / nrm : 1.0;
#pragma unroll
  for (int k = 0; k < 6; ++k) x[(size_t)j * 6 + k] = (nrm > 0.001) ? v[k] * sc : v[k];
}

// ---------------------------------------------------------------------------
// K7: pose update + pose part of the model change; trial cost; decision.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void update_poses_body(int blk, int N_total, const int *__restrict__ pose_opt,
                                                  const double *__restrict__ x, const double *__restrict__ A,
                                                  const double *__restrict__ a, const Params &prm, const ParamsW &prw,
                                                  double *__restrict__ partials, const LmState *__restrict__ st) {
  __shared__ double sm[kWarps][2];
  const int jt = blk * blockDim.x + threadIdx.x;
  double acc[2] = {0.0, 0.0};
  if (jt < N_total) {
    const double *Tc = prm.poses[st->cur] + (size_t)jt * 12;
    double *Tt = prw.poses[st->cur ^ 1] + (size_t)jt * 12;
    const int j = pose_opt[jt];
    if (j < 0) {
      for (int k = 0; k < 12; ++k) Tt[k] = Tc[k];
    } else {
      double xi[6], d[12], T[12];
      for (int k = 0; k < 6; ++k) xi[k] = x[(size_t)j * 6 + k];
      for (int k = 0; k < 12; ++k) T[k] = Tc[k];
      se3_exp(xi, d);
      // T_jw = delta * T_jw (:493): R = Rd R, t = Rd t + td
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c)
          Tt[r * 3 + c] = d[r * 3] * T[c] + d[r * 3 + 1] * T[3 + c] + d[r * 3 + 2] * T[6 + c];
        Tt[9 + r] = d[r * 3] * T[9] + d[r * 3 + 1] * T[10] + d[r * 3 + 2] * T[11] + d[9 + r];
      }
      // a.x + x^T A x (:438-440), damped A
      double m = 0.0, q = 0.0, nrm = 0.0;
      for (int r = 0; r < 6; ++r) {
        m += a[(size_t)j * 6 + r] * xi[r];
        double s = 0.0;
        for (int c = 0; c < 6; ++c) s += A[(size_t)j * 36 + r * 6 + c] * xi[c];
        q += xi[r] * s;
        nrm += xi[r] * xi[r];
      }
      acc[0] = m + q;
      acc[1] = sqrt(nrm);
    }
  }
  block_sum<2, kWarps>(acc, sm);
  if (threadIdx.x == 0) {
    partials[(size_t)blk * 2] = acc[0];
    partials[(size_t)blk * 2 + 1] = acc[1];
  }
}
// Back-substitution of the landmarks and the pose update in ONE launch: the two are independent (both only need x), the
// pose update is a single latency-bound CTA (9 us on C3) that now runs beside the landmark CTAs
__global__ void __launch_bounds__(kThreads)
k_backsub_points_update_poses(int point_blocks, int M_total, const int *__restrict__ point_has_pairs,
                              const uint8_t *__restrict__ point_free, const double *__restrict__ ptblk, size_t Mp,
                              const double *__restrict__ Btx, double *__restrict__ y, Params prm, ParamsW prw,
                              double *__restrict__ point_partials, int method, int N_total, const int *__restrict__ pose_opt,
                              const double *__restrict__ x, const double *__restrict__ A, const double *__restrict__ a,
                              double *__restrict__ pose_partials, const LmState *__restrict__ st) {
  if (st->done) return;
  if ((int)blockIdx.x < point_blocks)
    backsub_points_body(blockIdx.x, M_total, point_has_pairs, point_free, ptblk, Mp, Btx, y, prm, prw, point_partials, method, st);
  else
    update_poses_body(blockIdx.x - point_blocks, N_total, pose_opt, x, A, a, prm, prw, pose_partials, st);
}


// ---------------------------------------------------------------------------
// K4 for by-point landmarks when the reduced system is SMALL (dense co-visibility such as the test_ba.cpp scene:
// every landmark seen by half of the 55 free poses): S -= sum_i E_i B_i^T as a dense FP64 tensor-core GEMM instead
// of one FP64 red per block entry per landmark.  One CTA per (64 x 64 upper output tile, K split): the operands
// X[3 l + c][row] = -E_i(row, c), Y[3 l + c][col] = B_i(col, c) of 10 landmarks per pass are scattered into shared
// memory from the pair blocks (zeros where a pose does not see the landmark), E = B C^-1 formed on the fly; the rhs
// travels as column n = ld - 1 (Y = b_i).  One red per output entry per CTA at the end.  (:858-888)
// ---------------------------------------------------------------------------
constexpr int kDenseLm = 10;   // landmarks per pass: 30 of the kKH = 32 operand rows
constexpr int kDenseMaxPoses = 128;   // free poses (a landmark has at most one pair per pose): 6 N + 1 <= 769
// The by-point Schur products of a reduced system with N free poses go through k_schur_dense_gemm (ba_finalize sends
// every landmark there when most of them do not fit a window) rather than k_schur_pairs_list
inline bool dense_schur_fits(int N) { return N <= kDenseMaxPoses; }
__global__ void __launch_bounds__(256)
k_schur_dense_gemm(const int2 *__restrict__ groups /*pair range [x, y) of one landmark*/, int n_groups, int split_k,
                   const int *__restrict__ pair_pose, const int *__restrict__ pair_point,
                   const double *__restrict__ Bsoa, size_t Pp, const double *__restrict__ ptblk, size_t Mp,
                   double *__restrict__ Saug, int ld, const LmState *__restrict__ st) {
  if (st->done) return;
  __shared__ double X[kKH][kLdT];
  __shared__ double Y[kKH][kLdT];
  __shared__ int lm_first[kDenseLm + 1];   // prefix of the pair counts of the pass
  __shared__ int sq[kDenseLm * kDenseMaxPoses];
  __shared__ short sj[kDenseLm * kDenseMaxPoses];
  __shared__ unsigned char sl[kDenseLm * kDenseMaxPoses];
  const int n = ld - 1;
  const int tile_pair = blockIdx.x / split_k, ks = blockIdx.x - tile_pair * split_k;
  int ib = (int)((sqrt(8.0 * tile_pair + 1.0) - 1.0) * 0.5);
  while (ib * (ib + 1) / 2 > tile_pair) --ib;
  while ((ib + 1) * (ib + 2) / 2 <= tile_pair) ++ib;
  const int ia = tile_pair - ib * (ib + 1) / 2;        // ia <= ib: upper triangle, rows of tile ia, columns of tile ib
  const int r0 = 64 * ia, c0 = 64 * ib;
  const int per = (n_groups + split_k - 1) / split_k;
  const int g_begin = ks * per, g_end = min(n_groups, g_begin + per);
  double acc[2][4][2] = {};
  for (int g0 = g_begin; g0 < g_end; g0 += kDenseLm) {
    const int nl = min(kDenseLm, g_end - g0);
    __syncthreads();
    for (int e = threadIdx.x; e < kKH * kLdT; e += 256) { (&X[0][0])[e] = 0.0; (&Y[0][0])[e] = 0.0; }
    if (threadIdx.x == 0) {
      int run = 0;
      for (int l = 0; l < nl; ++l) { lm_first[l] = run; run += groups[g0 + l].y - groups[g0 + l].x; }
      lm_first[nl] = run;
    }
    __syncthreads();
    const int np = lm_first[nl];
    // stage the pass's pairs (global pair index, pose, landmark slot) so that the scatter below has ONE global
    // round trip per item and no data-dependent control flow in front of its loads
    for (int pl = threadIdx.x; pl < np; pl += 256) {
      int l = 0;
      while (pl >= lm_first[l + 1]) ++l;
      const int q = groups[g0 + l].x + (pl - lm_first[l]);
      sq[pl] = q;
      sj[pl] = (short)pair_pose[q];
      sl[pl] = (unsigned char)l;
    }
    __syncthreads();
    // one thread per (pair, row r of its 6 x 3 block); pairs fastest: Bsoa is component-major, so consecutive
    // threads read consecutive doubles.  Loads unconditional and unrolled (in flight together), stores predicated.
    const int items = np * 6;
#pragma unroll 4
    for (int e = threadIdx.x; e < items; e += 256) {
      const int r = e / np, pl = e - r * np;
      const int q = sq[pl], l = sl[pl];
      const int row = 6 * sj[pl] + r;
      const double b0 = Bsoa[(size_t)(r * 3 + 0) * Pp + q], b1 = Bsoa[(size_t)(r * 3 + 1) * Pp + q],
                   b2 = Bsoa[(size_t)(r * 3 + 2) * Pp + q];
      const bool in_r = row >= r0 && row < r0 + 64, in_c = row >= c0 && row < c0 + 64;
      if (in_c) { Y[3 * l][row - c0] = b0; Y[3 * l + 1][row - c0] = b1; Y[3 * l + 2][row - c0] = b2; }
      if (in_r) {
        const int pt = pair_point[q];
        double ci[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) ci[k] = ptblk[(PB_Cinv + k) * Mp + pt];
        X[3 * l][row - r0] = -(b0 * ci[0] + b1 * ci[1] + b2 * ci[2]);
        X[3 * l + 1][row - r0] = -(b0 * ci[1] + b1 * ci[3] + b2 * ci[4]);
        X[3 * l + 2][row - r0] = -(b0 * ci[2] + b1 * ci[4] + b2 * ci[5]);
      }
    }
    if (n >= c0 && n < c0 + 64 && threadIdx.x < 3 * nl) {   // rhs column: Y = b_i
      const int l = threadIdx.x / 3, c = threadIdx.x - 3 * l;
      Y[3 * l + c][n - c0] = ptblk[(PB_b + c) * Mp + pair_point[groups[g0 + l].x]];
    }
    __syncthreads();
    tile_mac_dmma(X, Y, acc);
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
        const double v = acc[i][j][e];
        if (rr < n && cc <= n && rr <= cc && v != 0.0) atomicAdd(&Saug[(size_t)rr * ld + cc], v);
      }
}

// peer exchange of the LM scalars (see SharedComm below)
constexpr int kMaxRanks = 16;
struct PeerExch {                       // one per rank, written by the peers
  double vals[2][kMaxRanks][8];         // [epoch parity][source rank][scalar]
  unsigned flag[2][kMaxRanks];          // epoch of the values
};
struct PeerTable {                      // device-side view
  PeerExch *peer[kMaxRanks];
  unsigned *epoch;                      // exchanges done so far (device counter, identical on all ranks)
  int *error;                           // sticky: a peer did not answer
  int rank, n_ranks;
};
struct DecideArgs {
  const double *cost_partials; int n_cost;
  const double *point_partials; int n_point;   // {model, step} per block
  const double *pose_partials; int n_pose;     // {model, step} per block
  double *scal;   // [8] reduced scalars {cost, model_point, step_point, model_pose, step_pose}
  double thr_step, thr_cost, dec_ratio, inc_ratio, inverse_scaler;
  double n_obs_global, n_params_global;  // num_observations ; N_opt + M_opt
  int max_iteration;
  int n_ranks;
  int method;   // BA_METHOD_*
};

// ordered (deterministic) sums of the per-block partials into scal[]
__global__ void __launch_bounds__(kThreads) k_reduce_scalars(DecideArgs g, int init_only,
                                                            const LmState *__restrict__ st) {
  if (!init_only && st->done) return;
  __shared__ double sm[kWarps][5];
  double acc[5] = {0, 0, 0, 0, 0};
  for (int i = threadIdx.x; i < g.n_cost; i += kThreads) acc[0] += g.cost_partials[i];
  if (!init_only) {
    for (int i = threadIdx.x; i < g.n_point; i += kThreads) {
      acc[1] += g.point_partials[2 * i];
      acc[2] += g.point_partials[2 * i + 1];
    }
    for (int i = threadIdx.x; i < g.n_pose; i += kThreads) {
      acc[3] += g.pose_partials[2 * i];
      acc[4] += g.pose_partials[2 * i + 1];
    }
  }
  block_sum<5, kWarps>(acc, sm);
  if (threadIdx.x == 0) {
    g.scal[0] = acc[0];
    g.scal[1] = acc[1];
    g.scal[2] = acc[2];
    // the pose part is computed redundantly on every rank from the replicated x and the rank's
    // PARTIAL A/a: the model term is additive over ranks, the step norm is not (divide it)
    g.scal[3] = acc[3];
    g.scal[4] = acc[4] / (double)g.n_ranks;
  }
}

__global__ void k_init_state(LmState *st, const double *scal, double lambda0) {
  st->lambda = lambda0;
  st->prev_cost = scal[0];
  st->cur = st->cur;  // keep
  st->done = 0;
  st->iteration = 0;
  st->converged = 0;
}

// trust-region decision (:930-1007), one thread.
__device__ __forceinline__ void decide(const DecideArgs &g, LmState *st, ba_iter_info *infos, int cap) {
  const double current_cost = g.scal[0];
  const double model = -(g.scal[3] + g.scal[1]);  // EvaluateCostChangeByQuadraticModel (:435-455)
  const double previous_cost = st->prev_cost;
  const double rho = (current_cost - previous_cost) * g.inverse_scaler / model;
  double lambda = st->lambda;
  st->last_cost_new = current_cost;
  st->last_model = model;
  st->last_rho = rho;
  st->last_lambda = lambda;
  int status;
  if (g.method != BA_METHOD_LEVENBERG_MARQUARDT) {
    // Gauss-Newton branch of the refactor class (full_bundle_adjustment_solver_refactor.cpp:976-982) and
    // SolveByGradientDescent (:1285-1289): the step is always kept, lambda stays where it is
    status = 0;
    st->cur ^= 1;
  } else {
    if (rho > 0.25) {
      status = 0;       // UPDATE: trial buffer becomes current
      st->cur ^= 1;
    } else {
      status = 2;       // SKIPPED: keep current (RevertToReservedParameters)
    }
    if (rho > 0.5) {
      lambda = fmax(1e-10, lambda * g.dec_ratio);
      status = 1;       // UPDATE_TRUST_MORE
    } else if (rho <= 0.25) {
      lambda = fmin(100.0, lambda * g.inc_ratio);
    }
  }
  const double average_error = current_cost / g.n_obs_global;
  const double cost_change = fabs(current_cost - previous_cost);
  // gradient descent starts both step sums at 0.01 (refactor.cpp:1296-1297)
  const double total_step = g.scal[2] + g.scal[4] + (g.method == BA_METHOD_GRADIENT_DESCENT ? 0.02 : 0.0);
  const double avg_step = total_step / g.n_params_global;
  bool converged = (avg_step < g.thr_step) || (cost_change < g.thr_cost);
  const int iteration = st->iteration;
  if (iteration >= g.max_iteration - 1) converged = false;
  if (infos != nullptr && iteration < cap) {
    ba_iter_info I;
    I.cost = current_cost;
    I.cost_change = cost_change;
    I.average_reprojection_error = average_error;
    I.abs_gradient = 0.0;
    I.abs_step = avg_step;
    I.damping_term = lambda;
    I.iter_time = 0.0;
    I.iteration_status = status;
    I._pad = 0;
    if (status == 2) {
      I.cost = previous_cost;
      I.cost_change = 0.0;
      I.average_reprojection_error = sqrt(previous_cost / g.n_obs_global);
    }
    infos[iteration] = I;
  }
  st->lambda = lambda;
  st->prev_cost = current_cost;  // unconditionally (:1005)
  st->iteration = iteration + 1;
  st->converged = converged ? 1 : 0;
  if (converged || iteration + 1 >= g.max_iteration) st->done = 1;
}

__global__ void k_decide(DecideArgs g, LmState *st, ba_iter_info *infos, int cap) {
  if (st->done) return;
  decide(g, st, infos, cap);
}

// K7, the trial cost AND the pose-side linearisation at the trial parameters in ONE pass over the observations in pose
// order (speculative pose side).  When the step is accepted the trial parameters are the next iteration's
// linearisation point, so its A / a sums are already there (Au[trial buffer]); when it is rejected the sums of the kept
// buffer are still valid (RevertToReservedParameters re-linearises at the same point, :939-953) -- either way the next
// iteration starts with k_pose_diag (or the storing k_tile_reduce) instead of a second pass over the observations.
// which = 0 (ignore_done) evaluates the accepted parameters instead: the initial cost and the sums the first iteration
// starts from.  Chunks of FIXED poses (j_opt < 0, at the end of the list) contribute to the cost only.  Per pose the
// last chunk to finish sums the pose's partials in chunk order (bit-reproducible); with decide_here the last CTA of the
// grid sums all the partials in their fixed order and takes the trust-region decision.
#ifndef BA_K7_MINB
#define BA_K7_MINB 2   // resident CTAs per SM the register allocation aims at (A/B builds: 3 -> 85 registers, spills)
#endif
__global__ void __launch_bounds__(kThreads, BA_K7_MINB)
k_cost_linearize_by_pose(const ChunkA *__restrict__ chunks, const double2 *__restrict__ uvA,
                         const int *__restrict__ pointA, const int *__restrict__ camA, const int *__restrict__ poseidA,
                         int n_chunks, Params prm, int which, const double *__restrict__ cams, double thres_huber,
                         double *__restrict__ partials /*[free chunks][27]*/, double *__restrict__ cost_partials /*[grid]*/,
                         const int *__restrict__ pose_chunk_ptr, unsigned *__restrict__ pose_ticket,
                         double *__restrict__ Au0, double *__restrict__ Au1, unsigned *__restrict__ ticket,
                         int decide_here, int ignore_done, DecideArgs g, LmState *st, ba_iter_info *infos, int cap) {
  if (!ignore_done && st->done) return;
  __shared__ double sm[kWarps][28];
  __shared__ int is_last_pose, is_last;
  // a problem without observations has no chunks: its grid is one CTA that contributes zeros and takes the decision
  const ChunkA ch = (int)blockIdx.x < n_chunks ? chunks[blockIdx.x] : ChunkA{0, 0, -1, 0};
  const int buf = st->cur ^ which;
  const double *poses = prm.poses[buf];
  const double *points = prm.points[buf];
  const bool free_pose = ch.j_opt >= 0;
  double T[12] = {};
  if (ch.obs_count > 0) {
    const double *Tp = poses + (size_t)poseidA[ch.obs_start] * 12;
#pragma unroll
    for (int i = 0; i < 12; ++i) T[i] = __ldg(Tp + i);
  }
  double acc[28];
#pragma unroll
  for (int i = 0; i < 28; ++i) acc[i] = 0.0;
  for (int t = threadIdx.x; t < ch.obs_count; t += kThreads) {
    const int k = ch.obs_start + t;
    const double2 uv = uvA[k];
    const int pt = pointA[k];
    const double *cam = cams + (camA[k] & kCamMask) * kCamStride;
    double X[3] = {__ldg(points + (size_t)pt * 3), __ldg(points + (size_t)pt * 3 + 1),
                   __ldg(points + (size_t)pt * 3 + 2)};
    Proj p;
    project(T, X, cam, uv.x, uv.y, p);
    acc[27] += sqrt(p.r0 * p.r0 + p.r1 * p.r1);   // EvaluateCurrentCost (:381-433)
    if (free_pose) {
      const double w = huber_weight(p.r0, p.r1, thres_huber);
      const double wr0 = w * p.r0, wr1 = w * p.r1;
      double G[6], Q[12];
      jac_G(p, cam, G);
      jac_Q(G, p.Xb, Q);
      // A_j(upper) += (w Q)^T Q (:519-556,807) ; a_j -= Q^T (w r) (:809)
      int e = 0;
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        const double wa0 = w * Q[r], wa1 = w * Q[6 + r];
#pragma unroll
        for (int c = r; c < 6; ++c) acc[e++] += wa0 * Q[c] + wa1 * Q[6 + c];
      }
#pragma unroll
      for (int r = 0; r < 6; ++r) acc[21 + r] -= Q[r] * wr0 + Q[6 + r] * wr1;
    }
  }
  block_sum<28, kWarps>(acc, sm);
  if (threadIdx.x == 0) {
    __stcg(cost_partials + blockIdx.x, acc[27]);
    is_last_pose = 0;
    if (free_pose) {
      double *o = partials + (size_t)blockIdx.x * 27;
#pragma unroll
      for (int i = 0; i < 27; ++i) __stcg(o + i, acc[i]);
    }
    __threadfence();
    if (free_pose) {
      const unsigned n_ck = (unsigned)(pose_chunk_ptr[ch.j_opt + 1] - pose_chunk_ptr[ch.j_opt]);
      is_last_pose = atomicAdd(pose_ticket + ch.j_opt, 1u) == n_ck - 1;
      if (is_last_pose) pose_ticket[ch.j_opt] = 0;
    }
    is_last = decide_here ? (atomicAdd(ticket, 1u) == gridDim.x - 1) : 0;
  }
  __syncthreads();
  if (is_last_pose && threadIdx.x < 32) {
    __threadfence();
    const double v = pose_partial_sum(ch.j_opt, threadIdx.x, pose_chunk_ptr, partials);
    if (threadIdx.x < 27) (buf ? Au1 : Au0)[(size_t)ch.j_opt * 27 + threadIdx.x] = v;
  }
  if (!is_last) return;
  __threadfence();
  __shared__ double sm2[kWarps][5];
  double red[5] = {0, 0, 0, 0, 0};
  for (int i = threadIdx.x; i < g.n_cost; i += kThreads) red[0] += __ldcg(g.cost_partials + i);
  for (int i = threadIdx.x; i < g.n_point; i += kThreads) {
    red[1] += __ldcg(g.point_partials + 2 * i);
    red[2] += __ldcg(g.point_partials + 2 * i + 1);
  }
  for (int i = threadIdx.x; i < g.n_pose; i += kThreads) {
    red[3] += __ldcg(g.pose_partials + 2 * i);
    red[4] += __ldcg(g.pose_partials + 2 * i + 1);
  }
  block_sum<5, kWarps>(red, sm2);
  if (threadIdx.x == 0) {
    *ticket = 0;
#pragma unroll
    for (int i = 0; i < 5; ++i) g.scal[i] = red[i];
    decide(g, st, infos, cap);
  }
}

// finalize: the pose-ordered copies of the observations, gathered from the point-ordered arrays
__global__ void k_gather_pose_order(long long nA, const int *__restrict__ perm, const double2 *__restrict__ uv,
                                    const int *__restrict__ obs_point, const int *__restrict__ camflags,
                                    const int *__restrict__ obs_pose, double2 *__restrict__ uvA, int *__restrict__ pointA,
                                    int *__restrict__ camA, int *__restrict__ poseidA) {
  for (long long w = blockIdx.x * (long long)blockDim.x + threadIdx.x; w < nA; w += (long long)gridDim.x * blockDim.x) {
    const int q = perm[w];
    uvA[w] = uv[q];
    pointA[w] = obs_point[q];
    camA[w] = camflags[q] & kCamMask;
    poseidA[w] = obs_pose[q];
  }
}

// ba_observation_residuals: residual and status of every observation at the accepted parameters (buffer cur), in one
// grid-stride pass over the point-ordered arrays; row_of maps a point-order position to its input row, the outputs are
// indexed by row.  The status counts are summed per block and added with integer atomics (exact, so deterministic).
// Any output may be null.
__global__ void __launch_bounds__(kThreads)
k_obs_residuals(long long n, const double2 *__restrict__ obs_uv, const int *__restrict__ obs_pose,
                const int *__restrict__ obs_point, const int *__restrict__ obs_camflags, const int *__restrict__ row_of,
                Params prm, const double *__restrict__ cams, double thres, const LmState *__restrict__ st,
                double2 *__restrict__ residuals, uint8_t *__restrict__ status, unsigned long long *__restrict__ counts) {
  __shared__ unsigned wsum[kWarps][3];
  const double *poses = prm.poses[st->cur];
  const double *points = prm.points[st->cur];
  unsigned cnt[3] = {0u, 0u, 0u};
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
    const int cf = obs_camflags[k];
    const int pt = obs_point[k];
    const double2 uv = obs_uv[k];
    double T[12];
    load_pose(poses + (size_t)obs_pose[k] * 12, T);
    const double X[3] = {__ldg(points + (size_t)pt * 3), __ldg(points + (size_t)pt * 3 + 1),
                         __ldg(points + (size_t)pt * 3 + 2)};
    const double *cam = cams + (cf & kCamMask) * kCamStride;
    Proj p;
    project(T, X, cam, uv.x, uv.y, p);
    int s;
    if (!(camera_depth(p, cam) > 0.0) || !isfinite(p.r0) || !isfinite(p.r1)) s = BA_OBS_BEHIND_CAMERA;
    else s = (fabs(p.r0) + fabs(p.r1) > thres) ? BA_OBS_OUTLIER : BA_OBS_INLIER;   // huber_weight's test
    cnt[0] += s == BA_OBS_INLIER;
    cnt[1] += s == BA_OBS_OUTLIER;
    cnt[2] += s == BA_OBS_BEHIND_CAMERA;
    const int r = row_of[k];
    if (residuals) residuals[r] = make_double2(p.r0, p.r1);
    if (status) status[r] = (uint8_t)s;
  }
  if (!counts) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const unsigned v = __reduce_add_sync(0xffffffffu, cnt[i]);
    if (lane == 0) wsum[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    unsigned long long tot = 0;
    for (int w = 0; w < kWarps; ++w) tot += wsum[w][threadIdx.x];
    if (tot) atomicAdd(counts + threadIdx.x, tot);
  }
}

// Multi-GPU: ordered sums of the partials, one-shot exchange of the five scalars through the peers' mapped buffers
// (one remote store per peer + a flag; the sum runs in rank order on every rank, so all ranks take bit-identical
// decisions) and the trust-region decision, in ONE launch.  Replaces k_reduce_scalars + ncclAllReduce + k_decide.
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__global__ void __launch_bounds__(kThreads) k_exchange_decide(DecideArgs g, PeerTable pt, LmState *st, ba_iter_info *infos,
                                                             int cap) {
  if (st->done) return;
  __shared__ double sm[kWarps][5];
  __shared__ double mine[5], all[kMaxRanks][5];
  double acc[5] = {0, 0, 0, 0, 0};
  for (int i = threadIdx.x; i < g.n_cost; i += kThreads) acc[0] += g.cost_partials[i];
  for (int i = threadIdx.x; i < g.n_point; i += kThreads) {
    acc[1] += g.point_partials[2 * i];
    acc[2] += g.point_partials[2 * i + 1];
  }
  for (int i = threadIdx.x; i < g.n_pose; i += kThreads) {
    acc[3] += g.pose_partials[2 * i];
    acc[4] += g.pose_partials[2 * i + 1];
  }
  block_sum<5, kWarps>(acc, sm);
  if (threadIdx.x == 0) {
    mine[0] = acc[0]; mine[1] = acc[1]; mine[2] = acc[2]; mine[3] = acc[3];
    mine[4] = acc[4] / (double)g.n_ranks;   // the pose step is computed redundantly on every rank (see k_reduce_scalars)
  }
  __syncthreads();
  const unsigned epoch = *pt.epoch + 1;
  const int par = epoch & 1;
  if (threadIdx.x < pt.n_ranks) {
    const int p = threadIdx.x;
    PeerExch *dst = pt.peer[p];
#pragma unroll
    for (int i = 0; i < 5; ++i) dst->vals[par][pt.rank][i] = mine[i];
    __threadfence_system();
    st_release_sys(&dst->flag[par][pt.rank], epoch);
    // the values of rank p arrive in MY buffer
    const PeerExch *own = pt.peer[pt.rank];
    long long spins = 0;
    bool ok = true;
    while (ld_acquire_sys(&own->flag[par][p]) != epoch) {
      if (++spins > (1ll << 28) || *((volatile int *)pt.error)) { ok = false; break; }
    }
    if (ok) {
#pragma unroll
      for (int i = 0; i < 5; ++i) all[p][i] = *((volatile const double *)&own->vals[par][p][i]);
    } else {
      *pt.error = 1;
#pragma unroll
      for (int i = 0; i < 5; ++i) all[p][i] = 0.0;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    *pt.epoch = epoch;
    if (*((volatile int *)pt.error)) {   // a peer is gone: stop the loop, the host reports it
      st->done = 1;
      return;
    }
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      double v = 0.0;
      for (int r = 0; r < pt.n_ranks; ++r) v += all[r][i];
      g.scal[i] = v;
    }
    decide(g, st, infos, cap);
  }
}

// band-only clearing of a large banded S: row r's columns r .. r + bw and its rhs entry (two strided 2-D memsets of
// 12 k short rows took 40 us on C4)
__global__ void __launch_bounds__(256) k_clear_band(double *__restrict__ S, int n, int ld, int bw, const LmState *__restrict__ st) {
  if (st->done) return;
  const int w = bw + 2;
  const long long total = (long long)n * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / w), t = (int)(i - (long long)r * w);
    if (t <= bw) { if (r + t < n) S[(size_t)r * ld + r + t] = 0.0; }
    else S[(size_t)r * ld + (ld - 1)] = 0.0;
  }
}

// Multi-GPU, banded reduced system, ranks with mapped peer memory: the band exchange as a TWO-SHOT all-reduce over
// NVLink, hand-written (BA_B200_BAND_XCHG=2; the default is the one-shot form below, see enqueue_allreduce_S).  The packed band (row r: columns r .. r + bw of the upper triangle + the rhs entry) is split by
// rows over the ranks.  k_band_push sends every row's partial to the row's OWNER (slot = my rank); k_band_reduce
// (owner) waits for the flags of all ranks, sums the slots in rank order and stores the result into EVERY rank's
// result buffer; k_band_pull waits for all owners and copies the result into S.  Bit-identical on every rank, no NCCL
// call; 2 (R-1)/R of the band leaves a rank instead of R-1 times the band with one-shot pushes (measured at R = 8 on
// C4: the one-shot exchange cost 0.10 ms).  Buffers are double-buffered by epoch parity.
struct BandPeers {
  double *buf[kMaxRanks];       // every rank's buffer: [2][ n_ranks x pslot partial slots | cap result ]
  unsigned *flag[kMaxRanks];    // every rank's flags: [2][2][kMaxRanks] (partials delivered, results delivered)
  unsigned *epoch;              // local: exchanges completed
  unsigned *counters;           // local: CTAs of the push / reduce / pull that finished
  int *error;
  long long cap, pslot;         // doubles of the result region / of one partial slot
  int rank, n_ranks;
};
__device__ __forceinline__ int band_row0(int n, int R, int p) { return (int)(((long long)n * p) / R); }
__device__ __forceinline__ bool band_wait_flags(const BandPeers &bp, const unsigned *flags, unsigned epoch) {
  if (threadIdx.x < bp.n_ranks) {
    const unsigned *f = flags + threadIdx.x;
    long long spins = 0;
    while (ld_acquire_sys(f) != epoch) {
      if (++spins > (1ll << 26) || *((volatile int *)bp.error)) { *bp.error = 1; break; }
    }
  }
  __syncthreads();
  return true;
}
// last CTA of a grid (ticket counter) publishes `epoch` into flags[...][my rank] of every peer
__device__ __forceinline__ void band_publish(const BandPeers &bp, unsigned *counter, int which, int par, unsigned epoch) {
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicAdd(counter, 1u);
    if (done == gridDim.x - 1) {
      *counter = 0;
      __threadfence_system();
      for (int p = 0; p < bp.n_ranks; ++p) st_release_sys(bp.flag[p] + (par * 2 + which) * kMaxRanks + bp.rank, epoch);
    }
  }
}
__global__ void __launch_bounds__(128) k_band_push(const double *__restrict__ S, int n, int ld, int bw, BandPeers bp,
                                                   const LmState *__restrict__ st) {
  if (st->done) return;
  const unsigned epoch = *bp.epoch + 1;
  const int par = epoch & 1, w = bw + 2, R = bp.n_ranks;
  const long long parstride = (long long)R * bp.pslot + bp.cap;
  const long long total = (long long)n * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / w), t = (int)(i - (long long)r * w);
    double v = 0.0;
    if (t <= bw) { if (r + t < n) v = S[(size_t)r * ld + r + t]; }
    else v = S[(size_t)r * ld + (ld - 1)];
    int p = (int)(((long long)r * R) / n);
    while (p > 0 && r < band_row0(n, R, p)) --p;
    while (p + 1 < R && r >= band_row0(n, R, p + 1)) ++p;
    bp.buf[p][par * parstride + (long long)bp.rank * bp.pslot + (long long)(r - band_row0(n, R, p)) * w + t] = v;
  }
  band_publish(bp, bp.counters, 0, par, epoch);
}
__global__ void __launch_bounds__(128) k_band_reduce(int n, int bw, BandPeers bp, const LmState *__restrict__ st) {
  if (st->done) return;
  const unsigned epoch = *bp.epoch + 1;
  const int par = epoch & 1, w = bw + 2, R = bp.n_ranks;
  const long long parstride = (long long)R * bp.pslot + bp.cap;
  band_wait_flags(bp, bp.flag[bp.rank] + (par * 2 + 0) * kMaxRanks, epoch);
  const int r0 = band_row0(n, R, bp.rank), r1 = band_row0(n, R, bp.rank + 1);
  const long long total = (long long)(r1 - r0) * w;
  const double *mine = bp.buf[bp.rank] + par * parstride;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    double vv[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) vv[p] = p < R ? __ldcg(mine + (long long)p * bp.pslot + i) : 0.0;
    double v = 0.0;
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) v += vv[p];      // rank order; the slots beyond n_ranks add exact zeros
    const long long o = par * parstride + (long long)R * bp.pslot + (long long)r0 * w + i;
    for (int q = 0; q < R; ++q) bp.buf[q][o] = v;
  }
  band_publish(bp, bp.counters + 1, 1, par, epoch);
}
__global__ void __launch_bounds__(128) k_band_pull(double *__restrict__ S, int n, int ld, int bw, BandPeers bp,
                                                   const LmState *__restrict__ st) {
  if (st->done) return;
  const unsigned epoch = *bp.epoch + 1;
  const int par = epoch & 1, w = bw + 2, R = bp.n_ranks;
  const long long parstride = (long long)R * bp.pslot + bp.cap;
  band_wait_flags(bp, bp.flag[bp.rank] + (par * 2 + 1) * kMaxRanks, epoch);
  const double *res = bp.buf[bp.rank] + par * parstride + (long long)R * bp.pslot;
  const long long total = (long long)n * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / w), t = (int)(i - (long long)r * w);
    const double v = __ldcg(res + i);
    if (t <= bw) { if (r + t < n) S[(size_t)r * ld + r + t] = v; }
    else S[(size_t)r * ld + (ld - 1)] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicAdd(bp.counters + 2, 1u);
    if (done == gridDim.x - 1) {
      bp.counters[2] = 0;
      *bp.epoch = epoch;
    }
  }
}

// One-shot form of the exchange (default): every rank pushes its whole packed band into every rank's receive buffer
// (slot = its rank) and publishes one epoch flag per peer; k_band_pull1 waits for all flags and writes S(band) = the
// sum of the slots in rank order.  One hand-over per exchange.
__global__ void __launch_bounds__(128) k_band_push1(const double *__restrict__ S, int n, int ld, int bw, BandPeers bp,
                                                   const LmState *__restrict__ st) {
  if (st->done) return;
  const unsigned epoch = *bp.epoch + 1;
  const int par = epoch & 1, w = bw + 2;
  const size_t slot = ((size_t)par * bp.n_ranks + bp.rank) * (size_t)bp.cap;
  // flat index over the packed band (row r, entry t): every lane busy, the stores of a warp are contiguous per peer
  const long long total = (long long)n * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / w), t = (int)(i - (long long)r * w);
    double v = 0.0;
    if (t <= bw) { if (r + t < n) v = S[(size_t)r * ld + r + t]; }
    else v = S[(size_t)r * ld + (ld - 1)];
    for (int p = 0; p < bp.n_ranks; ++p) bp.buf[p][slot + i] = v;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicAdd(bp.counters, 1u);
    if (done == gridDim.x - 1) {           // every CTA's stores are fenced: publish
      bp.counters[0] = 0;
      __threadfence_system();
      for (int p = 0; p < bp.n_ranks; ++p) st_release_sys(bp.flag[p] + par * kMaxRanks + bp.rank, epoch);
    }
  }
}
__global__ void __launch_bounds__(128) k_band_pull1(double *__restrict__ S, int n, int ld, int bw, BandPeers bp,
                                                   const LmState *__restrict__ st) {
  if (st->done) return;
  const unsigned epoch = *bp.epoch + 1;
  const int par = epoch & 1, w = bw + 2;
  if (threadIdx.x < bp.n_ranks) {
    const unsigned *f = bp.flag[bp.rank] + par * kMaxRanks + threadIdx.x;
    long long spins = 0;
    while (ld_acquire_sys(f) != epoch) {
      if (++spins > (1ll << 26) || *((volatile int *)bp.error)) { *bp.error = 1; break; }
    }
  }
  __syncthreads();
  const double *mine = bp.buf[bp.rank] + (size_t)par * bp.n_ranks * (size_t)bp.cap;
  const long long total = (long long)n * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / w), t = (int)(i - (long long)r * w);
    double vv[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) vv[p] = p < bp.n_ranks ? __ldcg(mine + (size_t)p * bp.cap + i) : 0.0;
    double v = 0.0;
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) v += vv[p];      // rank order; the slots beyond n_ranks add exact zeros
    if (t <= bw) { if (r + t < n) S[(size_t)r * ld + r + t] = v; }
    else S[(size_t)r * ld + (ld - 1)] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned done = atomicAdd(bp.counters + 2, 1u);
    if (done == gridDim.x - 1) {
      bp.counters[2] = 0;
      *bp.epoch = epoch;
    }
  }
}

// Multi-GPU, banded reduced system: only the band of S (row r: columns r .. r + bw of the upper triangle, what the
// build writes and the banded factorisation reads) and the rhs column take part in the all-reduce.
__global__ void k_band_pack(const double *__restrict__ S, int n, int ld, int bw, double *__restrict__ packed,
                            const LmState *__restrict__ st) {
  if (st->done) return;
  const int r = blockIdx.x, w = bw + 2;
  for (int t = threadIdx.x; t < w; t += blockDim.x) {
    double v = 0.0;
    if (t <= bw) { if (r + t < n) v = S[(size_t)r * ld + r + t]; }
    else v = S[(size_t)r * ld + (ld - 1)];
    packed[(size_t)r * w + t] = v;
  }
}
__global__ void k_band_unpack(double *__restrict__ S, int n, int ld, int bw, const double *__restrict__ packed,
                              const LmState *__restrict__ st) {
  if (st->done) return;
  const int r = blockIdx.x, w = bw + 2;
  for (int t = threadIdx.x; t < w; t += blockDim.x) {
    const double v = packed[(size_t)r * w + t];
    if (t <= bw) { if (r + t < n) S[(size_t)r * ld + r + t] = v; }
    else S[(size_t)r * ld + (ld - 1)] = v;
  }
}

}  // namespace ba

// =============================================================================
// Host side
// =============================================================================
using namespace ba;

#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      s->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                          \
      return BA_ERR_CUDA;                                                                   \
    }                                                                                       \
  } while (0)

namespace {

struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t,
                            cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  bool load() {
    if (lib) return true;
    // prefer a libnccl already loaded into the process (torch's), then the system one
    lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return false;
    GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
    AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
    AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
    return GetUniqueId && CommInitRank && AllReduce && CommDestroy;
  }
};
NcclApi g_nccl;

// One communicator per process and device, shared by the solvers that attach to it (creating an NCCL communicator
// costs ~0.4 s per rank: a process that solves problem after problem joins once).  Besides the NCCL handle it owns
// the PEER EXCHANGE buffers of the LM scalars: every rank maps every other rank's buffer (CUDA IPC over NVLink), so
// the five scalars of an iteration travel as one remote store per peer plus a flag instead of an NCCL all-reduce.
struct SharedComm {
  ncclComm_t comm = nullptr;
  int rank = 0, n_ranks = 1, device = 0;
  bool verbose = false;   // BA_B200_VERBOSE of the solver that created the communicator
  PeerExch *local = nullptr;
  PeerExch *peer[kMaxRanks] = {};
  unsigned *d_epoch = nullptr;
  int *d_error = nullptr;
  bool peer_ok = false;
  // band exchange through peer memory (k_band_push / k_band_pull): receive buffer [2][n_ranks][band_cap], flags
  double *band_local = nullptr, *band_peer[kMaxRanks] = {};
  unsigned *bflag_local = nullptr, *bflag_peer[kMaxRanks] = {};
  unsigned *d_band_epoch = nullptr, *d_band_counters = nullptr;
  long long band_cap = 0, band_pslot = 0;
  bool band_ok = false;
  struct RetiredBand { double *local; unsigned *flags, *epoch, *counters; double *peer[kMaxRanks]; unsigned *fpeer[kMaxRanks]; };
  std::vector<RetiredBand> retired;   // replaced by a larger set; kept alive for the graphs that captured it
  void retire_band() {
    RetiredBand rb{band_local, bflag_local, d_band_epoch, d_band_counters, {}, {}};
    for (int r = 0; r < kMaxRanks; ++r) { rb.peer[r] = band_peer[r]; rb.fpeer[r] = bflag_peer[r]; band_peer[r] = nullptr; bflag_peer[r] = nullptr; }
    retired.push_back(rb);
    band_local = nullptr; bflag_local = nullptr; d_band_epoch = nullptr; d_band_counters = nullptr;
    band_cap = 0; band_ok = false;
  }
  void close_band() {
    for (RetiredBand &rb : retired) {
      for (int r = 0; r < n_ranks && r < kMaxRanks; ++r) {
        if (rb.peer[r] && r != rank) cudaIpcCloseMemHandle(rb.peer[r]);
        if (rb.fpeer[r] && r != rank) cudaIpcCloseMemHandle(rb.fpeer[r]);
      }
      if (rb.local) cudaFree(rb.local);
      if (rb.flags) cudaFree(rb.flags);
      if (rb.epoch) cudaFree(rb.epoch);
      if (rb.counters) cudaFree(rb.counters);
    }
    retired.clear();
    for (int r = 0; r < n_ranks && r < kMaxRanks; ++r) {
      if (band_peer[r] && r != rank) cudaIpcCloseMemHandle(band_peer[r]);
      if (bflag_peer[r] && r != rank) cudaIpcCloseMemHandle(bflag_peer[r]);
      band_peer[r] = nullptr; bflag_peer[r] = nullptr;
    }
    if (band_local) cudaFree(band_local);
    if (bflag_local) cudaFree(bflag_local);
    if (d_band_epoch) cudaFree(d_band_epoch);
    if (d_band_counters) cudaFree(d_band_counters);
    band_local = nullptr; bflag_local = nullptr; d_band_epoch = nullptr; d_band_counters = nullptr;
    band_cap = 0; band_ok = false;
  }
  PeerTable table() const {
    PeerTable t{};
    for (int r = 0; r < kMaxRanks; ++r) t.peer[r] = peer[r];
    t.epoch = d_epoch; t.error = d_error; t.rank = rank; t.n_ranks = n_ranks;
    return t;
  }
  ~SharedComm() {
    cudaSetDevice(device);
    for (int r = 0; r < n_ranks && r < kMaxRanks; ++r)
      if (peer[r] && r != rank) cudaIpcCloseMemHandle(peer[r]);
    close_band();
    if (local) cudaFree(local);
    if (d_epoch) cudaFree(d_epoch);
    if (d_error) cudaFree(d_error);
    if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
  }
};
std::mutex g_comm_mu;
std::map<int, std::shared_ptr<SharedComm>> g_comm_registry;   // by device

// Device buffers come from the device's default stream-ordered memory pool (cudaMallocAsync) with the release
// threshold lifted, so the ~40 buffers of a problem cost a handful of driver allocations and a re-finalised or
// second solver reuses what an earlier one returned.  g_alloc_stream: stream of the entry point in progress.
thread_local cudaStream_t g_alloc_stream = nullptr;
inline void pool_setup(int device) {
  static bool done[64] = {};
  if (device < 0 || device >= 64 || done[device]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  done[device] = true;
}

// Host-side data-parallel loops of set_observations / finalize: plain threads that are joined at the end of the
// loop (at most 16).  An OpenMP team would keep spinning on every core after each of the dozen short regions, which
// starves the caller's own thread (and the driver's staging copies that follow) on hosts with a CPU quota.
static int host_threads() {
  static const int n = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  return n;
}
// Worker pool behind parallel_ranges / exclusive_scan_inplace: ba_finalize runs ~25 short data-parallel passes, and
// creating + joining 15 threads per pass cost more than some of the passes.  Workers sleep on a condition variable
// between jobs (no spinning: see host_threads), the pool lives for the process (leaked singleton).
class HostPool {
 public:
  static HostPool &get() { static HostPool *p = new HostPool(); return *p; }
  // runs job(t) for t in [0, nth), t = 0 on the caller; returns when all are done.  One job at a time (mutex).
  void run(int nth, const std::function<void(int)> &job) {
    if (nth <= 1) { job(0); return; }
    std::lock_guard<std::mutex> serial(run_mu_);
    {
      std::lock_guard<std::mutex> lk(mu_);
      grow(nth - 1);
      job_ = &job; n_active_ = nth - 1; pending_ = nth - 1; ++epoch_;
    }
    cv_.notify_all();
    job(0);
    std::unique_lock<std::mutex> lk(mu_);
    done_cv_.wait(lk, [&] { return pending_ == 0; });
    job_ = nullptr;
  }

 private:
  void grow(int n) {   // mu_ held
    while ((int)workers_.size() < n) {
      const int id = (int)workers_.size();
      workers_.emplace_back([this, id] { loop(id); });
      workers_.back().detach();
    }
  }
  void loop(int id) {
    unsigned long long seen = 0;
    for (;;) {
      const std::function<void(int)> *job = nullptr;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return epoch_ != seen; });
        seen = epoch_;
        if (id < n_active_) job = job_;
      }
      if (!job) continue;
      (*job)(id + 1);
      std::lock_guard<std::mutex> lk(mu_);
      if (--pending_ == 0) done_cv_.notify_one();
    }
  }
  std::mutex mu_, run_mu_;
  std::condition_variable cv_, done_cv_;
  std::vector<std::thread> workers_;
  const std::function<void(int)> *job_ = nullptr;
  int n_active_ = 0, pending_ = 0;
  unsigned long long epoch_ = 0;
};

template <typename F>
static void parallel_ranges(long long n, F &&fn /*(lo, hi, tid)*/, long long grain = 4096) {
  const int nth = (int)std::min<long long>(host_threads(), std::max<long long>(1, n / grain));
  if (nth <= 1) { fn(0LL, n, 0); return; }
  HostPool::get().run(nth, [&fn, n, nth](int t) { fn(n * t / nth, n * (t + 1) / nth, t); });
}

// exclusive prefix sum of v[0..n) in place (v has n + 1 entries; v[n] and the return value = total), two passes
static long long exclusive_scan_inplace(int *v, long long n) {
  const int nth = (int)std::min<long long>(host_threads(), std::max<long long>(1, n / 4096));
  std::vector<long long> part(nth + 1, 0);
  auto range = [&](int t, long long &lo, long long &hi) { lo = n * t / nth; hi = n * (t + 1) / nth; };
  auto run = [&](auto &&body) { HostPool::get().run(nth, [&body](int t) { body(t); }); };
  run([&](int t) { long long lo, hi; range(t, lo, hi); long long sum = 0; for (long long q = lo; q < hi; ++q) sum += v[q]; part[t + 1] = sum; });
  for (int k = 0; k < nth; ++k) part[k + 1] += part[k];
  run([&](int t) { long long lo, hi; range(t, lo, hi); long long acc = part[t]; for (long long q = lo; q < hi; ++q) { const int x = v[q]; v[q] = (int)acc; acc += x; } });
  v[n] = (int)part[nth];
  return part[nth];
}

// Small pinned blocks (the 64-byte LM state / scalar read-backs) are recycled process-wide: cudaMallocHost costs
// about a millisecond, a solver is often created per problem.
static std::mutex g_pinned_mu;
static std::vector<void *> g_pinned_free;
constexpr size_t kPinnedBlock = 256;
static cudaError_t pinned_get(void **p) {
  {
    std::lock_guard<std::mutex> lk(g_pinned_mu);
    if (!g_pinned_free.empty()) { *p = g_pinned_free.back(); g_pinned_free.pop_back(); return cudaSuccess; }
  }
  return cudaMallocHost(p, kPinnedBlock);
}
static void pinned_put(void *p) {
  if (!p) return;
  std::lock_guard<std::mutex> lk(g_pinned_mu);
  g_pinned_free.push_back(p);
}

// Host scratch arrays of ba_finalize: blocks come from a process-wide cache and are NOT zero-filled -- value-initialised
// std::vectors of 50 MB (zero fill + first-touch page faults on fresh pages) were a quarter of the finalisation time
// of a process that solves problem after problem.
struct HostScratchCache {
  std::mutex mu;
  std::vector<std::pair<void *, size_t>> free_blocks;
  size_t cached = 0;
  void *get(size_t bytes, size_t *got) {
    bytes = (bytes + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
    {
      std::lock_guard<std::mutex> lk(mu);
      int best = -1;
      for (int i = 0; i < (int)free_blocks.size(); ++i)
        if (free_blocks[i].second >= bytes && (best < 0 || free_blocks[i].second < free_blocks[best].second)) best = i;
      if (best >= 0 && free_blocks[best].second <= 2 * bytes + (8u << 20)) {
        void *p = free_blocks[best].first;
        *got = free_blocks[best].second;
        cached -= *got;
        free_blocks.erase(free_blocks.begin() + best);
        return p;
      }
    }
    *got = bytes;
    void *p = std::malloc(bytes);
    if (!p) throw std::bad_alloc();
    // page-locked once, reused by every later problem of the process: the uploads out of these arrays then run at
    // the link rate and really overlap the host work (a failed registration only costs that)
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) cudaGetLastError();
    return p;
  }
  void put(void *p, size_t bytes) {
    std::lock_guard<std::mutex> lk(mu);
    if (cached + bytes > ((size_t)2 << 30) || free_blocks.size() > 64) {   // keep at most 2 GB
      if (cudaHostUnregister(p) != cudaSuccess) cudaGetLastError();
      std::free(p);
      return;
    }
    free_blocks.emplace_back(p, bytes);
    cached += bytes;
  }
};
inline HostScratchCache &host_scratch() { static HostScratchCache c; return c; }
template <typename T>
struct ScratchAlloc {
  using value_type = T;
  ScratchAlloc() = default;
  template <typename U> ScratchAlloc(const ScratchAlloc<U> &) {}
  T *allocate(size_t n) {
    size_t got = 0;
    char *raw = static_cast<char *>(host_scratch().get(n * sizeof(T) + 64, &got));
    *reinterpret_cast<size_t *>(raw) = got;      // block size in front of the array (64 B keeps the alignment)
    return reinterpret_cast<T *>(raw + 64);
  }
  void deallocate(T *p, size_t) {
    char *raw = reinterpret_cast<char *>(p) - 64;
    host_scratch().put(raw, *reinterpret_cast<size_t *>(raw));
  }
  template <typename U> void construct(U *p) { ::new ((void *)p) U; }                 // default-init: no zero fill
  template <typename U, typename... A> void construct(U *p, A &&...a) { ::new ((void *)p) U(std::forward<A>(a)...); }
  template <typename U> bool operator==(const ScratchAlloc<U> &) const { return true; }
  template <typename U> bool operator!=(const ScratchAlloc<U> &) const { return false; }
};
template <typename T> using hvec = std::vector<T, ScratchAlloc<T>>;

template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  cudaError_t alloc(size_t count) {
    if (count <= n && p) return cudaSuccess;
    release();
    n = count;
    if (count == 0) return cudaSuccess;
    return cudaMallocAsync((void **)&p, count * sizeof(T), g_alloc_stream);
  }
  template <typename V>
  cudaError_t upload(const V &h, cudaStream_t st) {
    cudaError_t e = alloc(h.size());
    if (e != cudaSuccess || h.empty()) return e;
    return cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, st);
  }
  void release() {
    if (p) cudaFreeAsync(p, g_alloc_stream);
    p = nullptr;
    n = 0;
  }
};

// A/B and diagnostic switches (DESIGN §4.0).  read_switches() holds the engine's only getenv calls; ba_create takes
// one snapshot per solver, so a switch applies to the solvers created after it is set and never changes under a
// solver that exists.  The defaults are the shipped path.
struct EngineSwitches {
  int band_mode = 6;             // BA_B200_BAND_MODE: 6 partitioned, one persistent launch; 5 partitioned, one launch
                                 // per level; <= 4 the serial window kernel
  int chol_mode = -1;            // BA_B200_CHOL_MODE: -1 auto, 0 dense multi-kernel, 1 cluster (cholesky_make_plan)
  int nd_depth = -1, nd_chunk = -1;   // BA_B200_ND_DEPTH / BA_B200_ND_CHUNK: force the partition (tests)
  bool reduce_stores = true;     // BA_B200_REDUCE_STORES=0: clear of S + k_pose_diag + adding k_tile_reduce instead
                                 // of the storing reduce on banded plans (the two forms are bit-identical)
  size_t band_clear_min = (size_t)64 << 20;   // BA_B200_BAND_CLEAR_MIN_MB: dense S above this clears only its band
  int band_xchg = 1;             // BA_B200_BAND_XCHG: 1 one-shot, 2 two-shot band exchange over peer memory
  bool no_peer_exchange = false; // BA_B200_NO_PEER_EXCHANGE: NCCL for the scalars and the band (ba_comm_init)
  bool verbose = false;          // BA_B200_VERBOSE: finalisation laps, the solve plan, in-kernel solve timing
};

static EngineSwitches read_switches() {
  EngineSwitches w;
  if (const char *e = getenv("BA_B200_BAND_MODE")) w.band_mode = atoi(e);
  if (const char *e = getenv("BA_B200_CHOL_MODE")) w.chol_mode = atoi(e);
  if (const char *e = getenv("BA_B200_ND_DEPTH")) w.nd_depth = atoi(e);
  if (const char *e = getenv("BA_B200_ND_CHUNK")) w.nd_chunk = atoi(e);
  if (const char *e = getenv("BA_B200_REDUCE_STORES")) w.reduce_stores = atoi(e) != 0;
  if (const char *e = getenv("BA_B200_BAND_CLEAR_MIN_MB")) w.band_clear_min = (size_t)atoi(e) << 20;
  if (const char *e = getenv("BA_B200_BAND_XCHG")) w.band_xchg = atoi(e) ? atoi(e) : 1;
  w.no_peer_exchange = getenv("BA_B200_NO_PEER_EXCHANGE") != nullptr;
  w.verbose = getenv("BA_B200_VERBOSE") != nullptr;
  return w;
}

}  // namespace

struct ba_solver {
  int device = 0;
  EngineSwitches sw;   // read once by ba_create
  std::string err;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool profile = false, debug_keep = false;

  // host problem
  std::unordered_map<int, int> cam_slot;
  std::vector<double> h_cams;
  int n_cam = 0;
  std::vector<double> h_poses, h_points;
  std::vector<uint8_t> h_pose_fixed, h_point_fixed;
  std::vector<int> h_obs_cam, h_obs_pose, h_obs_point;
  std::vector<double> h_obs_uv;
  long long n_obs = 0;
  // rows of the last ba_set_observations call (ba_observation_residuals): how many were passed in, the input row of
  // every kept observation when some were dropped (empty: the identity), and the kept index of every point-order
  // position (written by ba_finalize, uploaded on the first ba_observation_residuals after it)
  long long n_rows = 0;
  std::vector<int> h_kept_row;
  hvec<int> h_kept_of_pos;
  DevBuf<int> d_row_of_pos;
  bool row_map_uploaded = false;
  int N_total = 0, M_total = 0, N = 0, M = 0;
  long long P = 0;
  bool finalized = false;
  std::vector<int> h_pose_opt, h_point_opt, h_opt_pose, h_opt_point;
  std::vector<int> h_pair_pose, h_pair_point;  // j_opt, original point id
  std::vector<int> h_first_pose;               // per free pose: first co-visible free pose (envelope of S)
  int n_chunksA = 0, n_split = 0, n_split_pairs = 0;

  // device problem
  DevBuf<double> d_cams, d_poses[2], d_points[2];
  DevBuf<double2> d_obs_uv, d_uvA;
  DevBuf<int> d_obs_pose, d_obs_point, d_obs_camflags;
  DevBuf<int> d_pointA, d_camA, d_poseidA;
  DevBuf<int2> d_pair_obs;
  DevBuf<ChunkA> d_chunksA;
  DevBuf<int> d_pose_chunk_ptr, d_pose_opt, d_pair_pose, d_pair_point, d_pair_end, d_point_has_pairs;
  DevBuf<uint8_t> d_point_free;
  DevBuf<int> d_split_points;
  DevBuf<SchurChunk> d_schur_chunks;
  DevBuf<int> d_tpt_point, d_tpt_inc_start, d_fallback_pairs;
  DevBuf<int2> d_fb_groups;   // pair range of every by-point landmark (dense-GEMM Schur path of small systems)
  int n_fb_groups = 0;
  DevBuf<int4> d_inc_a, d_tile_batches;
  int n_tpt = 0;   // tile landmarks
  DevBuf<int2> d_inc_b;
  DevBuf<int> d_cta_batch_ptr;
  // deterministic tile flush: one staging window per (CTA, chunk) segment of the batch list
  DevBuf<int> d_cta_seg_ptr;     // first segment of every CTA
  DevBuf<long long> d_seg_off;   // window offset in d_stage (doubles)
  DevBuf<int4> d_seg_win;        // 6 jmin, rows, offset (lo, hi)
  DevBuf<int2> d_pose_seg;       // per free pose: range of segments whose window may hold it
  DevBuf<double> d_stage;
  int stage_span = 0;
  TileLaunch tile_launch{};
  DevBuf<Chunk> d_chunks_fb;
  DevBuf<int2> d_chunk_pts_fb;
  DevBuf<ChunkPoint> d_cpts_fb;
  DevBuf<int> d_chunk_pair_count_fb;
  DevBuf<uint8_t> d_point_fb;
  int n_chunks_fb = 0;
  int n_schur_chunks = 0, n_fallback_pairs = 0;
  CholeskyPlan chol;
  DevBuf<int> d_chol_rows, d_chol_first, d_chol_rows_ptr;
  DevBuf<NdNode> d_nd_nodes;                       // partitioned banded solve (ba_cholesky_nd.cuh)
  DevBuf<int> d_nd_level_nodes, d_nd_cta_nodes, d_nd_cta_ptr, d_nd_flags, d_nd_helpers;
  DevBuf<double> d_nd_L, d_nd_U;
  DevBuf<double> d_band;   // multi-GPU, banded S: band rows + rhs packed for the all-reduce
  bool S_clean_outside_band = false;   // Saug was fully cleared since it was allocated / the plan changed
  // blocks
  size_t Mp = 0, Pp = 0;
  DevBuf<double> d_ptblk, d_Bsoa, d_A, d_a, d_partialsA, d_Saug, d_Scopy, d_x, d_z, d_linv, d_Btx, d_y;
  DevBuf<double> d_point_partials, d_pose_partials, d_scal;
  DevBuf<LmState> d_state;
  DevBuf<unsigned> d_ticket;        // k_cost_linearize_by_pose: CTAs that have finished
  DevBuf<unsigned> d_pose_ticket;   // k_cost_linearize_by_pose: chunks of every pose that have finished
  DevBuf<double> d_Au[2];           // speculative pose side: undamped A (21) / a (6) sums per free pose and parameter buffer
  DevBuf<double> d_cost_partialsA;  // cost partials of k_cost_linearize_by_pose, one per pose-order chunk
  int n_chunksA_all = 0;            // free-pose chunks (the first n_chunksA) + fixed-pose chunks
  DevBuf<ba_iter_info> d_infos;
  int point_grid = 0, pose_grid = 0;
  LmState *h_state = nullptr;  // pinned
  double *h_scal = nullptr;    // pinned

  // graph
  cudaGraphExec_t graph_exec = nullptr;
  ba_options graph_opt{};       // kernel arguments are baked into the graph: rebuilt when options change
  long long graph_nodes = 0;    // kernel nodes per replay

  // comm
  std::shared_ptr<SharedComm> shared;   // keeps the communicator alive; `comm` mirrors shared->comm
  BandPeers band_peers{};               // snapshot taken when the plan was agreed (cap == 0: NCCL all-reduce of the band)
  ncclComm_t comm = nullptr;
  int rank = 0, n_ranks = 1;
  long long global_M = -1, global_n_obs = -1;

  long long launches = 0;
  std::vector<cudaEvent_t> ev;
};

static int ensure_stream(ba_solver *s) {
  if (!s->stream) {
    CUDA_TRY(cudaSetDevice(s->device));
    CUDA_TRY(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    s->own_stream = true;
  }
  pool_setup(s->device);
  g_alloc_stream = s->stream;
  return BA_OK;
}

static void destroy_graph(ba_solver *s) {
  if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
  s->graph_exec = nullptr;
}

extern "C" {

const char *ba_version(void) { return "ba_b200 0.1 (sm_100a)"; }

int ba_create(ba_solver **out, int device) {
  if (!out) return BA_ERR_INVALID;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    // fail loudly: there is no CPU fallback
    fprintf(stderr, "ba_b200: no CUDA device available (%s); the engine has no CPU fallback\n",
            e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    *out = nullptr;
    return BA_ERR_CUDA;
  }
  if (device < 0 || device >= count) return BA_ERR_INVALID;
  ba_solver *s = new ba_solver();
  s->device = device;
  s->sw = read_switches();
  *out = s;
  return BA_OK;
}

static void free_device(ba_solver *s) {
  destroy_graph(s);
  s->d_cams.release();
  for (int i = 0; i < 2; ++i) { s->d_poses[i].release(); s->d_points[i].release(); }
  s->d_obs_uv.release(); s->d_uvA.release(); s->d_obs_pose.release(); s->d_obs_point.release();
  s->d_obs_camflags.release(); s->d_pointA.release(); s->d_camA.release();
  s->d_poseidA.release(); s->d_pair_obs.release(); s->d_chunksA.release();
  s->d_pose_chunk_ptr.release(); s->d_pose_opt.release(); s->d_pair_pose.release(); s->d_pair_point.release();
  s->d_pair_end.release(); s->d_point_has_pairs.release(); s->d_point_free.release();
  s->d_split_points.release(); s->d_schur_chunks.release();
  s->d_tpt_point.release(); s->d_tpt_inc_start.release(); s->d_fallback_pairs.release(); s->d_fb_groups.release();
  s->d_inc_a.release(); s->d_inc_b.release(); s->d_tile_batches.release(); s->d_cta_batch_ptr.release(); s->d_cta_seg_ptr.release(); s->d_seg_off.release(); s->d_seg_win.release(); s->d_pose_seg.release(); s->d_stage.release(); s->d_chunks_fb.release(); s->d_chunk_pts_fb.release(); s->d_cpts_fb.release(); s->d_chunk_pair_count_fb.release(); s->d_point_fb.release();
  s->d_chol_rows.release(); s->d_chol_first.release(); s->d_chol_rows_ptr.release(); s->d_band.release();
  s->d_nd_nodes.release(); s->d_nd_level_nodes.release(); s->d_nd_cta_nodes.release(); s->d_nd_cta_ptr.release();
  s->d_nd_flags.release(); s->d_nd_helpers.release(); s->d_nd_L.release(); s->d_nd_U.release();
  s->d_ptblk.release(); s->d_Bsoa.release();
  s->d_A.release(); s->d_a.release(); s->d_partialsA.release(); s->d_Saug.release(); s->d_Scopy.release();
  s->d_x.release(); s->d_z.release(); s->d_linv.release(); s->d_Btx.release(); s->d_y.release();
  s->d_point_partials.release(); s->d_pose_partials.release(); s->d_scal.release(); s->d_state.release(); s->d_ticket.release(); s->d_pose_ticket.release();
  s->d_Au[0].release(); s->d_Au[1].release(); s->d_cost_partialsA.release();
  s->d_infos.release();
  s->d_row_of_pos.release();
}

void ba_destroy(ba_solver *s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  g_alloc_stream = s->stream;
  free_device(s);
  if (s->stream) cudaStreamSynchronize(s->stream);
  for (auto e : s->ev) cudaEventDestroy(e);
  pinned_put(s->h_state);
  pinned_put(s->h_scal);
  s->comm = nullptr;
  s->shared.reset();
  if (s->own_stream && s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

int ba_reset(ba_solver *s) {
  if (!s) return BA_ERR_INVALID;
  s->cam_slot.clear(); s->h_cams.clear(); s->n_cam = 0;
  s->h_poses.clear(); s->h_points.clear(); s->h_pose_fixed.clear(); s->h_point_fixed.clear();
  s->h_obs_cam.clear(); s->h_obs_pose.clear(); s->h_obs_point.clear(); s->h_obs_uv.clear();
  s->n_obs = 0; s->N_total = s->M_total = s->N = s->M = 0; s->P = 0;
  s->n_rows = 0; s->h_kept_row.clear(); s->h_kept_of_pos.clear();
  s->finalized = false;
  destroy_graph(s);
  return BA_OK;
}

const char *ba_last_error(const ba_solver *s) { return s ? s->err.c_str() : "null handle"; }

int ba_set_stream(ba_solver *s, void *cuda_stream) {
  if (!s) return BA_ERR_INVALID;
  if (s->own_stream && s->stream) cudaStreamDestroy(s->stream);
  s->stream = (cudaStream_t)cuda_stream;
  s->own_stream = false;
  destroy_graph(s);
  return BA_OK;
}
int ba_set_profile(ba_solver *s, int enable) { if (!s) return BA_ERR_INVALID; s->profile = enable != 0; return BA_OK; }
int ba_set_debug(ba_solver *s, int keep) { if (!s) return BA_ERR_INVALID; s->debug_keep = keep != 0; destroy_graph(s); return BA_OK; }

int ba_set_cameras(ba_solver *s, int n_cam, const int *ids, const double *intr, const double *T) {
  if (!s || n_cam <= 0 || n_cam > 256 || !ids || !intr || !T) return BA_ERR_INVALID;
  s->cam_slot.clear();
  s->h_cams.clear();
  s->n_cam = 0;
  for (int k = 0; k < n_cam; ++k) {
    if (s->cam_slot.count(ids[k])) continue;  // duplicate ids ignored (unordered_map::insert, :80)
    s->cam_slot[ids[k]] = s->n_cam++;
    for (int i = 0; i < 4; ++i) s->h_cams.push_back(intr[4 * k + i]);
    for (int i = 0; i < 12; ++i) s->h_cams.push_back(T[12 * k + i]);
  }
  s->finalized = false;
  return BA_OK;
}

int ba_set_poses(ba_solver *s, int n, const double *T_jw, const uint8_t *fixed) {
  if (!s || n < 0 || (n > 0 && !T_jw)) return BA_ERR_INVALID;
  s->h_poses.assign(T_jw, T_jw + (size_t)n * 12);
  s->h_pose_fixed.assign(n, 0);
  if (fixed) s->h_pose_fixed.assign(fixed, fixed + n);
  s->N_total = n;
  s->finalized = false;
  return BA_OK;
}

int ba_set_points(ba_solver *s, int m, const double *X, const uint8_t *fixed) {
  if (!s || m < 0 || (m > 0 && !X)) return BA_ERR_INVALID;
  s->h_points.assign(X, X + (size_t)m * 3);
  s->h_point_fixed.assign(m, 0);
  if (fixed) s->h_point_fixed.assign(fixed, fixed + m);
  s->M_total = m;
  s->finalized = false;
  return BA_OK;
}

int ba_set_observations(ba_solver *s, long long n_obs, const int *cam_id, const int *pose, const int *point,
                        const double *uv, long long *n_kept) {
  return ba_set_observations_scaled(s, n_obs, cam_id, pose, point, uv, 1.0, n_kept);
}

// pixels in the caller's units: multiplied by uv_scale (the reference's scaler_, full...cpp:176) during the copy
int ba_set_observations_scaled(ba_solver *s, long long n_obs, const int *cam_id, const int *pose, const int *point,
                               const double *uv, double uv_scale, long long *n_kept) {
  if (!s || n_obs < 0 || (n_obs > 0 && (!cam_id || !pose || !point || !uv))) return BA_ERR_INVALID;
  if (n_obs > 2000000000LL) { s->err = "too many observations for 32-bit indexing"; return BA_ERR_INVALID; }
  s->h_obs_cam.clear(); s->h_obs_pose.clear(); s->h_obs_point.clear(); s->h_obs_uv.clear();
  s->n_rows = n_obs;
  s->h_kept_row.clear();
  // fast path: every row valid (the common case) -> bulk copies and a table look-up of the camera slot
  {
    int max_id = -1, min_id = 0;
    for (auto &kv : s->cam_slot) { max_id = std::max(max_id, kv.first); min_id = std::min(min_id, kv.first); }
    if (min_id >= 0 && max_id < 4096) {
      std::vector<int> table(max_id + 1, -1);
      for (auto &kv : s->cam_slot) table[kv.first] = kv.second;
      const int Nt = s->N_total, Mt = s->M_total;
      long long bad = 0;
      std::atomic<long long> bad_total{0};
      parallel_ranges(n_obs, [&](long long lo_, long long hi_, int) {
        long long bad = 0;
        for (long long k = (long long)lo_; k < (long long)hi_; ++k) {
          const int c = cam_id[k];
          bad += (c < 0 || c > max_id || table[c] < 0 || pose[k] < 0 || pose[k] >= Nt || point[k] < 0 || point[k] >= Mt);
        }
        bad_total += bad;
      });
      bad = bad_total.load();
      if (bad == 0) {
        s->h_obs_cam.resize(n_obs);
        parallel_ranges(n_obs, [&](long long lo_, long long hi_, int) {
          for (long long k = (long long)lo_; k < (long long)hi_; ++k) s->h_obs_cam[k] = table[cam_id[k]];
        });
        s->h_obs_pose.resize(n_obs); s->h_obs_point.resize(n_obs); s->h_obs_uv.resize(2 * n_obs);
        parallel_ranges(n_obs, [&](long long lo_, long long hi_, int) {
          std::memcpy(s->h_obs_pose.data() + lo_, pose + lo_, (size_t)(hi_ - lo_) * sizeof(int));
          std::memcpy(s->h_obs_point.data() + lo_, point + lo_, (size_t)(hi_ - lo_) * sizeof(int));
          if (uv_scale == 1.0) std::memcpy(s->h_obs_uv.data() + 2 * lo_, uv + 2 * lo_, (size_t)(hi_ - lo_) * 2 * sizeof(double));
          else for (long long k = 2 * lo_; k < 2 * hi_; ++k) s->h_obs_uv[k] = uv[k] * uv_scale;
        });
        s->n_obs = n_obs;
        if (n_kept) *n_kept = s->n_obs;
        s->finalized = false;
        return BA_OK;
      }
    }
  }
  s->h_obs_cam.reserve(n_obs); s->h_obs_pose.reserve(n_obs); s->h_obs_point.reserve(n_obs);
  s->h_obs_uv.reserve(2 * n_obs); s->h_kept_row.reserve(n_obs);
  for (long long k = 0; k < n_obs; ++k) {
    auto it = s->cam_slot.find(cam_id[k]);
    if (it == s->cam_slot.end()) continue;                       // "Invalid camera index." (:160-163)
    if (pose[k] < 0 || pose[k] >= s->N_total) continue;          // "Nonexisting pose." (:164-167)
    if (point[k] < 0 || point[k] >= s->M_total) continue;        // "Nonexisting point." (:168-171)
    s->h_obs_cam.push_back(it->second);
    s->h_obs_pose.push_back(pose[k]);
    s->h_obs_point.push_back(point[k]);
    s->h_obs_uv.push_back(uv[2 * k] * uv_scale);
    s->h_obs_uv.push_back(uv[2 * k + 1] * uv_scale);
    s->h_kept_row.push_back((int)k);
  }
  s->n_obs = (long long)s->h_obs_cam.size();
  if (n_kept) *n_kept = s->n_obs;
  s->finalized = false;
  return BA_OK;
}

// device copies of the envelope plan; again after ba_comm_init agreed on the global envelope
static int upload_cholesky_plan(ba_solver *s) {
  cudaStream_t st = s->stream;
  s->S_clean_outside_band = false;
  std::vector<int> rows = s->chol.rows;
  rows.push_back(0);
  CUDA_TRY(s->d_chol_rows.upload(rows, st));
  CUDA_TRY(s->d_chol_first.upload(s->chol.first_tile, st));
  CUDA_TRY(s->d_chol_rows_ptr.upload(s->chol.rows_ptr, st));
  s->chol.d_rows = s->d_chol_rows.p;
  s->chol.d_first_tile = s->d_chol_first.p;
  s->chol.d_rows_ptr = s->d_chol_rows_ptr.p;
  // partitioned banded solve: node table, level / CTA lists, factor and contribution-block workspaces
  NdPlan &nd = s->chol.nd;
  s->chol.nd_dev = NdDevice();
  if (s->chol.banded && nd.valid) {
    NdDevice &dv = s->chol.nd_dev;
    dv.smem = nd_smem_bytes(nd);
    dv.tpw = nd_tpw_for(nd.max_BT);
    if (dv.smem > kNdSmemLimit || dv.tpw < 0) {
      nd.valid = false;
    } else {
      CUDA_TRY(s->d_nd_nodes.upload(nd.nodes, st));
      CUDA_TRY(s->d_nd_level_nodes.upload(nd.level_nodes, st));
      CUDA_TRY(s->d_nd_cta_nodes.upload(nd.cta_nodes, st));
      CUDA_TRY(s->d_nd_cta_ptr.upload(nd.cta_ptr, st));
      CUDA_TRY(s->d_nd_flags.alloc(2 * nd.nodes.size() + nd.n_step_flags + 2));
      CUDA_TRY(s->d_nd_helpers.upload(nd.helper_nodes, st));
      CUDA_TRY(s->d_nd_L.alloc((size_t)nd.L_doubles));
      CUDA_TRY(s->d_nd_U.alloc((size_t)std::max<long long>(1, nd.U_doubles)));
      // entries of a parent's front that a child does not cover are never written: they must read as zero
      CUDA_TRY(cudaMemsetAsync(s->d_nd_U.p, 0, s->d_nd_U.n * sizeof(double), st));
      CUDA_TRY(cudaMemsetAsync(s->d_nd_flags.p, 0, s->d_nd_flags.n * sizeof(int), st));
      NdArgs a{};
      a.nodes = s->d_nd_nodes.p;
      a.n = nd.n; a.ld = nd.n + 1; a.bw = nd.bw;      // S and x are patched in at enqueue time
      a.Lws = s->d_nd_L.p; a.Uws = s->d_nd_U.p;
      a.flags = s->d_nd_flags.p; a.n_nodes = (int)nd.nodes.size();
      a.max_R8 = nd.max_R8; a.max_tiles = nd.max_tiles; a.max_KT = nd.max_KT;
      a.step_base = 2 * (int)nd.nodes.size();
      a.abort_idx = a.step_base + nd.n_step_flags;
      a.n_main = nd.n_ctas;
      a.helper_list = s->d_nd_helpers.p;
      a.use_helpers = 0;
      dv.level_args = a; dv.level_args.list = s->d_nd_level_nodes.p; dv.level_args.list_ptr = nullptr;
      dv.cta_args = a; dv.cta_args.list = s->d_nd_cta_nodes.p; dv.cta_args.list_ptr = s->d_nd_cta_ptr.p;
      dv.cta_args.use_helpers = nd.n_helpers > 0;
    }
  }
  // the reduced solve: BA_B200_BAND_MODE picks between the partition (if it is valid) and the serial window kernel
  CholeskyPlan &pl = s->chol;
  if (pl.banded && nd.valid && s->sw.band_mode >= 5)
    pl.path = s->sw.band_mode == 6 ? SolvePath::NdPersistent : SolvePath::NdLevels;
  else if (pl.banded)
    pl.path = SolvePath::Banded;
  else
    pl.path = pl.cluster_size > 0 ? SolvePath::Cluster : SolvePath::Dense;
  return BA_OK;
}

// Multi-GPU: the reduced solve is replicated, so every rank must factor the all-reduced S with the SAME plan, built
// from the co-visibility of ALL landmarks, not of its shard: min over ranks of the first co-visible pose.  Called by
// whichever comes second, ba_comm_init or ba_finalize.
static void ensure_band_exchange(SharedComm &sc, cudaStream_t st, long long count);
static int agree_on_envelope(ba_solver *s) {
  if (!s->comm || s->N <= 0) return BA_OK;
  cudaStream_t st = s->stream;
  g_alloc_stream = st;
  DevBuf<int> d_fp;
  CUDA_TRY(d_fp.upload(s->h_first_pose, st));
  ncclResult_t r = g_nccl.AllReduce(d_fp.p, d_fp.p, (size_t)s->N, ncclInt, ncclMin, s->comm, st);
  if (r != ncclSuccess) { s->err = "ncclAllReduce(envelope) failed"; return BA_ERR_NCCL; }
  CUDA_TRY(cudaMemcpyAsync(s->h_first_pose.data(), d_fp.p, (size_t)s->N * sizeof(int), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  d_fp.release();
  cholesky_make_plan(s->chol, 6 * s->N, s->h_first_pose, s->sw.chol_mode, s->sw.nd_depth, s->sw.nd_chunk);
  if (int rc = upload_cholesky_plan(s)) return rc;
  CUDA_TRY(cudaStreamSynchronize(st));
  // band exchange through peer memory (same count on every rank: the plan is global now)
  s->band_peers = BandPeers{};
  if (s->shared && s->chol.banded) {
    SharedComm &sc = *s->shared;
    const long long count = (long long)6 * s->N * (s->chol.bw + 2);
    ensure_band_exchange(sc, st, count);
    if (sc.band_ok && count <= sc.band_cap) {
      BandPeers bp{};
      for (int r = 0; r < kMaxRanks; ++r) { bp.buf[r] = sc.band_peer[r]; bp.flag[r] = sc.bflag_peer[r]; }
      bp.epoch = sc.d_band_epoch; bp.counters = sc.d_band_counters; bp.error = sc.d_error;
      bp.cap = sc.band_cap; bp.pslot = sc.band_pslot; bp.rank = sc.rank; bp.n_ranks = sc.n_ranks;
      s->band_peers = bp;
    }
  }
  return BA_OK;
}

int ba_finalize(ba_solver *s) {
  if (!s) return BA_ERR_INVALID;
  if (s->finalized) return BA_OK;
  if (s->n_cam == 0) { s->err = "no cameras"; return BA_ERR_STATE; }
  CUDA_TRY(cudaSetDevice(s->device));
  if (int rc = ensure_stream(s)) return rc;
  destroy_graph(s);
  const bool verbose = s->sw.verbose;
  auto tp0 = std::chrono::high_resolution_clock::now();
  auto lap = [&](const char *what) {
    if (!verbose) return;
    const auto now = std::chrono::high_resolution_clock::now();
    fprintf(stderr, "[ba_b200] finalize %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - tp0).count());
    tp0 = now;
  };
  const int Nt = s->N_total, Mt = s->M_total;
  const long long n = s->n_obs;
  // --- free indices in id order (FinalizeParameters :182-206; insertion order replaces hash order)
  s->h_pose_opt.assign(Nt, -1); s->h_point_opt.assign(Mt, -1);
  s->h_opt_pose.clear(); s->h_opt_point.clear();
  for (int j = 0; j < Nt; ++j) if (!s->h_pose_fixed[j]) { s->h_pose_opt[j] = (int)s->h_opt_pose.size(); s->h_opt_pose.push_back(j); }
  for (int i = 0; i < Mt; ++i) if (!s->h_point_fixed[i]) { s->h_point_opt[i] = (int)s->h_opt_point.size(); s->h_opt_point.push_back(i); }
  s->N = (int)s->h_opt_pose.size();
  s->M = (int)s->h_opt_point.size();
  // --- stable counting sort by pose, then by point  => order (point, pose, insertion)
  hvec<int> by_pose(n);
  std::vector<long long> pose_begin(Nt + 1, 0);   // observation range of every pose in by_pose order
  hvec<int> pose_to_point_order(n);               // position in POINT order of the q-th observation of the POSE order
  std::vector<long long> pt_q0;                   // observation range of every landmark in point order
  // point-ordered observation arrays: written by the scatter pass of the second sort
  hvec<double2> uv(n);
  hvec<int> o_pose(n), o_point(n), o_cf(n), o_pair(n);
  s->h_kept_of_pos.resize(n);
  s->d_row_of_pos.release();
  s->row_map_uploaded = false;
  {
    // both sorts: per-thread histograms over contiguous ranges of the input, bucket offsets per thread, parallel
    // scatter -- stable because every thread's range is contiguous and the ranges are ordered
    std::vector<long long> starts;
    auto counting_sort = [&](long long count, int n_buckets, auto &&key_of /*(q) -> bucket*/, auto &&place /*(q, position)*/) {
      const int nth = (int)std::min<long long>(host_threads(), std::max<long long>(1, count / 65536));
      std::vector<std::vector<int>> hist(nth, std::vector<int>((size_t)n_buckets, 0));
      parallel_ranges(nth, [&](long long t0, long long t1, int) {
        for (long long t = t0; t < t1; ++t) {
          std::vector<int> &h = hist[t];
          for (long long q = count * t / nth; q < count * (t + 1) / nth; ++q) h[key_of(q)]++;
        }
      }, 1);
      starts.assign((size_t)n_buckets + 1, 0);
      for (int b = 0; b < n_buckets; ++b) {
        long long run = starts[b];
        for (int t = 0; t < nth; ++t) { const int c = hist[t][b]; hist[t][b] = (int)run; run += c; }
        starts[b + 1] = run;
      }
      parallel_ranges(nth, [&](long long t0, long long t1, int) {
        for (long long t = t0; t < t1; ++t) {
          std::vector<int> &h = hist[t];
          for (long long q = count * t / nth; q < count * (t + 1) / nth; ++q) place(q, h[key_of(q)]++);
        }
      }, 1);
    };
    counting_sort(n, Nt, [&](long long k) { return s->h_obs_pose[k]; }, [&](long long k, int pos) { by_pose[pos] = (int)k; });
    pose_begin = starts;
    // the second scatter writes the point-ordered arrays directly (one random pass instead of sort + gather)
    counting_sort(n, Mt, [&](long long q) { return s->h_obs_point[by_pose[q]]; }, [&](long long q, int pos) {
      const int k = by_pose[q];
      const int ps = s->h_obs_pose[k], pt = s->h_obs_point[k];
      const bool pf = s->h_pose_opt[ps] >= 0, qf = s->h_point_opt[pt] >= 0;
      pose_to_point_order[q] = pos;
      s->h_kept_of_pos[pos] = k;
      uv[pos] = make_double2(s->h_obs_uv[2 * (size_t)k], s->h_obs_uv[2 * (size_t)k + 1]);
      o_pose[pos] = ps; o_point[pos] = pt;
      o_cf[pos] = s->h_obs_cam[k] | (pf ? kFlagPoseFree : 0) | (qf ? kFlagPointFree : 0);
    });
    pt_q0 = starts;                  // the bucket offsets of this sort ARE the observation range of every landmark
  }
  lap("counting sorts");
  // --- pairs, last-writer flags
  s->h_pair_pose.clear(); s->h_pair_point.clear();
  std::vector<int> point_has_pairs(Mt, 0);
  {
    // a pair starts at every free (pose, point) observation whose predecessor in point order belongs to another
    // (point, pose): flags, exclusive scan, fill -- three parallel passes instead of one serial scan
    hvec<int> pair_rank(n + 1);
    pair_rank[n] = 0;
    parallel_ranges(n, [&](long long lo_, long long hi_, int) {
      for (long long q = (long long)lo_; q < (long long)hi_; ++q) {
        const bool both = (o_cf[q] & kFlagPoseFree) && (o_cf[q] & kFlagPointFree);
        pair_rank[q] = (both && (q == 0 || o_point[q] != o_point[q - 1] || o_pose[q] != o_pose[q - 1])) ? 1 : 0;
      }
    });
    const long long n_pairs = exclusive_scan_inplace(pair_rank.data(), n);
    s->h_pair_pose.resize(n_pairs); s->h_pair_point.resize(n_pairs);
    parallel_ranges(n, [&](long long lo_, long long hi_, int) {
      for (long long q = (long long)lo_; q < (long long)hi_; ++q) {
        const bool both = (o_cf[q] & kFlagPoseFree) && (o_cf[q] & kFlagPointFree);
        const bool is_new = (q + 1 < n ? pair_rank[q + 1] : (int)n_pairs) != pair_rank[q];
        if (is_new) {
          s->h_pair_pose[pair_rank[q]] = s->h_pose_opt[o_pose[q]];
          s->h_pair_point[pair_rank[q]] = o_point[q];
          point_has_pairs[o_point[q]] = 1;
        }
        // rank counts the pairs that started before q: an observation of a pair that started earlier has index rank - 1
        o_pair[q] = both ? (is_new ? pair_rank[q] : pair_rank[q] - 1) : -1;
      }
    });
  }
  s->P = (long long)s->h_pair_pose.size();
  const long long P = s->P;
  std::vector<int2> pair_obs(P);
  // first / last observation of every pair (last = last inserted: stable sort) and the last-writer flag
  parallel_ranges(n, [&](long long lo_, long long hi_, int) {
    for (long long q = (long long)lo_; q < (long long)hi_; ++q) {
      const int pr = o_pair[q];
      if (pr < 0) continue;
      if (q == 0 || o_pair[q - 1] != pr) pair_obs[pr].x = (int)q;
      if (q + 1 == n || o_pair[q + 1] != pr) { pair_obs[pr].y = (int)q; o_cf[q] |= kFlagLastOfPair; }
    }
  });
  // pairs of one landmark are contiguous: group starts, then one past the last pair of the landmark for every pair
  std::vector<int> pair_end(P), grp_start;
  {
    hvec<int> gflag(P + 1);     // flags, exclusive scan, fill (parallel) instead of one serial pass over the pairs
    gflag[P] = 0;
    parallel_ranges(P, [&](long long lo_, long long hi_, int) {
      for (long long p = lo_; p < hi_; ++p) gflag[p] = (p == 0 || s->h_pair_point[p] != s->h_pair_point[p - 1]) ? 1 : 0;
    });
    const long long ng = exclusive_scan_inplace(gflag.data(), P);
    grp_start.resize((size_t)ng + 1);
    parallel_ranges(P, [&](long long lo_, long long hi_, int) {
      for (long long p = lo_; p < hi_; ++p)
        if ((p + 1 < P ? gflag[p + 1] : (int)ng) != gflag[p]) grp_start[gflag[p]] = (int)p;
    });
    grp_start[ng] = (int)P;
  }
  const long long n_grp = (long long)grp_start.size() - 1;
  parallel_ranges(n_grp, [&](long long lo_, long long hi_, int) {
    for (long long g = (long long)lo_; g < (long long)hi_; ++g)
      for (int p = grp_start[g]; p < grp_start[g + 1]; ++p) pair_end[p] = grp_start[g + 1];
  });
  lap("point order, pairs");
  // The point-ordered observation arrays (most of what this function uploads) are final: a helper thread sends them
  // while this thread builds the tile / chunk structures.  +1 sentinel so that obs_point[k+1] reads of the kernels
  // stay in bounds (the host code below never reads past n).
  cudaStream_t st = s->stream;
  o_point.push_back(-1);
  cudaError_t early_err = cudaSuccess;
  std::thread early_upload([&]() {
    cudaSetDevice(s->device);
    g_alloc_stream = st;
    cudaError_t e = s->d_obs_uv.upload(uv, st);
    if (e == cudaSuccess) e = s->d_obs_pose.upload(o_pose, st);
    if (e == cudaSuccess) e = s->d_obs_point.upload(o_point, st);
    if (e == cudaSuccess) e = s->d_pair_obs.upload(pair_obs, st);
    if (e == cudaSuccess) e = s->d_pair_end.upload(pair_end, st);
    early_err = e;
  });
  struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } early_joiner{early_upload};
  // --- observation range of every landmark in point order
  if ((long long)pt_q0.size() != (long long)Mt + 1) pt_q0.assign((size_t)Mt + 1, 0);   // (no observations at all)
  // --- tile chunks: runs of consecutive landmarks whose free poses fit one window of kTileW poses
  std::vector<SchurChunk> schur_chunks;
  std::vector<int> tpt_point, tpt_inc_start, fallback_pairs;
  hvec<int4> inc_a;
  hvec<int2> inc_b;
  std::vector<uint8_t> is_tile_point(Mt, 0);
  {
    struct Cand { int point, p0, p1, jmin, jmax, n_inc, ok; };
    // one candidate per landmark with pairs (parallel): window of its free poses, incidences = distinct poses
    // (free or fixed) observing it; pairs of a point are ascending in j_opt
    std::vector<Cand> all(n_grp);
    parallel_ranges(n_grp, [&](long long lo_, long long hi_, int) {
      for (long long g = (long long)lo_; g < (long long)hi_; ++g) {
        const int p0 = grp_start[g], p1 = grp_start[g + 1];
        Cand c{s->h_pair_point[p0], p0, p1, s->h_pair_pose[p0], s->h_pair_pose[p1 - 1], 0, 0};
        int prev = -1;
        for (long long q = pt_q0[c.point]; q < pt_q0[c.point + 1]; ++q)
          if (o_pose[q] != prev) { ++c.n_inc; prev = o_pose[q]; }
        c.ok = (c.jmax - c.jmin + 1 <= kTileW && c.n_inc <= kTileMaxInc) ? 1 : 0;
        all[g] = c;
      }
    });
    // Landmarks are grouped by (first pose, last pose) rather than by id: consecutive landmarks then share their
    // window, so a chunk's window is as narrow as its tracks and the GEMM operands are dense (mixed track lengths
    // in id order would widen every chunk to the longest track in it).  Stable counting sort on jmin * W + span.
    std::vector<Cand> cands;
    {
      std::vector<int> key_cnt((size_t)std::max(1, s->N) * kTileW + 1, 0);
      for (const Cand &c : all) {
        if (c.ok) key_cnt[(size_t)c.jmin * kTileW + (c.jmax - c.jmin) + 1]++;
        else for (int q = c.p0; q < c.p1; ++q) fallback_pairs.push_back(q);
      }
      for (size_t k = 1; k < key_cnt.size(); ++k) key_cnt[k] += key_cnt[k - 1];
      cands.resize(key_cnt.back());
      for (const Cand &c : all)
        if (c.ok) cands[key_cnt[(size_t)c.jmin * kTileW + (c.jmax - c.jmin)]++] = c;
    }
    // Small reduced system whose landmarks mostly do NOT fit a window (dense co-visibility, test_ba.cpp): the
    // by-point path ends in one dense tensor-core GEMM (k_schur_dense_gemm) that takes the few window landmarks
    // along for free, while a second, nearly empty persistent tile launch would cost its fixed 30 us
    if (dense_schur_fits(s->N) && 2 * (long long)cands.size() < n_grp) {
      for (const Cand &c : cands)
        for (int q = c.p0; q < c.p1; ++q) fallback_pairs.push_back(q);
      cands.clear();
    }
    // Greedy runs.  A run keeps growing while its pose window stays within kTileW; once it holds enough
    // landmarks to amortise the final flush it is also cut when the next landmark would WIDEN the window,
    // so that most chunks are exactly as wide as their landmarks' tracks (dense GEMM operands).
    constexpr int kMinPts = 6, kMinStart = 32, kGoodPts = 64, kMaxPts = 128;
    std::vector<int> tpt_cand, tpt_lo;   // candidate and window start of every tile landmark
    size_t i = 0;
    while (i < cands.size()) {
      int lo = cands[i].jmin, hi = cands[i].jmax;
      size_t e = i + 1;
      while (e < cands.size() && (int)(e - i) < kMaxPts) {
        const int nlo = std::min(lo, cands[e].jmin), nhi = std::max(hi, cands[e].jmax);
        if (nhi - nlo + 1 > kTileW) break;
        if ((int)(e - i) >= kGoodPts && (nlo != lo || nhi != hi)) break;
        if ((int)(e - i) >= kMinStart && cands[e].jmin != cands[i].jmin) break;  // keep a common first pose
        lo = nlo; hi = nhi; ++e;
      }
      if ((int)(e - i) >= kMinPts) {
        schur_chunks.push_back(SchurChunk{(int)tpt_cand.size(), (int)(e - i), lo, hi - lo + 1});
        for (size_t k = i; k < e; ++k) { tpt_cand.push_back((int)k); tpt_lo.push_back(lo); }
      } else {
        for (size_t k = i; k < e; ++k)
          for (int q = cands[k].p0; q < cands[k].p1; ++q) fallback_pairs.push_back(q);
      }
      i = e;
    }
    // incidence records of the tile landmarks: offsets by a scan over the incidence counts, then a parallel fill
    const long long n_tpt = (long long)tpt_cand.size();
    tpt_point.resize(n_tpt);
    tpt_inc_start.assign(n_tpt + 1, 0);
    for (long long t = 0; t < n_tpt; ++t) tpt_inc_start[t + 1] = tpt_inc_start[t] + cands[tpt_cand[t]].n_inc;
    inc_a.resize(tpt_inc_start[n_tpt]);
    inc_b.resize(tpt_inc_start[n_tpt]);
    parallel_ranges(n_tpt, [&](long long lo_, long long hi_, int) {
      for (long long t = (long long)lo_; t < (long long)hi_; ++t) {
        const int pt = cands[tpt_cand[t]].point, lo = tpt_lo[t];
        is_tile_point[pt] = 1;
        tpt_point[t] = pt;
        int w = tpt_inc_start[t];
        for (long long q = pt_q0[pt]; q < pt_q0[pt + 1];) {
          long long r = q;
          while (r < pt_q0[pt + 1] && o_pose[r] == o_pose[q]) ++r;
          const int pair = o_pair[q];
          inc_a[w] = make_int4((int)q, (int)(r - q), o_pose[q], pair);
          // .y: camera slots of the first two observations, so that the camera block can be fetched before the
          // observation's own record arrives
          inc_b[w] = make_int2(pair >= 0 ? s->h_pair_pose[pair] - lo : -1,
                               (o_cf[q] & kCamMask) | ((r - q > 1 ? (o_cf[q + 1] & kCamMask) : 0) << 8));
          ++w;
          q = r;
        }
      }
    });
    std::sort(fallback_pairs.begin(), fallback_pairs.end());
  }
  // --- flat list of 8-landmark batches over the tile chunks, split evenly over one persistent CTA per SM
  std::vector<int4> tile_batches;
  std::vector<int> cta_batch_ptr;
  std::vector<int> cta_seg_ptr;
  std::vector<long long> seg_off;
  std::vector<int4> seg_win;
  std::vector<int2> pose_seg;
  long long stage_doubles = 0;
  {
    int nt_max = 1;
    for (size_t c = 0; c < schur_chunks.size(); ++c) {
      const SchurChunk &sc = schur_chunks[c];
      nt_max = std::max(nt_max, (6 * sc.width + 7) / 8);
      for (int o = 0; o < sc.pt_count; o += kT2LB)
        tile_batches.push_back(make_int4(sc.pt_start + o, std::min(kT2LB, sc.pt_count - o), (int)c, (8 * ((6 * sc.width + 7) / 8)) | (sc.width << 16)));
    }
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device);
    TileLaunch &tl = s->tile_launch;
    tl.nt_max = nt_max;
    tl.ldE = 16 * ((nt_max + 1) / 2) + 4;   // whole super-tiles; 4 mod 16: conflict-free fragment reads
    tl.ldB = 16 * ((nt_max + 2) / 2) + 4;   // window + rhs tile column
    tl.bufD = kT2K * (tl.ldE + tl.ldB);
    tl.G = std::min(kT2MaxGroups, kT2SmemDoubles / tl.bufD);
    const long long nbt = (long long)tile_batches.size();
    tl.n_cta = (int)std::min<long long>(sms, std::max<long long>(1, (nbt + tl.G - 1) / tl.G));
    cta_batch_ptr.resize(tl.n_cta + 1);
    for (int k = 0; k <= tl.n_cta; ++k) cta_batch_ptr[k] = (int)(nbt * k / tl.n_cta);
    // deterministic flush: every (CTA, chunk) run of the batch list owns a staging window
    cta_seg_ptr.assign(tl.n_cta + 1, 0);
    pose_seg.assign(std::max(1, s->N), make_int2(0, 0));
    long long off = 0;
    int span = 0;
    for (int c = 0; c < tl.n_cta; ++c) {
      cta_seg_ptr[c] = (int)seg_off.size();
      int prev = -1;
      for (int fb = cta_batch_ptr[c]; fb < cta_batch_ptr[c + 1]; ++fb) {
        const int chunk = tile_batches[fb].z;
        if (chunk == prev) continue;
        prev = chunk;
        const SchurChunk &ch = schur_chunks[chunk];
        const int sg = (int)seg_off.size(), nr = 6 * ch.width;
        seg_off.push_back(off);
        seg_win.push_back(make_int4(6 * ch.jmin, nr, (int)(unsigned)(off & 0xffffffffLL), (int)(off >> 32)));
        off += (long long)nr * (nr + 1);
        span = std::max(span, nr - 1);
        for (int j = ch.jmin; j < ch.jmin + ch.width && j < s->N; ++j) {
          if (pose_seg[j].y == 0) pose_seg[j].x = sg;
          pose_seg[j].y = sg + 1;
        }
      }
    }
    cta_seg_ptr[tl.n_cta] = (int)seg_off.size();
    stage_doubles = off;
    s->stage_span = span;
  }
  lap("tile chunks, incidences");
  // --- Cholesky envelope plan from the co-visibility structure (first co-visible pose of every free pose)
  {
    std::vector<int> &first_pose = s->h_first_pose;
    first_pose.resize(s->N);
    for (int j = 0; j < s->N; ++j) first_pose[j] = j;
    for (long long g = 0; g < n_grp; ++g) {
      const int jmin = s->h_pair_pose[grp_start[g]];
      for (int q = grp_start[g]; q < grp_start[g + 1]; ++q) first_pose[s->h_pair_pose[q]] = std::min(first_pose[s->h_pair_pose[q]], jmin);
    }
    cholesky_make_plan(s->chol, 6 * s->N, first_pose, s->sw.chol_mode, s->sw.nd_depth, s->sw.nd_chunk);
  }
  s->n_schur_chunks = (int)schur_chunks.size();
  s->n_fallback_pairs = (int)fallback_pairs.size();
  lap("cholesky plan");
  // --- chunks of whole points (<= kThreads observations) of the by-point path (linearisation, back-substitution);
  //     longer points are split
  struct PointChunks {
    std::vector<Chunk> chunks;
    std::vector<int> chunk_pair_count, split_points, split_pairs;
    std::vector<int2> chunk_pts;
    std::vector<ChunkPoint> cpts;
  };
  auto build_point_chunks = [&](long long q_begin, long long q_end) {
    PointChunks pc;
    long long q = q_begin;
    const long long n = q_end;     // this part's observations end here (shadows the total on purpose)
    Chunk cur{0, 0, 0, 0};
    int cur_pairs_first = -1, cur_pairs_last = -1;
    long long cur_end = 0;
    auto flush = [&]() {
      if (cur.obs_count == 0) return;
      cur.pair_start = cur_pairs_first < 0 ? 0 : cur_pairs_first;
      pc.chunks.push_back(cur);
      pc.chunk_pair_count.push_back(cur_pairs_first < 0 ? 0 : cur_pairs_last - cur_pairs_first + 1);
      cur = Chunk{0, 0, 0, 0};
      cur_pairs_first = cur_pairs_last = -1;
    };
    auto add_range = [&](long long a, long long b) {  // obs [a,b) appended to the current chunk
      if (cur.obs_count == 0) cur.obs_start = (int)a;
      cur.obs_count += (int)(b - a);
      cur_end = b;
      for (long long r = a; r < b; ++r)
        if (o_pair[r] >= 0 && (o_cf[r] & kFlagLastOfPair)) { if (cur_pairs_first < 0) cur_pairs_first = o_pair[r]; cur_pairs_last = o_pair[r]; }
    };
    while (q < n) {
      long long e = q;
      while (e < n && o_point[e] == o_point[q]) ++e;
      const long long len = e - q;
      if (is_tile_point[o_point[q]]) { flush(); q = e; continue; }
      if (len > kThreads) {
        flush();
        if (s->h_point_opt[o_point[q]] >= 0) pc.split_points.push_back(o_point[q]);
        for (long long a = q; a < e; a += kThreads) {
          const long long b = std::min(e, a + kThreads);
          add_range(a, b);
          cur.flags = kChunkSplit;
          flush();
        }
        for (long long r = q; r < e; ++r)
          if (o_pair[r] >= 0 && (pc.split_pairs.empty() || pc.split_pairs.back() != o_pair[r])) pc.split_pairs.push_back(o_pair[r]);
      } else {
        // a chunk is a CONTIGUOUS observation range: close it when skipped landmarks lie in between
        if (cur.obs_count + len > kThreads || (cur.obs_count > 0 && cur_end != q)) flush();
        add_range(q, e);
      }
      q = e;
    }
    flush();
    // landmarks of each chunk (runs of equal point id inside the chunk's observation range)
    pc.chunk_pts.resize(pc.chunks.size());
    for (size_t c = 0; c < pc.chunks.size(); ++c) {
      pc.chunk_pts[c].x = (int)pc.cpts.size();
      const long long a = pc.chunks[c].obs_start, b = a + pc.chunks[c].obs_count;
      for (long long r = a; r < b;) {
        long long e = r;
        while (e < b && o_point[e] == o_point[r]) ++e;
        pc.cpts.push_back(ChunkPoint{o_point[r], (int)(r - a), (int)(e - r), s->h_point_opt[o_point[r]] >= 0 ? 1 : 0});
        r = e;
      }
      pc.chunk_pts[c].y = (int)pc.cpts.size() - pc.chunk_pts[c].x;
    }
    return pc;
  };
  // A serial scan; the landmark sequence is cut into kParts parts of about equal observation count (always kParts,
  // whatever the number of host threads: the chunking, hence the summation order on the device, must not depend on
  // the machine) that are scanned independently and concatenated
  PointChunks pc_fb;
  {
    constexpr int kParts = 16;
    long long cut[kParts + 1];
    cut[0] = 0; cut[kParts] = n;
    for (int p = 1; p < kParts; ++p) {
      const long long target = n * p / kParts;
      const int lm = (int)(std::lower_bound(pt_q0.begin(), pt_q0.end(), target) - pt_q0.begin());
      cut[p] = std::max(cut[p - 1], pt_q0[std::min(lm, Mt)]);
    }
    std::vector<PointChunks> parts(kParts);
    parallel_ranges(kParts, [&](long long lo_, long long hi_, int) {
      for (long long j = lo_; j < hi_; ++j) parts[j] = build_point_chunks(cut[j], cut[j + 1]);
    }, 1);
    for (PointChunks &src : parts) {
      PointChunks &dst = pc_fb;
      const int cp0 = (int)dst.cpts.size();
      dst.chunks.insert(dst.chunks.end(), src.chunks.begin(), src.chunks.end());
      dst.chunk_pair_count.insert(dst.chunk_pair_count.end(), src.chunk_pair_count.begin(), src.chunk_pair_count.end());
      dst.split_points.insert(dst.split_points.end(), src.split_points.begin(), src.split_points.end());
      dst.split_pairs.insert(dst.split_pairs.end(), src.split_pairs.begin(), src.split_pairs.end());
      for (int2 cp : src.chunk_pts) dst.chunk_pts.push_back(make_int2(cp.x + cp0, cp.y));
      dst.cpts.insert(dst.cpts.end(), src.cpts.begin(), src.cpts.end());
    }
  }
  s->n_chunks_fb = (int)pc_fb.chunks.size();
  s->n_split = (int)pc_fb.split_points.size();
  s->n_split_pairs = (int)pc_fb.split_pairs.size();
  lap("point chunks");
  // --- pose-ordered arrays (free poses only) and their chunks
  // the pose-ordered copies of the observations (uvA, pointA, camA, poseidA) are gathered ON THE DEVICE from the
  // point-ordered arrays through permA (position in point order of every pose-ordered slot): 4 B/obs instead of 28
  hvec<int> permA;
  std::vector<ChunkA> chunksA; std::vector<int> pose_chunk_ptr(s->N + 1, 0);
  {
    // A-order = the by_pose order restricted to free poses: offsets per pose, chunks per pose (serial over poses),
    // then a parallel gather of the observations
    std::vector<long long> a_begin(Nt + 1, 0);
    for (int ps = 0; ps < Nt; ++ps)
      a_begin[ps + 1] = a_begin[ps] + (s->h_pose_opt[ps] >= 0 ? pose_begin[ps + 1] - pose_begin[ps] : 0);
    const long long nA = a_begin[Nt];
    permA.resize(pose_begin[Nt]);   // free poses first (nA slots), the observations of fixed poses behind them
    // Chunk size: enough observations per thread to amortise the 27-value block reduction at the end of a chunk
    // (it costs as much as two observations), while the grid still fills the GPU (two 256-thread CTAs per SM);
    // a pose's observations are split evenly over its chunks.
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device);
    // measured on B200 (C3: 4 / 8 / 13 observations per thread -> 55 / 47 / 56 us; C4: 4 / 8 / 16 -> 0.46 / 0.41 /
    // 0.39 ms): about three CTAs per slot, between 4 and 16 observations per thread
    const int per_thread = (int)std::min<long long>(16, std::max<long long>(4, nA / ((long long)3 * sms * kThreads)));
    const long long chunk_cap = (long long)kThreads * per_thread;
    for (int ps = 0; ps < Nt; ++ps) {
      const int j = s->h_pose_opt[ps];
      const long long len = a_begin[ps + 1] - a_begin[ps];
      if (j < 0 || len == 0) continue;
      pose_chunk_ptr[j] = (int)chunksA.size();
      const long long nck = (len + chunk_cap - 1) / chunk_cap;
      const long long sz = ((len + nck - 1) / nck + 31) / 32 * 32;
      for (long long a = a_begin[ps]; a < a_begin[ps + 1]; a += sz)
        chunksA.push_back(ChunkA{(int)a, (int)(std::min(a_begin[ps + 1], a + sz) - a), j, 0});
    }
    parallel_ranges(Nt, [&](long long lo_, long long hi_, int) {
      for (int ps = (int)lo_; ps < (int)hi_; ++ps) {
        if (s->h_pose_opt[ps] < 0) continue;
        const long long len = pose_begin[ps + 1] - pose_begin[ps];
        for (long long r = 0; r < len; ++r) {
          permA[a_begin[ps] + r] = pose_to_point_order[pose_begin[ps] + r];
        }
      }
    }, 1);
    // poses without observations keep an empty chunk range: fix up the CSR (chunks are in pose order)
    std::vector<int> cnt(s->N, 0);
    for (auto &c : chunksA) cnt[c.j_opt]++;
    pose_chunk_ptr[0] = 0;
    for (int j = 0; j < s->N; ++j) pose_chunk_ptr[j + 1] = pose_chunk_ptr[j] + cnt[j];
    // observations of FIXED poses, behind the free ones (chunks with j_opt = -1): k_cost_linearize_by_pose walks them
    // for the cost only, so the first n_chunksA chunks are the ones with pose-side partials (d_partialsA)
    s->n_chunksA = (int)chunksA.size();
    long long f_at = nA;
    std::vector<long long> f_begin(Nt, -1);
    for (int ps = 0; ps < Nt; ++ps) {
      const long long len = pose_begin[ps + 1] - pose_begin[ps];
      if (s->h_pose_opt[ps] >= 0 || len == 0) continue;
      f_begin[ps] = f_at;
      const long long nck = (len + chunk_cap - 1) / chunk_cap;
      const long long sz = ((len + nck - 1) / nck + 31) / 32 * 32;
      for (long long a = f_at; a < f_at + len; a += sz)
        chunksA.push_back(ChunkA{(int)a, (int)(std::min(f_at + len, a + sz) - a), -1, 0});
      f_at += len;
    }
    if (f_at > nA) {
      for (int ps = 0; ps < Nt; ++ps) {
        if (f_begin[ps] < 0) continue;
        const long long len = pose_begin[ps + 1] - pose_begin[ps];
        for (long long r = 0; r < len; ++r) permA[f_begin[ps] + r] = pose_to_point_order[pose_begin[ps] + r];
      }
    }
  }
  s->n_chunksA_all = (int)chunksA.size();
  lap("pose order");
  // --- upload
  early_upload.join();
  if (early_err != cudaSuccess) { s->err = std::string("upload of the observation arrays: ") + cudaGetErrorString(early_err); return BA_ERR_CUDA; }
  std::vector<uint8_t> point_free(Mt);
  for (int i = 0; i < Mt; ++i) point_free[i] = s->h_point_fixed[i] ? 0 : 1;
  CUDA_TRY(s->d_cams.upload(s->h_cams, st));
  CUDA_TRY(s->d_poses[0].upload(s->h_poses, st));
  CUDA_TRY(s->d_poses[1].upload(s->h_poses, st));
  CUDA_TRY(s->d_points[0].upload(s->h_points, st));
  CUDA_TRY(s->d_points[1].upload(s->h_points, st));
  CUDA_TRY(s->d_obs_camflags.upload(o_cf, st));
  {
    const size_t nA = permA.size();
    DevBuf<int> d_perm;
    CUDA_TRY(d_perm.upload(permA, st));
    CUDA_TRY(s->d_uvA.alloc(nA)); CUDA_TRY(s->d_pointA.alloc(nA)); CUDA_TRY(s->d_camA.alloc(nA)); CUDA_TRY(s->d_poseidA.alloc(nA));
    if (nA > 0)
      k_gather_pose_order<<<(unsigned)std::min<size_t>((nA + 255) / 256, 148 * 16), 256, 0, st>>>(
          (long long)nA, d_perm.p, s->d_obs_uv.p, s->d_obs_point.p, s->d_obs_camflags.p, s->d_obs_pose.p, s->d_uvA.p,
          s->d_pointA.p, s->d_camA.p, s->d_poseidA.p);
    CUDA_TRY(cudaGetLastError());
    d_perm.release();   // stream-ordered: freed after the gather
  }
  CUDA_TRY(s->d_chunksA.upload(chunksA, st));
  CUDA_TRY(s->d_pose_chunk_ptr.upload(pose_chunk_ptr, st));
  CUDA_TRY(s->d_pose_opt.upload(s->h_pose_opt, st));
  CUDA_TRY(s->d_pair_pose.upload(s->h_pair_pose, st));
  {
    std::vector<int> pp = s->h_pair_point;
    pp.push_back(-1);
    CUDA_TRY(s->d_pair_point.upload(pp, st));
  }
  CUDA_TRY(s->d_point_has_pairs.upload(point_has_pairs, st));
  CUDA_TRY(s->d_point_free.upload(point_free, st));
  if (int rc = upload_cholesky_plan(s)) return rc;
  CUDA_TRY(s->d_schur_chunks.upload(schur_chunks, st));
  CUDA_TRY(s->d_tpt_point.upload(tpt_point, st));
  s->n_tpt = (int)tpt_point.size();
  CUDA_TRY(s->d_tpt_inc_start.upload(tpt_inc_start, st));
  CUDA_TRY(s->d_inc_a.upload(inc_a, st));
  CUDA_TRY(s->d_inc_b.upload(inc_b, st));
  CUDA_TRY(s->d_tile_batches.upload(tile_batches, st));
  CUDA_TRY(s->d_cta_batch_ptr.upload(cta_batch_ptr, st));
  CUDA_TRY(s->d_cta_seg_ptr.upload(cta_seg_ptr, st));
  CUDA_TRY(s->d_seg_off.upload(seg_off, st));
  CUDA_TRY(s->d_seg_win.upload(seg_win, st));
  CUDA_TRY(s->d_pose_seg.upload(pose_seg, st));
  CUDA_TRY(s->d_stage.alloc((size_t)std::max<long long>(1, stage_doubles)));
  CUDA_TRY(s->d_chunks_fb.upload(pc_fb.chunks, st));
  CUDA_TRY(s->d_chunk_pts_fb.upload(pc_fb.chunk_pts, st));
  CUDA_TRY(s->d_cpts_fb.upload(pc_fb.cpts, st));
  CUDA_TRY(s->d_chunk_pair_count_fb.upload(pc_fb.chunk_pair_count, st));
  {
    std::vector<uint8_t> point_fb(Mt);
    for (int i = 0; i < Mt; ++i) point_fb[i] = (!s->h_point_fixed[i] && !is_tile_point[i]) ? 1 : 0;
    CUDA_TRY(s->d_point_fb.upload(point_fb, st));
  }
  CUDA_TRY(s->d_fallback_pairs.upload(fallback_pairs, st));
  {
    // the pairs of a landmark are contiguous in the pair numbering: ranges of the sorted fallback list
    std::vector<int2> fb_groups;
    for (size_t k = 0; k < fallback_pairs.size();) {
      size_t e = k + 1;
      while (e < fallback_pairs.size() && fallback_pairs[e] == fallback_pairs[e - 1] + 1 &&
             s->h_pair_point[fallback_pairs[e]] == s->h_pair_point[fallback_pairs[k]]) ++e;
      fb_groups.push_back(make_int2(fallback_pairs[k], fallback_pairs[k] + (int)(e - k)));
      k = e;
    }
    s->n_fb_groups = (int)fb_groups.size();
    CUDA_TRY(s->d_fb_groups.upload(fb_groups, st));
  }
  CUDA_TRY(s->d_split_points.upload(pc_fb.split_points, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  lap("uploads");
  // --- block storage
  s->Mp = ((size_t)Mt + 31) / 32 * 32;
  s->Pp = ((size_t)P + 31) / 32 * 32;
  const size_t nS = (size_t)6 * s->N + 1;
  CUDA_TRY(s->d_ptblk.alloc(std::max<size_t>(1, kPtBlk * s->Mp)));
  // B blocks in global memory: by-point pairs, and every pair when they are kept for ba_debug_dump (the tile build
  // keeps its blocks on chip, their back-substitution forms them again)
  const bool keep_B = s->n_fallback_pairs > 0 || s->debug_keep;
  if (keep_B) CUDA_TRY(s->d_Bsoa.alloc(std::max<size_t>(1, 18 * s->Pp)));
  else s->d_Bsoa.release();
  CUDA_TRY(s->d_A.alloc(std::max<size_t>(1, (size_t)s->N * 36)));
  CUDA_TRY(s->d_a.alloc(std::max<size_t>(1, (size_t)s->N * 6)));
  CUDA_TRY(s->d_partialsA.alloc(std::max<size_t>(1, (size_t)s->n_chunksA * 27)));
  CUDA_TRY(s->d_Saug.alloc(nS * nS));
  s->S_clean_outside_band = false;
  CUDA_TRY(s->d_x.alloc(std::max<size_t>(1, (size_t)6 * s->N)));
  CUDA_TRY(s->d_z.alloc(std::max<size_t>(1, (size_t)6 * s->N)));
  CUDA_TRY(s->d_linv.alloc(std::max<size_t>(1, cholesky_linv_doubles(6 * s->N))));
  CUDA_TRY(s->d_Btx.alloc(std::max<size_t>(1, 3 * s->Mp)));
  CUDA_TRY(s->d_y.alloc(std::max<size_t>(1, (size_t)Mt * 3)));
  CUDA_TRY(cudaMemsetAsync(s->d_ptblk.p, 0, s->d_ptblk.n * sizeof(double), st));
  if (keep_B) CUDA_TRY(cudaMemsetAsync(s->d_Bsoa.p, 0, s->d_Bsoa.n * sizeof(double), st));
  CUDA_TRY(cudaMemsetAsync(s->d_x.p, 0, s->d_x.n * sizeof(double), st));
  CUDA_TRY(cudaMemsetAsync(s->d_y.p, 0, s->d_y.n * sizeof(double), st));
  CUDA_TRY(cudaMemsetAsync(s->d_Btx.p, 0, s->d_Btx.n * sizeof(double), st));
  CUDA_TRY(cudaMemsetAsync(s->d_A.p, 0, s->d_A.n * sizeof(double), st));
  CUDA_TRY(cudaMemsetAsync(s->d_a.p, 0, s->d_a.n * sizeof(double), st));
  s->point_grid = std::max(1, (Mt + kThreads - 1) / kThreads);
  s->pose_grid = std::max(1, (Nt + kThreads - 1) / kThreads);
  CUDA_TRY(s->d_point_partials.alloc(2 * (size_t)s->point_grid));
  CUDA_TRY(s->d_pose_partials.alloc(2 * (size_t)s->pose_grid));
  CUDA_TRY(s->d_scal.alloc(8));
  CUDA_TRY(s->d_state.alloc(1));
  CUDA_TRY(s->d_ticket.alloc(1));
  CUDA_TRY(cudaMemsetAsync(s->d_ticket.p, 0, sizeof(unsigned), st));
  CUDA_TRY(s->d_pose_ticket.alloc(std::max(1, s->N)));
  CUDA_TRY(cudaMemsetAsync(s->d_pose_ticket.p, 0, s->d_pose_ticket.n * sizeof(unsigned), st));
  for (int b = 0; b < 2; ++b) {   // a pose without observations keeps its zeros
    CUDA_TRY(s->d_Au[b].alloc(std::max<size_t>(1, (size_t)s->N * 27)));
    CUDA_TRY(cudaMemsetAsync(s->d_Au[b].p, 0, s->d_Au[b].n * sizeof(double), st));
  }
  CUDA_TRY(s->d_cost_partialsA.alloc(std::max(1, s->n_chunksA_all)));
  CUDA_TRY(cudaMemsetAsync(s->d_state.p, 0, sizeof(LmState), st));
  CUDA_TRY(cudaMemsetAsync(s->d_scal.p, 0, 8 * sizeof(double), st));
  static_assert(sizeof(LmState) <= kPinnedBlock, "pinned block");
  lap("block storage: device");
  if (!s->h_state) CUDA_TRY(pinned_get((void **)&s->h_state));
  if (!s->h_scal) CUDA_TRY(pinned_get((void **)&s->h_scal));
  CUDA_TRY(cudaStreamSynchronize(st));
  lap("block storage");
  s->finalized = true;
  return agree_on_envelope(s);   // no-op on a single GPU
}

int ba_update_parameters(ba_solver *s, const double *T_jw, const double *X) {
  if (!s || !s->finalized) return BA_ERR_STATE;
  CUDA_TRY(cudaSetDevice(s->device));
  // the accepted parameters live in buffer `cur`; reset to buffer 0.  A set that is not supplied keeps its accepted
  // values: they are copied from buffer `cur` into the other buffer before `cur` is reset
  if (!T_jw || !X) {
    LmState hs;
    CUDA_TRY(cudaMemcpyAsync(&hs, s->d_state.p, sizeof(hs), cudaMemcpyDeviceToHost, s->stream));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    const int cur = hs.cur & 1;
    if (!T_jw)
      CUDA_TRY(cudaMemcpyAsync(s->d_poses[cur ^ 1].p, s->d_poses[cur].p, (size_t)s->N_total * 12 * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
    if (!X)
      CUDA_TRY(cudaMemcpyAsync(s->d_points[cur ^ 1].p, s->d_points[cur].p, (size_t)s->M_total * 3 * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
  }
  if (T_jw) {
    s->h_poses.assign(T_jw, T_jw + (size_t)s->N_total * 12);
    CUDA_TRY(cudaMemcpyAsync(s->d_poses[0].p, T_jw, (size_t)s->N_total * 12 * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->d_poses[1].p, s->d_poses[0].p, (size_t)s->N_total * 12 * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
  }
  if (X) {
    s->h_points.assign(X, X + (size_t)s->M_total * 3);
    CUDA_TRY(cudaMemcpyAsync(s->d_points[0].p, X, (size_t)s->M_total * 3 * sizeof(double), cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->d_points[1].p, s->d_points[0].p, (size_t)s->M_total * 3 * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
  }
  CUDA_TRY(cudaMemsetAsync(s->d_state.p, 0, sizeof(LmState), s->stream));
  return BA_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// iteration enqueue
// ---------------------------------------------------------------------------
namespace {

struct Phase { enum { Lin = 0, Schur, Solve, Backsub, Update, End, Count }; };

static DecideArgs make_decide_args(ba_solver *s, const ba_options *opt) {
  DecideArgs g;
  g.cost_partials = s->d_cost_partialsA.p; g.n_cost = s->n_chunksA_all;
  g.point_partials = s->d_point_partials.p; g.n_point = s->point_grid;
  g.pose_partials = s->d_pose_partials.p; g.n_pose = s->pose_grid;
  g.scal = s->d_scal.p;
  g.thr_step = (double)opt->threshold_step_size;
  g.thr_cost = (double)opt->threshold_cost_change;
  g.dec_ratio = (double)opt->decrease_ratio_lambda;
  g.inc_ratio = (double)opt->increase_ratio_lambda;
  g.inverse_scaler = opt->inverse_scaler;
  const long long gM = s->global_M >= 0 ? s->global_M : s->M;
  const long long gO = s->global_n_obs >= 0 ? s->global_n_obs : s->n_obs;
  g.n_obs_global = (double)gO;
  g.n_params_global = (double)(s->N + gM);
  g.max_iteration = opt->max_num_iterations;
  g.n_ranks = s->n_ranks;
  g.method = opt->method;
  return g;
}

// Banded plans clear only the band of Saug per iteration (enqueue_build); everything else is cleared once here,
// before the first iteration (and before the iteration is captured into a graph).
static int ensure_S_clean(ba_solver *s) {
  if (!s->chol.banded || s->S_clean_outside_band) return BA_OK;
  const size_t ld = (size_t)6 * s->N + 1;
  CUDA_TRY(cudaMemsetAsync(s->d_Saug.p, 0, ld * ld * sizeof(double), s->stream));
  s->S_clean_outside_band = true;
  return BA_OK;
}

// Large banded reduced systems (C4: 1.15 GB dense) clear only the band of S per iteration: everything outside it stays
// zero once ensure_S_clean has cleared it.  A small one is cleared faster by one linear memset.
static bool clears_band_only(const ba_solver *s) {
  const size_t ld = (size_t)s->chol.n + 1;
  return s->chol.banded && ld * ld * sizeof(double) > s->sw.band_clear_min;
}

// Enqueue the build (K1..K4) on the stream.  ev: optional events at phase boundaries.
static int enqueue_build(ba_solver *s, const ba_options *opt, cudaEvent_t *ev) {
  cudaStream_t st = s->stream;
  const Params prm{{s->d_poses[0].p, s->d_poses[1].p}, {s->d_points[0].p, s->d_points[1].p}};
  const double thres = (double)opt->threshold_huber_loss;
  const LmState *dst = s->d_state.p;
  const int ld = 6 * s->N + 1;
  if (ev) cudaEventRecord(ev[Phase::Lin], st);
  // On a banded plan k_tile_reduce WRITES every band entry and rhs entry of S (damped pose-side sums + windows) and
  // the rows of A / a, so nothing is cleared here and k_pose_diag is not launched (BA_B200_REDUCE_STORES=0: clear +
  // k_pose_diag + adding reduce)
  const bool reduce_stores = s->sw.reduce_stores && s->N > 0 && s->n_schur_chunks > 0 && s->chol.banded &&
                             s->S_clean_outside_band && std::max(s->stage_span, s->chol.bw) + 2 <= 2 * 96;
  if (reduce_stores) {
    // nothing to clear
  } else if (clears_band_only(s) && s->S_clean_outside_band) {
    // the build, the factorisation and the exchange only touch row r's columns r .. r + bw and the last column
    const int n = 6 * s->N;
    const long long total = (long long)n * (s->chol.bw + 2);
    k_clear_band<<<(int)std::min<long long>(148 * 8, (total + 255) / 256), 256, 0, st>>>(s->d_Saug.p, n, ld, s->chol.bw, dst);
    s->launches++;
  } else {
    cudaMemsetAsync(s->d_Saug.p, 0, (size_t)ld * ld * sizeof(double), st);
  }
  if (s->n_split > 0) {
    k_zero_split<<<(s->n_split + 127) / 128, 128, 0, st>>>(s->d_split_points.p, s->n_split, s->d_ptblk.p, s->Mp, dst);
    s->launches++;
  }
  // pose side first: k_pose_diag STORES the damped diagonal blocks and the rhs, everything after it adds.  The sums
  // of the accepted buffer are there (the trial-cost pass of the previous iteration, or the initial pass)
  if (s->N > 0 && !reduce_stores) {
    k_pose_diag<<<(s->N + 3) / 4, 128, 0, st>>>(s->N, s->d_Au[0].p, s->d_Au[1].p, s->d_A.p, s->d_a.p, s->d_Saug.p, ld, dst);
    s->launches++;
  }
  // landmarks on the by-point path (poses do not fit a window, or not enough neighbours for a chunk)
  if (s->n_chunks_fb > 0) {
    k_linearize_by_point<<<s->n_chunks_fb, kThreads, 0, st>>>(s->d_chunks_fb.p, s->d_chunk_pts_fb.p, s->d_cpts_fb.p,
                                                              s->d_obs_uv.p, s->d_obs_pose.p, s->d_obs_point.p,
                                                              s->d_obs_camflags.p, prm, s->d_cams.p, thres,
                                                              s->d_ptblk.p, s->Mp, dst);
    s->launches++;
  }
  // B of the by-point pairs; with debug_keep, of every pair (the tile build keeps its own on chip), for ba_debug_dump
  const int n_blk = s->debug_keep ? (int)s->P : s->n_fallback_pairs;
  if (n_blk > 0) {
    const int grid = (n_blk + kThreads - 1) / kThreads;
    const int *list = s->debug_keep ? nullptr : s->d_fallback_pairs.p;
    if (opt->b_accumulate)
      k_pair_blocks<true><<<grid, kThreads, 0, st>>>(n_blk, list, s->d_pair_obs.p, s->d_obs_uv.p, s->d_obs_pose.p,
                                                     s->d_obs_point.p, s->d_obs_camflags.p, prm, s->d_cams.p, thres,
                                                     s->d_Bsoa.p, s->Pp, dst);
    else
      k_pair_blocks<false><<<grid, kThreads, 0, st>>>(n_blk, list, s->d_pair_obs.p, s->d_obs_uv.p, s->d_obs_pose.p,
                                                      s->d_obs_point.p, s->d_obs_camflags.p, prm, s->d_cams.p, thres,
                                                      s->d_Bsoa.p, s->Pp, dst);
    s->launches++;
  }
  if (s->n_chunks_fb > 0) {
    k_finish_points<<<(s->M_total + 127) / 128, 128, 0, st>>>(s->M_total, s->d_point_fb.p, s->d_ptblk.p, s->Mp, dst);
    s->launches++;
  }
  if (ev) cudaEventRecord(ev[Phase::Schur], st);
  // tile landmarks: linearisation + C^-1 + Schur products fused (DMMA)
  if (s->n_schur_chunks > 0) {
    static PerDeviceOnce once;
    if (once.first()) {
      cudaFuncSetAttribute(k_build_tiles<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kT2SmemBytes);
      cudaFuncSetAttribute(k_build_tiles<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kT2SmemBytes);
    }
    const TileLaunch &tl = s->tile_launch;
    const size_t smem = (size_t)tl.G * tl.bufD * sizeof(double);
    if (opt->b_accumulate)
      k_build_tiles<true><<<tl.n_cta, kT2Threads, smem, st>>>(
          s->d_schur_chunks.p, s->d_tile_batches.p, s->d_cta_batch_ptr.p, tl, s->d_tpt_point.p, s->d_tpt_inc_start.p,
          s->d_inc_a.p, s->d_inc_b.p, s->d_obs_uv.p, s->d_obs_camflags.p, prm, s->d_cams.p, thres,
          s->d_ptblk.p, s->Mp, s->d_cta_seg_ptr.p, s->d_seg_off.p, s->d_stage.p, dst);
    else
      k_build_tiles<false><<<tl.n_cta, kT2Threads, smem, st>>>(
          s->d_schur_chunks.p, s->d_tile_batches.p, s->d_cta_batch_ptr.p, tl, s->d_tpt_point.p, s->d_tpt_inc_start.p,
          s->d_inc_a.p, s->d_inc_b.p, s->d_obs_uv.p, s->d_obs_camflags.p, prm, s->d_cams.p, thres,
          s->d_ptblk.p, s->Mp, s->d_cta_seg_ptr.p, s->d_seg_off.p, s->d_stage.p, dst);
    s->launches++;
    if (s->N > 0) {
      k_tile_reduce<<<6 * s->N, 96, 0, st>>>(6 * s->N, ld, s->stage_span, s->d_seg_win.p, s->d_pose_seg.p, s->d_stage.p,
                                             s->d_Saug.p, reduce_stores ? s->chol.bw : -1, s->d_Au[0].p, s->d_Au[1].p,
                                             s->d_A.p, s->d_a.p, dst);
      s->launches++;
    }
  }
  if (s->n_fallback_pairs > 0 && dense_schur_fits(s->N)) {
    // small reduced system (dense co-visibility): the products as a tensor-core GEMM over 64 x 64 tiles
    const int nT = (ld + 63) / 64, tile_pairs = nT * (nT + 1) / 2;
    const int split_k = std::max(1, std::min((s->n_fb_groups + kDenseLm - 1) / kDenseLm, (2 * 148 + tile_pairs - 1) / tile_pairs));
    k_schur_dense_gemm<<<tile_pairs * split_k, 256, 0, st>>>(s->d_fb_groups.p, s->n_fb_groups, split_k, s->d_pair_pose.p,
                                                           s->d_pair_point.p, s->d_Bsoa.p, s->Pp, s->d_ptblk.p, s->Mp,
                                                           s->d_Saug.p, ld, dst);
    s->launches++;
  } else if (s->n_fallback_pairs > 0) {
    k_schur_pairs_list<<<(s->n_fallback_pairs + 127) / 128, 128, 0, st>>>(
        s->n_fallback_pairs, s->d_fallback_pairs.p, s->d_pair_pose.p, s->d_pair_point.p, s->d_pair_end.p,
        s->d_Bsoa.p, s->Pp, s->d_ptblk.p, s->Mp, s->d_Saug.p, ld, dst);
    s->launches++;
  }
  return BA_OK;
}

static int enqueue_allreduce_S(ba_solver *s) {
  if (!s->comm) return BA_OK;
  const int n = 6 * s->N;
  const size_t ld = (size_t)n + 1;
  ncclResult_t r;
  if (s->chol.banded && n > 0 && s->band_peers.cap > 0) {
    const int grid = (int)std::min<long long>(148 * 8, ((long long)n * (s->chol.bw + 2) + 127) / 128);
    // BA_B200_BAND_XCHG: 1 (default) one-shot pushes, 2 two-shot (reduce-scatter + all-gather).  Measured on 8 B200:
    // C4 (3.5 MB band) 0.507 vs 0.502 ms per iteration, weak C3 (0.7 MB) 0.487 vs 0.507 ms; on 2 B200 the two-shot form
    // is 0.1 ms slower on C4 -- the exchange is bound by its hand-overs, not by NVLink bytes, so fewer hand-overs win
    if (s->sw.band_xchg == 1) {
      k_band_push1<<<grid, 128, 0, s->stream>>>(s->d_Saug.p, n, (int)ld, s->chol.bw, s->band_peers, s->d_state.p);
      k_band_pull1<<<grid, 128, 0, s->stream>>>(s->d_Saug.p, n, (int)ld, s->chol.bw, s->band_peers, s->d_state.p);
      s->launches += 2;
      return BA_OK;
    }
    const int grid_r = (int)std::min<long long>(148 * 8, ((long long)(n / s->n_ranks + 1) * (s->chol.bw + 2) + 127) / 128);
    k_band_push<<<grid, 128, 0, s->stream>>>(s->d_Saug.p, n, (int)ld, s->chol.bw, s->band_peers, s->d_state.p);
    k_band_reduce<<<grid_r, 128, 0, s->stream>>>(n, s->chol.bw, s->band_peers, s->d_state.p);
    k_band_pull<<<grid, 128, 0, s->stream>>>(s->d_Saug.p, n, (int)ld, s->chol.bw, s->band_peers, s->d_state.p);
    s->launches += 3;
    return BA_OK;
  }
  if (s->chol.banded && n > 0) {
    // every rank holds the same plan (ba_comm_init agreed on the global envelope): band + rhs only
    const int bw = s->chol.bw;
    const size_t count = (size_t)n * (bw + 2);
    if (s->d_band.n < count) { s->err = "band exchange buffer not allocated"; return BA_ERR_STATE; }
    k_band_pack<<<n, 128, 0, s->stream>>>(s->d_Saug.p, n, (int)ld, bw, s->d_band.p, s->d_state.p);
    r = g_nccl.AllReduce(s->d_band.p, s->d_band.p, count, ncclDouble, ncclSum, s->comm, s->stream);
    k_band_unpack<<<n, 128, 0, s->stream>>>(s->d_Saug.p, n, (int)ld, bw, s->d_band.p, s->d_state.p);
    s->launches += 2;
  } else {
    r = g_nccl.AllReduce(s->d_Saug.p, s->d_Saug.p, ld * ld, ncclDouble, ncclSum, s->comm, s->stream);
  }
  if (r != ncclSuccess) { s->err = "ncclAllReduce(S) failed"; return BA_ERR_NCCL; }
  return BA_OK;
}
static int enqueue_allreduce_scal(ba_solver *s) {
  if (!s->comm) return BA_OK;
  ncclResult_t r = g_nccl.AllReduce(s->d_scal.p, s->d_scal.p, 5, ncclDouble, ncclSum, s->comm, s->stream);
  if (r != ncclSuccess) { s->err = "ncclAllReduce(scalars) failed"; return BA_ERR_NCCL; }
  return BA_OK;
}

static int enqueue_solve_backsub(ba_solver *s, const ba_options *opt, cudaEvent_t *ev) {
  cudaStream_t st = s->stream;
  const Params prm{{s->d_poses[0].p, s->d_poses[1].p}, {s->d_points[0].p, s->d_points[1].p}};
  const ParamsW prw{{s->d_poses[0].p, s->d_poses[1].p}, {s->d_points[0].p, s->d_points[1].p}};
  const LmState *dst = s->d_state.p;
  const int n = 6 * s->N, ld = n + 1;
  if (ev) cudaEventRecord(ev[Phase::Solve], st);
  if (s->debug_keep && s->d_Scopy.p) {
    cudaMemcpyAsync(s->d_Scopy.p, s->d_Saug.p, (size_t)ld * ld * sizeof(double), cudaMemcpyDeviceToDevice, st);
  }
  const bool gd = opt->method == BA_METHOD_GRADIENT_DESCENT;
  if (gd) {
    if (s->N > 0) { k_gd_poses<<<(s->N + 127) / 128, 128, 0, st>>>(s->N, s->d_a.p, s->d_x.p, dst); s->launches++; }
  } else if (n > 0) {
    cholesky_solve_enqueue(s->chol, s->d_Saug.p, s->d_x.p, s->d_z.p, s->d_linv.p, dst, st, &s->launches, s->sw.verbose);
  }
  if (ev) cudaEventRecord(ev[Phase::Backsub], st);
  // sum_j B^T x_j of every landmark with pairs: plain stores, except the pieces of a split by-point landmark (reds;
  // tile landmarks are never split)
  if (!gd && s->n_split_pairs > 0) cudaMemsetAsync(s->d_Btx.p, 0, 3 * s->Mp * sizeof(double), st);
  if (!gd && s->n_tpt > 0) {
    const int grid = (4 * s->n_tpt + kThreads - 1) / kThreads;
    const double thres = (double)opt->threshold_huber_loss;
    if (opt->b_accumulate)
      k_backsub_tiles<true><<<grid, kThreads, 0, st>>>(
          s->n_tpt, s->d_tpt_point.p, s->d_tpt_inc_start.p, s->d_inc_a.p, s->d_inc_b.p, s->d_obs_uv.p,
          s->d_obs_camflags.p, s->d_pose_opt.p, prm, s->d_cams.p, thres, s->d_x.p, s->d_Btx.p, s->Mp, dst);
    else
      k_backsub_tiles<false><<<grid, kThreads, 0, st>>>(
          s->n_tpt, s->d_tpt_point.p, s->d_tpt_inc_start.p, s->d_inc_a.p, s->d_inc_b.p, s->d_obs_uv.p,
          s->d_obs_camflags.p, s->d_pose_opt.p, prm, s->d_cams.p, thres, s->d_x.p, s->d_Btx.p, s->Mp, dst);
    s->launches++;
  }
  if (!gd && s->n_fallback_pairs > 0) {
    k_backsub_pairs<<<s->n_chunks_fb, kThreads, 0, st>>>(s->d_chunks_fb.p, s->d_chunk_pair_count_fb.p, s->d_pair_pose.p,
                                                         s->d_pair_point.p, s->d_Bsoa.p, s->Pp, s->d_x.p,
                                                         s->d_Btx.p, s->Mp, dst);
    s->launches++;
  }
  k_backsub_points_update_poses<<<s->point_grid + s->pose_grid, kThreads, 0, st>>>(
      s->point_grid, s->M_total, s->d_point_has_pairs.p, s->d_point_free.p, s->d_ptblk.p, s->Mp, s->d_Btx.p, s->d_y.p, prm,
      prw, s->d_point_partials.p, opt->method, s->N_total, s->d_pose_opt.p, s->d_x.p, s->d_A.p, s->d_a.p,
      s->d_pose_partials.p, dst);
  s->launches++;
  return BA_OK;
}

// trial cost (which = 1) or initial cost (which = 0, ignore_done) together with the pose-side sums at those parameters
static void launch_cost_linearize(ba_solver *s, const ba_options *opt, int which, int decide_here, int ignore_done,
                                  const DecideArgs &g) {
  const Params prm{{s->d_poses[0].p, s->d_poses[1].p}, {s->d_points[0].p, s->d_points[1].p}};
  k_cost_linearize_by_pose<<<std::max(1, s->n_chunksA_all), kThreads, 0, s->stream>>>(
      s->d_chunksA.p, s->d_uvA.p, s->d_pointA.p, s->d_camA.p, s->d_poseidA.p, s->n_chunksA_all, prm, which, s->d_cams.p,
      (double)opt->threshold_huber_loss, s->d_partialsA.p, s->d_cost_partialsA.p, s->d_pose_chunk_ptr.p,
      s->d_pose_ticket.p, s->d_Au[0].p, s->d_Au[1].p, s->d_ticket.p, decide_here, ignore_done, g, s->d_state.p,
      s->d_infos.p, (int)s->d_infos.n);
}

static int enqueue_update_decide(ba_solver *s, const ba_options *opt, cudaEvent_t *ev) {
  cudaStream_t st = s->stream;
  LmState *dst = s->d_state.p;
  if (ev) cudaEventRecord(ev[Phase::Update], st);
  // the pose update (se3Exp, pose part of the model change) ran with the back-substitution of the landmarks
  // (k_backsub_points_update_poses; a forked graph branch for it cost more than the 9 us it hid)
  DecideArgs g = make_decide_args(s, opt);
  // single GPU: the trial-cost pass also takes the decision; several GPUs exchange the partial sums first
  launch_cost_linearize(s, opt, 1, s->comm ? 0 : 1, 0, g);
  s->launches++;
  if (s->comm && s->shared && s->shared->peer_ok) {
    k_exchange_decide<<<1, kThreads, 0, st>>>(g, s->shared->table(), dst, s->d_infos.p, (int)s->d_infos.n);
    s->launches++;
  } else if (s->comm) {
    k_reduce_scalars<<<1, kThreads, 0, st>>>(g, 0, dst);
    if (int rc = enqueue_allreduce_scal(s)) return rc;
    k_decide<<<1, 1, 0, st>>>(g, dst, s->d_infos.p, (int)s->d_infos.n);
    s->launches += 2;
  }
  if (ev) cudaEventRecord(ev[Phase::End], st);
  return BA_OK;
}

// the persistent partitioned solve hands over between CTAs through flags with a bounded spin; a lost hand-over
// (CTAs not co-resident) is reported instead of hanging the device
static int check_nd_error(ba_solver *s) {
  if (s->shared && s->shared->peer_ok) {
    int perr = 0;
    CUDA_TRY(cudaMemcpy(&perr, s->shared->d_error, sizeof(int), cudaMemcpyDeviceToHost));
    if (perr) { s->err = "multi-GPU scalar exchange: a peer rank did not answer"; return BA_ERR_NCCL; }
  }
  if (!s->chol.nd.valid || !s->d_nd_flags.p) return BA_OK;
  int err = 0;
  CUDA_TRY(cudaMemcpy(&err, s->d_nd_flags.p + 2 * s->chol.nd.nodes.size() + s->chol.nd.n_step_flags + 1, sizeof(int), cudaMemcpyDeviceToHost));
  if (err) { s->err = "partitioned reduced solve: hand-over between CTAs timed out"; return BA_ERR_CUDA; }
  return BA_OK;
}

static int enqueue_iteration(ba_solver *s, const ba_options *opt, cudaEvent_t *ev) {
  if (int rc = enqueue_build(s, opt, ev)) return rc;
  if (int rc = enqueue_allreduce_S(s)) return rc;
  if (int rc = enqueue_solve_backsub(s, opt, ev)) return rc;
  return enqueue_update_decide(s, opt, ev);
}

// Cost of the accepted parameters (buffer cur) into scal[0], ordered over the pose-order chunks (and summed over the
// ranks), together with their pose-side sums in Au[cur]: the initial cost of ba_solve and the sums its first
// iteration starts from.  Ignores `done`.
static int enqueue_current_cost(ba_solver *s, const ba_options *opt) {
  DecideArgs g = make_decide_args(s, opt);
  launch_cost_linearize(s, opt, 0, 0, 1, g);
  k_reduce_scalars<<<1, kThreads, 0, s->stream>>>(g, 1, s->d_state.p);
  s->launches += 2;
  return enqueue_allreduce_scal(s);
}

}  // namespace

extern "C" {

int ba_cost(ba_solver *s, double *cost) {
  if (!s || !cost) return BA_ERR_INVALID;
  if (int rc = ba_finalize(s)) return rc;
  CUDA_TRY(cudaSetDevice(s->device));
  // no options here, so no Huber threshold: the pose-side sums this leaves in Au[cur] are not meaningful.  Nothing
  // reads them -- ba_solve and ba_build_only form Au[cur] again before they use it
  ba_options o{};
  o.max_num_iterations = 1;
  if (int rc = enqueue_current_cost(s, &o)) return rc;
  CUDA_TRY(cudaMemcpyAsync(s->h_scal, s->d_scal.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  *cost = s->h_scal[0];
  return BA_OK;
}

int ba_observation_residuals(ba_solver *s, double threshold, double *residuals, uint8_t *status, long long *counts) {
  if (!s) return BA_ERR_INVALID;
  if (!(threshold >= 0.0)) { s->err = "ba_observation_residuals: threshold must be >= 0 (NaN is invalid)"; return BA_ERR_INVALID; }
  if (int rc = ba_finalize(s)) return rc;
  CUDA_TRY(cudaSetDevice(s->device));
  if (int rc = ensure_stream(s)) return rc;
  cudaStream_t st = s->stream;
  const long long n = s->n_obs, n_rows = s->n_rows;
  if (!s->row_map_uploaded) {
    // point-order position -> input row: the kept index, or the input row of the kept row when some were dropped
    if (s->h_kept_row.empty()) {
      CUDA_TRY(s->d_row_of_pos.upload(s->h_kept_of_pos, st));
    } else {
      hvec<int> row(n);
      parallel_ranges(n, [&](long long lo_, long long hi_, int) {
        for (long long q = lo_; q < hi_; ++q) row[q] = s->h_kept_row[s->h_kept_of_pos[q]];
      });
      CUDA_TRY(s->d_row_of_pos.upload(row, st));
      CUDA_TRY(cudaStreamSynchronize(st));   // `row` is freed on return
    }
    s->row_map_uploaded = true;
  }
  DevBuf<double2> d_res;
  DevBuf<uint8_t> d_status;
  DevBuf<unsigned long long> d_counts;
  struct Release {   // stream-ordered frees on every return path
    DevBuf<double2> &a; DevBuf<uint8_t> &b; DevBuf<unsigned long long> &c;
    ~Release() { a.release(); b.release(); c.release(); }
  } release{d_res, d_status, d_counts};
  const bool dropped = n_rows > n;
  if (residuals) {
    CUDA_TRY(d_res.alloc((size_t)n_rows));
    if (dropped) CUDA_TRY(cudaMemsetAsync(d_res.p, 0xff, (size_t)n_rows * sizeof(double2), st));   // all-ones: NaN
  }
  if (status) {
    CUDA_TRY(d_status.alloc((size_t)n_rows));
    if (dropped) CUDA_TRY(cudaMemsetAsync(d_status.p, BA_OBS_DROPPED, (size_t)n_rows, st));
  }
  if (counts) {
    CUDA_TRY(d_counts.alloc(3));
    CUDA_TRY(cudaMemsetAsync(d_counts.p, 0, 3 * sizeof(unsigned long long), st));
  }
  if (n > 0) {
    const Params prm{{s->d_poses[0].p, s->d_poses[1].p}, {s->d_points[0].p, s->d_points[1].p}};
    const unsigned grid = (unsigned)std::min<long long>((n + kThreads - 1) / kThreads, 148LL * 8);
    k_obs_residuals<<<grid, kThreads, 0, st>>>(n, s->d_obs_uv.p, s->d_obs_pose.p, s->d_obs_point.p, s->d_obs_camflags.p,
                                               s->d_row_of_pos.p, prm, s->d_cams.p, threshold, s->d_state.p, d_res.p,
                                               d_status.p, d_counts.p);
    CUDA_TRY(cudaGetLastError());
  }
  unsigned long long h_counts[3] = {0, 0, 0};
  if (residuals && n_rows > 0)
    CUDA_TRY(cudaMemcpyAsync(residuals, d_res.p, (size_t)n_rows * sizeof(double2), cudaMemcpyDeviceToHost, st));
  if (status && n_rows > 0)
    CUDA_TRY(cudaMemcpyAsync(status, d_status.p, (size_t)n_rows, cudaMemcpyDeviceToHost, st));
  if (counts) CUDA_TRY(cudaMemcpyAsync(h_counts, d_counts.p, sizeof(h_counts), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (counts) {
    for (int i = 0; i < 3; ++i) counts[i] = (long long)h_counts[i];
    counts[BA_OBS_DROPPED] = n_rows - n;
  }
  return BA_OK;
}

int ba_solve(ba_solver *s, const ba_options *opt_in, ba_iter_info *infos, int cap, ba_result *result) {
  if (!s || !opt_in) return BA_ERR_INVALID;
  const auto t0 = std::chrono::high_resolution_clock::now();
  if (int rc = ba_finalize(s)) return rc;
  CUDA_TRY(cudaSetDevice(s->device));
  if (int rc = ensure_stream(s)) return rc;
  ba_options opt = *opt_in;
  if (opt.inverse_scaler == 0.0) opt.inverse_scaler = 100.0;
  if (opt.check_every <= 0) opt.check_every = 8;
  if (opt.method < 0 || opt.method > BA_METHOD_GRADIENT_DESCENT) { s->err = "unknown ba_options.method"; return BA_ERR_INVALID; }
  if (opt.method == BA_METHOD_GRADIENT_DESCENT && s->comm) { s->err = "gradient descent is single-GPU only"; return BA_ERR_STATE; }
  const int max_it = opt.max_num_iterations;
  cudaStream_t st = s->stream;
  s->launches = 0;
  CUDA_TRY(s->d_infos.alloc(std::max(1, max_it)));
  if (int rc = ensure_S_clean(s)) return rc;
  // --- initial cost (:707), the pose-side sums of the initial parameters, and the state
  if (int rc = enqueue_current_cost(s, &opt)) return rc;
  k_init_state<<<1, 1, 0, st>>>(s->d_state.p, s->d_scal.p, (double)opt.initial_lambda);
  s->launches++;
  CUDA_TRY(cudaMemcpyAsync(s->h_scal, s->d_scal.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, st));
  struct EventPair {   // destroyed on every return path
    cudaEvent_t a = nullptr, b = nullptr;
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
  } ev_pair;
  CUDA_TRY(cudaEventCreate(&ev_pair.a));
  CUDA_TRY(cudaEventCreate(&ev_pair.b));
  cudaEvent_t ev_begin = ev_pair.a, ev_end = ev_pair.b;
  CUDA_TRY(cudaEventRecord(ev_begin, st));
  double phase_ms[Phase::Count] = {0};
  int it_launched = 0;
  int n_done = 0, converged = 0;
  const bool use_graph = opt.use_graph != 0 && !s->profile;   // NCCL collectives are captured with the kernels
  if (s->debug_keep) {   // (debug switched on after ba_finalize: the B blocks may not be allocated yet)
    const size_t ld = (size_t)6 * s->N + 1;
    CUDA_TRY(s->d_Scopy.alloc(ld * ld));
    CUDA_TRY(s->d_Bsoa.alloc(std::max<size_t>(1, 18 * s->Pp)));
  }
  if (s->comm && s->chol.banded && s->N > 0) {
    // exchange buffer of the band: allocated HERE, outside the capture (an allocation inside would become a graph
    // node that allocates again at every replay)
    const size_t count = (size_t)6 * s->N * (s->chol.bw + 2);
    if (s->d_band.n < count) CUDA_TRY(s->d_band.alloc(count));
  }
  if (use_graph && max_it > 0) {
    ba_options key = opt;
    key.check_every = 0;
    if (!s->graph_exec || std::memcmp(&s->graph_opt, &key, sizeof(key)) != 0) {
      destroy_graph(s);
      cudaGraph_t graph;
      const long long l0 = s->launches;
      CUDA_TRY(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
      const int rc = enqueue_iteration(s, &opt, nullptr);
      const cudaError_t e = cudaStreamEndCapture(st, &graph);
      if (rc) return rc;
      if (e != cudaSuccess) { s->err = std::string("graph capture: ") + cudaGetErrorString(e); return BA_ERR_CUDA; }
      s->graph_nodes = s->launches - l0;
      s->launches = l0;
      CUDA_TRY(cudaGraphInstantiate(&s->graph_exec, graph, 0));
      cudaGraphDestroy(graph);
      s->graph_opt = key;
    }
  }
  std::vector<cudaEvent_t> &evp = s->ev;
  while (it_launched < max_it) {
    const int batch = std::min(opt.check_every, max_it - it_launched);
    for (int b = 0; b < batch; ++b) {
      if (use_graph) {
        CUDA_TRY(cudaGraphLaunch(s->graph_exec, st));
      } else {
        cudaEvent_t *ev = nullptr;
        if (s->profile) {
          const size_t need = (size_t)(it_launched + b + 1) * Phase::Count;
          while (evp.size() < need) { cudaEvent_t e; CUDA_TRY(cudaEventCreate(&e)); evp.push_back(e); }
          ev = &evp[(size_t)(it_launched + b) * Phase::Count];
        }
        if (int rc = enqueue_iteration(s, &opt, ev)) return rc;
      }
    }
    it_launched += batch;
    CUDA_TRY(cudaMemcpyAsync(s->h_state, s->d_state.p, sizeof(LmState), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (s->h_state->done) break;
  }
  CUDA_TRY(cudaEventRecord(ev_end, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { s->err = std::string("kernel failure: ") + cudaGetErrorString(e); return BA_ERR_CUDA; }
  }
  if (int rc = check_nd_error(s)) return rc;
  if (max_it > 0) {
    n_done = s->h_state->iteration;
    converged = s->h_state->converged;
  }
  float dev_ms = 0.f;
  cudaEventElapsedTime(&dev_ms, ev_begin, ev_end);
  if (use_graph) s->launches += s->graph_nodes * it_launched;
  if (s->profile && !use_graph) {
    for (int it = 0; it < std::min(n_done, it_launched); ++it) {
      for (int ph = 0; ph < Phase::End; ++ph) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, evp[(size_t)it * Phase::Count + ph], evp[(size_t)it * Phase::Count + ph + 1]);
        phase_ms[ph] += ms;
      }
    }
  }
  std::vector<ba_iter_info> h_infos(std::max(1, n_done));
  if (n_done > 0)
    CUDA_TRY(cudaMemcpy(h_infos.data(), s->d_infos.p, (size_t)n_done * sizeof(ba_iter_info), cudaMemcpyDeviceToHost));
  const double per_iter_ms = n_done > 0 ? dev_ms / n_done : 0.0;
  for (int i = 0; i < n_done; ++i) h_infos[i].iter_time = per_iter_ms;
  if (infos) for (int i = 0; i < std::min(n_done, cap); ++i) infos[i] = h_infos[i];
  if (result) {
    std::memset(result, 0, sizeof(*result));
    result->n_iterations = n_done;
    result->converged = converged;
    result->initial_cost = s->h_scal[0];
    result->final_cost = max_it > 0 ? s->h_state->prev_cost : s->h_scal[0];
    result->device_time_ms = dev_ms;
    result->t_linearize_ms = phase_ms[Phase::Lin];
    result->t_schur_ms = phase_ms[Phase::Schur];
    result->t_solve_ms = phase_ms[Phase::Solve];
    result->t_backsub_ms = phase_ms[Phase::Backsub];
    result->t_update_cost_ms = phase_ms[Phase::Update];
    result->kernel_launches = s->launches;
    result->total_time_ms =
        std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t0).count();
  }
  return BA_OK;
}

int ba_build_only(ba_solver *s, const ba_options *opt_in, double lambda, int do_solve) {
  if (!s || !opt_in) return BA_ERR_INVALID;
  if (int rc = ba_finalize(s)) return rc;
  CUDA_TRY(cudaSetDevice(s->device));
  if (int rc = ensure_stream(s)) return rc;
  ba_options opt = *opt_in;
  cudaStream_t st = s->stream;
  // state: keep `cur`, set lambda, not done
  CUDA_TRY(cudaMemcpyAsync(s->h_state, s->d_state.p, sizeof(LmState), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  s->h_state->lambda = lambda;
  s->h_state->done = 0;
  CUDA_TRY(cudaMemcpyAsync(s->d_state.p, s->h_state, sizeof(LmState), cudaMemcpyHostToDevice, st));
  if (s->debug_keep) {
    const size_t ldc = (size_t)6 * s->N + 1;
    CUDA_TRY(s->d_Scopy.alloc(ldc * ldc));
    CUDA_TRY(s->d_Bsoa.alloc(std::max<size_t>(1, 18 * s->Pp)));
  }
  if (int rc = ensure_S_clean(s)) return rc;
  // the pose-side sums at the accepted parameters (Au[cur]), then the build of an iteration
  DecideArgs g = make_decide_args(s, &opt);
  launch_cost_linearize(s, &opt, 0, /*decide_here*/0, /*ignore_done*/1, g);
  if (int rc = enqueue_build(s, &opt, nullptr)) return rc;
  if (int rc = enqueue_allreduce_S(s)) return rc;
  if (do_solve) {
    if (int rc = enqueue_solve_backsub(s, &opt, nullptr)) return rc;
  } else if (s->debug_keep) {
    const size_t ld = (size_t)6 * s->N + 1;
    CUDA_TRY(s->d_Scopy.alloc(ld * ld));
    CUDA_TRY(cudaMemcpyAsync(s->d_Scopy.p, s->d_Saug.p, ld * ld * sizeof(double), cudaMemcpyDeviceToDevice, st));
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { s->err = std::string("kernel failure: ") + cudaGetErrorString(e); return BA_ERR_CUDA; }
  return check_nd_error(s);
}

static int current_buffer(ba_solver *s, int *cur) {
  CUDA_TRY(cudaMemcpy(s->h_state, s->d_state.p, sizeof(LmState), cudaMemcpyDeviceToHost));
  *cur = s->h_state->cur & 1;
  return BA_OK;
}

int ba_get_poses(ba_solver *s, double *T_jw) {
  if (!s || !s->finalized || !T_jw) return BA_ERR_STATE;
  CUDA_TRY(cudaSetDevice(s->device));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  int cur;
  if (int rc = current_buffer(s, &cur)) return rc;
  CUDA_TRY(cudaMemcpy(T_jw, s->d_poses[cur].p, (size_t)s->N_total * 12 * sizeof(double), cudaMemcpyDeviceToHost));
  return BA_OK;
}

int ba_get_points(ba_solver *s, double *X) {
  if (!s || !s->finalized || !X) return BA_ERR_STATE;
  CUDA_TRY(cudaSetDevice(s->device));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  int cur;
  if (int rc = current_buffer(s, &cur)) return rc;
  CUDA_TRY(cudaMemcpy(X, s->d_points[cur].p, (size_t)s->M_total * 3 * sizeof(double), cudaMemcpyDeviceToHost));
  return BA_OK;
}

int ba_get_sizes(ba_solver *s, long long *o) {
  if (!s || !o) return BA_ERR_INVALID;
  if (int rc = ba_finalize(s)) return rc;
  o[0] = s->N; o[1] = s->M; o[2] = s->P; o[3] = s->n_obs; o[4] = s->N_total; o[5] = s->M_total;
  return BA_OK;
}

long long ba_debug_dump(ba_solver *s, int which, double *buf) {
  if (!s || !s->finalized) return BA_ERR_STATE;
  cudaSetDevice(s->device);
  cudaStreamSynchronize(s->stream);
  const int N = s->N, M = s->M, n = 6 * N, ld = n + 1;
  const long long P = s->P;
  auto fetch = [&](const double *d, size_t cnt) {
    std::vector<double> h(cnt);
    if (cnt) cudaMemcpy(h.data(), d, cnt * sizeof(double), cudaMemcpyDeviceToHost);
    return h;
  };
  switch (which) {
    case 0: if (buf) { auto h = fetch(s->d_A.p, (size_t)N * 36); std::copy(h.begin(), h.end(), buf); } return (long long)N * 36;
    case 1: if (buf) { auto h = fetch(s->d_a.p, (size_t)N * 6); std::copy(h.begin(), h.end(), buf); } return (long long)N * 6;
    case 2: case 3: case 4: {
      const int w = which == 3 ? 3 : 9;
      if (buf) {
        auto h = fetch(s->d_ptblk.p, kPtBlk * s->Mp);
        const int sym[9] = {0, 1, 2, 1, 3, 4, 2, 4, 5};
        for (int io = 0; io < M; ++io) {
          const int i = s->h_opt_point[io];
          if (which == 3) for (int k = 0; k < 3; ++k) buf[(size_t)io * 3 + k] = h[(PB_b + k) * s->Mp + i];
          else {
            const int base = which == 2 ? PB_Cd : PB_Cinv;
            for (int k = 0; k < 9; ++k) buf[(size_t)io * 9 + k] = h[(base + sym[k]) * s->Mp + i];
          }
        }
      }
      return (long long)M * w;
    }
    case 5:   // every pair's B is stored only with debug_keep (the tile build keeps its blocks on chip)
      if (P > 0 && (!s->debug_keep || s->d_Bsoa.n < 18 * s->Pp)) return BA_ERR_STATE;
      if (buf) {
        auto h = fetch(s->d_Bsoa.p, 18 * s->Pp);
        for (long long p = 0; p < P; ++p)
          for (int k = 0; k < 18; ++k) buf[p * 18 + k] = h[(size_t)k * s->Pp + p];
      }
      return P * 18;
    case 6: case 7: {
      if (!s->d_Scopy.p) return BA_ERR_STATE;
      if (buf) {
        auto h = fetch(s->d_Scopy.p, (size_t)ld * ld);
        if (which == 6) {
          for (int r = 0; r < n; ++r)
            for (int c = 0; c < n; ++c) {
              const int a = std::min(r, c), b = std::max(r, c);
              buf[(size_t)c * n + r] = h[(size_t)a * ld + b];  // symmetric; row-major upper is filled
            }
        } else {
          for (int r = 0; r < n; ++r) buf[r] = h[(size_t)r * ld + n];
        }
      }
      return which == 6 ? (long long)n * n : n;
    }
    case 8: if (buf) { auto h = fetch(s->d_x.p, (size_t)n); std::copy(h.begin(), h.end(), buf); } return n;
    case 9:
      if (buf) {
        auto h = fetch(s->d_y.p, (size_t)s->M_total * 3);
        for (int io = 0; io < M; ++io)
          for (int k = 0; k < 3; ++k) buf[(size_t)io * 3 + k] = h[(size_t)s->h_opt_point[io] * 3 + k];
      }
      return (long long)M * 3;
    case 10:
      if (buf) {
        LmState h;
        cudaMemcpy(&h, s->d_state.p, sizeof(h), cudaMemcpyDeviceToHost);
        buf[0] = 0.0; buf[1] = h.last_cost_new; buf[2] = h.last_model; buf[3] = h.last_rho; buf[4] = h.last_lambda;
      }
      return 5;
    case 11:  // raw factor buffer after the last solve: (n+1)^2 doubles, column-major lower + z row
      if (buf) { auto h = fetch(s->d_Saug.p, (size_t)ld * ld); std::copy(h.begin(), h.end(), buf); }
      return (long long)ld * ld;
    default: return BA_ERR_INVALID;
  }
}

// In-situ timing of parts of the reduced solve on whatever S currently holds (numerically meaningless,
// timing only): parts bit 0 diag, 1 trsm, 2 syrk, 3 backward.  Graph-replayed `reps` times.
int ba_debug_time_solve(ba_solver *s, int parts, int reps, float *ms_per_rep) {
  if (!s || !s->finalized || !ms_per_rep) return BA_ERR_STATE;
  CUDA_TRY(cudaSetDevice(s->device));
  cudaStream_t st = s->stream;
  CUDA_TRY(cudaMemsetAsync(s->d_state.p, 0, sizeof(LmState), st));
  cudaGraph_t graph;
  cudaGraphExec_t exec;
  CUDA_TRY(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
  cholesky_solve_enqueue(s->chol, s->d_Saug.p, s->d_x.p, s->d_z.p, s->d_linv.p, s->d_state.p, st, nullptr, s->sw.verbose,
                         parts);
  CUDA_TRY(cudaStreamEndCapture(st, &graph));
  CUDA_TRY(cudaGraphInstantiate(&exec, graph, 0));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int i = 0; i < 3; ++i) cudaGraphLaunch(exec, st);
  cudaEventRecord(e0, st);
  for (int i = 0; i < reps; ++i) cudaGraphLaunch(exec, st);
  cudaEventRecord(e1, st);
  CUDA_TRY(cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  *ms_per_rep = ms / reps;
  const SolvePath path = s->chol.path;
  if (s->sw.verbose) {
    unsigned long long dbg[8];
    cudaMemcpyFromSymbol(dbg, g_cl_dbg, sizeof(dbg));
    if (path == SolvePath::NdPersistent || path == SolvePath::NdLevels) {
      unsigned long long d3[16];
      cudaMemcpyFromSymbol(d3, g_nd_dbg, 16 * sizeof(unsigned long long));
      const double r = 1.0 / (3.0 + reps);   // accumulated over warm-up + timed replays
      fprintf(stderr, "[ba_b200] partitioned banded (n=%d bw=%d depth=%d leaves=%d nodes=%zu): CTA 0 forward %llu ns, forward+backward %llu ns | per-level front ns (sum over nodes / replays):",
              s->chol.n, s->chol.bw, s->chol.nd.depth, s->chol.nd.n_leaves, s->chol.nd.nodes.size(), d3[0], d3[1]);
      for (int l = 0; l < 7; ++l) fprintf(stderr, " L%d %.0f", l, (double)d3[2 + l] * r);
      fprintf(stderr, " | CTA 0 per replay: wait %.0f assemble %.0f (staged at %.0f, own columns at %.0f) factor %.0f flag %.0f | root diagonal warp cycles: waiting %.0f working %.0f\n", (double)d3[9] * r, (double)d3[10] * r,
              (double)d3[13] * r, (double)d3[14] * r, (double)d3[11] * r, (double)d3[12] * r, (double)d3[8] * r, (double)d3[15] * r);
      unsigned long long z[16] = {0};
      cudaMemcpyToSymbol(g_nd_dbg, z, sizeof(z));
    } else if (path == SolvePath::Banded) {
      unsigned long long d2[16];
      cudaMemcpyFromSymbol(d2, g_band_dbg, 16 * sizeof(unsigned long long));
      fprintf(stderr, "[ba_b200] banded ns: factor %llu backward %llu (n=%d bw=%d) | cycles: producer wait %llu work %llu | consumer0 loads %llu waitL %llu priority %llu bulk %llu endbar %llu\n",
              d2[0], d2[1], s->chol.n, s->chol.bw, d2[2], d2[3], d2[4], d2[5], d2[6], d2[7], d2[8]);
    } else
    fprintf(stderr, "[ba_b200] cluster ns: diag %llu sync %llu trsm %llu sync %llu syrk %llu sync %llu backward %llu\n", dbg[0], dbg[1], dbg[2], dbg[3], dbg[4], dbg[5], dbg[6]);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaGraphExecDestroy(exec); cudaGraphDestroy(graph);
  return BA_OK;
}

// Which reduced-solve path the plan selected and what it costs (bench.py's roofline accounting).
//   vals[0] algorithmic flops: Cholesky of S inside its row envelope (sum over rows of width^2) + the two
//           triangular solves -- the work the PROBLEM needs, independent of the kernel
//   vals[1] executed flops of the selected path (partitioned: partial factorisations of all fronts incl. fill and
//           padding; serial banded: n (W^2); cluster / dense: envelope tiles)
//   vals[2] dense equivalent n^3 / 3 + 2 n^2     vals[3] half-bandwidth bw      vals[4] CTAs of the launch
//   vals[5] dependent 8-column panel steps on the critical path     vals[6] 1 if S is cleared band-only
//   vals[7] algorithmic bytes of the solve: the envelope of S read once + rhs + x
int ba_debug_solve_info(ba_solver *s, char *name, int cap, double *vals) {
  if (!s || !s->finalized || !vals) return BA_ERR_STATE;
  const CholeskyPlan &pl = s->chol;
  const int n = pl.n;
  double alg = 0.0, env_entries = 0.0;
  for (int j = 0; j < s->N; ++j) {
    const double w = 6.0 * (j - s->h_first_pose[j]);
    for (int r = 0; r < 6; ++r) { alg += (w + r + 1) * (w + r + 1); env_entries += w + r + 1; }
  }
  alg += 4.0 * env_entries;
  std::string nm;
  double exec = 0.0, ctas = 1.0, chain = 0.0;
  const bool persistent = pl.path == SolvePath::NdPersistent;
  if (persistent || pl.path == SolvePath::NdLevels) {
    for (const NdNode &nd : pl.nd.nodes) {
      const double R = nd.k8 + nd.b8;
      for (int c = 0; c < nd.k8; ++c) exec += (R - c) * (R - c);
    }
    chain = nd_plan_cost(pl.nd);
    ctas = persistent ? pl.nd.n_ctas + pl.nd.n_helpers : pl.nd.n_leaves;
    char buf[256];
    snprintf(buf, sizeof(buf), "%s<%d,%d> (partitioned banded Cholesky: nested dissection depth %d, %d fronts, DMMA panel solves and updates)",
             persistent ? "k_nd_persistent" : "k_nd_forward_level+k_nd_backward_level", pl.nd_dev.tpw, nd_cons_for(pl.nd.max_BT),
             pl.nd.depth, (int)pl.nd.nodes.size());
    nm = buf;
  } else if (pl.path == SolvePath::Banded) {
    const double W = pl.bw + 16.0;
    exec = (double)n * W * W;
    chain = n / 8.0;
    nm = "k_chol_banded_smem (serial banded Cholesky, one CTA, DMMA window update)";
  } else {
    for (int k = 0; k < pl.T; ++k) {
      const double m = pl.rows_ptr[k + 1] - pl.rows_ptr[k];
      exec += (double)kNB * kNB * kNB * (1.0 / 3.0 + m + m * (m + 1) / 2.0);
    }
    chain = n / 8.0;
    ctas = pl.path == SolvePath::Cluster ? pl.cluster_size : 148;
    nm = pl.path == SolvePath::Cluster ? "k_chol_cluster (blocked Cholesky in one thread-block-cluster launch)"
                             : "k_chol_diag+k_chol_trsm+k_syrk_update (blocked dense Cholesky, DMMA TRSM and trailing update)";
  }
  const bool band_clear = clears_band_only(s);   // steady state of the LM loop
  vals[0] = alg; vals[1] = exec; vals[2] = (double)n * n * n / 3.0 + 2.0 * n * n; vals[3] = pl.bw; vals[4] = ctas;
  vals[5] = chain; vals[6] = band_clear ? 1.0 : 0.0; vals[7] = 8.0 * (env_entries + 2.0 * n);
  if (name && cap > 0) { strncpy(name, nm.c_str(), cap - 1); name[cap - 1] = 0; }
  return BA_OK;
}

// Host-only: the partition plan of the banded reduced solve for N free poses and track span b (no device needed).
// nodes_out: [cap][20] = own0 k k8 rb0 wr lb0 wl b8 child0 child1 parent rb_off lb_off rhs_off level cta seq L_off U_off helper
// meta: [8] = valid depth n_leaves n_levels n_ctas max_tiles max_R8 smem_bytes.  Returns the number of nodes.
int ba_debug_nd_plan(int N, int b, int max_ctas, int force_depth, int force_chunk, long long *meta,
                     long long *nodes_out, int cap) {
  NdPlan pl;
  nd_make_plan(pl, N, b, max_ctas, force_depth, force_chunk);
  if (meta) {
    meta[0] = pl.valid; meta[1] = pl.depth; meta[2] = pl.n_leaves; meta[3] = pl.n_levels; meta[4] = pl.n_ctas;
    meta[5] = pl.max_tiles; meta[6] = pl.max_R8; meta[7] = (long long)nd_smem_bytes(pl);
  }
  const int nn = (int)pl.nodes.size();
  for (int i = 0; i < std::min(nn, cap) && nodes_out; ++i) {
    const NdNode &d = pl.nodes[i];
    const long long v[20] = {d.own0, d.k, d.k8, d.rb0, d.wr, d.lb0, d.wl, d.b8, d.child[0], d.child[1], d.parent,
                             d.rb_off, d.lb_off, d.rhs_off, d.level, d.cta, d.seq, d.L_off, d.U_off, d.helper};
    std::copy(v, v + 20, nodes_out + (size_t)i * 20);
  }
  return nn;
}

int ba_debug_pairs(ba_solver *s, int *pair_pose_id, int *pair_point_id) {
  if (!s || !s->finalized) return BA_ERR_STATE;
  for (long long p = 0; p < s->P; ++p) {
    pair_pose_id[p] = s->h_opt_pose[s->h_pair_pose[p]];
    pair_point_id[p] = s->h_pair_point[p];
  }
  return BA_OK;
}

int ba_comm_get_unique_id(void *id128) {
  if (!id128) return BA_ERR_INVALID;
  if (!g_nccl.load()) return BA_ERR_NCCL;
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return BA_ERR_NCCL;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  std::memcpy(id128, &id, 128);
  return BA_OK;
}

// peer exchange set-up: every rank allocates its PeerExch, the IPC handles travel by ncclAllGather, every rank maps
// the others.  All-or-nothing: the ranks agree (min-reduce) and fall back to the NCCL all-reduce of the scalars.
// Collective over the communicator: every rank contributes one device allocation (`local`, nullptr = this rank failed
// to allocate), receives the IPC handles of all ranks and maps them.  All-or-nothing: returns true on every rank or
// on none (min-reduce of the per-rank outcome).
static bool ipc_map_all(SharedComm &sc, cudaStream_t st, void *local, void **mapped /*[n_ranks]*/) {
  for (int r = 0; r < sc.n_ranks; ++r) mapped[r] = nullptr;
  if (!g_nccl.AllGather) return false;
  cudaIpcMemHandle_t mine{};
  int ok = local != nullptr;
  if (ok && cudaIpcGetMemHandle(&mine, local) != cudaSuccess) ok = 0;
  cudaGetLastError();
  const size_t rec = sizeof(cudaIpcMemHandle_t) + 8;
  unsigned char *d_send = nullptr, *d_recv = nullptr;
  if (cudaMalloc(&d_send, rec) != cudaSuccess || cudaMalloc(&d_recv, rec * sc.n_ranks) != cudaSuccess) {
    cudaGetLastError();
    if (d_send) cudaFree(d_send);
    return false;   // cannot even talk: every rank fails the same way only by luck, so never use the peers
  }
  std::vector<unsigned char> h_send(rec, 0), h_recv(rec * sc.n_ranks, 0);
  std::memcpy(h_send.data(), &mine, sizeof(mine));
  h_send[sizeof(mine)] = (unsigned char)ok;
  cudaMemcpyAsync(d_send, h_send.data(), rec, cudaMemcpyHostToDevice, st);
  bool talked = g_nccl.AllGather(d_send, d_recv, rec, ncclChar, sc.comm, st) == ncclSuccess;
  cudaMemcpyAsync(h_recv.data(), d_recv, rec * sc.n_ranks, cudaMemcpyDeviceToHost, st);
  talked = talked && cudaStreamSynchronize(st) == cudaSuccess;
  int all_ok = talked ? 1 : 0;
  for (int r = 0; r < sc.n_ranks && all_ok; ++r) all_ok = h_recv[r * rec + sizeof(mine)] ? 1 : 0;
  if (all_ok) {
    for (int r = 0; r < sc.n_ranks; ++r) {
      if (r == sc.rank) { mapped[r] = local; continue; }
      cudaIpcMemHandle_t h;
      std::memcpy(&h, h_recv.data() + r * rec, sizeof(h));
      void *ptr = nullptr;
      if (cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); all_ok = 0; break; }
      mapped[r] = ptr;
    }
  }
  bool agreed_ok = false;
  if (talked) {   // second round: did every rank map every peer?
    int *d_flag = reinterpret_cast<int *>(d_send);
    cudaMemcpyAsync(d_flag, &all_ok, sizeof(int), cudaMemcpyHostToDevice, st);
    if (g_nccl.AllReduce(d_flag, d_flag, 1, ncclInt, ncclMin, sc.comm, st) != ncclSuccess) all_ok = 0;
    int agreed = 0;
    cudaMemcpyAsync(&agreed, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) agreed = 0;
    agreed_ok = all_ok && agreed;
  }
  cudaFree(d_send);
  cudaFree(d_recv);
  if (!agreed_ok)
    for (int r = 0; r < sc.n_ranks; ++r) {
      if (mapped[r] && r != sc.rank) cudaIpcCloseMemHandle(mapped[r]);
      mapped[r] = nullptr;
    }
  return agreed_ok;
}

// peer exchange of the LM scalars: every rank allocates its PeerExch and maps the others'; falls back to the NCCL
// all-reduce of the scalars when that fails anywhere
static void setup_peer_exchange(SharedComm &sc, cudaStream_t st, bool no_peer_exchange) {
  sc.peer_ok = false;
  if (no_peer_exchange || sc.n_ranks > kMaxRanks) return;
  bool ok = true;
  if (cudaMalloc(&sc.local, sizeof(PeerExch)) != cudaSuccess) { sc.local = nullptr; ok = false; }
  if (cudaMalloc(&sc.d_epoch, sizeof(unsigned)) != cudaSuccess) { sc.d_epoch = nullptr; ok = false; }
  if (cudaMalloc(&sc.d_error, sizeof(int)) != cudaSuccess) { sc.d_error = nullptr; ok = false; }
  if (ok) {
    cudaMemset(sc.local, 0, sizeof(PeerExch));
    cudaMemset(sc.d_epoch, 0, sizeof(unsigned));
    cudaMemset(sc.d_error, 0, sizeof(int));
  }
  cudaGetLastError();
  void *mapped[kMaxRanks] = {};
  sc.peer_ok = ipc_map_all(sc, st, ok ? sc.local : nullptr, mapped);
  for (int r = 0; r < sc.n_ranks; ++r) sc.peer[r] = sc.peer_ok ? static_cast<PeerExch *>(mapped[r]) : nullptr;
  if (sc.verbose) fprintf(stderr, "[ba_b200] rank %d/%d: scalar exchange over %s\n", sc.rank, sc.n_ranks, sc.peer_ok ? "peer memory (CUDA IPC)" : "ncclAllReduce");
}

// band exchange through peer memory: (re)allocated when a problem needs more than the current capacity.  Collective:
// every rank calls it at the same point (agree_on_envelope) with the same count (same global plan).
static void ensure_band_exchange(SharedComm &sc, cudaStream_t st, long long count) {
  if (!sc.peer_ok || count <= 0) return;
  if (sc.band_ok && count <= sc.band_cap) return;
  if (sc.band_local) sc.retire_band();           // graphs of earlier solvers keep using the old set
  const long long cap = (count + 511) / 512 * 512;
  bool ok = true;
  const long long pslot = (cap + sc.n_ranks - 1) / sc.n_ranks + 1024;     // one rank's rows of the band (+ one row of slack)
  const size_t band_doubles = (size_t)2 * ((size_t)sc.n_ranks * cap + cap + (size_t)sc.n_ranks * 1024);   // room for either layout
  if (cudaMalloc(&sc.band_local, sizeof(double) * band_doubles) != cudaSuccess) { sc.band_local = nullptr; ok = false; }
  if (cudaMalloc(&sc.bflag_local, sizeof(unsigned) * 4 * kMaxRanks) != cudaSuccess) { sc.bflag_local = nullptr; ok = false; }
  if (cudaMalloc(&sc.d_band_epoch, sizeof(unsigned)) != cudaSuccess) { sc.d_band_epoch = nullptr; ok = false; }
  if (cudaMalloc(&sc.d_band_counters, 4 * sizeof(unsigned)) != cudaSuccess) { sc.d_band_counters = nullptr; ok = false; }
  if (ok) {
    cudaMemset(sc.bflag_local, 0, sizeof(unsigned) * 4 * kMaxRanks);
    cudaMemset(sc.d_band_epoch, 0, sizeof(unsigned));
    cudaMemset(sc.d_band_counters, 0, 4 * sizeof(unsigned));
  }
  cudaGetLastError();
  void *m1[kMaxRanks] = {}, *m2[kMaxRanks] = {};
  const bool ok1 = ipc_map_all(sc, st, ok ? (void *)sc.band_local : nullptr, m1);
  const bool ok2 = ipc_map_all(sc, st, ok ? (void *)sc.bflag_local : nullptr, m2);
  sc.band_ok = ok1 && ok2;
  for (int r = 0; r < sc.n_ranks; ++r) {
    sc.band_peer[r] = sc.band_ok ? static_cast<double *>(m1[r]) : nullptr;
    sc.bflag_peer[r] = sc.band_ok ? static_cast<unsigned *>(m2[r]) : nullptr;
    if (!sc.band_ok) {   // one of the two mapped: undo
      if (m1[r] && r != sc.rank) cudaIpcCloseMemHandle(m1[r]);
      if (m2[r] && r != sc.rank) cudaIpcCloseMemHandle(m2[r]);
    }
  }
  sc.band_cap = sc.band_ok ? cap : 0;
  sc.band_pslot = pslot;
  if (sc.verbose) fprintf(stderr, "[ba_b200] rank %d/%d: band exchange over %s (%lld doubles per slot)\n", sc.rank, sc.n_ranks, sc.band_ok ? "peer memory (CUDA IPC)" : "ncclAllReduce", cap);
}

static int adopt_comm(ba_solver *s, const std::shared_ptr<SharedComm> &sc, long long global_M, long long global_n_obs) {
  s->shared = sc;
  s->comm = sc->comm;
  s->rank = sc->rank; s->n_ranks = sc->n_ranks; s->global_M = global_M; s->global_n_obs = global_n_obs;
  destroy_graph(s);
  if (s->finalized) return agree_on_envelope(s);
  return BA_OK;
}

int ba_comm_init(ba_solver *s, const void *id128, int rank, int nranks, long long global_M,
                 long long global_n_obs) {
  if (!s || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return BA_ERR_INVALID;
  if (!g_nccl.load()) { s->err = "libnccl.so.2 not found"; return BA_ERR_NCCL; }
  CUDA_TRY(cudaSetDevice(s->device));
  if (int rc = ensure_stream(s)) return rc;
  ncclUniqueId id;
  std::memcpy(&id, id128, 128);
  s->comm = nullptr;
  s->shared.reset();                       // re-initialisation: the old communicator goes when its last user does
  auto sc = std::make_shared<SharedComm>();
  sc->device = s->device; sc->rank = rank; sc->n_ranks = nranks; sc->verbose = s->sw.verbose;
  ncclResult_t r = g_nccl.CommInitRank(&sc->comm, nranks, id, rank);
  if (r != ncclSuccess) { s->err = "ncclCommInitRank failed"; sc->comm = nullptr; return BA_ERR_NCCL; }
  setup_peer_exchange(*sc, s->stream, s->sw.no_peer_exchange);
  {
    std::lock_guard<std::mutex> lk(g_comm_mu);
    g_comm_registry[s->device] = sc;       // the device's communicator for later ba_comm_attach calls
  }
  return adopt_comm(s, sc, global_M, global_n_obs);
}

int ba_comm_attach(ba_solver *s, long long global_M, long long global_n_obs) {
  if (!s) return BA_ERR_INVALID;
  CUDA_TRY(cudaSetDevice(s->device));
  if (int rc = ensure_stream(s)) return rc;
  std::shared_ptr<SharedComm> sc;
  {
    std::lock_guard<std::mutex> lk(g_comm_mu);
    auto it = g_comm_registry.find(s->device);
    if (it != g_comm_registry.end()) sc = it->second;
  }
  if (!sc) { s->err = "ba_comm_attach: no communicator on this device (call ba_comm_init once first)"; return BA_ERR_STATE; }
  return adopt_comm(s, sc, global_M, global_n_obs);
}

int ba_comm_destroy(ba_solver *s) {
  if (!s) return BA_ERR_INVALID;
  s->comm = nullptr;
  s->shared.reset();
  s->rank = 0; s->n_ranks = 1; s->global_M = s->global_n_obs = -1;
  destroy_graph(s);
  return BA_OK;
}

int ba_comm_shutdown(int device) {
  std::shared_ptr<SharedComm> sc;
  {
    std::lock_guard<std::mutex> lk(g_comm_mu);
    auto it = g_comm_registry.find(device);
    if (it == g_comm_registry.end()) return BA_OK;
    sc = it->second;
    g_comm_registry.erase(it);
  }
  return BA_OK;   // destroyed here unless a solver still holds it
}

}  // extern "C"
