// ba_device.cuh -- device-side math shared by the full-BA kernels (FP64).
// Arithmetic follows core/full_bundle_adjustment_solver.cpp (file:line cited per function).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ba {

constexpr int kCamStride = 16;  // fx fy cx cy | R_c row-major 9 | t_c 3

// flags packed with the camera slot in obs_camflags
constexpr int kFlagPoseFree = 1 << 8;
constexpr int kFlagPointFree = 1 << 9;
constexpr int kFlagLastOfPair = 1 << 10;
constexpr int kCamMask = 0xff;

// chunk flags
constexpr int kChunkSplit = 1;  // chunk holds a piece of a point that spans several chunks

struct __align__(16) Chunk {
  int obs_start;
  int obs_count;
  int pair_start;
  int flags;
};

// Device-resident LM state; every kernel of the loop reads it, only k_decide writes it.
struct LmState {
  double lambda;
  double prev_cost;
  double last_cost_new, last_model, last_rho, last_lambda;  // debug (oracle dump 10)
  int cur;        // which parameter buffer holds the accepted parameters
  int done;       // 1 once converged or max iterations reached: later kernels are no-ops
  int iteration;  // LM iterations executed so far
  int converged;
};

// Projection + residual at one observation (full...cpp:733-760 / :403-425).
//   Xb = R_jw X + t_jw ; Xc = R_c Xb + t_c ; r = (fx x/z + cx - u, fy y/z + cy - v)
struct Proj {
  double Xb[3];
  double r0, r1;
  double fxinvz, fyinvz, fx_xinvz2, fy_yinvz2;
};

__device__ __forceinline__ void project(const double *__restrict__ T, const double *__restrict__ X,
                                        const double *__restrict__ cam, double u, double v, Proj &p) {
  const double X0 = X[0], X1 = X[1], X2 = X[2];
  p.Xb[0] = T[0] * X0 + T[1] * X1 + T[2] * X2 + T[9];
  p.Xb[1] = T[3] * X0 + T[4] * X1 + T[5] * X2 + T[10];
  p.Xb[2] = T[6] * X0 + T[7] * X1 + T[8] * X2 + T[11];
  const double *Rc = cam + 4;
  const double xc = Rc[0] * p.Xb[0] + Rc[1] * p.Xb[1] + Rc[2] * p.Xb[2] + cam[13];
  const double yc = Rc[3] * p.Xb[0] + Rc[4] * p.Xb[1] + Rc[5] * p.Xb[2] + cam[14];
  const double zc = Rc[6] * p.Xb[0] + Rc[7] * p.Xb[1] + Rc[8] * p.Xb[2] + cam[15];
  const double invz = 1.0 / zc;
  p.fxinvz = cam[0] * invz;
  p.fyinvz = cam[1] * invz;
  const double xinvz = xc * invz, yinvz = yc * invz;
  p.fx_xinvz2 = p.fxinvz * xinvz;
  p.fy_yinvz2 = p.fyinvz * yinvz;
  p.r0 = cam[0] * xinvz + cam[2] - u;
  p.r1 = cam[1] * yinvz + cam[3] - v;
}

// Depth zc of a projected observation in its camera: the expression project() divides by (kept apart from Proj so
// that the kernels which inline project() are unchanged).
__device__ __forceinline__ double camera_depth(const Proj &p, const double *__restrict__ cam) {
  const double *Rc = cam + 4;
  return Rc[6] * p.Xb[0] + Rc[7] * p.Xb[1] + Rc[8] * p.Xb[2] + cam[15];
}

// Viewing ray of one observation in the world frame (ba_triangulate_points): the observing camera is R_k = R_c R_jw,
// t_k = R_c t_jw + t_c (the transform project() applies); its centre is c = -R_k^T t_k and the unit ray through the
// pixel is d = R_k^T m / ||m||, m = ((u - cx) / fx, (v - cy) / fy, 1).
__device__ __forceinline__ void obs_ray(const double *__restrict__ T, const double *__restrict__ cam, double u,
                                        double v, double *c, double *d) {
  const double *Rc = cam + 4;
  double Rk[9], tk[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int col = 0; col < 3; ++col)
      Rk[r * 3 + col] = Rc[r * 3] * T[col] + Rc[r * 3 + 1] * T[3 + col] + Rc[r * 3 + 2] * T[6 + col];
    tk[r] = Rc[r * 3] * T[9] + Rc[r * 3 + 1] * T[10] + Rc[r * 3 + 2] * T[11] + cam[13 + r];
  }
  const double m0 = (u - cam[2]) / cam[0], m1 = (v - cam[3]) / cam[1];
  const double norm = sqrt(m0 * m0 + m1 * m1 + 1.0);
#pragma unroll
  for (int col = 0; col < 3; ++col) {
    c[col] = -(Rk[col] * tk[0] + Rk[3 + col] * tk[1] + Rk[6 + col] * tk[2]);
    d[col] = (Rk[col] * m0 + Rk[3 + col] * m1 + Rk[6 + col]) / norm;
  }
}

// Huber-style weight by the L1 norm (full...cpp:763-766); thres is the float option promoted.
__device__ __forceinline__ double huber_weight(double r0, double r1, double thres) {
  const double absrxry = fabs(r0) + fabs(r1);
  return (absrxry > thres) ? (thres / absrxry) : 1.0;
}

// G = D R_c (2x3), D = d(pixel)/d(Xc)  (full...cpp:770-787)
__device__ __forceinline__ void jac_G(const Proj &p, const double *__restrict__ cam, double *G) {
  const double *Rc = cam + 4;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    G[c] = p.fxinvz * Rc[c] + (-p.fx_xinvz2) * Rc[6 + c];
    G[3 + c] = p.fyinvz * Rc[3 + c] + (-p.fy_yinvz2) * Rc[6 + c];
  }
}

// Q = [G, G K], K = -[Xb]x  (full...cpp:797-800), 2x6 row-major
__device__ __forceinline__ void jac_Q(const double *G, const double *Xb, double *Q) {
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const double g0 = G[r * 3], g1 = G[r * 3 + 1], g2 = G[r * 3 + 2];
    Q[r * 6 + 0] = g0;
    Q[r * 6 + 1] = g1;
    Q[r * 6 + 2] = g2;
    // K = [0 z -y; -z 0 x; y -x 0]
    Q[r * 6 + 3] = g1 * (-Xb[2]) + g2 * Xb[1];
    Q[r * 6 + 4] = g0 * Xb[2] + g2 * (-Xb[0]);
    Q[r * 6 + 5] = g0 * (-Xb[1]) + g1 * Xb[0];
  }
}

// Rm = G R_jw (2x3)  (full...cpp:814)
__device__ __forceinline__ void jac_R(const double *G, const double *__restrict__ T, double *Rm) {
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c)
      Rm[r * 3 + c] = G[r * 3] * T[c] + G[r * 3 + 1] * T[3 + c] + G[r * 3 + 2] * T[6 + c];
}

// One observation linearised for the landmark side: residual, Huber weight, G and Rm (full...cpp:733-814).
struct ObsLin {
  Proj pr;
  double w;
  double G[6], Rm[6];
};
__device__ __forceinline__ void linearize_obs(const double *__restrict__ T, const double *__restrict__ X,
                                              const double *__restrict__ cam, double u, double v, double thres,
                                              ObsLin &o) {
  project(T, X, cam, u, v, o.pr);
  o.w = huber_weight(o.pr.r0, o.pr.r1, thres);
  jac_G(o.pr, cam, o.G);
  jac_R(o.G, T, o.Rm);
}
// Bv (6x3 row-major) += w Q^T Rm, the observation's share of the pose-landmark block B_ji (:826).  Every kernel that
// forms B calls this, so the Schur complement, the back-substitution and the debug dump see the same B.
__device__ __forceinline__ void add_B(const ObsLin &o, double *Bv) {
  double Q[12];
  jac_Q(o.G, o.pr.Xb, Q);
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) Bv[r * 3 + c] += o.w * (Q[r] * o.Rm[c] + Q[6 + r] * o.Rm[3 + c]);
}

// se3Exp (full...cpp:1046-1082), xi = [v; w]; out = R row-major 9 | t 3
__device__ __forceinline__ void se3_exp(const double *xi, double *out) {
  const double v0 = xi[0], v1 = xi[1], v2 = xi[2];
  const double w0 = xi[3], w1 = xi[4], w2 = xi[5];
  const double theta = sqrt(w0 * w0 + w1 * w1 + w2 * w2);
  const double wx[9] = {0.0, -w2, w1, w2, 0.0, -w0, -w1, w0, 0.0};
  double wx2[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c)
      wx2[r * 3 + c] = wx[r * 3] * wx[c] + wx[r * 3 + 1] * wx[3 + c] + wx[r * 3 + 2] * wx[6 + c];
  double a, b, g;
  if (theta < 1e-7) {
    a = 1.0;
    b = 0.5;
    g = 0.33333333333333333333333333;
  } else {
    double s, c;
    sincos(theta, &s, &c);
    a = s / theta;
    b = (1.0 - c) / (theta * theta);
    g = (theta - s) / (theta * theta * theta);
  }
  double V[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const double I = (i % 4 == 0) ? 1.0 : 0.0;
    out[i] = I + a * wx[i] + b * wx2[i];
    V[i] = I + b * wx[i] + g * wx2[i];
  }
  out[9] = V[0] * v0 + V[1] * v1 + V[2] * v2;
  out[10] = V[3] * v0 + V[4] * v1 + V[5] * v2;
  out[11] = V[6] * v0 + V[7] * v1 + V[8] * v2;
}

// 3x3 symmetric inverse through Eigen's diagonal-pivoted, left-looking LDL^T with the
// |D| <= DBL_MIN -> 0 pseudo-inverse rule (full...cpp:854 `C.ldlt().solve(I)`), fully in
// registers (no dynamic indexing).  in: c = {c00,c01,c02,c11,c12,c22}; out: inv row-major 9.
__device__ __forceinline__ void swapd(double &a, double &b) {
  const double t = a;
  a = b;
  b = t;
}
__device__ __forceinline__ void ldlt3_inverse(const double *c, double *inv) {
  double a00 = c[0], a10 = c[1], a20 = c[2], a11 = c[3], a21 = c[4], a22 = c[5];
  // k = 0: largest |diagonal| (first maximum wins)
  int p0 = 0;
  double best = fabs(a00);
  if (fabs(a11) > best) { best = fabs(a11); p0 = 1; }
  if (fabs(a22) > best) { p0 = 2; }
  if (p0 == 1) { swapd(a00, a11); swapd(a20, a21); }
  else if (p0 == 2) { swapd(a00, a22); swapd(a10, a21); }
  // one reciprocal per pivot instead of twelve divisions (differs from a true division by <= 1 ulp)
  const double tol = 2.2250738585072014e-308;
  const double d0 = a00;
  const double r0 = (fabs(d0) > 0.0) ? 1.0 / d0 : 1.0;
  double l10 = a10 * r0, l20 = a20 * r0;
  if (!(fabs(d0) > 0.0)) { l10 = a10; l20 = a20; }
  // k = 1: compares the not-yet-updated diagonals (Eigen's unblocked kernel is left-looking)
  int p1 = 1;
  if (fabs(a22) > fabs(a11)) p1 = 2;
  if (p1 == 2) { swapd(a11, a22); swapd(l10, l20); }
  const double t0 = d0 * l10;
  const double d1 = a11 - l10 * t0;
  double l21 = a21 - l20 * t0;
  const double r1 = (fabs(d1) > 0.0) ? 1.0 / d1 : 1.0;
  l21 *= r1;
  // k = 2
  const double u0 = d0 * l20, u1 = d1 * l21;
  const double d2 = a22 - (l20 * u0 + l21 * u1);
  const double r2 = (fabs(d2) > 0.0) ? 1.0 / d2 : 1.0;
  const double q0 = (fabs(d0) > tol) ? r0 : 0.0, q1 = (fabs(d1) > tol) ? r1 : 0.0, q2 = (fabs(d2) > tol) ? r2 : 0.0;
#pragma unroll
  for (int col = 0; col < 3; ++col) {
    double v0 = (col == 0) ? 1.0 : 0.0, v1 = (col == 1) ? 1.0 : 0.0, v2 = (col == 2) ? 1.0 : 0.0;
    // P b
    if (p0 == 1) swapd(v0, v1); else if (p0 == 2) swapd(v0, v2);
    if (p1 == 2) swapd(v1, v2);
    // L^-1
    v1 -= l10 * v0;
    v2 -= l20 * v0;
    v2 -= l21 * v1;
    // D^+
    v0 *= q0;
    v1 *= q1;
    v2 *= q2;
    // L^-T
    v1 -= l21 * v2;
    v0 -= l10 * v1 + l20 * v2;
    // P^T
    if (p1 == 2) swapd(v1, v2);
    if (p0 == 1) swapd(v0, v1); else if (p0 == 2) swapd(v0, v2);
    inv[0 * 3 + col] = v0;
    inv[1 * 3 + col] = v1;
    inv[2 * 3 + col] = v2;
  }
}

// ---------------------------------------------------------------------------
// Block-wide segmented sum over threads whose segments are delimited by `head`.
// After the call, the thread flagged `tail` holds the sum of its whole segment, provided the
// segment lies inside the block.  K values per thread.  smem: (nwarps*(K) doubles + nwarps ints).
// ---------------------------------------------------------------------------
template <int K, int NWARPS>
struct SegSmem {
  double tailv[NWARPS][K];
  int has_head[NWARPS];
};

template <int K, int NWARPS>
__device__ __forceinline__ void block_segmented_sum(double (&v)[K], bool head, bool tail,
                                                    SegSmem<K, NWARPS> &sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned heads = __ballot_sync(0xffffffffu, head);
  // closest head at or before this lane (-1: the segment started in an earlier warp)
  const unsigned below = heads & (0xffffffffu >> (31 - lane));
  const int seg_lane = below ? (31 - __clz(below)) : -1;
  const int lo = seg_lane < 0 ? 0 : seg_lane;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const bool take = (lane - d) >= lo;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double o = __shfl_up_sync(0xffffffffu, v[k], d);
      if (take) v[k] += o;
    }
  }
  if (lane == 31) {
#pragma unroll
    for (int k = 0; k < K; ++k) sm.tailv[warp][k] = v[k];
    sm.has_head[warp] = heads != 0u;
  }
  __syncthreads();
  if (tail && seg_lane < 0) {
    for (int w = warp - 1; w >= 0; --w) {
#pragma unroll
      for (int k = 0; k < K; ++k) v[k] += sm.tailv[w][k];
      if (sm.has_head[w]) break;
    }
  }
}

// plain block sum of K values; result valid in thread 0.  NWARPS warps.
template <int K, int NWARPS>
__device__ __forceinline__ void block_sum(double (&v)[K], double (*sm)[K]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1)
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] += __shfl_down_sync(0xffffffffu, v[k], d);
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < K; ++k) sm[warp][k] = v[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < NWARPS; ++w)
#pragma unroll
      for (int k = 0; k < K; ++k) v[k] += sm[w][k];
  }
}

}  // namespace ba
