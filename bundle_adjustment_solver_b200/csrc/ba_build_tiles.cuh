// ba_build_tiles.cuh -- K1b+K3+K4 fused for "tile" landmarks: persistent CTAs, barrier-free producers (included by
// ba_engine.cu inside namespace ba, after Params / SchurChunk / load_pose / damp_invert / bar_* helpers).
//
// Same arithmetic as core/full_bundle_adjustment_solver.cpp:716-831 (point side), :846-856, :858-888.  Layout of the
// work:
//   * the tile chunks are cut into batches of 8 landmarks (K = 24 operand rows); the flat list of batches is split
//     evenly over one persistent CTA per SM, so the producer/consumer pipeline never drains between chunks
//     (a chunk that straddles two CTAs is flushed into two staging segments);
//   * a landmark is owned by 4 adjacent lanes of one warp; lane `sub` linearises incidences sub, sub+4, ... of the
//     landmark, the 9 C/b partials are combined with an xor-butterfly (bitwise identical on the 4 lanes, so each
//     lane inverts the damped C redundantly and forms E = B C^-1 for its own incidences): no CTA barrier, no
//     shared-memory staging of partials, no idle threads while one thread per landmark inverts;
//   * every producer warp is its own group with its own operand buffer (G = 5..7 buffers, sized by the widest
//     window of the launch in whole 2 x 2 super-tiles, leading dimensions = 4 mod 16 -> conflict-free DMMA fragment
//     reads) and runs ahead on its own batch; the eighth warp owns no buffer and prefetches the batch list's
//     gathers into L2; the index records of the next round / next batch are prefetched,
//     the next batch's landmark data only after the observation loop (live across it, it would be spilled, and a
//     spill waits for the load);
//   * the four DMMA warps consume the buffers round-robin (2 x 2 super-tiles: every fragment read feeds two DMMAs,
//     accumulators in registers across all batches of a chunk, flushed into a staging window when the chunk changes)
//     and hand them back: full[g] / empty[g] named barriers, nothing else; a producer clears the few window slots its
//     landmark does not cover instead of anybody clearing whole buffers.
// B is never stored to global memory: k_backsub_tiles (end of this file) forms it again for the back-substitution.
#pragma once

constexpr int kT2LB = 8;                  // landmarks per batch (one producer warp, 4 lanes per landmark)
constexpr int kT2K = 3 * kT2LB;           // 24 operand rows
constexpr int kT2ProdWarps = 8;           // warps 0..7 (two warpgroups for setmaxnreg); at most 7 of them produce
constexpr int kT2MaxGroups = 7;           // named barriers: full 1..7, empty 8..14
constexpr int kT2Cons = 128;              // 4 DMMA warps
constexpr int kT2Threads = kT2ProdWarps * 32 + kT2Cons;
constexpr int kT2SmemBytes = 227 * 1024;  // everything an SM has: one CTA per SM
constexpr int kT2SmemDoubles = kT2SmemBytes / 8;
#ifndef BA_T2_PROD_REGS
#define BA_T2_PROD_REGS 160
#endif
// register split (setmaxnreg): the consumers can only take what the producers gave back to the CTA pool.
// Measured (C3 / C4 tile kernel): 144/216 0.151 / 1.31 ms, 152/200 0.138 / 1.21, 160/184 0.125 / 1.09, 168/168 0.158 / 1.36
constexpr int kT2ProdRegs = BA_T2_PROD_REGS;
constexpr int kT2ConsRegs = 168 + 2 * (168 - kT2ProdRegs);
static_assert(kT2ProdWarps * (168 - kT2ProdRegs) >= 4 * (kT2ConsRegs - 168) && kT2ProdRegs % 8 == 0, "register pool");
constexpr int kT2SPW = 7;                 // 2 x 2 super-tiles per DMMA warp at the widest window (27 over 4 warps)

struct TileLaunch {   // uniform per launch, fixed at finalize
  int nt_max;         // 8x8 tiles across the widest chunk window
  int ldE, ldB;       // operand leading dimensions (doubles): whole 2 x 2 super-tiles, = 4 mod 16
  int bufD;           // doubles per operand buffer
  int G;              // buffers = producer warps in use
  int n_cta;
};

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void dmma_884nv2(double &c0, double &c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <bool ACCUM_B>
__global__ void __launch_bounds__(kT2Threads, 1)
k_build_tiles(const SchurChunk *__restrict__ chunks, const int4 *__restrict__ batches /*ti0, nb, chunk, rhs column*/,
               const int *__restrict__ cta_batch_ptr, TileLaunch tl, const int *__restrict__ tpt_point,
               const int *__restrict__ tpt_inc_start, const int4 *__restrict__ inc_a /*obs_first, n_obs, pose, pair*/,
               const int2 *__restrict__ inc_b /*slot (-1: fixed pose), camera slots of obs 0 | obs 1 << 8*/,
               const double2 *__restrict__ obs_uv, const int *__restrict__ obs_camflags, Params prm,
               const double *__restrict__ cams, double thres_huber, double *__restrict__ ptblk, size_t Mp,
               const int *__restrict__ cta_seg_ptr /*first staging segment of every CTA*/,
               const long long *__restrict__ seg_off, double *__restrict__ stage, const LmState *__restrict__ st) {
  if (st->done) return;
  extern __shared__ double tsm[];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int b0 = cta_batch_ptr[blockIdx.x], b1 = cta_batch_ptr[blockIdx.x + 1];
  const int ldE = tl.ldE, ldB = tl.ldB, bufD = tl.bufD, G = tl.G;
  const int bar_cnt = 32 + kT2Cons;
  {
    double2 *z = reinterpret_cast<double2 *>(tsm);
    for (int e = t; e < G * bufD / 2; e += kT2Threads) z[e] = make_double2(0.0, 0.0);
  }
  __syncthreads();

  if (warp < kT2ProdWarps) {
    // ===================================================== producers =====================================
    // asking for more than the pool holds spins forever in TRY_ALLOC (static_assert above)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kT2ProdRegs));
    const int grp = warp;
    if (grp >= G) {
      // The last producer warp never owns a buffer (named barriers allow 7 groups): it walks the CTA's batch list
      // ahead of the others and pulls what they will gather -- incidence records, pixels, points --
      // into L2, so that their dependent round trips hit L2 instead of DRAM.  Hints only: no synchronisation.
      // (C3 / C4 / C5 tile kernel -1.6 / -4 / -3 %; prefetching into L1 instead measured the same.)
      if (warp == kT2ProdWarps - 1) {
        const int li = lane >> 2, sub = lane & 3;
        const double *points = prm.points[st->cur];
#pragma unroll 2
        for (int fb = b0; fb < b1; ++fb) {
          const int4 rec = __ldg(batches + fb);
          if (li < rec.y) {
            const int ti = rec.x + li;
            const int a = __ldg(tpt_inc_start + ti), b = __ldg(tpt_inc_start + ti + 1);
            if (sub == 0) prefetch_l2(points + (size_t)__ldg(tpt_point + ti) * 3);
            for (int ii = a + sub; ii < b; ii += 4) {
              const int4 ia = __ldg(inc_a + ii);
              prefetch_l2(inc_b + ii);
              prefetch_l2(obs_uv + ia.x);
              prefetch_l2(obs_uv + ia.x + ia.y - 1);
            }
          }
        }
      }
      return;
    }
    const int sub = lane & 3;
    const int li = lane >> 2;   // landmark of the batch
    const double *poses = prm.poses[st->cur];
    const double *points = prm.points[st->cur];
    const double lambda = st->lambda;
    double *Ebase = tsm + grp * bufD;
    double *Bbase = Ebase + kT2K * ldE;
    // software pipeline over the warp's batches: rec_n = record of the next batch, (a, b, pt, X) of the current one
    int a = 0, b = 0, pt = 0;
    double X[3] = {0.0, 0.0, 0.0};
    bool live = false;
    int rhs_n = 0, nb_n = 0;   // rec.w = rhs column of the chunk's B operand (8 nt) | window width << 16; rec.y = landmarks
    auto load_landmark = [&](int4 rec) {
      live = li < rec.y;
      rhs_n = rec.w;
      nb_n = rec.y;
      a = b = pt = 0;
      if (live) {
        const int ti = rec.x + li;
        a = __ldg(tpt_inc_start + ti);
        b = __ldg(tpt_inc_start + ti + 1);
        pt = __ldg(tpt_point + ti);
        X[0] = __ldg(points + (size_t)pt * 3);
        X[1] = __ldg(points + (size_t)pt * 3 + 1);
        X[2] = __ldg(points + (size_t)pt * 3 + 2);
      }
    };
    int fb = b0 + grp;
    int4 rec_n = make_int4(0, 0, 0, 0);
    if (fb < b1) {
      load_landmark(__ldg(batches + fb));
      if (fb + G < b1) rec_n = __ldg(batches + fb + G);
    }
    int4 ia_b = make_int4(0, 0, 0, 0);   // first incidence record of the lane in the coming batch
    int2 sc_b = make_int2(-1, 0);
    if (a + sub < b) { ia_b = __ldg(inc_a + a + sub); sc_b = __ldg(inc_b + a + sub); }
    for (; fb < b1; fb += G) {
      const bool cur_live = live;
      const int ca = a, cb = b, cpt = pt;
      const int rhs_col = rhs_n & 0xffff, W = rhs_n >> 16, cur_nb = nb_n;
      const double X0 = X[0], X1 = X[1], X2 = X[2];
      // the lane's first incidence record was requested at the end of the previous batch
      int4 ia_n = ia_b;
      int2 sc_n = sc_b;
      double cp[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) cp[i] = 0.0;
      const double Xc[3] = {X0, X1, X2};
      // ---- 1. incidences sub, sub + 4, ... of the landmark, in warp-uniform rounds.  The buffer is only needed
      //         when the first round is stored: its loads and arithmetic run while the consumers still read it
      const int rounds = __reduce_max_sync(0xffffffffu, (cb - ca + 3) >> 2);
      unsigned covered = 0u;   // window slots of the landmark that receive a B / E block
      unsigned slots = 0u;     // (slot + 1) of the lane's incidence in round rd, 5 bits each
      for (int rd = 0; rd < rounds; ++rd) {
        const int ii = ca + sub + 4 * rd;
        const bool act = ii < cb;
        const int4 ia = ia_n;
        const int slot = act ? sc_n.x : -1;
        const int cams01 = sc_n.y;
        if (ii + 4 < cb) { ia_n = __ldg(inc_a + ii + 4); sc_n = __ldg(inc_b + ii + 4); }
        double Bv[18];
#pragma unroll
        for (int i = 0; i < 18; ++i) Bv[i] = 0.0;
        if (act) {
        double T[12];
        load_pose(poses + (size_t)ia.z * 12, T);
        for (int k = ia.x; k < ia.x + ia.y; ++k) {
          const double2 uv = obs_uv[k];
          const int kk = k - ia.x;
          const int cid = (kk == 0) ? (cams01 & 0xff) : (kk == 1) ? (cams01 >> 8) : (obs_camflags[k] & kCamMask);
          ObsLin o;
          linearize_obs(T, Xc, cams + cid * kCamStride, uv.x, uv.y, thres_huber, o);
          const double w = o.w, wr0 = w * o.pr.r0, wr1 = w * o.pr.r1;
          const double *Rm = o.Rm;
          cp[0] += w * (Rm[0] * Rm[0] + Rm[3] * Rm[3]);
          cp[1] += w * (Rm[0] * Rm[1] + Rm[3] * Rm[4]);
          cp[2] += w * (Rm[0] * Rm[2] + Rm[3] * Rm[5]);
          cp[3] += w * (Rm[1] * Rm[1] + Rm[4] * Rm[4]);
          cp[4] += w * (Rm[1] * Rm[2] + Rm[4] * Rm[5]);
          cp[5] += w * (Rm[2] * Rm[2] + Rm[5] * Rm[5]);
          cp[6] -= Rm[0] * wr0 + Rm[3] * wr1;
          cp[7] -= Rm[1] * wr0 + Rm[4] * wr1;
          cp[8] -= Rm[2] * wr0 + Rm[5] * wr1;
          if (slot >= 0 && (ACCUM_B || k == ia.x + ia.y - 1)) add_B(o, Bv);
        }
        }
        if (rd == 0 && fb - b0 >= G) bar_sync(8 + grp, bar_cnt);   // the consumers have read this buffer
        if (slot >= 0) {
          covered |= 1u << slot;
          slots |= (unsigned)(slot + 1) << (5 * rd);
#pragma unroll
          for (int r = 0; r < 6; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) Bbase[(3 * li + c) * ldB + 6 * slot + r] = Bv[r * 3 + c];
        }
      }
      if (rounds == 0 && fb - b0 >= G) bar_sync(8 + grp, bar_cnt);
      // the next batch's landmark data is requested only now: in flight during the sums / inverse / E phase, but
      // not live across the observation loop above (where it would be spilled -- a spill waits for the load)
      if (fb + G < b1) {
        load_landmark(rec_n);
        if (fb + 2 * G < b1) rec_n = __ldg(batches + fb + 2 * G);
      }
      // ---- 2. landmark sums over its 4 lanes: xor butterfly, bitwise identical on every lane of the landmark
#pragma unroll
      for (int i = 0; i < 9; ++i) {
        cp[i] += __shfl_xor_sync(0xffffffffu, cp[i], 1);
        cp[i] += __shfl_xor_sync(0xffffffffu, cp[i], 2);
      }
      // ---- the buffer still holds the previous batch: clear the window slots this landmark does not cover (few:
      //      chunks group landmarks of the same window) and, on a partial batch, the rows of the first unused
      //      landmark (the GEMM runs over whole k-steps of 4 rows); its rhs entries are cleared by the store below
      covered |= __shfl_xor_sync(0xffffffffu, covered, 1);
      covered |= __shfl_xor_sync(0xffffffffu, covered, 2);
      const bool zrow = cur_live || li == cur_nb;
      if (zrow) {
        for (int sl = sub; sl < W; sl += 4) {
          if ((covered >> sl) & 1u) continue;
          double *Bz = Bbase + (3 * li) * ldB + 6 * sl;
          double *Ez = Ebase + (3 * li) * ldE + 6 * sl;
#pragma unroll
          for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int r = 0; r < 6; r += 2) {
              *reinterpret_cast<double2 *>(Bz + c * ldB + r) = make_double2(0.0, 0.0);
              *reinterpret_cast<double2 *>(Ez + c * ldE + r) = make_double2(0.0, 0.0);
            }
        }
        if (!cur_live && sub == 0) {
#pragma unroll
          for (int c = 0; c < 3; ++c) Bbase[(3 * li + c) * ldB + rhs_col] = 0.0;
        }
      }
      if (cur_live) {
        // ---- damping + Eigen-style pivoted 3x3 LDLT inverse, redundantly on the 4 lanes (:846-856)
        double cd[6], ci[6];
        damp_invert(cp, lambda, cd, ci);
        // the 18 per-landmark values are spread over the 4 lanes of the landmark
        if (sub == 0) {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            ptblk[(PB_b + c) * Mp + cpt] = cp[6 + c];
            Bbase[(3 * li + c) * ldB + rhs_col] = cp[6 + c];
          }
          ptblk[(PB_Cd + 0) * Mp + cpt] = cd[0];
          ptblk[(PB_Cd + 1) * Mp + cpt] = cd[1];
        } else if (sub == 1) {
#pragma unroll
          for (int i = 2; i < 6; ++i) ptblk[(PB_Cd + i) * Mp + cpt] = cd[i];
          ptblk[(PB_Cinv + 0) * Mp + cpt] = ci[0];
        } else if (sub == 2) {
#pragma unroll
          for (int i = 1; i < 6; ++i) ptblk[(PB_Cinv + i) * Mp + cpt] = ci[i];
        } else {
          ptblk[(PB_Cinvb + 0) * Mp + cpt] = ci[0] * cp[6] + ci[1] * cp[7] + ci[2] * cp[8];
          ptblk[(PB_Cinvb + 1) * Mp + cpt] = ci[1] * cp[6] + ci[3] * cp[7] + ci[4] * cp[8];
          ptblk[(PB_Cinvb + 2) * Mp + cpt] = ci[2] * cp[6] + ci[4] * cp[7] + ci[5] * cp[8];
        }
        // ---- 3. E = B Cinv for the lane's own incidences (B read back from the operand the lane wrote); the
        //         operand holds -E so that the GEMM accumulates S -= E B^T directly
        for (; slots != 0u; slots >>= 5) {
          const int slot = (int)(slots & 31u) - 1;
          if (slot < 0) continue;
          const double *Bc = Bbase + (3 * li) * ldB + 6 * slot;
          double *Ec = Ebase + (3 * li) * ldE + 6 * slot;
#pragma unroll
          for (int r = 0; r < 6; ++r) {
            const double v0 = Bc[r], v1 = Bc[ldB + r], v2 = Bc[2 * ldB + r];
            Ec[r] = -(v0 * ci[0] + v1 * ci[1] + v2 * ci[2]);
            Ec[ldE + r] = -(v0 * ci[1] + v1 * ci[3] + v2 * ci[4]);
            Ec[2 * ldE + r] = -(v0 * ci[2] + v1 * ci[4] + v2 * ci[5]);
          }
        }
      }
      ia_b = make_int4(0, 0, 0, 0);
      sc_b = make_int2(-1, 0);
      if (a + sub < b) { ia_b = __ldg(inc_a + a + sub); sc_b = __ldg(inc_b + a + sub); }   // round 0 of the next batch
      bar_arrive(1 + grp, bar_cnt);   // operands of this batch are complete
    }
  } else {
    // ===================================================== consumers =====================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kT2ConsRegs));
    const int cw = warp - kT2ProdWarps;
    const int fr = lane >> 2, fc = 2 * (lane & 3), kq = lane & 3;
    const double *Afrag0 = tsm + kq * ldE + fr;                 // + 8 ti
    const double *Bfrag0 = tsm + kT2K * ldE + kq * ldB + fr;    // + 8 tj
    // The window is cut into 2 x 2 super-tiles (16 x 16 entries) so that every fragment read from shared memory
    // feeds two DMMAs: super-tile (I, J), J >= I, holds tiles (2I + p, 2J + q); the rhs travels as tile column nt.
    int sdesc[kT2SPW];               // I | J << 8 | diagonal << 16 of the warp's super-tiles; mycnt of them are live
    int aofs[kT2SPW], bofs[kT2SPW];  // 16 I, 16 J
    double acc[kT2SPW][4][2];
    int mycnt = 0, cur_chunk = -1, nrows = 0, nt = 0;
    // flush: upper triangle of the chunk's window (row-major) and its rhs column.  Every (CTA, chunk) SEGMENT of the
    // batch list owns a private staging window, written with plain stores (every entry, zeros included, so nothing has
    // to be cleared); k_tile_reduce then adds the windows into S in segment order and S is bit-reproducible.
    int seg = __ldg(cta_seg_ptr + blockIdx.x) - 1;
    double *stg = stage;
    auto flush = [&]() {
      const int ldc = nrows + 1;
#pragma unroll
      for (int i = 0; i < kT2SPW; ++i) {
        if (i >= mycnt) continue;
        const int I = sdesc[i] & 0xff, J = (sdesc[i] >> 8) & 0xff;
#pragma unroll
        for (int p = 0; p < 2; ++p)
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const int tj = 2 * J + q;
            const int lr = 8 * (2 * I + p) + fr;
            if (lr >= nrows || tj > nt) continue;
            double *srow = stg + (size_t)lr * ldc;
            if (tj == nt) {
              if (fc == 0) __stcg(srow + nrows, acc[i][2 * p + q][0]);
            } else {
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const int lc = 8 * tj + fc + e;
                if (lc < nrows && lc >= lr) __stcg(srow + lc, acc[i][2 * p + q][e]);
              }
            }
          }
      }
    };
    int4 rec = make_int4(0, 0, 0, 0);
    if (b0 < b1) rec = __ldg(batches + b0);
    int buf = 0;
    for (int fb = b0; fb < b1; ++fb) {
      const int4 rec_n = (fb + 1 < b1) ? __ldg(batches + fb + 1) : rec;
      if (rec.z != cur_chunk) {
        if (cur_chunk >= 0) flush();
        cur_chunk = rec.z;
        stg = stage + __ldg(seg_off + (++seg));
        const SchurChunk ch = chunks[cur_chunk];
        nrows = 6 * ch.width;
        nt = (nrows + 7) >> 3;
        const int nI = (nt + 1) >> 1, nJ = (nt + 2) >> 1;          // super-rows, super-columns (rhs included)
        const int nst = nI * nJ - nI * (nI - 1) / 2;
        const int cnt = (nst + 3) >> 2;
        mycnt = max(0, min(cnt, nst - cw * cnt));
#pragma unroll
        for (int i = 0; i < kT2SPW; ++i) {
          int e = cw * cnt + i, I = 0, len = nJ;
          if (i < mycnt) {
            while (e >= len) { e -= len; ++I; --len; }
          } else {
            e = 0;
          }
          const int J = I + e;
          sdesc[i] = I | (J << 8) | ((I == J) ? (1 << 16) : 0);
          aofs[i] = 16 * I;
          bofs[i] = 16 * J;
#pragma unroll
          for (int u = 0; u < 4; ++u) acc[i][u][0] = acc[i][u][1] = 0.0;
        }
      }
      const double *Ab = Afrag0 + buf * bufD, *Bb = Bfrag0 + buf * bufD;
      bar_sync(1 + buf, bar_cnt);
      // window += (-E_all) B_all^T  (K = 3 nb, zero padded)
      const int ksteps = (3 * rec.y + 3) >> 2;
#pragma unroll 2
      for (int ks = 0; ks < ksteps; ++ks) {
        const double *Ak = Ab + ks * 4 * ldE, *Bk = Bb + ks * 4 * ldB;
#pragma unroll
        for (int i = 0; i < kT2SPW; ++i) {
          if (i >= mycnt) break;   // uniform
          const double *pa = Ak + aofs[i], *pb = Bk + bofs[i];
          const double a0 = pa[0], a1 = pa[8], v0 = pb[0], v1 = pb[8];
          dmma_884nv2(acc[i][0][0], acc[i][0][1], a0, v0);
          dmma_884nv2(acc[i][1][0], acc[i][1][1], a0, v1);
          if (!(sdesc[i] >> 16)) dmma_884nv2(acc[i][2][0], acc[i][2][1], a1, v0);   // below the diagonal: not needed
          dmma_884nv2(acc[i][3][0], acc[i][3][1], a1, v1);
        }
      }
      if (fb + G < b1) bar_arrive(8 + buf, bar_cnt);   // hand the buffer back to its producer warp
      buf = (buf + 1 == G) ? 0 : buf + 1;
      rec = rec_n;
    }
    if (cur_chunk >= 0) flush();
  }
}

// Second stage of the deterministic flush: S(r, c) += sum over the staging segments whose window holds (r, c), in
// segment order.  One CTA per scalar row; segments are sorted by their first pose, so the candidates of a row are a
// contiguous range (pose_seg).
// STORE form (store_bw >= 0; banded plans, ba_engine.cu enqueue_build): the row is WRITTEN
// instead of added to -- band entries r .. r + store_bw and the rhs entry get (damped pose-side sums of the accepted
// parameter buffer, Au) + (sum of the windows), everything else of the band gets the plain sum (zero where no window
// reaches) -- so neither the clearing of S nor k_pose_diag is launched; the row's CTA also stores the row of A and the
// entry of a that the back-substitution reads.  Same values as clear + k_pose_diag + add, bit for bit.
__global__ void __launch_bounds__(96) k_tile_reduce(int n, int ld, int span /*largest column distance written*/,
                                                     const int4 *__restrict__ seg_win /*6 jmin, rows, offset lo, offset hi*/,
                                                     const int2 *__restrict__ pose_seg,
                                                     const double *__restrict__ stage, double *__restrict__ Saug,
                                                     int store_bw, const double *__restrict__ Au0,
                                                     const double *__restrict__ Au1, double *__restrict__ A,
                                                     double *__restrict__ a, const LmState *__restrict__ st) {
  if (st->done) return;
  const int r = blockIdx.x;
  const int2 range = __ldg(pose_seg + r / 6);
  const int cover = store_bw > span ? store_bw : span;   // column distances handled by this CTA (+ the rhs entry)
  // the segment records that hold this row, once per CTA and in segment order (read per entry they would be the bulk
  // of the traffic), kKeep at a time
  constexpr int kKeep = 128;
  __shared__ int4 rec[kKeep];
  __shared__ int n_rec;
  double sum[2] = {0.0, 0.0};                 // up to two columns per thread (cover + 2 <= 2 x 96)
  for (int s0 = range.x; s0 < range.y; s0 += kKeep) {
    __syncthreads();
    if (threadIdx.x < 32) {       // ordered compaction of the segments that hold row r (warp 0, ballots)
      const int lane = threadIdx.x, end = min(range.y, s0 + kKeep);
      int cnt = 0;
      for (int base = s0; base < end; base += 32) {
        const int sg = base + lane;
        int4 w = make_int4(0, 0, 0, 0);
        if (sg < end) w = __ldg(seg_win + sg);
        const bool hit = sg < end && r - w.x >= 0 && r - w.x < w.y;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (hit) rec[cnt + __popc(m & ((1u << lane) - 1u))] = w;
        cnt += __popc(m);
      }
      if (lane == 0) n_rec = cnt;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int t = threadIdx.x + u * blockDim.x;
      if (t > cover + 1) continue;
      const bool rhs = t == cover + 1;
      const int c = rhs ? n : r + t;
      if (!rhs && c >= n) continue;
      for (int k0 = 0; k0 < n_rec; k0 += 8) {        // eight loads in flight, summed in segment order
        double v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int4 w = rec[min(k0 + q, n_rec - 1)];
          const bool ok = k0 + q < n_rec && (rhs || c - w.x < w.y);
          const long long off = ((long long)w.w << 32) | (unsigned)w.z;
          v[q] = ok ? __ldcg(stage + off + (size_t)(r - w.x) * (w.y + 1) + (rhs ? w.y : c - w.x)) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) sum[u] += v[q];
      }
    }
  }
  const int j = r / 6, rr = r - 6 * j;
  const double *Au = nullptr;
  double lp1 = 1.0;
  if (store_bw >= 0) {
    Au = (st->cur ? Au1 : Au0) + (size_t)j * 27;
    lp1 = 1.0 + st->lambda;
    if (threadIdx.x < 6) {       // row rr of the damped 6 x 6 block A_j (both triangles)
      const int cc = threadIdx.x, lo = rr < cc ? rr : cc, hi = rr < cc ? cc : rr;
      double v = Au[lo * 6 - lo * (lo - 1) / 2 + (hi - lo)];
      if (cc == rr) v *= lp1;
      A[(size_t)j * 36 + rr * 6 + cc] = v;
    }
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int t = threadIdx.x + u * blockDim.x;
    if (t > cover + 1) continue;
    const bool rhs = t == cover + 1;
    const int c = rhs ? n : r + t;
    if (!rhs && c >= n) continue;
    double *dst = Saug + (size_t)r * ld + (rhs ? ld - 1 : c);
    if (store_bw >= 0 && (rhs || t <= store_bw)) {
      double base = 0.0;
      if (rhs) {
        base = Au[21 + rr];
        a[(size_t)j * 6 + rr] = base;
      } else if (t < 6 - rr) {   // (rr, rr + t) of the diagonal block, packed upper index
        base = Au[rr * 6 - rr * (rr - 1) / 2 + t];
        if (t == 0) base *= lp1;
      }
      *dst = base + sum[u];
    } else if (sum[u] != 0.0) {
      *dst += sum[u];
    }
  }
}

// K6 for the tile landmarks: Btx[pt] = sum_j B_ji^T x_j.  k_build_tiles keeps B only in its shared-memory operands;
// here B is formed again at the accepted parameters by the same linearize_obs / add_B (last observation of the
// incidence, or all of them when ACCUM_B), which reads ~40 B per incidence instead of storing and reading back 144 B
// per pair (C3: 72 MB written by the build + 76 MB read here, per iteration).  4 adjacent lanes per tile landmark, in
// tile order, as in the producers of k_build_tiles: lane sub takes incidences sub, sub + 4, ...; the 4 partials are
// combined with the xor butterfly (fixed order: bit-reproducible, no atomics) and stored, zeros for a landmark without
// a free incidence.  The kernel is bound by its chain of dependent gathers (landmark -> incidences -> pose, pixel ->
// x), so the landmarks are numbered directly rather than through the batch list, and the free-pose index of x comes
// from pose_opt (same level as the pose) rather than from the chunk's window.
// Registers: reference mode runs three CTAs per SM (80 registers, 56 B of spill stores) because that measured faster
// than two CTAs without spills (108 registers); back-substitution phase on one B200 at 1000 W, C3 / C4 / C5: 29.7 /
// 232 / 373 us against 29.7 / 268 / 412 us (profiles/r03_bench_*_backsub_2cta.json).  Corrected mode keeps two CTAs
// (128 registers, 24 B of spill stores; at three it spills 364 B).
template <bool ACCUM_B>
__global__ void __launch_bounds__(256, ACCUM_B ? 2 : 3)
k_backsub_tiles(int n_tpt, const int *__restrict__ tpt_point, const int *__restrict__ tpt_inc_start,
                const int4 *__restrict__ inc_a, const int2 *__restrict__ inc_b, const double2 *__restrict__ obs_uv,
                const int *__restrict__ obs_camflags, const int *__restrict__ pose_opt, Params prm,
                const double *__restrict__ cams, double thres_huber, const double *__restrict__ x,
                double *__restrict__ Btx /*[3][Mp]*/, size_t Mp, const LmState *__restrict__ st) {
  if (st->done) return;
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  if ((gt & ~31) >= 4 * n_tpt) return;   // whole warps
  const int ti = gt >> 2, sub = gt & 3;
  const bool live = ti < n_tpt;
  int pt = 0;
  double v[3] = {0.0, 0.0, 0.0};
  if (live) {
    const int a = __ldg(tpt_inc_start + ti), b = __ldg(tpt_inc_start + ti + 1);
    pt = __ldg(tpt_point + ti);
    const double *poses = prm.poses[st->cur];
    const double *points = prm.points[st->cur];
    const double X[3] = {__ldg(points + (size_t)pt * 3), __ldg(points + (size_t)pt * 3 + 1),
                         __ldg(points + (size_t)pt * 3 + 2)};
    for (int ii = a + sub; ii < b; ii += 4) {
      const int2 sc = __ldg(inc_b + ii);
      const int4 ia = __ldg(inc_a + ii);
      if (sc.x < 0) continue;   // fixed pose: no B block
      const int j = __ldg(pose_opt + ia.z);   // = window start + sc.x
      double T[12];
      load_pose(poses + (size_t)ia.z * 12, T);
      double Bv[18];
#pragma unroll
      for (int i = 0; i < 18; ++i) Bv[i] = 0.0;
      for (int k = ACCUM_B ? ia.x : ia.x + ia.y - 1; k < ia.x + ia.y; ++k) {
        const double2 uv = obs_uv[k];
        const int kk = k - ia.x;   // camera: the producers' rule
        const int cid = (kk == 0) ? (sc.y & 0xff) : (kk == 1) ? (sc.y >> 8) : (obs_camflags[k] & kCamMask);
        ObsLin o;
        linearize_obs(T, X, cams + cid * kCamStride, uv.x, uv.y, thres_huber, o);
        add_B(o, Bv);
      }
      const double *xj = x + (size_t)6 * j;
      double xv[6];
#pragma unroll
      for (int r = 0; r < 6; ++r) xv[r] = __ldg(xj + r);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < 6; ++r) s += Bv[r * 3 + c] * xv[r];
        v[c] += s;
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    v[c] += __shfl_xor_sync(0xffffffffu, v[c], 1);
    v[c] += __shfl_xor_sync(0xffffffffu, v[c], 2);
  }
  if (live && sub == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) Btx[(size_t)c * Mp + pt] = v[c];
  }
}
