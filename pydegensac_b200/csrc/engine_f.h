// engine_f.h -- LO-RANSAC / DEGENSAC for the fundamental matrix, one CTA per image pair.
//
// Replaces the reference's sequential driver exp_ransacFcustomLAF (exp_ranF.c:1244-1767) and its LO
// (exp_inFranicustom :745-806, exp_iterFcustom :621-743) by a two-phase design:
//
//   WAVE   (parallel, speculative)  a chunk of iterations is hypothesised at once: one THREAD draws the
//          Philox sample, solves the 7-point problem in registers/local memory and applies the oriented
//          epipolar test; surviving models are queued and one WARP per model scores them over all
//          correspondences of the FP32 tile (lane-strided, shuffle reduction).  Only models whose MSAC
//          score can beat the running thresholds survive the wave.
//   REPLAY (ordered, exact)         survivors are re-evaluated in iteration order with the reference's
//          control flow: so-far-the-best bookkeeping, symmetric gate, LO scheduling (first-50 rule),
//          iterated re-weighted 8-point LSQ with hash de-duplication, adaptive termination.
//
// Why this is equivalent: WHICH models get scored depends only on the sampling stream; the running best
// only decides acceptance / LO / termination (exp_ranF.c:1381-1499,1571-1576), and a model can change
// state only if J > min(best.J, bestSample.J), a bound that never decreases inside a chunk (if it
// does -- DEGENSAC branch -- the chunk is re-waved).  The first ITER_SAM iterations are replayed
// unfiltered because the reference's forced LO at sample 50 reads a residual row that later models of
// the same root index have overwritten (errs[4] aliasing, exp_ranF.c:1375,1486,1497-1508).
#pragma once
#include "common.h"
#include "rng.h"
#include "la.h"
#include "fgeom.h"
#include "block.h"
#include "ffit.h"
#include "hfit.h"
#include "degensac.h"
#include "filter32.h"

namespace dg {

#ifdef DG_FILTER_CHECK
static long g_filter_checked = 0, g_filter_violations = 0;
static double g_filter_maxslack = 0.0;
#endif

// ---------------------------------------------------------------------------------------------
// Iterated re-weighted LSQ with shrinking threshold (reference exp_iterFcustom, exp_ranF.c:621-743).
// e[] are the physical ids behind the reference's errs[] pointers; e[4] holds the residual row of the
// starting model.  With the binding's inlLimit=0 every fit uses a random 8-subset (SURVEY App. A#5).
// ---------------------------------------------------------------------------------------------
DG_ENGN Score lo_iter_F(const Ctx& c, const FParams& P, Workspace& W, int* e, int* inl, double th,
                              double ths, double* Fio, int iterID, DrawCursor& cur, HashTab& ht) {
  int d = e[1];
  double f[9];
  const double dth = (ths - th) / kIlsqIters;
  Score S = make_score(), Ss, maxS;
  maxS = blk_inlidxs(c, W.err[e[4]], th, inl);
  if (maxS.I < 8) return S;
  S = blk_inlidxs(c, W.err[e[4]], th * kMWM, inl);
  if (8 >= S.I) {
    blk_fit_F(c, inl, (int)S.I, nullptr, f);
  } else {
    blk_sample8_fit_F(c, inl, (int)S.I, nullptr, cur, f);
  }
  #pragma unroll 1
  for (int it = 0; it < kIlsqIters; ++it) {
    blk_resid_w_F(c, P.metric, f, W.err[d], W.w);
    // The support at the wider threshold is needed on the SAME row unless this iteration improves the score (then
    // the reference's pointer rotation moves `d` to the previous best row): both lists are built in one pass, the
    // second one speculatively into a side buffer, and copied over `inl` when it is the one the reference would
    // have built (the copy keeps `inl` byte-identical to the reference's buffer, whose stale tail is read later by
    // the caller -- SURVEY App. A).
    int* spec = W.itmp[0];
    Score Sspec;
    blk_inlidxs2(c, W.err[d], th, inl, &S, ths * kMWM, spec, &Sspec);
#if DG_DEVICE_PASS
    if (!score_less(maxS, S) && Sspec.I > 8 && c.nw >= 2) {
      // no improvement: the next fit uses the speculative list; run it next to the hash chain (see ffit.h)
      if (blk_hash_and_fit8_F(c, W, ht, inl, (int)S.I, iterID, spec, (int)Sspec.I, W.w, cur, inl, f)) return make_score();
      ths -= dth;
      continue;
    }
#endif
    if (hash_seen_elsewhere(c, W, ht, inl, (int)S.I, iterID)) return make_score();
    if (score_less(maxS, S)) {
      maxS = S;
      e[1] = e[0];
      e[0] = d;
      d = e[1];
      for (int i = 0; i < 9; ++i) Fio[i] = f[i];
      Ss = blk_inlidxs(c, W.err[d], ths * kMWM, inl);
    } else {
      Ss = Sspec;
      #pragma unroll 1
      for (int j = c.tid; j < (int)Ss.I; j += c.nt) inl[j] = spec[j];
      DG_SYNC();
    }
    if (Ss.I < 8) return maxS;
    if (8 >= Ss.I) {
      blk_fit_F(c, inl, (int)Ss.I, W.w, f);
    } else {
      blk_sample8_fit_F(c, inl, (int)Ss.I, W.w, cur, f);
    }
    ths -= dth;
  }
  blk_resid_F(c, P.metric, f, W.err[d]);
  S = blk_inlidxs(c, W.err[d], th, inl);
  if (score_less(maxS, S)) {
    maxS = S;
    e[1] = e[0];
    e[0] = d;
    for (int i = 0; i < 9; ++i) Fio[i] = f[i];
  }
  return maxS;
}

// Inner RANSAC of the LO step (reference exp_inFranicustom, exp_ranF.c:745-806).
DG_ENGN Score lo_inner_F(const Ctx& c, const FParams& P, Workspace& W, int* e, int* inliers, int ninl,
                               double th, double* Fout, int& iterID, DrawCursor& cur, HashTab& ht) {
  Score S, maxS = make_score();
  if (ninl < 16) return maxS;
  int ssiz = ninl / 2;
  if (ssiz > 14) ssiz = 14;
  int t = e[2]; e[2] = e[0]; e[0] = t;
  double f[9];
  #pragma unroll 1
  for (int rep = 0; rep < kRanRep; ++rep) {
    blk_randsubset(c, inliers, ninl, ssiz, cur);
    blk_fit_F(c, inliers + ninl - ssiz, ssiz, nullptr, f);
    blk_resid_F(c, P.metric, f, W.err[e[0]]);
    e[4] = e[0];
    ++iterID;
    S = lo_iter_F(c, P, W, e, W.intbuff, th, kTC * th, f, iterID, cur, ht);
    if (score_less(maxS, S)) {
      maxS = S;
      t = e[2]; e[2] = e[0]; e[0] = t;
      for (int i = 0; i < 9; ++i) Fout[i] = f[i];
      #pragma unroll 1
      for (int j = c.tid; j < (int)maxS.I; j += c.nt) W.intbuff_best[j] = W.intbuff[j];
      DG_SYNC();
    }
  }
  t = e[2]; e[2] = e[0]; e[0] = t;
  #pragma unroll 1
  for (int j = c.tid; j < (int)maxS.I; j += c.nt) inliers[j] = W.intbuff_best[j];
  DG_SYNC();
  return maxS;
}

// Running state of one pair (replicated in every thread; all values are block-uniform).
struct FState {
  Score maxS, maxSs;
  int e[5];
  double F[9], FBest[9];
  int samidxBest[7];
  int max_sam, iter_cnt, degen_cnt, non_degen, iterID, Ihmax;
  HashTab ht;
  DrawCursor cur;
};

// "LSQ before LO" + LO + acceptance (exp_ranF.c:1501-1577 in the loop, :1630-1696 post-loop).
// src_row: residual row the LSQ support is taken from (errs[4] in the loop, errorsBest post-loop).
DG_ENGN bool run_lo_F(const Ctx& c, const FParams& P, Workspace& W, FState& st, const double* src_row) {
  double f[9];
  bool new_max = false;
  DG_PROF_BEGIN(3);
  ++st.iter_cnt;
  const int d = st.e[0];
  Score S = blk_inlidxs(c, src_row, kTC * P.th * kMWM, W.inliers);
  blk_fit_F(c, W.inliers, (int)S.I, nullptr, f);
  blk_resid_F(c, P.metric, f, W.err[d]);
  S = blk_inlidxs(c, W.err[d], P.th, W.inliers);
  S = lo_inner_F(c, P, W, st.e, W.inliers, (int)S.I, P.th, f, st.iterID, st.cur, st.ht);
  if (score_less(st.maxS, S)) {
    bool do_update = true;
    if (P.do_sym) {
      S.Is = blk_sym_count_F(c, f, W.inliers, (int)S.I, P.sym_th);
      if (S.Is < st.maxS.Is) do_update = false;
    }
    if (P.do_laf && do_update) {   // exp_ranF.c:1536-1555 / 1664-1683
      S.Ilafs = blk_laf_count_F(c, P.metric, f, W.inliers, (int)S.I, P.th_laf);
      if (S.Ilafs < st.maxS.Ilafs) do_update = false;
    }
    if (do_update) {
      const int t = st.e[0]; st.e[0] = st.e[3]; st.e[3] = t;
      st.maxS = S;
      for (int i = 0; i < 9; ++i) st.F[i] = f[i];
      new_max = true;
    }
  }
  DG_PROF_END(3);
  return new_max;
}

#if DG_DEVICE_PASS
// ---------------------------------------------------------------------------------------------
// Wave stage A1 (device): Gauss-Jordan of the 7x9 sample systems with TWO THREADS PER SAMPLE, the matrix held in
// registers (thread h of a lane pair owns columns 5h..5h+4 as a[lc][row]; pivots, pivot row choice and the six
// multipliers travel through warp shuffles).  Every entry sees exactly the operations of the reference's
// `nullspace` in the same order (utools.c:97-167: partial pivoting from the diagonal, pivot row divided, all other
// rows eliminated), so the two null vectors are bit-identical to the one-thread routine (nullspace9) that the
// host emulation and the non-generic fallback use -- without its 1.3 KB of local memory per thread.
// Output per iteration k: W.nsbuf[16*(k-kbeg) + ..] = {-col7[0..6], -col8[0..6], generic?1:0}.
// ---------------------------------------------------------------------------------------------
// One pivot column of the pair elimination.  A template (not a loop) so that every index into `a` is a literal
// in each instantiation: with the seven columns as an unrolled loop the compiler left the whole matrix in local
// memory (280-byte depot, ~800 local loads/stores per sample).
template <int COL>
__device__ __forceinline__ void pairsolve_step(double (&a)[5][7], int h, int lane, bool& generic) {
  constexpr int owner = (COL < 5) ? 0 : 1;
  constexpr int lc = COL - 5 * owner;
  const unsigned full = 0xffffffffu;
  int best = COL;
  double mag = 0.0;
  if (h == owner) {
    mag = fabs(a[lc][COL]);
#pragma unroll
    for (int r = COL + 1; r < 7; ++r) {
      const double t = fabs(a[lc][r]);
      if (mag < t) { mag = t; best = r; }
    }
  }
  const int src = (lane & ~1) | owner;
  best = __shfl_sync(full, best, src);
  mag = __shfl_sync(full, mag, src);
  if (mag < 1e-12) generic = false;
#pragma unroll
  for (int r = COL + 1; r < 7; ++r) {
    if (best == r) {
#pragma unroll
      for (int q = 0; q < 5; ++q) { const double t = a[q][COL]; a[q][COL] = a[q][r]; a[q][r] = t; }
    }
  }
  const double p = __shfl_sync(full, a[lc][COL], src);
  // (dividing the pivot row through one shared reciprocal, as hgeom.h does for pinvJ, was measured 1.7 % SLOWER here:
  //  at most five quotients per thread share the reciprocal and the range guards cost more than they save)
  double m[7];
#pragma unroll
  for (int r = 0; r < 7; ++r) m[r] = (r == COL) ? 0.0 : __shfl_sync(full, a[lc][r], src);
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    const int gc = 5 * h + q;
    if (gc >= COL && gc < 9) {
      a[q][COL] /= p;
#pragma unroll
      for (int r = 0; r < 7; ++r)
        if (r != COL) a[q][r] -= m[r] * a[q][COL];
    }
  }
}

__device__ __noinline__ void wave_F_pairsolve(const Ctx& c, const FParams& P, Workspace& W, int kbeg, int kend) {
  const int h = c.lane & 1;
  const int slot = c.lane >> 1;
  const int per_pass = c.nw * 16;
#pragma unroll 1
  for (int base = kbeg + c.wid * 16; base <= kend; base += per_pass) {
    const int k = base + slot;
    const bool live = k <= kend;
    int sel[7];
    minimal_sample<7>(P.seed, (uint32_t)(live ? k : kbeg), c.N, sel);
    double a[5][7];
#define DG_PS_ROW(r)                                                                                             \
    {                                                                                                            \
      const int p = sel[r];                                                                                      \
      const double x1 = c.x1[p], y1 = c.y1[p], x2 = c.x2[p], y2 = c.y2[p];                                       \
      a[0][r] = h ? y2 : x2 * x1; a[1][r] = h ? x1 : x2 * y1; a[2][r] = h ? y1 : x2;                              \
      a[3][r] = h ? 1.0 : y2 * x1; a[4][r] = h ? 0.0 : y2 * y1;                                                  \
    }
    DG_PS_ROW(0) DG_PS_ROW(1) DG_PS_ROW(2) DG_PS_ROW(3) DG_PS_ROW(4) DG_PS_ROW(5) DG_PS_ROW(6)
#undef DG_PS_ROW
    bool generic = true;
    pairsolve_step<0>(a, h, c.lane, generic);
    pairsolve_step<1>(a, h, c.lane, generic);
    pairsolve_step<2>(a, h, c.lane, generic);
    pairsolve_step<3>(a, h, c.lane, generic);
    pairsolve_step<4>(a, h, c.lane, generic);
    pairsolve_step<5>(a, h, c.lane, generic);
    pairsolve_step<6>(a, h, c.lane, generic);
    if (live && h == 1) {
      double* o = W.nsbuf + (size_t)(k - kbeg) * 16;
      o[0] = -a[2][0]; o[1] = -a[2][1]; o[2] = -a[2][2]; o[3] = -a[2][3]; o[4] = -a[2][4]; o[5] = -a[2][5]; o[6] = -a[2][6];
      o[7] = -a[3][0]; o[8] = -a[3][1]; o[9] = -a[3][2]; o[10] = -a[3][3]; o[11] = -a[3][4]; o[12] = -a[3][5]; o[13] = -a[3][6];
      o[14] = generic ? 1.0 : 0.0;
    }
  }
}
#endif

// Null-space basis of a 7-point sample by the one-thread routine (host emulation; device: only the rare samples
// whose pair elimination met a tiny pivot).  Returned by value so that the caller's copies stay in registers.
struct NullPair { double v[18]; int n; };
DG_ENGN NullPair nullspace_of_sample(const Ctx& c, int p0, int p1, int p2, int p3, int p4, int p5, int p6) {
  double M[81], full[81];
  const int ps[7] = {p0, p1, p2, p3, p4, p5, p6};
  #pragma unroll 1
  for (int i = 0; i < 7; ++i) {
    const int p = ps[i];
    f_lin_row(c.x1[p], c.y1[p], c.x2[p], c.y2[p], M + 9 * i);
  }
  #pragma unroll 1
  for (int i = 63; i < 81; ++i) M[i] = 0.0;
  NullPair r;
  r.n = nullspace9(M, full);
  #pragma unroll 1
  for (int i = 0; i < 18; ++i) r.v[i] = full[i];
  return r;
}

// ---------------------------------------------------------------------------------------------
// WAVE: hypothesise iterations kbeg..kend (1-based), queue oriented-valid models, score them one
// warp per model, keep those with J > T (or all when passall).  Returns the number kept; W.pass holds
// their indices into W.cand sorted by (iteration, root).  valid_itersam reports whether iteration
// ITER_SAM produced a two-dimensional null space (needed for the forced-LO rule).
// ---------------------------------------------------------------------------------------------
DG_ENGN int wave_F(const Ctx& c, const FParams& P, Workspace& W, int kbeg, int kend, double T, bool passall,
                         bool* valid_itersam) {
  DG_SYNC();
  if (c.tid == 0) { c.sc->counter[0] = 0; c.sc->counter[1] = 0; c.sc->counter[2] = 0; }
  // (an L1 prefetch of the whole SoA in front of the gathers of stage A was measured neutral-to-negative once the
  //  streaming passes stopped polluting L1 -- the lines it displaced, stack and lists, cost as much as it saved)
  DG_SYNC();
  // stage A: minimal solvers.  Device: A1 = two threads per sample eliminate in registers (wave_F_pairsolve),
  // A2 = one thread per sample takes the null-space basis through the cubic and the oriented test.
  DG_PROF_BEGIN(0);
  DG_PROF_COUNT(9, 1);
  DG_PROF_COUNT(12, kend - kbeg + 1);
#if DG_DEVICE_PASS
  DG_PROF_BEGIN(10);
  wave_F_pairsolve(c, P, W, kbeg, kend);
  DG_SYNC();
  DG_PROF_END(10);
#endif
  #pragma unroll 1
  for (int k = kbeg + c.tid; k <= kend; k += c.nt) {
    int sel[7];
    minimal_sample<7>(P.seed, (uint32_t)k, c.N, sel);
    // every array below is indexed by literals only (after unrolling) so that it lives in registers
    double f1[9], f2[9];
    int nullsize = 2;
#if DG_DEVICE_PASS
    const double* ns = W.nsbuf + (size_t)(k - kbeg) * 16;
    if (ns[14] != 0.0) {
#pragma unroll
      for (int i = 0; i < 7; ++i) { f1[i] = ns[i]; f2[i] = ns[7 + i]; }
      f1[7] = 1.0; f1[8] = 0.0; f2[7] = 0.0; f2[8] = 1.0;
    } else
#endif
    {
      const NullPair np = nullspace_of_sample(c, sel[0], sel[1], sel[2], sel[3], sel[4], sel[5], sel[6]);
      nullsize = np.n;
#pragma unroll
      for (int i = 0; i < 9; ++i) { f1[i] = np.v[i]; f2[i] = np.v[9 + i]; }
    }
    if (nullsize != 2) continue;
    if (k == kIterSam) c.sc->counter[2] = 1;
    double poly[4], roots[3];
    seven_pt_cubic_inl(f1, f2, poly);
    roots[1] = 0.0; roots[2] = 0.0;
    const int nsol = cubic_real_roots_inl(poly, roots);
    double sy1[7], sx2[7], sy2[7];
#pragma unroll
    for (int t = 0; t < 7; ++t) {  // reference samidx order = reverse draw order
      const int p = sel[6 - t];
      sy1[t] = c.y1[p]; sx2[t] = c.x2[p]; sy2[t] = c.y2[p];
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (i < nsol) {
        double f[9];
#pragma unroll
        for (int j = 0; j < 9; ++j) f[j] = f1[j] * roots[i] + f2[j] * (1 - roots[i]);
        if (oriented_ok_F7(f, sy1, sx2, sy2)) {
          const int slot = atomic_inc_shared(&c.sc->counter[0]);
          if (slot < W.cand_cap) {
            Cand& cd = W.cand[slot];
#pragma unroll
            for (int j = 0; j < 9; ++j) cd.f[j] = f[j];
            cd.k = k;
            cd.root = i;
          }
        }
      }
    }
  }
  DG_SYNC();
  DG_PROF_END(0);
  DG_PROF_BEGIN(1);
  DG_PROF_COUNT(13, c.sc->counter[0]);
  int ncand = c.sc->counter[0];
  *valid_itersam = (c.sc->counter[2] != 0);
  if (ncand > W.cand_cap) { DG_SYNC(); return -1; }   // queue overflow: the driver splits the wave
  // stage B: one warp per model, lanes stride the correspondences
  const double w94 = P.th * 9 / 4;
  #pragma unroll 1
  for (int ci = c.wid; ci < ncand; ci += c.nw) {
    bool keep = passall;
    if (!passall) {
      double f[9];
      for (int j = 0; j < 9; ++j) f[j] = W.cand[ci].f[j];
      if (c.t32) {
        // FP32 upper bound of the MSAC score (filter32.h): a superset of the models that matter survives
        FFilter32 ff;
        f_filter_setup(P.metric, f, *c.t32, w94, &ff);
        float J = 0.0f;
#if DG_DEVICE_PASS
        {  // packed pairs (FFMA2), two independent pair chains per lane and trip
          FFilter32x2 f2;
          f_filter_pack(ff, &f2);
          const float4* tp = reinterpret_cast<const float4*>(c.t32->pts);
          const int npair = (c.N + 1) >> 1;
          const int last = (c.N & 1) ? npair - 1 : -1;     // pair whose second slot is padding
          f32x2 Ja = pk2(0.0f, 0.0f), Jb = pk2(0.0f, 0.0f);
          int i = c.lane;
          #pragma unroll 1
          for (; i + 32 < npair; i += 64) {
            const float4 A0 = tp[2 * i], B0 = tp[2 * i + 1], A1 = tp[2 * i + 64], B1 = tp[2 * i + 65];
            Ja = add2(Ja, f_filter_gain2(f2, A0, B0, i != last));
            Jb = add2(Jb, f_filter_gain2(f2, A1, B1, i + 32 != last));
          }
          if (i < npair) Ja = add2(Ja, f_filter_gain2(f2, tp[2 * i], tp[2 * i + 1], i != last));
          float j0, j1;
          upk2(add2(Ja, Jb), j0, j1);
          J = j0 + j1;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) J += __shfl_xor_sync(0xffffffffu, J, o);
        }
#else
        const Pt32* pts = c.t32->pts;
        for (int i = 0; i < c.N; ++i) J += f_filter_gain(ff, pts[i]);
#endif
        const double Jup = (double)J * (1.0 + 1.52587890625e-05) + 1e-3;
#ifdef DG_FILTER_CHECK
        {
          double J64 = 0.0;
          for (int i = 0; i < c.N; ++i) {
            const double e = f_resid(P.metric, f, c.x1[i], c.y1[i], c.x2[i], c.y2[i]);
            if (e < w94) J64 += 1 - (e / w94);
          }
          if (c.lane == 0) { ++g_filter_checked; if (!(Jup >= J64) && J64 == J64) ++g_filter_violations; if (Jup - J64 > g_filter_maxslack) g_filter_maxslack = Jup - J64; }
        }
#endif
        keep = Jup > T - 1e-9 * (1.0 + fabs(T));
      } else {
        double J = 0.0;
#if DG_DEVICE_PASS
        for (int i = c.lane; i < c.N; i += 32) {
#else
        for (int i = 0; i < c.N; ++i) {
#endif
          const double e = f_resid(P.metric, f, c.x1[i], c.y1[i], c.x2[i], c.y2[i]);
          if (e < w94) J += 1 - (e / w94);
        }
        J = warp_sum(J);
        keep = J > T - 1e-9 * (1.0 + fabs(T));
      }
    }
    if (c.lane == 0 && keep) {
      const int slot = atomic_inc_shared(&c.sc->counter[1]);
      W.pass[slot] = ci;
    }
  }
  DG_SYNC();
  DG_PROF_END(1);
  const int npass = c.sc->counter[1];
  // order survivors by (iteration, root): small list, thread 0 insertion sort
  if (c.tid == 0) {
    #pragma unroll 1
    for (int a = 1; a < npass; ++a) {
      const int v = W.pass[a];
      const long key = (long)W.cand[v].k * 4 + W.cand[v].root;
      int b = a - 1;
      while (b >= 0) {
        const int u = W.pass[b];
        const long kb = (long)W.cand[u].k * 4 + W.cand[u].root;
        if (kb <= key) break;
        W.pass[b + 1] = u;
        --b;
      }
      W.pass[b + 1] = v;
    }
  }
  DG_SYNC();
  return npass;
}

// Final inlier mask (exp_ranF.c:1699-1723) incl. the reference's indexing quirk in the symmetric prune
// (it clears mask[j] for the j-th LIST POSITION instead of mask[inliers[j]]; SURVEY App. A#4).
DG_ENGN void final_mask_F(const Ctx& c, const FParams& P, Workspace& W, FState& st, unsigned char* mask) {
  double* d = W.err[st.e[3]];
  if (P.final_lsq) {   // exp_ranF.c:1701-1705: LSQ on all inliers of the best model, residuals (and the mask) from it
    const Score Sl = blk_inlidxs(c, d, P.th, W.inliers);
    blk_fit_F(c, W.inliers, (int)Sl.I, nullptr, st.F);
    blk_resid_F(c, P.metric, st.F, d);
  }
  #pragma unroll 1
  for (int j = c.tid; j < c.N; j += c.nt) mask[j] = (d[j] <= P.th) ? 1 : 0;
  DG_SYNC();
  if (P.do_sym) {
    const Score S = blk_inlidxs(c, d, P.th, W.inliers);
    #pragma unroll 1
    for (int j = c.tid; j < (int)S.I; j += c.nt) {
      const int i = W.inliers[j];
      if (f_resid_symepi(st.F, c.x1[i], c.y1[i], c.x2[i], c.y2[i]) > P.sym_th) mask[j] = 0;
    }
    DG_SYNC();
  }
}

// ---------------------------------------------------------------------------------------------
// REPLAY of one iteration (the body of the reference's while loop, exp_ranF.c:1334-1578) restricted to
// the models that survived the wave (`cnt` entries of W.pass starting at `pos`, ascending root order).
// ---------------------------------------------------------------------------------------------
DG_ENGN void replay_iteration_F(const Ctx& c, const FParams& P, Workspace& W, FState& st, int k, int pos,
                                      int cnt) {
  bool new_max = false, do_iterate = false;
  DG_PROF_BEGIN(2);
  DG_PROF_COUNT(14, 1);
  DG_PROF_COUNT(15, cnt);
  int sel[7], samidx[7];
  minimal_sample<7>(P.seed, (uint32_t)k, c.N, sel);
  for (int t = 0; t < 7; ++t) samidx[t] = sel[6 - t];
  st.cur.seed = P.seed; st.cur.k = (uint32_t)k; st.cur.j = 8;
  #pragma unroll 1
  for (int q = 0; q < cnt; ++q) {
    const Cand& cd = W.cand[W.pass[pos + q]];
    const int i = cd.root;
    double f[9];
    for (int j = 0; j < 9; ++j) f[j] = cd.f[j];
    int d = st.e[i];
    blk_resid_F(c, P.metric, f, W.err[d]);
    Score S = blk_inlidxs(c, W.err[d], P.th, W.inliers);
    if (score_less(st.maxS, S)) {
      bool ok = true;
      if (P.do_sym) {
        S.Is = blk_sym_count_F(c, f, W.inliers, (int)S.I, P.sym_th);
        if (S.Is < st.maxS.Is) ok = false;
      }
      if (ok && P.do_laf) {   // LAF gate (exp_ranF.c:1394-1412)
        S.Ilafs = blk_laf_count_F(c, P.metric, f, W.inliers, (int)S.I, P.th_laf);
        if (S.Ilafs < st.maxS.Ilafs) ok = false;
      }
      if (!ok) continue;  // the reference `continue`s: the best-sample test below is skipped too
      st.e[i] = st.e[3];
      st.e[3] = d;
      st.maxS = S;
      for (int j = 0; j < 9; ++j) st.F[j] = f[j];
      new_max = true;
    }
    if (score_less(st.maxSs, S)) {
#ifdef DG_TRACE
      fprintf(stderr, "BS k=%d root=%d S.I=%u S.J=%.17g maxS.J=%.17g\n", k, i, S.I, S.J, st.maxS.J);
#endif
      st.maxSs = S;
      DG_PROF_COUNT(16, 1);
      bool degenerate = false;
      double H[9];
      if (P.degen) {
        double u7[28];
        for (int t = 0; t < 7; ++t) {
          const int p = samidx[t];
          u7[4 * t] = c.x1[p]; u7[4 * t + 1] = c.y1[p]; u7[4 * t + 2] = c.x2[p]; u7[4 * t + 3] = c.y2[p];
        }
        DG_PROF_BEGIN(5);
        degenerate = blk_checksample(c, f, u7, 3 * P.th, H);
        DG_PROF_END(5);
      }
      if (degenerate) {
        DG_PROF_BEGIN(6);
        blk_resid_H_sampson(c, H, W.dtmp[4]);
        unsigned I = (unsigned)blk_count_lt(c, W.dtmp[4], P.th * 3);
        if (I < 8) { DG_PROF_END(6); break; }
        { DG_PROF_BEGIN(25); I = blk_inner_H(c, W, H, 16 * P.th, 10, W.btmp[0], st.cur); DG_PROF_END(25); }
        DG_PROF_COUNT(30, 1);
        if ((int)I > st.Ihmax) st.Ihmax = (int)I;
        if (I > 6) {
          { DG_PROF_BEGIN(26); I = blk_rFtH(c, W, W.btmp[0], P.th, H, f, st.cur); DG_PROF_END(26); }
          DG_PROF_COUNT(31, 1);
          if (I > st.maxS.I) {
            blk_resid_F(c, P.metric, f, W.err[st.e[3]]);
            st.maxS.I = I;
            for (int j = 0; j < 9; ++j) st.F[j] = f[j];
            new_max = true;
            d = st.e[3];
          } else {
            blk_resid_F(c, P.metric, f, W.err[st.e[i]]);
            d = st.e[i];
          }
          double jj = 0.0;
          {  // J of the row in index order per thread segment (exp_ranF.c:1470-1477)
            const Score t = blk_inlidxs(c, W.err[d], P.th, W.inliers);
            jj = t.J;
          }
          if (new_max) st.maxS.J = jj;
          ++st.degen_cnt;
        }
        DG_PROF_END(6);
      } else {
        do_iterate = (k > kIterSam);
        st.e[4] = d;
        ++st.non_degen;
        for (int t = 0; t < 7; ++t) st.samidxBest[t] = samidx[t];
        #pragma unroll 1
        for (int j = c.tid; j < c.N; j += c.nt) st_row(W.errBest + j, ld_row(W.err[d] + j));
        DG_SYNC();
        for (int j = 0; j < 9; ++j) st.FBest[j] = f[j];
      }
    }
  }
  if (k == kIterSam && st.non_degen) do_iterate = true;
  if (do_iterate) {
    DG_PROF_COUNT(17, 1);
    if (run_lo_F(c, P, W, st, W.err[st.e[4]])) new_max = true;
    if (new_max) {
      const int new_sam = nsamples((int)st.maxS.I + 1, c.N, 7, P.conf);
      if (new_sam < st.max_sam) st.max_sam = new_sam;
    }
  }
  DG_PROF_END(2);
}

// ---------------------------------------------------------------------------------------------
// One image pair, whole RANSAC.  Outputs: F (row-major, zero when no model), mask, stats
// {samples drawn, LO runs, plane inliers (Ihmax), inlier count of the returned model}.
// ---------------------------------------------------------------------------------------------
DG_ENGN void ransac_F_pair(const Ctx& c, const FParams& P, Workspace& W, double* F_out, unsigned char* mask_out,
                                 int* stats_out) {
  FState st;
  st.maxS = make_score(); st.maxSs = make_score();
  st.maxS.I = 8; st.maxSs.I = 8;
  for (int i = 0; i < 4; ++i) st.e[i] = i;
  st.e[4] = 3;
  for (int i = 0; i < 9; ++i) { st.F[i] = 0.0; st.FBest[i] = 0.0; }
  for (int i = 0; i < 7; ++i) st.samidxBest[i] = 0;
  st.max_sam = P.max_iters; st.iter_cnt = 0; st.degen_cnt = 0; st.non_degen = 0; st.iterID = 0; st.Ihmax = 0;
  st.ht.n = 0;
  st.cur.seed = P.seed; st.cur.k = 0; st.cur.j = 1;
  // residual rows start zeroed (the reference reads uninitialised malloc memory if no model is ever scored)
  for (int r = 0; r < 4; ++r)
    #pragma unroll 1
    for (int j = c.tid; j < c.N; j += c.nt) W.err[r][j] = 0.0;
  #pragma unroll 1
  for (int j = c.tid; j < c.N; j += c.nt) W.errBest[j] = 0.0;
  DG_SYNC();

  int k0 = 0, no_sam = 0;
  bool finished = false;
  while (!finished && k0 < st.max_sam) {
    int kend = k0 + P.chunk;
    if (kend > st.max_sam) kend = st.max_sam;
    const bool passall = k0 < kIterSam;
    if (passall && kend > kIterSam) kend = kIterSam;
    const double T = st.maxS.J < st.maxSs.J ? st.maxS.J : st.maxSs.J;
    bool valid_itersam = false;
    int npass = wave_F(c, P, W, k0 + 1, kend, T, passall, &valid_itersam);
    while (npass < 0) {   // more oriented-valid models than the queue holds (up to 3 per iteration): halve the wave
      kend = k0 + ((kend - k0) > 1 ? (kend - k0) / 2 : 1);
      npass = wave_F(c, P, W, k0 + 1, kend, T, passall, &valid_itersam);
    }
    int pos = 0;
    bool rewave = false, did_itersam = false;
    while (pos < npass) {
      const int k = W.cand[W.pass[pos]].k;
      if (k > st.max_sam) break;
      int cnt = 1;
      while (pos + cnt < npass && W.cand[W.pass[pos + cnt]].k == k) ++cnt;
      replay_iteration_F(c, P, W, st, k, pos, cnt);
      if (k == kIterSam) did_itersam = true;
      pos += cnt;
      if (k >= st.max_sam) { finished = true; no_sam = k; break; }
      const double Tn = st.maxS.J < st.maxSs.J ? st.maxS.J : st.maxSs.J;
      if (Tn < T && k < kend) { rewave = true; k0 = k; DG_PROF_COUNT(18, 1); break; }
    }
    if (finished) break;
    if (rewave) continue;
    if (kend == kIterSam && kIterSam <= st.max_sam && valid_itersam && !did_itersam) {
      // iteration ITER_SAM had a valid null space but no oriented-valid model: only the forced-LO rule applies
      replay_iteration_F(c, P, W, st, kIterSam, 0, 0);
      if (kIterSam >= st.max_sam) { finished = true; no_sam = kIterSam; break; }
    }
    k0 = kend;
  }
  if (!finished) no_sam = st.max_sam;
  if ((int)st.cur.k != no_sam) { st.cur.k = (uint32_t)no_sam; st.cur.j = 8; }

  // post-loop LO when none ran (exp_ranF.c:1580-1697)
  if (!st.iter_cnt && !st.degen_cnt && st.non_degen) {
    bool degenerate = false;
    double H[9], f[9];
    if (P.degen) {
      double u7[28];
      for (int t = 0; t < 7; ++t) {
        const int p = st.samidxBest[t];
        u7[4 * t] = c.x1[p]; u7[4 * t + 1] = c.y1[p]; u7[4 * t + 2] = c.x2[p]; u7[4 * t + 3] = c.y2[p];
      }
      degenerate = blk_checksample(c, st.FBest, u7, 3 * P.th, H);
    }
    if (degenerate) {
      blk_resid_H_sampson(c, H, W.dtmp[4]);
      unsigned I = (unsigned)blk_count_lt(c, W.dtmp[4], P.th * 3);
      if (I >= 8) I = blk_inner_H(c, W, H, 16 * P.th, 10, W.btmp[0], st.cur);
      else { for (int j = c.tid; j < c.N; j += c.nt) W.btmp[0][j] = 0; DG_SYNC(); }
      if ((int)I > st.Ihmax) st.Ihmax = (int)I;
      if (I > 6) {
        bool new_max = false;
        for (int j = 0; j < 9; ++j) f[j] = st.FBest[j];  // the reference's `f` is whatever the last iteration left
        I = blk_rFtH(c, W, W.btmp[0], P.th, H, f, st.cur);
        int d;
        if (I > st.maxS.I) {
          blk_resid_F(c, P.metric, f, W.err[st.e[3]]);
          st.maxS.I = I;
          for (int j = 0; j < 9; ++j) st.F[j] = f[j];
          new_max = true;
          d = st.e[3];
        } else {
          blk_resid_F(c, P.metric, f, W.err[st.e[0]]);  // reference: errs[i] with a stale loop index
          d = st.e[0];
        }
        const Score t = blk_inlidxs(c, W.err[d], P.th, W.inliers);
        if (new_max) st.maxS.J = t.J;
        ++st.degen_cnt;
      }
    } else {
      run_lo_F(c, P, W, st, W.errBest);
    }
  }

  final_mask_F(c, P, W, st, mask_out);
  if (c.tid == 0) {
    for (int i = 0; i < 9; ++i) F_out[i] = st.F[i];
    stats_out[0] = no_sam;
    stats_out[1] = st.iter_cnt;
    stats_out[2] = st.Ihmax;
    stats_out[3] = (int)st.maxS.I;
  }
  DG_SYNC();
}

}  // namespace dg
