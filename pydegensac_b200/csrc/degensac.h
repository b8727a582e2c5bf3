// degensac.h -- DEGENSAC: H-degeneracy test of a 7-point sample, plane consensus + LO of the plane
// homography, plane-and-parallax recovery of F.  Replaces DegUtils.c (checksample :42, Hdetect :93,
// dHDs :186, rFtH :254, innerFH :488, dual_sample :596, u2Fit :635, innerH :693) and the old LO it
// reaches in ranH.c (iterH :18, inHrani :88).
//
// B200 mapping: the 5 sample triplets of checksample are tested by 5 warps in parallel (first success in
// triplet order wins, as in the reference's sequential loop); every O(N) pass (plane consensus, residual
// rows, masks, ordered compactions) is CTA-parallel; the plane-and-parallax loop (<= 20k two-point
// samples, each a Sampson pass over the off-plane correspondences) runs as speculative waves of one WARP
// per two-point hypothesis with an ordered replay of the rare "new best" events, mirroring the main loop.
#pragma once
#include "common.h"
#include "rng.h"
#include "la.h"
#include "fgeom.h"
#include "hgeom.h"
#include "block.h"
#include "ffit.h"
#include "hfit.h"
#include "filter32.h"

namespace dg {

#ifdef DG_FILTER_CHECK
static long g_pp_checked = 0, g_pp_violations = 0, g_pp_settled = 0;   // plane-and-parallax count bound (host emulation)
#endif

// ------------------------------------------------------------------------------------------------
// Homography compatible with F through 3 correspondences (Hartley & Zisserman p.318; reference Hdetect,
// DegUtils.c:93-161).  u7 holds the sample as 7 x (x1,y1,x2,y2); H is column-major, image2 -> image1.
// ------------------------------------------------------------------------------------------------
DG_HDN void h_from_F_3pts(const double* F, const double* u7, const int* tri, double* H) {
  double ec[3];
  gkr_third_right_vector3(F, ec);  // column 2 of CCMATH's V (usually, not always, F ec = 0)
  const double Ex[9] = {0, -ec[2], ec[1], ec[2], 0, -ec[0], -ec[1], ec[0], 0};
  double A[9];  // A = [ec]x * F^T
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      for (int k = 0; k < 3; ++k) s += Ex[3 * i + k] * F[3 * j + k];
      A[3 * i + j] = s;
    }
  double b[3], M[9];
  for (int t = 0; t < 3; ++t) {
    const double* p = u7 + 4 * tri[t];
    const double a1[3] = {p[0], p[1], 1.0};
    const double a2[3] = {p[2], p[3], 1.0};
    double Ab[3], p1[3], p2[3];
    for (int i = 0; i < 3; ++i) {
      double s = 0.0;
      for (int k = 0; k < 3; ++k) s += A[3 * i + k] * a2[k];
      Ab[i] = s;
    }
    cross3(p1, a1, Ab);
    for (int i = 0; i < 3; ++i) {
      double s = 0.0;
      for (int k = 0; k < 3; ++k) s += (-Ex[3 * i + k]) * a1[k];
      p2[i] = s;
    }
    b[t] = (p1[0] * p2[0] + p1[1] * p2[1] + p1[2] * p2[2]) / (p2[0] * p2[0] + p2[1] * p2[1] + p2[2] * p2[2]);
    M[3 * t] = a2[0]; M[3 * t + 1] = a2[1]; M[3 * t + 2] = a2[2];
  }
  const int sing = minv3(M);   // CCMATH minv, bit for bit (DegUtils.c:141)
  double v[3];
  for (int i = 0; i < 3; ++i) v[i] = M[3 * i] * b[0] + M[3 * i + 1] * b[1] + M[3 * i + 2] * b[2];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) H[i + 3 * j] = A[3 * i + j] - ec[i] * v[j];
  if (isnan(H[0]) || isinf(H[0]) || sing) {
    for (int i = 0; i < 9; ++i) H[i] = 0.0;
    H[0] = H[4] = H[8] = 1.0;
  }
}

// Normalised DLT on a handful of points of the sample (the 5-point refit of checksample), warp-cooperative:
// lane 0 normalises and writes the 2*len DLT rows, the lanes form the normal matrix and run the Jacobi sweeps.
// Result (lane 0): h[9].
DG_ENGN void warp_h_fit_small(WarpScratch* ws, const double* u7, const int* idx, int len, double* h, int lane, int W) {
  double A1[3] = {0, 0, 0}, A2[3] = {0, 0, 0};
  double* rows = ws->aux;   // 2*len x 9, len <= 6
  if (lane == 0) {
    #pragma unroll 1
    for (int j = 0; j < len; ++j) {
      const double* p = u7 + 4 * idx[j];
      A1[1] += p[0]; A1[2] += p[1]; A2[1] += p[2]; A2[2] += p[3];
    }
    for (int i = 1; i < 3; ++i) { A1[i] /= len; A2[i] /= len; }
    #pragma unroll 1
    for (int j = 0; j < len; ++j) {
      const double* p = u7 + 4 * idx[j];
      double a = p[0] - A1[1], b = p[1] - A1[2];
      A1[0] += sqrt(a * a + b * b);
      a = p[2] - A2[1]; b = p[3] - A2[2];
      A2[0] += sqrt(a * a + b * b);
    }
    if (A1[0] != 0) A1[0] = len * sqrt(2.0) / A1[0];
    if (A2[0] != 0) A2[0] = len * sqrt(2.0) / A2[0];
    A1[1] *= -A1[0]; A1[2] *= -A1[0];
    A2[1] *= -A2[0]; A2[2] *= -A2[0];
    #pragma unroll 1
    for (int j = 0; j < len; ++j) {
      const double* p = u7 + 4 * idx[j];
      double a[3], b[3];
      a[0] = p[0] * A1[0] + A1[1]; a[1] = p[1] * A1[0] + A1[2]; a[2] = 1.0;
      b[0] = p[2] * A2[0] + A2[1]; b[1] = p[3] * A2[0] + A2[2]; b[2] = 1.0;
      double* r0 = rows + 18 * j;
      double* r1 = r0 + 9;
      for (int t = 0; t < 3; ++t) {
        r0[3 * t] = b[t]; r0[3 * t + 1] = 0.0; r0[3 * t + 2] = -a[0] * b[t];
        r1[3 * t] = 0.0;  r1[3 * t + 1] = b[t]; r1[3 * t + 2] = -a[1] * b[t];
      }
    }
  }
  DG_WSYNC();
  #pragma unroll 1
  for (int t = lane; t < 45; t += W) {
    int i = 0;
    while ((i + 1) * (i + 2) / 2 <= t) ++i;
    const int jj = t - i * (i + 1) / 2;
    double s = 0.0;
    #pragma unroll 1
    for (int r = 0; r < 2 * len; ++r) s += rows[9 * r + i] * rows[9 * r + jj];
    ws->A[9 * i + jj] = s;
    ws->A[9 * jj + i] = s;
  }
  DG_WSYNC();
  warp_smallest_eigvec9(ws, lane, W);
  if (lane == 0) {
    for (int i = 0; i < 9; ++i) h[i] = ws->cs[i];
    denorm_H(h, A1, A2);
  }
  DG_WSYNC();
}

// One triplet of the degeneracy test (body of the loop in checksample, DegUtils.c:55-80), one warp.
// Verdict and H are valid on lane 0.
DG_ENGN bool warp_checksample_triplet(WarpScratch* ws, const double* F, const double* u7, int t, double th, double* H,
                                      int lane, int W) {
  const int TRI[5][3] = {{0, 1, 2}, {3, 4, 5}, {0, 1, 6}, {3, 4, 6}, {2, 5, 6}};
  int* idx = reinterpret_cast<int*>(ws->cs + 8);   // 7 ints shared with the other lanes
  if (lane == 0) {
    h_from_F_3pts(F, u7, TRI[t], H);
#ifdef DG_TRACE
    if (t == 0) {
      fprintf(stderr, "CSIN F=");
      for (int i = 0; i < 9; ++i) fprintf(stderr, "%.17g ", F[i]);
      fprintf(stderr, "u7=");
      #pragma unroll 1
      for (int i = 0; i < 28; ++i) fprintf(stderr, "%.17g ", u7[i]);
      fprintf(stderr, "\n");
    }
    fprintf(stderr, "HDET t=%d H=%.10g %.10g %.10g %.10g\n", t, H[0], H[1], H[2], H[8]);
#endif
    double Ds[7];
    for (int j = 0; j < 7; ++j) {
      Ds[j] = h_resid_sampson(H, u7[4 * j], u7[4 * j + 1], u7[4 * j + 2], u7[4 * j + 3]);
      idx[j] = j;
    }
    for (int i = 0; i < 7; ++i)      // exchange sort of the reference's sortDs (DegUtils.c:164-183)
      #pragma unroll 1
      for (int j = i + 1; j < 7; ++j)
        if (Ds[j] < Ds[i]) {
          const double td = Ds[j]; Ds[j] = Ds[i]; Ds[i] = td;
          const int ti = idx[j]; idx[j] = idx[i]; idx[i] = ti;
        }
  }
  DG_WSYNC();
  warp_h_fit_small(ws, u7, idx, 5, H, lane, W);
  int cnt = 0;
  if (lane == 0)
    for (int j = 0; j < 7; ++j)
      if (h_resid_sampson(H, u7[4 * j], u7[4 * j + 1], u7[4 * j + 2], u7[4 * j + 3]) < th) ++cnt;
#ifdef DG_TRACE
  if (lane == 0) {
    double Ds[7];
    for (int j = 0; j < 7; ++j) Ds[j] = h_resid_sampson(H, u7[4 * j], u7[4 * j + 1], u7[4 * j + 2], u7[4 * j + 3]);
    fprintf(stderr, "CS trip=%d cnt=%d Ds=%.6g %.6g %.6g %.6g %.6g %.6g %.6g H=%.10g %.10g %.10g\n", t, cnt, Ds[0], Ds[1], Ds[2], Ds[3], Ds[4], Ds[5], Ds[6], H[0] / H[8], H[1] / H[8], H[2] / H[8]);
  }
#endif
  return cnt > 4;
}

// checksample: 5 warps test the 5 triplets concurrently; the first successful triplet (reference order)
// provides H.  Returns the verdict to every thread, H in every thread's copy.
DG_ENGN bool blk_checksample(const Ctx& c, const double* F, const double* u7, double th, double* H) {
  DG_SYNC();
  const int par = (c.nw >= 5) ? 5 : 1;
  const int W = DG_DEVICE_PASS ? 32 : 1;
  if (c.wid < par) {
    #pragma unroll 1
    for (int t = c.wid; t < 5; t += par) {
      double Ht[9];
      const bool ok = warp_checksample_triplet(c.sc->warp_tile(c.wid), F, u7, t, th, Ht, c.lane, W);
      if (c.lane == 0) {
        c.sc->bci[t] = ok ? 1 : 0;
        if (t < 3) { for (int i = 0; i < 9; ++i) c.sc->bc[9 * t + i] = Ht[i]; }
        else { for (int i = 0; i < 9; ++i) c.sc->vec_out[9 * (t - 3) + i] = Ht[i]; }
      }
    }
  }
  DG_SYNC();
  int win = -1;
  for (int t = 0; t < 5; ++t)
    if (c.sc->bci[t]) { win = t; break; }
  // the reference leaves the LAST tested triplet's H in the buffer when none succeeds; it is unused then
  const int src = win < 0 ? 4 : win;
  for (int i = 0; i < 9; ++i) H[i] = (src < 3) ? c.sc->bc[9 * src + i] : c.sc->vec_out[9 * (src - 3) + i];
  DG_SYNC();
  return win >= 0;
}

// ------------------------------------------------------------------------------------------------
// LO of the plane homography: reference innerH (DegUtils.c:693-731) -> inHrani / iterH (ranH.c:88,18),
// Sampson metric, threshold 16*th, inlLimit = 10.  Uses its own four residual rows (W.dtmp[0..3]).
// Writes the plane-inlier mask, returns its population.
// ------------------------------------------------------------------------------------------------
DG_ENGN Score plane_iter_H(const Ctx& c, Workspace& W, int* e, double** rows, int* inl, double th, double ths,
                                 double* Hio, unsigned inlLimit, DrawCursor& cur) {
  int d = e[1];
  double h[9];
  const double dth = (ths - th) / kIlsqIters;
  Score S = make_score(), Ss, maxS;
  maxS = blk_inlidxs(c, rows[e[4]], th, inl);
  if (maxS.I < 4) return S;
  for (int i = 0; i < 9; ++i) h[i] = Hio[i];
  if (maxS.I <= inlLimit) {
    blk_fit_H(c, inl, (int)maxS.I, h);
  } else {
    blk_randsubset(c, inl, (int)maxS.I, (int)inlLimit, cur);
    blk_fit_H(c, inl + maxS.I - inlLimit, (int)inlLimit, h);
  }
  #pragma unroll 1
  for (int it = 0; it < kIlsqIters; ++it) {
    blk_resid_H_sampson(c, h, rows[d]);
    S = blk_inlidxs(c, rows[d], th, inl);
    Ss = blk_inlidxs(c, rows[d], ths, inl);
    if (score_less(maxS, S)) {
      maxS = S;
      e[1] = e[0];
      e[0] = d;
      d = e[1];
      for (int i = 0; i < 9; ++i) Hio[i] = h[i];
    }
    if (Ss.I < 4) return maxS;
    if (Ss.I <= inlLimit) {
      blk_fit_H(c, inl, (int)Ss.I, h);
    } else {
      blk_randsubset(c, inl, (int)Ss.I, (int)inlLimit, cur);
      blk_fit_H(c, inl + Ss.I - inlLimit, (int)inlLimit, h);
    }
    ths -= dth;
  }
  blk_resid_H_sampson(c, h, rows[d]);
  S = blk_inlidxs(c, rows[d], th, inl);
  if (score_less(maxS, S)) {
    maxS = S;
    e[1] = e[0];
    e[0] = d;
    for (int i = 0; i < 9; ++i) Hio[i] = h[i];
  }
  return maxS;
}

DG_ENGN unsigned blk_inner_H(const Ctx& c, Workspace& W, double* H, double th, unsigned inlLimit,
                                   unsigned char* mask, DrawCursor& cur) {
  double* rows[4] = {W.dtmp[0], W.dtmp[1], W.dtmp[2], W.dtmp[3]};
  int e[5] = {0, 1, 2, 3, 3};
  int* inliers = W.itmp[0];
  int* intbuff = W.itmp[1];
  blk_resid_H_sampson(c, H, rows[e[0]]);
  Score S = blk_inlidxs(c, rows[e[0]], th, inliers);
  const int ninl = (int)S.I;
#ifdef DG_TRACE
  fprintf(stderr, "innerH start I=%u\n", S.I);
#endif
  if (ninl >= 8) {  // inHrani
    Score maxS = make_score();
    int ssiz = ninl / 2;
    if (ssiz > 12) ssiz = 12;
    int t = e[2]; e[2] = e[0]; e[0] = t;
    double h[9];
    for (int i = 0; i < 9; ++i) h[i] = H[i];
    #pragma unroll 1
    for (int rep = 0; rep < kRanRep; ++rep) {
      blk_randsubset(c, inliers, ninl, ssiz, cur);
      blk_fit_H(c, inliers + ninl - ssiz, ssiz, h);
      blk_resid_H_sampson(c, h, rows[e[0]]);
      e[4] = e[0];
      S = plane_iter_H(c, W, e, rows, intbuff, th, kTC * th, h, inlLimit, cur);
      if (score_less(maxS, S)) {
        maxS = S;
        t = e[2]; e[2] = e[0]; e[0] = t;
        for (int i = 0; i < 9; ++i) H[i] = h[i];
      }
    }
    t = e[2]; e[2] = e[0]; e[0] = t;
  }
  const double* d = rows[e[0]];
  int cnt = 0;
  #pragma unroll 1
  for (int j = c.tid; j < c.N; j += c.nt) {
    const unsigned char m = (d[j] <= th) ? 1 : 0;
    mask[j] = m;
    cnt += m;
  }
  const int I = blk_sum_i(c, cnt);
  DG_SYNC();
  return (unsigned)I;
}

// ordered compaction of {i : flag(i)} into list; returns count
template <class Pred>
DG_ENGN int blk_compact(const Ctx& c, int n, int* list, Pred pred) {
  const int per = (n + c.nt - 1) / c.nt;
  const int beg = c.tid * per;
  const int end = (beg + per < n) ? beg + per : n;
  int cnt = 0;
  #pragma unroll 1
  for (int i = beg; i < end; ++i)
    if (pred(i)) ++cnt;
  int total;
  int off = blk_excl_scan_i(c, cnt, &total);
  #pragma unroll 1
  for (int i = beg; i < end; ++i)
    if (pred(i)) list[off++] = i;
  DG_SYNC();
  return total;
}

// ------------------------------------------------------------------------------------------------
// Iterated LSQ of F on all inliers with shrinking strict threshold (reference u2Fit, DegUtils.c:635-690).
// F in/out; mask out; returns population.  Ds row = W.dtmp[5], list = W.itmp[3].
// ------------------------------------------------------------------------------------------------
DG_ENGN unsigned blk_u2Fit(const Ctx& c, Workspace& W, double* F, unsigned char* mask, double th, double ths,
                                 unsigned iters) {
  const double dth = (ths - th) / (iters - 1);
  double* Ds = W.dtmp[5];
  int* inlI = W.itmp[3];
  #pragma unroll 1
  for (unsigned iter = 0; iter < iters; ++iter) {
    blk_resid_F(c, F_SAMPSON, F, Ds);
    const double tcur = ths;
    int cnt = 0;
    #pragma unroll 1
    for (int i = c.tid; i < c.N; i += c.nt) {
      const unsigned char m = (Ds[i] < tcur) ? 1 : 0;
      mask[i] = m;
      cnt += m;
    }
    const int no_i = blk_sum_i(c, cnt);
    DG_SYNC();
    if (no_i < 8) return (unsigned)no_i;
    blk_compact(c, c.N, inlI, [&](int i) { return mask[i] != 0; });
    blk_fit_F(c, inlI, no_i, nullptr, F);
    ths -= dth;
  }
  blk_resid_F(c, F_SAMPSON, F, Ds);
  int cnt = 0;
  #pragma unroll 1
  for (int i = c.tid; i < c.N; i += c.nt) {
    const unsigned char m = (Ds[i] < th) ? 1 : 0;
    mask[i] = m;
    cnt += m;
  }
  const int no_i = blk_sum_i(c, cnt);
  DG_SYNC();
  return (unsigned)no_i;
}

#if DG_DEVICE_PASS
// Positions 0..S-1 of an identity permutation after the swaps `pos <-> idx[pos]` (pos = 0..S-1), replayed on a
// register log of writes (later entries override earlier ones).  idx[pos] comes from lane base+pos.
template <int S>
__device__ __forceinline__ void identity_swaps(int drawmod, int base, int lane, int& mine) {
  const unsigned full = 0xffffffffu;
  int tp[2 * S], tv[2 * S];
#pragma unroll
  for (int pos = 0; pos < S; ++pos) {
    const int idx = __shfl_sync(full, drawmod, base + pos);
    int vp = pos, vi = idx;
#pragma unroll
    for (int t = 0; t < 2 * pos; ++t) {
      if (tp[t] == pos) vp = tv[t];
      if (tp[t] == idx) vi = tv[t];
    }
    tp[2 * pos] = pos;     tv[2 * pos] = vi;
    tp[2 * pos + 1] = idx; tv[2 * pos + 1] = vp;
  }
#pragma unroll
  for (int pos = 0; pos < S; ++pos) {
    int v = pos;
#pragma unroll
    for (int t = 0; t < 2 * S; ++t) if (tp[t] == pos) v = tv[t];
    if (lane == base + pos) mine = v;    // lane base+pos keeps entry `pos`
  }
}
// dual_sample on one warp: the ten draws are generated by ten lanes at once, the swaps replayed in registers.
__device__ __noinline__ void warp_dual_sample(const int* uH, int nH, const int* uO, int nO, int* usam, uint64_t seed,
                                              uint32_t k, uint32_t j0, int lane) {
  int dm = 0;
  if (lane < 10) dm = (int)(value31(seed, k, j0 + (uint32_t)lane) % (uint32_t)(lane < 6 ? nH : nO));
  int mine = 0;
  identity_swaps<6>(dm, 0, lane, mine);
  identity_swaps<4>(dm, 6, lane, mine);
  if (lane < 6) usam[lane] = uH[mine];
  else if (lane < 10) usam[lane] = uO[mine];
}
#endif

// ------------------------------------------------------------------------------------------------
// LO of F from plane + off-plane correspondences (reference innerFH + dual_sample, DegUtils.c:488-632).
// uH list (plane inliers, nH), uO list (off-plane support, nO), 15 reps of 6 + 4 points.
// Output: F (9) and inlier mask `inl` (N).  Scratch masks: W.btmp[2] (v).  Returns nothing (max_i unused).
// ------------------------------------------------------------------------------------------------
DG_ENGN void blk_inner_FH(const Ctx& c, Workspace& W, const int* uH, int nH, const int* uO, int nO, double th,
                                double* F, unsigned char* inl, DrawCursor& cur) {
  unsigned char* v = W.btmp[2];
  double* Ds = W.dtmp[5];
  int* usam = W.itmp[2];  // 10 indices
  unsigned max_i = 0, max_s = 0;
  for (int i = 0; i < 9; ++i) F[i] = 1.0;
  #pragma unroll 1
  for (int i = c.tid; i < c.N; i += c.nt) inl[i] = 0;
  DG_SYNC();
#if DG_DEVICE_PASS
  // The fifteen repetitions are INDEPENDENT up to the bookkeeping: every one consumes exactly ten draws and fits its own
  // 6 + 4 sample; only "best so far" (max_i, max_s) and the rare u2Fit are order-dependent.  So the samples, the ten-point
  // fits (one warp each, five side by side -- the tiles of the checksample triplets) and the support counts (one warp
  // per model) are computed up front, and the reference's loop is then replayed in order on the stored (model, count)
  // pairs; a full residual row is produced only for the repetitions that improve on the best (a handful of fifteen).
  {
    double* fhF = c.sc->fh_F;
    int* fhC = c.sc->fh_cnt;
    const int nfit = (c.nw >= 5) ? 5 : 1;   // warp tiles available side by side
    #pragma unroll 1
    for (int base = 0; base < 15; base += nfit) {
      DG_SYNC();
      if (c.wid < nfit) {
        const int rep = base + c.wid;
        WarpScratch* ws = c.sc->warp_tile(c.wid);
        int* usam_w = reinterpret_cast<int*>(ws->V);
        warp_dual_sample(uH, nH, uO, nO, usam_w, cur.seed, cur.k, cur.j + 10u * (uint32_t)rep, c.lane);
        __syncwarp();
        warp_fit_F_small(c, ws, ws->aux, usam_w, 10, nullptr, fhF + 9 * rep);
      }
    }
    DG_SYNC();
    #pragma unroll 1
    for (int rep = c.wid; rep < 15; rep += c.nw) {
      double aF[9];
      for (int i = 0; i < 9; ++i) aF[i] = fhF[9 * rep + i];
      int cnt = 0;
      #pragma unroll 1
      for (int i = c.lane; i < c.N; i += 32)
        cnt += (f_resid(F_SAMPSON, aF, ld_soa(c.x1 + i), ld_soa(c.y1 + i), ld_soa(c.x2 + i), ld_soa(c.y2 + i)) < th) ? 1 : 0;
      cnt = warp_sum_i(cnt);
      if (c.lane == 0) fhC[rep] = cnt;
    }
    DG_SYNC();
    cur.j += 150;
    #pragma unroll 1
    for (unsigned rep = 0; rep < 15; ++rep) {
      unsigned no_i = (unsigned)fhC[rep];
      if (!(max_i < no_i) && !(no_i > max_s)) continue;
      double aF[9];
      for (int i = 0; i < 9; ++i) aF[i] = fhF[9 * rep + i];
      blk_resid_F(c, F_SAMPSON, aF, Ds);
      #pragma unroll 1
      for (int i = c.tid; i < c.N; i += c.nt) v[i] = (Ds[i] < th) ? 1 : 0;
      DG_SYNC();
      if (max_i < no_i) {
        #pragma unroll 1
        for (int i = c.tid; i < c.N; i += c.nt) inl[i] = v[i];
        for (int i = 0; i < 9; ++i) F[i] = aF[i];
        max_i = no_i;
        DG_SYNC();
      }
      if (no_i > max_s) {
        max_s = no_i;
        DG_PROF_COUNT(38, 1);
        { DG_PROF_BEGIN(37); no_i = blk_u2Fit(c, W, aF, v, th, th * 3, 4); DG_PROF_END(37); }
        if (max_i < no_i) {
          #pragma unroll 1
          for (int i = c.tid; i < c.N; i += c.nt) inl[i] = v[i];
          for (int i = 0; i < 9; ++i) F[i] = aF[i];
          max_i = no_i;
          DG_SYNC();
        }
      }
    }
  }
#else
  #pragma unroll 1
  for (unsigned rep = 0; rep < 15; ++rep) {
    // dual_sample: fresh identity permutations, `pos <-> rand()%len` swaps (DegUtils.c:596-632)
    DG_PROF_BEGIN(36);
    DG_SYNC();
#if DG_DEVICE_PASS
    if (c.wid == 0) warp_dual_sample(uH, nH, uO, nO, usam, cur.seed, cur.k, cur.j, c.lane);
#else
    if (c.tid == 0) {
      DrawCursor t = cur;
      int tp[12], tv[12], nt;
      for (int side = 0; side < 2; ++side) {
        const int len = side ? nO : nH, s = side ? 4 : 6;
        const int* src = side ? uO : uH;
        nt = 0;
        #pragma unroll 1
        for (int pos = 0; pos < s; ++pos) {
          const int idx = (int)(next_draw(t) % (uint32_t)len);
          int vp = pos, vi = idx;
          #pragma unroll 1
          for (int q = 0; q < nt; ++q) { if (tp[q] == pos) vp = tv[q]; if (tp[q] == idx) vi = tv[q]; }
          int q = 0;
          while (q < nt && tp[q] != pos) ++q;
          if (q == nt) { tp[nt] = pos; ++nt; }
          tv[q] = vi;
          q = 0;
          while (q < nt && tp[q] != idx) ++q;
          if (q == nt) { tp[nt] = idx; ++nt; }
          tv[q] = vp;
        }
        #pragma unroll 1
        for (int pos = 0; pos < s; ++pos) {
          int vp = pos;
          #pragma unroll 1
          for (int q = 0; q < nt; ++q) if (tp[q] == pos) vp = tv[q];
          usam[(side ? 6 : 0) + pos] = src[vp];
        }
      }
    }
#endif
    cur.j += 10;
    DG_SYNC();
    DG_PROF_END(36);
    double aF[9];
    blk_fit_F(c, usam, 10, nullptr, aF);
    blk_resid_F(c, F_SAMPSON, aF, Ds);
    int cnt = 0;
    #pragma unroll 1
    for (int i = c.tid; i < c.N; i += c.nt) {
      const unsigned char m = (Ds[i] < th) ? 1 : 0;
      v[i] = m;
      cnt += m;
    }
    unsigned no_i = (unsigned)blk_sum_i(c, cnt);
    DG_SYNC();
    if (max_i < no_i) {
      #pragma unroll 1
      for (int i = c.tid; i < c.N; i += c.nt) inl[i] = v[i];
      for (int i = 0; i < 9; ++i) F[i] = aF[i];
      max_i = no_i;
      DG_SYNC();
    }
    if (no_i > max_s) {
      max_s = no_i;
      DG_PROF_COUNT(38, 1);
      { DG_PROF_BEGIN(37); no_i = blk_u2Fit(c, W, aF, v, th, th * 3, 4); DG_PROF_END(37); }
      if (max_i < no_i) {
        #pragma unroll 1
        for (int i = c.tid; i < c.N; i += c.nt) inl[i] = v[i];
        for (int i = 0; i < 9; ++i) F[i] = aF[i];
        max_i = no_i;
        DG_SYNC();
      }
    }
  }
#endif
}

// F = transpose( [e]x * H^T ) for the epipole e through two off-plane correspondences
// (reference rFtH inner loop, DegUtils.c:353-371).  H column-major.
DG_HD void f_from_plane_parallax(const double* H, double ax1, double ay1, double ax2, double ay2, double bx1,
                                 double by1, double bx2, double by2, double* F) {
  double ua[3] = {ax1, ay1, 1.0}, ub[3] = {bx1, by1, 1.0}, ha[3], hb[3], c1[3], c2[3], ec[3];
  ha[0] = H[0] * ax2 + H[3] * ay2 + H[6] * 1.0;
  ha[1] = H[1] * ax2 + H[4] * ay2 + H[7] * 1.0;
  ha[2] = H[2] * ax2 + H[5] * ay2 + H[8] * 1.0;
  hb[0] = H[0] * bx2 + H[3] * by2 + H[6] * 1.0;
  hb[1] = H[1] * bx2 + H[4] * by2 + H[7] * 1.0;
  hb[2] = H[2] * bx2 + H[5] * by2 + H[8] * 1.0;
  cross3(c1, ua, ha);
  cross3(c2, ub, hb);
  cross3(ec, c1, c2);
  const double n = sqrt(ec[0] * ec[0] + ec[1] * ec[1] + ec[2] * ec[2]);
  ec[0] = ec[0] / n; ec[1] = ec[1] / n; ec[2] = ec[2] / n;
  const double S[9] = {0, -ec[2], ec[1], ec[2], 0, -ec[0], -ec[1], ec[0], 0};
  // Ht (row-major transpose of the column-major array, i.e. Ht[i][j] = H[j*3+i]); G = S * Ht ; F = G^T
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      for (int k = 0; k < 3; ++k) s += S[3 * i + k] * H[j * 3 + k];
      F[3 * j + i] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// Plane-and-parallax: reference rFtH (DegUtils.c:254-444).  hinl = plane-inlier mask (from innerH).
// Returns max_i; F written only when a better model was found (as in the reference).
// ------------------------------------------------------------------------------------------------
DG_ENGN unsigned blk_rFtH(const Ctx& c, Workspace& W, const unsigned char* hinl, double th, const double* H,
                                double* F, DrawCursor& cur) {
  double* Ds = W.dtmp[4];
  unsigned char* nhinl = W.btmp[1];
  unsigned char* inl = W.btmp[3];
  int* uN = W.inliers;        // ordered off-plane indices (main-loop lists are dead at this point)
  int* uHl = W.intbuff;       // ordered plane-inlier indices
  int* uV = W.intbuff_best;   // ordered support of the current 2-point model
  int* ptr = W.itmp[0];       // persistent permutation over uN positions (innerH's list is dead here)
  blk_resid_H_sampson(c, H, Ds);
  #pragma unroll 1
  for (int i = c.tid; i < c.N; i += c.nt) nhinl[i] = (Ds[i] > 100 * th) ? 1 : 0;
  DG_SYNC();
  const int nN = blk_compact(c, c.N, uN, [&](int i) { return nhinl[i] != 0; });
  const int nH = blk_compact(c, c.N, uHl, [&](int i) { return hinl[i] != 0; });
  unsigned max_i = 3, m_i = 4, max_sam = 10000, maxni = 0;
  if (nN < 4 || nH < 6) return 0;
  #pragma unroll 1
  for (int i = c.tid; i < nN; i += c.nt) ptr[i] = i;
#if DG_DEVICE_PASS
  // FP32 tile of the OFF-PLANE correspondences only, in list order, pair-interleaved like the main tile (filter32.h);
  // lives in the first two residual rows of the plane LO, which are dead here (16 (nN + 1) <= 16 N bytes, nN <= N - 6)
  float* tileN = reinterpret_cast<float*>(W.dtmp[0]);
  if (c.t32) {
    const float* tf = reinterpret_cast<const float*>(c.t32->pts);
    #pragma unroll 1
    for (int i = c.tid; i < nN; i += c.nt) {
      const int p = uN[i];
      const float* src = tf + 8 * (p >> 1) + (p & 1);
      float* dst = tileN + 8 * (i >> 1) + (i & 1);
      dst[0] = src[0]; dst[2] = src[2]; dst[4] = src[4]; dst[6] = src[6];
      if (i == nN - 1 && !(i & 1)) { dst[1] = 0.f; dst[3] = 0.f; dst[5] = 0.f; dst[7] = 0.f; }
    }
  }
#endif
  DG_SYNC();
  const double th2 = th * 2;
  const int WAVE = c.nw * 8;
  int* pairs = W.itmp[2] + 16;   // WAVE x 2 sampled positions
  int* counts = W.itmp[2] + 16 + 2 * 128;
  int* idxs = reinterpret_cast<int*>(c.sc->vec);   // 2 x 128 swap partners of the current wave (block scratch is idle here)
  int* vals = idxs + 256;                          // permutation entries they address, as they were before the wave
  int* wrote = idxs + 512;                         // value each access stores
  int* prevq = idxs + 768;                         // latest earlier access of the wave to the same entry (-1: none)
  unsigned no_sam = 1;
  while (no_sam < 2 * max_sam) {
    int nw = (int)(2 * max_sam - no_sam);
    if (nw > WAVE) nw = WAVE;
    if (nw > 128) nw = 128;
    // All threads: the 2*nw draws of the speculative iterations (swap partners) go to shared memory together with the
    // permutation entries they address (one round of independent loads) and, per access, the latest EARLIER access of
    // this wave to the same entry.  Thread 0 then replays the swaps in order on shared memory only -- ptr[0], ptr[1] in
    // registers, an entry touched twice read from the log -- and nothing is written to the permutation until the
    // outcome of the wave is known (no rewind; the serial chain no longer waits on global memory).
    DG_PROF_BEGIN(32);
    DG_SYNC();
    #pragma unroll 1
    for (int q = c.tid; q < 2 * nw; q += c.nt) {
      const int pos = q & 1;
      const int idx = pos + 1 + (int)(value31(cur.seed, cur.k, cur.j + (uint32_t)q) % (uint32_t)(nN - pos - 1));
      idxs[q] = idx;
      vals[q] = ptr[idx];
    }
    DG_SYNC();
    #pragma unroll 1
    for (int q = c.tid; q < 2 * nw; q += c.nt) {
      const int idx = idxs[q];
      int pr = -1;
      if (idx != 1) {
        #pragma unroll 4
        for (int t = q - 1; t >= 0; --t)
          if (idxs[t] == idx) { pr = t; break; }
      }
      prevq[q] = pr;
    }
    DG_SYNC();
    DG_PROF_BEGIN(47);
    if (c.tid == 0) {
      int p0 = ptr[0], p1 = ptr[1];
      #pragma unroll 1
      for (int s = 0; s < nw; ++s) {
        const int q0 = 2 * s, q1 = 2 * s + 1;
        int v;
        if (idxs[q0] == 1) { v = p1; p1 = p0; }
        else { const int pr = prevq[q0]; v = pr >= 0 ? wrote[pr] : vals[q0]; wrote[q0] = p0; }
        p0 = v;
        { const int pr = prevq[q1]; v = pr >= 0 ? wrote[pr] : vals[q1]; wrote[q1] = p1; p1 = v; }
        pairs[2 * s] = p0;
        pairs[2 * s + 1] = p1;
      }
    }
    DG_SYNC();
    DG_PROF_END(47);
    DG_PROF_BEGIN(48);
    // One warp per two-point hypothesis: support count over the off-plane correspondences.  The count only matters
    // when it EXCEEDS the best support so far (m_i) -- a few dozen of the thousands of hypotheses.  An FP32 UPPER BOUND
    // of the count (filter32.h: a lower bound of every Sampson error on the centred single-precision tile, counted when
    // it is below the threshold) settles the rest at a fifth of the instructions; hypotheses whose bound exceeds m_i
    // are recounted exactly.
    auto exact_count = [&](const double* aF) -> int {
      int cnt = 0;
#if DG_DEVICE_PASS
      {  // two gathers + two residual chains in flight per lane
        int i = c.lane;
        #pragma unroll 1
        for (; i + 32 < nN; i += 64) {
          const int p = uN[i], q = uN[i + 32];
          const double a1 = c.x1[p], b1 = c.y1[p], a2 = c.x2[p], b2 = c.y2[p];
          const double e1 = c.x1[q], g1 = c.y1[q], e2 = c.x2[q], g2 = c.y2[q];
          const double r0 = f_resid_sampson(aF, a1, b1, a2, b2);
          const double r1 = f_resid_sampson(aF, e1, g1, e2, g2);
          if (r0 < th2) ++cnt;
          if (r1 < th2) ++cnt;
        }
        if (i < nN) {
          const int p = uN[i];
          if (f_resid_sampson(aF, c.x1[p], c.y1[p], c.x2[p], c.y2[p]) < th2) ++cnt;
        }
      }
#else
      for (int i = 0; i < nN; ++i) {
        const int p = uN[i];
        if (f_resid_sampson(aF, c.x1[p], c.y1[p], c.x2[p], c.y2[p]) < th2) ++cnt;
      }
#endif
      return warp_sum_i(cnt);
    };
#if DG_DEVICE_PASS
    if (c.t32) {
      // The per-hypothesis preparation (epipole and F from the plane and two points, constants of the FP32 bound) is a
      // few hundred dependent FP64 instructions and three levels of dependent loads: the (up to) eight hypotheses of
      // this warp are prepared SIDE BY SIDE, one per lane, and handed to the whole warp through shuffles one at a time.
      const unsigned full = 0xffffffffu;
      const int myS = c.wid + c.lane * c.nw;
      double aFl[9];
      FFilter32 ffl;
#pragma unroll
      for (int i = 0; i < 9; ++i) { aFl[i] = 0.0; ffl.F[i] = 0.f; }
      ffl.Er = 0.f; ffl.c1 = 1.f; ffl.c2 = 1.f; ffl.winv = 0.f; ffl.sym = 0;
      if (c.lane < 8 && myS < nw) {
        const int a = uN[pairs[2 * myS]], b = uN[pairs[2 * myS + 1]];
        f_from_plane_parallax(H, c.x1[a], c.y1[a], c.x2[a], c.y2[a], c.x1[b], c.y1[b], c.x2[b], c.y2[b], aFl);
        f_filter_setup(F_SAMPSON, aFl, *c.t32, th2, &ffl);
      }
      __syncwarp();
      const float4* tp = reinterpret_cast<const float4*>(tileN);
      const int npair = (nN + 1) >> 1;
      const int last = (nN & 1) ? npair - 1 : -1;
      #pragma unroll 1
      for (int l = 0; l < 8; ++l) {
        const int s = c.wid + l * c.nw;
        if (s >= nw) break;
        FFilter32 ff;
#pragma unroll
        for (int i = 0; i < 9; ++i) ff.F[i] = __shfl_sync(full, ffl.F[i], l);
        ff.Er = __shfl_sync(full, ffl.Er, l); ff.c1 = __shfl_sync(full, ffl.c1, l);
        ff.c2 = __shfl_sync(full, ffl.c2, l); ff.winv = __shfl_sync(full, ffl.winv, l);
        ff.sym = 0;
        FFilter32x2 f2;
        f_filter_pack(ff, &f2);
        int ub = 0;
        int i = c.lane;
        #pragma unroll 1
        for (; i + 32 < npair; i += 64) {
          const float4 A0 = tp[2 * i], B0 = tp[2 * i + 1], A1 = tp[2 * i + 64], B1 = tp[2 * i + 65];
          float g0, g1, g2, g3;
          upk2(f_filter_gain2(f2, A0, B0, i != last), g0, g1);
          upk2(f_filter_gain2(f2, A1, B1, i + 32 != last), g2, g3);
          ub += (g0 > 0.0f ? 1 : 0) + (g1 > 0.0f ? 1 : 0) + (g2 > 0.0f ? 1 : 0) + (g3 > 0.0f ? 1 : 0);
        }
        if (i < npair) {
          float g0, g1;
          upk2(f_filter_gain2(f2, tp[2 * i], tp[2 * i + 1], i != last), g0, g1);
          ub += (g0 > 0.0f ? 1 : 0) + (g1 > 0.0f ? 1 : 0);
        }
        ub = warp_sum_i(ub);
        int cnt = ub;
        if ((unsigned)ub > m_i) {
          double aF[9];
#pragma unroll
          for (int k = 0; k < 9; ++k) aF[k] = shfl_d(aFl[k], l);
          cnt = exact_count(aF);
        }
        if (c.lane == 0) counts[s] = cnt;
      }
    } else
#endif
    {
      #pragma unroll 1
      for (int s = c.wid; s < nw; s += c.nw) {
        const int a = uN[pairs[2 * s]], b = uN[pairs[2 * s + 1]];
        double aF[9];
        f_from_plane_parallax(H, c.x1[a], c.y1[a], c.x2[a], c.y2[a], c.x1[b], c.y1[b], c.x2[b], c.y2[b], aF);
        int cnt = -1;
#if !DG_DEVICE_PASS
        if (c.t32) {   // host emulation: the same bound, one correspondence at a time
          FFilter32 ff;
          f_filter_setup(F_SAMPSON, aF, *c.t32, th2, &ff);
          int ub = 0;
          for (int i = 0; i < nN; ++i) ub += (f_filter_gain(ff, c.t32->pts[uN[i]]) > 0.0f) ? 1 : 0;
          if ((unsigned)ub <= m_i) cnt = ub;
#ifdef DG_FILTER_CHECK
          { const int ex = exact_count(aF); ++g_pp_checked; if (ub < ex) ++g_pp_violations; if (cnt >= 0) ++g_pp_settled; }
#endif
        }
#endif
        if (cnt < 0) cnt = exact_count(aF);
        if (c.lane == 0) counts[s] = cnt;
      }
    }
    DG_SYNC();
    DG_PROF_END(48);
    int ev = -1;
    #pragma unroll 1
    for (int s = 0; s < nw; ++s)
      if ((unsigned)counts[s] > m_i) { ev = s; break; }
    DG_PROF_END(32);
    DG_PROF_COUNT(35, nw);
    // commit the swaps of the iterations that count: all of them, or those up to the event
    {
      const int upto = (ev < 0) ? nw : ev + 1;
      if (c.tid == 0) {
        #pragma unroll 1
        for (int q = 0; q < 2 * upto; ++q)
          if (idxs[q] != 1) ptr[idxs[q]] = wrote[q];
        ptr[0] = pairs[2 * (upto - 1)];
        ptr[1] = pairs[2 * (upto - 1) + 1];
      }
      DG_SYNC();
    }
    if (ev < 0) {
      cur.j += 2u * (uint32_t)nw;
      no_sam += (unsigned)nw;
      continue;
    }
    cur.j += 2u * (uint32_t)(ev + 1);
    no_sam += (unsigned)(ev + 1);
    // event: new best two-point support -> LO from plane + parallax points
    {
      const int a = uN[pairs[2 * ev]], b = uN[pairs[2 * ev + 1]];
      double aF[9];
      f_from_plane_parallax(H, c.x1[a], c.y1[a], c.x2[a], c.y2[a], c.x1[b], c.y1[b], c.x2[b], c.y2[b], aF);
      const int no_i = blk_compact(c, nN, uV, [&](int i) {
        const int p = uN[i];
        return f_resid_sampson(aF, c.x1[p], c.y1[p], c.x2[p], c.y2[p]) < th2;
      });
      // uV currently holds POSITIONS in uN; convert to correspondence indices
      #pragma unroll 1
      for (int i = c.tid; i < no_i; i += c.nt) uV[i] = uN[uV[i]];
      DG_SYNC();
      m_i = (unsigned)no_i;
      double Fnew[9];
      DG_PROF_COUNT(33, 1);
      { DG_PROF_BEGIN(34); blk_inner_FH(c, W, uHl, nH, uV, no_i, th, Fnew, inl, cur); DG_PROF_END(34); }
      int cnt = 0, cnt2 = 0;
      #pragma unroll 1
      for (int i = c.tid; i < c.N; i += c.nt) {
        if (inl[i]) { ++cnt; if (nhinl[i]) ++cnt2; }
      }
      const unsigned ninl = (unsigned)blk_sum_i(c, cnt);
      const unsigned both = (unsigned)blk_sum_i(c, cnt2);
      if (ninl > max_i) {
        max_i = ninl;
        for (int i = 0; i < 9; ++i) F[i] = Fnew[i];
        maxni = both;
        const unsigned ns = (unsigned)nsamples((int)maxni, nN, 2, 0.999);
        if (ns < max_sam) max_sam = ns;
      }
    }
  }
  (void)maxni;
  return max_i;
}

}  // namespace dg
