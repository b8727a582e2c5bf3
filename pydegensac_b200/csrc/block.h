// block.h -- CTA-cooperative primitives for the per-pair engine: deterministic block reductions,
// ordered inlier compaction (the reference's `inlidxs`, rtools.c:160-171, done by a block scan) and
// the execution context.  One CTA owns one image pair; every thread runs the same scalar control
// flow on identical values (block reductions broadcast their result), so RANSAC state is replicated
// in registers and only tiny solves are single-threaded.
#pragma once
#include "common.h"
#include "la.h"
#include "warpla.h"

namespace dg {

// The CTA has 8 warps.  red_d / red_i have 16 slots because blk_inlidxs_ballot<2> uses the two halves of red_i as
// the warp counts of its two thresholds.
constexpr int kMaxWarps = 16;
constexpr int kVecRed = 48;        // widest vector reduction (45 covariance entries)
// `vec` doubles as the row buffer of the one-warp small fits (hfit.h: 2 x 32 DLT rows of 9) and as the swap-partner
// buffer of the plane-and-parallax waves, hence at least 576 doubles.
constexpr int kVecDoubles = kMaxWarps * kVecRed;
static_assert(kVecDoubles >= 576, "vec holds the small fits' rows and the plane-and-parallax swap partners");

struct BlockScratch {
  double red_d[kMaxWarps];
  int red_i[kMaxWarps];
  double vec_out[kVecRed];
  double bc[32];                   // broadcast area for small results (models, scalars)
  int bci[16];
  int counter[4];                  // atomic counters of the hypothesis wave
  int pair, ok;                    // the group's current image pair / "its input has landed" flag
  int stats[4];
  int fh_cnt[16];                  // blk_inner_FH: support of the fifteen repetitions' models ...
  double fh_F[15 * 9];             // ... and the models
  WarpScratch ws[1];               // warp 0's tile for the cooperative 9x9 / 8x9 solves
  union {                          // never live at the same time:
    WarpScratch wsx[4];            //   tiles of warps 1..4 (the five checksample triplets run side by side)
    double vec[kVecDoubles];       //   per-warp slots of the wide block reductions
  };
  DG_ENG WarpScratch* warp_tile(int wid) { return wid == 0 ? &ws[0] : &wsx[wid - 1]; }
};

struct Tile32;
struct Ctx {
  int tid, nt, lane, wid, nw;
  int N;
  const double* x1; const double* y1; const double* x2; const double* y2;   // SoA correspondences
  BlockScratch* sc;
  const Tile32* t32;   // FP32 upper-bound filter tile (nullptr: the wave scores in FP64)
  // LAF helper correspondences (laf_coef > 0, [N,6] input): p1 = x + (a12, a22), p2 = x + (a11, a21) in each image
  // (bindings.cpp:337-389); rows {p1: x1,y1,x2,y2, p2: x1,y1,x2,y2}, nullptr when the gate is off
  const double* laf[8];
};

#if DG_DEVICE_PASS
DG_ENG inline double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
DG_ENG inline int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
DG_ENG inline int warp_incl_scan_i(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}
DG_ENG inline int atomic_inc_shared(int* p) { return atomicAdd(p, 1); }
#else
inline double warp_sum(double v) { return v; }
inline int warp_sum_i(int v) { return v; }
inline int warp_incl_scan_i(int v, int) { return v; }
inline int atomic_inc_shared(int* p) { return (*p)++; }
#endif

// Sum over the CTA, same value returned to every thread, fixed combination order.
DG_ENG inline double blk_sum(const Ctx& c, double v) {
  v = warp_sum(v);
  DG_SYNC();
  if (c.lane == 0) c.sc->red_d[c.wid] = v;
  DG_SYNC();
  double s = 0.0;
  #pragma unroll 1
  for (int w = 0; w < c.nw; ++w) s += c.sc->red_d[w];
  return s;
}
DG_ENG inline int blk_sum_i(const Ctx& c, int v) {
  v = warp_sum_i(v);
  DG_SYNC();
  if (c.lane == 0) c.sc->red_i[c.wid] = v;
  DG_SYNC();
  int s = 0;
  #pragma unroll 1
  for (int w = 0; w < c.nw; ++w) s += c.sc->red_i[w];
  return s;
}
// Exclusive prefix over threads (thread order) + total.
DG_ENG inline int blk_excl_scan_i(const Ctx& c, int v, int* total) {
  const int incl = warp_incl_scan_i(v, c.lane);
  DG_SYNC();
  if (c.lane == 31 || c.tid == c.nt - 1) c.sc->red_i[c.wid] = incl;
  DG_SYNC();
  int base = 0, tot = 0;
  #pragma unroll 1
  for (int w = 0; w < c.nw; ++w) {
    const int t = c.sc->red_i[w];
    if (w < c.wid) base += t;
    tot += t;
  }
  *total = tot;
  return base + incl - v;
}
// k-wide vector sum (k <= kVecRed); result in c.sc->vec_out[0..k), visible to all threads on return.
DG_ENGN void blk_sum_vec(const Ctx& c, double* v, int k) {
  DG_SYNC();
  #pragma unroll 1
  for (int i = 0; i < k; ++i) {
    const double s = warp_sum(v[i]);
    if (c.lane == 0) c.sc->vec[c.wid * kVecRed + i] = s;
  }
  DG_SYNC();
  #pragma unroll 1
  for (int i = c.tid; i < k; i += c.nt) {
    double s = 0.0;
    #pragma unroll 1
    for (int w = 0; w < c.nw; ++w) s += c.sc->vec[w * kVecRed + i];
    c.sc->vec_out[i] = s;
  }
  DG_SYNC();
}
// Broadcast n doubles computed by thread 0 (already stored in c.sc->bc) to every thread's `dst`.
DG_ENG inline void bc_fetch(const Ctx& c, double* dst, int n) {
  DG_SYNC();
  #pragma unroll 1
  for (int i = 0; i < n; ++i) dst[i] = c.sc->bc[i];
  DG_SYNC();
}

// Exclusive scan of an int and sum of a double over the CTA in ONE barrier pair (both results to every thread).
DG_ENG inline void blk_scan_sum(const Ctx& c, int cnt, double J, int* off, int* total, double* Jtot) {
  const int incl = warp_incl_scan_i(cnt, c.lane);
  const double js = warp_sum(J);
  DG_SYNC();
  if (c.lane == 31 || c.tid == c.nt - 1) c.sc->red_i[c.wid] = incl;
  if (c.lane == 0) c.sc->red_d[c.wid] = js;
  DG_SYNC();
  int base = 0, tot = 0;
  double jt = 0.0;
  for (int w = 0; w < c.nw; ++w) {
    const int t = c.sc->red_i[w];
    if (w < c.wid) base += t;
    tot += t;
    jt += c.sc->red_d[w];
  }
  *off = base + incl - cnt;
  *total = tot;
  *Jtot = jt;
}

// MSAC score + ascending inlier index list of a residual row (reference inlidxs, rtools.c:160-171):
// J = sum truncQuad(err, th), list = {i : err[i] <= th}.  Threads own contiguous index segments so the list comes
// out ordered after one block scan; up to 8 residuals per thread stay in registers between counting and writing
// (one global read of the row, two barriers).
#if DG_DEVICE_PASS
// residual rows are streamed (written once, read once or twice): keep them out of L1 so the correspondences stay there
DG_ENG inline double ld_row(const double* p) { return __ldcg(p); }
DG_ENG inline void st_row(double* p, double v) { __stcg(p, v); }
DG_ENG inline void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
// correspondences read by the streaming O(N) passes (every residual row reads all four SoA rows once): L2 only
// (ld.cg; measured +5 % over default caching: the L1 lines the serial steps live on -- stack, lists, hypothesis
// queue -- are no longer swept out by every residual row)
DG_ENG inline double ld_soa(const double* p) { return __ldcg(p); }
#else
inline double ld_row(const double* p) { return *p; }
inline void st_row(double* p, double v) { *p = v; }
inline void prefetch_l1(const void*) {}
inline double ld_soa(const double* p) { return *p; }
#endif


#if DG_DEVICE_PASS
// Ordered compaction for rows whose per-thread segment would exceed the 8 register-resident residuals of the fast
// path (long rows: N > 8 x CTA size, e.g. the 5000-correspondence homography batches).  Warp w owns the contiguous
// chunk [w*chunk, (w+1)*chunk) of the row (chunk a multiple of 32); its lanes stride the chunk 32 residuals at a time,
// so the loads are coalesced and the ballot of "e <= th" IS the order.  The ballot word of trip j is parked on lane j
// (chunks up to 1024 residuals), the warp totals are scanned across the CTA, then the parked words are replayed to
// write the indices -- the row is read once (the host emulation's thread-segment loop below reads it twice).
// NTH = 1: (S[0], lists[0]) for th[0];  NTH = 2: both thresholds from the same pass.
template <int NTH>
__device__ __noinline__ void blk_inlidxs_ballot(const Ctx& c, const double* __restrict__ err, const double* th,
                                                int* const* lists, Score* S) {
  const unsigned full = 0xffffffffu;
  const unsigned lt = (1u << c.lane) - 1u;
  double wq[NTH], winv[NTH], J[NTH];
  int off[NTH], cnt[NTH];
  unsigned parked[NTH];
#pragma unroll
  for (int t = 0; t < NTH; ++t) {
    wq[t] = th[t] * 9 / 4;
    winv[t] = (th[t] == 0) ? 0.0 : 1.0 / wq[t];
    J[t] = 0.0; off[t] = 0; cnt[t] = 0; parked[t] = 0u;
  }
  const int chunk = (((c.N + c.nw - 1) / c.nw) + 31) & ~31;
  const int wbeg = c.wid * chunk;
  const int wend = (wbeg + chunk < c.N) ? wbeg + chunk : c.N;
  const bool park = chunk <= 1024;
  #pragma unroll 1
  for (int base = wbeg, trip = 0; base < wend; base += 32, ++trip) {
    const int i = base + c.lane;
    const double e = (i < wend) ? ld_row(err + i) : INFINITY;
#pragma unroll
    for (int t = 0; t < NTH; ++t) {
      if (th[t] != 0 && !(e >= wq[t])) J[t] += 1 - e * winv[t];
      const unsigned m = __ballot_sync(full, e <= th[t]);
      if (c.lane == trip) parked[t] = m;
      cnt[t] += __popc(m);
    }
  }
  DG_SYNC();
#pragma unroll
  for (int t = 0; t < NTH; ++t) {
    const double js = warp_sum(J[t]);
    if (c.lane == 0) {
      c.sc->red_i[t * (kMaxWarps / 2) + c.wid] = cnt[t];
      if (t == 0) c.sc->red_d[c.wid] = js; else c.sc->bc[c.wid] = js;
    }
  }
  DG_SYNC();
#pragma unroll
  for (int t = 0; t < NTH; ++t) {
    int base_off = 0, tot = 0;
    double jt = 0.0;
    for (int w = 0; w < c.nw; ++w) {
      const int v = c.sc->red_i[t * (kMaxWarps / 2) + w];
      if (w < c.wid) base_off += v;
      tot += v;
      jt += (t == 0) ? c.sc->red_d[w] : c.sc->bc[w];
    }
    S[t] = make_score(); S[t].J = jt; S[t].I = (unsigned)tot;
    off[t] = base_off;
  }
  if (park) {
    #pragma unroll 1
    for (int base = wbeg, trip = 0; base < wend; base += 32, ++trip) {
#pragma unroll
      for (int t = 0; t < NTH; ++t) {
        const unsigned m = __shfl_sync(full, parked[t], trip);
        if ((m >> c.lane) & 1u) lists[t][off[t] + __popc(m & lt)] = base + c.lane;
        off[t] += __popc(m);
      }
    }
  } else {
    #pragma unroll 1
    for (int base = wbeg; base < wend; base += 32) {
      const int i = base + c.lane;
      const double e = (i < wend) ? ld_row(err + i) : INFINITY;
#pragma unroll
      for (int t = 0; t < NTH; ++t) {
        const unsigned m = __ballot_sync(full, e <= th[t]);
        if ((m >> c.lane) & 1u) lists[t][off[t] + __popc(m & lt)] = i;
        off[t] += __popc(m);
      }
    }
  }
  DG_SYNC();
}
#endif

DG_ENGN Score blk_inlidxs(const Ctx& c, const double* err, double th, int* list) {
  DG_PROF_BEGIN(21);
  DG_PROF_COUNT(22, 1);
  const int per = (c.N + c.nt - 1) / c.nt;
  const int beg = c.tid * per;
  const int end = (beg + per < c.N) ? beg + per : c.N;
  int cnt = 0;
  double J = 0.0;
  // MSAC gain 1 - e/(9 th / 4) (reference truncQuad, rtools.c:228-236) with the division hoisted out of the loop
  const double wq = th * 9 / 4;
  const double winv = (th == 0) ? 0.0 : 1.0 / wq;
  Score s = make_score();
  int off, total;
  double Jtot;
  if (per <= 8) {
    double e[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = beg + j;
      e[j] = (i < end) ? ld_row(err + i) : INFINITY;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (th != 0 && !(e[j] >= wq)) J += 1 - e[j] * winv;   // NaN -> NaN score, as the reference's truncQuad
      if (e[j] <= th) ++cnt;
    }
    blk_scan_sum(c, cnt, J, &off, &total, &Jtot);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (e[j] <= th) list[off++] = beg + j;
  } else {
#if DG_DEVICE_PASS
    const double tha[1] = {th};
    int* const la[1] = {list};
    Score Sa[1];
    blk_inlidxs_ballot<1>(c, err, tha, la, Sa);
    DG_PROF_END(21);
    return Sa[0];
#else
    #pragma unroll 1
    for (int i = beg; i < end; ++i) {
      const double e = ld_row(err + i);
      if (th != 0 && !(e >= wq)) J += 1 - e * winv;
      if (e <= th) ++cnt;
    }
    blk_scan_sum(c, cnt, J, &off, &total, &Jtot);
    #pragma unroll 1
    for (int i = beg; i < end; ++i)
      if (ld_row(err + i) <= th) list[off++] = i;
#endif
  }
  s.J = Jtot;
  s.I = (unsigned)total;
  DG_SYNC();
  DG_PROF_END(21);
  return s;
}

// Two thresholds in one pass over the same row: (SA, listA) = blk_inlidxs(err, thA, listA) and
// (SB, listB) = blk_inlidxs(err, thB, listB), bit-identical to the two separate calls (same per-thread segments,
// same summation order), one read of the row and one barrier pair instead of two.  Counts are packed in one int
// for the scan (N < 65536; larger inputs take the two-call route).
DG_ENGN void blk_inlidxs2(const Ctx& c, const double* err, double thA, int* listA, Score* SA, double thB, int* listB,
                          Score* SB) {
  const int per = (c.N + c.nt - 1) / c.nt;
  if (per > 8 || c.N >= 65536) {
#if DG_DEVICE_PASS
    const double tha[2] = {thA, thB};
    int* const la[2] = {listA, listB};
    Score Sa[2];
    blk_inlidxs_ballot<2>(c, err, tha, la, Sa);
    *SA = Sa[0]; *SB = Sa[1];
#else
    *SA = blk_inlidxs(c, err, thA, listA);
    *SB = blk_inlidxs(c, err, thB, listB);
#endif
    return;
  }
  DG_PROF_BEGIN(21);
  DG_PROF_COUNT(22, 1);
  const int beg = c.tid * per;
  const int end = (beg + per < c.N) ? beg + per : c.N;
  const double wqA = thA * 9 / 4, wqB = thB * 9 / 4;
  const double winvA = (thA == 0) ? 0.0 : 1.0 / wqA, winvB = (thB == 0) ? 0.0 : 1.0 / wqB;
  double e[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int i = beg + j;
    e[j] = (i < end) ? ld_row(err + i) : INFINITY;
  }
  int cA = 0, cB = 0;
  double JA = 0.0, JB = 0.0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (thA != 0 && !(e[j] >= wqA)) JA += 1 - e[j] * winvA;
    if (thB != 0 && !(e[j] >= wqB)) JB += 1 - e[j] * winvB;
    if (e[j] <= thA) ++cA;
    if (e[j] <= thB) ++cB;
  }
  // one scan for both counts, both gains reduced in the same barrier pair
  const int packed = cA | (cB << 16);
  const int incl = warp_incl_scan_i(packed, c.lane);
  const double ja = warp_sum(JA), jb = warp_sum(JB);
  DG_SYNC();
  if (c.lane == 31 || c.tid == c.nt - 1) c.sc->red_i[c.wid] = incl;
  if (c.lane == 0) { c.sc->red_d[c.wid] = ja; c.sc->bc[c.wid] = jb; }
  DG_SYNC();
  int base = 0, tot = 0;
  double jta = 0.0, jtb = 0.0;
  for (int w = 0; w < c.nw; ++w) {
    const int t = c.sc->red_i[w];
    if (w < c.wid) base += t;
    tot += t;
    jta += c.sc->red_d[w];
    jtb += c.sc->bc[w];
  }
  const int excl = base + incl - packed;
  int offA = excl & 0xffff, offB = excl >> 16;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (e[j] <= thA) listA[offA++] = beg + j;
    if (e[j] <= thB) listB[offB++] = beg + j;
  }
  *SA = make_score(); SA->J = jta; SA->I = (unsigned)(tot & 0xffff);
  *SB = make_score(); SB->J = jtb; SB->I = (unsigned)(tot >> 16);
  DG_SYNC();
  DG_PROF_END(21);
}

// count of err[i] < th (strict) or <= th over all points
DG_ENG inline int blk_count_lt(const Ctx& c, const double* err, double th) {
  int cnt = 0;
  #pragma unroll 1
  for (int i = c.tid; i < c.N; i += c.nt)
    if (err[i] < th) ++cnt;
  return blk_sum_i(c, cnt);
}

}  // namespace dg
