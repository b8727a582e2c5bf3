// workspace.h -- carving of the per-CTA scratch slab (global memory, L2 resident) into the rows,
// index lists, hypothesis queue and LO hash table the engines use.  Same layout on the device and in
// the one-thread host emulation used by the tests.
#pragma once
#include "common.h"
#include "ffit.h"

namespace dg {

constexpr int kHashCap = 2048;
constexpr int kListPad = 512;

DG_HD size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// `laf`: the eight rows of LAF helper correspondences are only allocated for [N,6] inputs with the gate on.
// Hypothesis queue: `chunk` entries (about one iteration in four yields an oriented-valid model; a wave that would
// overflow is split by the driver).
DG_HD size_t workspace_bytes(int N, int chunk, bool laf) {
  size_t b = 0;
  b += align_up(sizeof(double) * (size_t)N, 128) * (laf ? 20 : 12);   // err[4], errBest, w, dtmp[6] (, laf[8])
  b += align_up(sizeof(int) * (size_t)(N + kListPad), 128) * 7;   // inliers, intbuff, intbuff_best, itmp[4]
  b += align_up((size_t)N, 128) * 4;                              // btmp[4]
  b += align_up(sizeof(Cand) * (size_t)chunk, 128);               // hypothesis queue
  b += align_up(sizeof(int) * (size_t)chunk, 128);                // survivors
  b += align_up(sizeof(double) * 16 * (size_t)chunk, 128);        // null-space bases of the wave
  b += align_up(sizeof(uint32_t) * kHashCap, 128) * 3;            // hash table
  b += align_up(sizeof(double) * (size_t)N, 128) * 4;             // SoA correspondences of the pair
  b += align_up(16 * ((size_t)N + 1), 128);                       // FP32 filter tile (pair-interleaved, N+1 slots)
  return b;
}

DG_HD void workspace_carve(unsigned char* base, int N, int chunk, bool laf, Workspace* W, double** pts_soa) {
  unsigned char* p = base;
  const size_t rowd = align_up(sizeof(double) * (size_t)N, 128);
  const size_t rowi = align_up(sizeof(int) * (size_t)(N + kListPad), 128);
  const size_t rowb = align_up((size_t)N, 128);
  #pragma unroll 1
  for (int i = 0; i < 4; ++i) { W->err[i] = (double*)p; p += rowd; }
  W->errBest = (double*)p; p += rowd;
  W->w = (double*)p; p += rowd;
  #pragma unroll 1
  for (int i = 0; i < 6; ++i) { W->dtmp[i] = (double*)p; p += rowd; }
  #pragma unroll 1
  for (int i = 0; i < 8; ++i) { W->laf[i] = laf ? (double*)p : nullptr; if (laf) p += rowd; }
  W->inliers = (int*)p; p += rowi;
  W->intbuff = (int*)p; p += rowi;
  W->intbuff_best = (int*)p; p += rowi;
  #pragma unroll 1
  for (int i = 0; i < 4; ++i) { W->itmp[i] = (int*)p; p += rowi; }
  #pragma unroll 1
  for (int i = 0; i < 4; ++i) { W->btmp[i] = p; p += rowb; }
  W->cand = (Cand*)p; p += align_up(sizeof(Cand) * (size_t)chunk, 128);
  W->pass = (int*)p; p += align_up(sizeof(int) * (size_t)chunk, 128);
  W->nsbuf = (double*)p; p += align_up(sizeof(double) * 16 * (size_t)chunk, 128);
  W->cand_cap = chunk;
  W->hhash = (uint32_t*)p; p += align_up(sizeof(uint32_t) * kHashCap, 128);
  W->hlen = (int*)p; p += align_up(sizeof(uint32_t) * kHashCap, 128);
  W->hid = (int*)p; p += align_up(sizeof(uint32_t) * kHashCap, 128);
  W->hcap = kHashCap;
  *pts_soa = (double*)p;
}
DG_HD unsigned char* workspace_tile32(unsigned char* base, int N, int chunk, bool laf) {
  return base + workspace_bytes(N, chunk, laf) - align_up(16 * ((size_t)N + 1), 128);
}

// Threshold conventions of the reference's binding layer (bindings.cpp:64-107, 297-318).
DG_HD void f_thresholds(double px_th, int sym_check, double* th, double* sym_th) {
  *th = px_th * px_th;
  *sym_th = px_th * px_th * (3.0 * (sym_check ? 1 : 0));
}
DG_HD int h_thresholds(int metric, double px_th, int sym_check, double* th, double* sym_th) {
  const double coef = 3.0 * (sym_check ? 1 : 0);
  switch (metric) {
    case H_SAMPSON: *th = px_th * px_th; *sym_th = px_th * coef; return 0;
    case H_SYMM_SQ_MAX: *th = px_th * px_th; *sym_th = 0; return 0;
    case H_SYMM_MAX: *th = px_th; *sym_th = 0; return 0;
    case H_SYMM_SQ_SUM: *th = px_th * px_th; *sym_th = px_th * coef; return 0;
    case H_SYMM_SUM: *th = px_th; *sym_th = px_th * coef; return 0;
  }
  return -1;
}

}  // namespace dg
