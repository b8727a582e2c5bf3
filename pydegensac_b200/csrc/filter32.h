// filter32.h -- FP32 UPPER-BOUND MSAC score used by the hypothesis wave to discard models.
//
// The wave only has to answer "can this model's MSAC score J exceed the running threshold T?".  Models that
// cannot are dropped; the few that might are re-scored exactly in FP64 by the ordered replay, so the wave may
// use any arithmetic as long as it never UNDER-estimates J.  Here J_up >= J is computed in FP32 (FMA, approximate
// division) on centroid-centred single-precision coordinates, with explicit rounding-error budgets:
//
//   exact (real arithmetic, centred form):  e = r^2 / |g|^2,  r = X2c^T F' X1c,  g = (d r/d x1, d r/d y1, d r/d x2, d r/d y2),
//                                           F' = T2^T F T1 (Sampson error is translation invariant)
//   FP32 evaluation errors:                 |r^ - r| <= Er = c_r * 2^-24 * sum_ij |F'_ij| b2_i b1_j     (b = max |coord| per axis, 1)
//                                           | |g^| - |g| | <= 2 Eg,  Eg = c_g * 2^-24 * max_k sum |F'_.k| b
//   lower bound of the residual:            D = |g^| (1 + 2^-20) + 2 Eg >= |g|;  e >= ((|r^| - Er)_+ / D)^2, and, SQUARE-ROOT FREE,
//                                           D^2 <= |g^|^2 c1 + c2  with  c1 = (1 + 2^-19)(1 + 2^-12), c2 = (2 Eg)^2 (1 + 2^12)
//                                           (2ab <= 2^-12 a^2 + 2^12 b^2), so  e_lo = (|r^| - Er)_+^2 / (|g^|^2 c1 + c2) (1 - 2^-17) <= e
//   upper bound of the gain:                g_up = max(0, 1 - e_lo / w) >= truncQuad(e, th)              (w = 9 th / 4)
//   J_up = sum g_up (1 + 2^-16) + 1e-3 >= J.
// On the device the loop runs on PACKED pairs of correspondences with Blackwell's two-wide FP32 instructions
// (fma.rn.f32x2 / mul / add -> FFMA2, FMUL2, FADD2 in SASS): the tile is stored pair-interleaved
// {u0 u1 v0 v1 | s0 s1 t0 t1} so that two LDS.128 deliver the four operand pairs, ~16 instructions per (model,
// correspondence) instead of ~34.
// c_r = 16 and c_g = 8 are several times the number of roundings on each path (input conversion, 8 fused
// multiply-adds for r, 2 for each gradient component).  tests/ check J_up >= J(FP64) on every scored model.
// Cost: ~16 FP32 instructions per (model, correspondence) instead of ~75 FP64 ones, half the shared-memory bytes.
#pragma once
#include "common.h"
#include "block.h"

namespace dg {

struct alignas(16) Pt32 { float u, v, s, t; };   // (x1 - c1x, y1 - c1y, x2 - c2x, y2 - c2y)

struct Tile32 {
  const Pt32* pts;    // centred single-precision correspondences (in the CTA's slab)
  double cen[4];      // centroids c1x, c1y, c2x, c2y
  double bnd[4];      // max |u|, |v|, |s|, |t|
};

// Fill the FP32 tile of the current pair (block-wide) and its error-model constants.
DG_ENGN void blk_prepare_tile32(const Ctx& c, Pt32* dst, Tile32* T) {
  double v[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
  for (int i = c.tid; i < c.N; i += c.nt) { v[0] += c.x1[i]; v[1] += c.y1[i]; v[2] += c.x2[i]; v[3] += c.y2[i]; }
  blk_sum_vec(c, v, 4);
  for (int k = 0; k < 4; ++k) T->cen[k] = c.sc->vec_out[k] / c.N;
  double m[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
  for (int i = c.tid; i < c.N; i += c.nt) {
    Pt32 p;
    p.u = (float)(c.x1[i] - T->cen[0]); p.v = (float)(c.y1[i] - T->cen[1]);
    p.s = (float)(c.x2[i] - T->cen[2]); p.t = (float)(c.y2[i] - T->cen[3]);
#if DG_DEVICE_PASS
    {   // pair-interleaved: correspondences 2q and 2q+1 share two float4 {u0 u1 v0 v1} {s0 s1 t0 t1}
      float* base = reinterpret_cast<float*>(dst) + 8 * (i >> 1) + (i & 1);
      base[0] = p.u; base[2] = p.v; base[4] = p.s; base[6] = p.t;
      if (i == c.N - 1 && !(i & 1)) { base[1] = 0.f; base[3] = 0.f; base[5] = 0.f; base[7] = 0.f; }   // odd N: padding slot (masked in the loop)
    }
#else
    dst[i] = p;
#endif
    m[0] = fmax(m[0], fabs((double)p.u)); m[1] = fmax(m[1], fabs((double)p.v));
    m[2] = fmax(m[2], fabs((double)p.s)); m[3] = fmax(m[3], fabs((double)p.t));
  }
  // block max through the sum-reduction scratch: max == -min(-x); done with one lane per warp then a scan
  DG_SYNC();
#if DG_DEVICE_PASS
#pragma unroll
  for (int k = 0; k < 4; ++k)
    for (int o = 16; o > 0; o >>= 1) m[k] = fmax(m[k], __shfl_xor_sync(0xffffffffu, m[k], o));
#endif
  if (c.lane == 0) for (int k = 0; k < 4; ++k) c.sc->vec[c.wid * kVecRed + k] = m[k];
  DG_SYNC();
  for (int k = 0; k < 4; ++k) {
    double mm = 0.0;
    for (int w = 0; w < c.nw; ++w) mm = fmax(mm, c.sc->vec[w * kVecRed + k]);
    T->bnd[k] = mm;
  }
  DG_SYNC();
  T->pts = dst;
}

struct FFilter32 {
  float F[9];
  float Er, c1, c2, winv;
  int sym;    // 0: Sampson (FDs), 1: symmetric epipolar (FDsSym):  e = r^2 (1/|g1|^2 + 1/|g2|^2)
};

// Per-model constants (every lane computes them redundantly: they are warp-uniform).
DG_HD void f_filter_setup(int metric, const double* F, const Tile32& T, double w, FFilter32* o) {
  o->sym = (metric == F_SYMM_EPI) ? 1 : 0;
  double G[9], Fp[9];
  for (int i = 0; i < 3; ++i) {
    G[3 * i] = F[3 * i];
    G[3 * i + 1] = F[3 * i + 1];
    G[3 * i + 2] = F[3 * i] * T.cen[0] + F[3 * i + 1] * T.cen[1] + F[3 * i + 2];
  }
  for (int j = 0; j < 3; ++j) {
    Fp[j] = G[j];
    Fp[3 + j] = G[3 + j];
    Fp[6 + j] = T.cen[2] * G[j] + T.cen[3] * G[3 + j] + G[6 + j];
  }
  double mx = 0.0;
  for (int i = 0; i < 9; ++i) mx = fmax(mx, fabs(Fp[i]));
  const double sc = (mx > 0.0 && mx < 1e300) ? 1.0 / mx : 1.0;
  double a[9];
  for (int i = 0; i < 9; ++i) { o->F[i] = (float)(Fp[i] * sc); a[i] = fabs((double)o->F[i]); }
  const double b1[3] = {T.bnd[0], T.bnd[1], 1.0}, b2[3] = {T.bnd[2], T.bnd[3], 1.0};
  double Kr = 0.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Kr += a[3 * i + j] * b2[i] * b1[j];
  // gradient components: d/dx1 = column 0 of F' against X2, d/dy1 = column 1; d/dx2 = row 0 against X1, d/dy2 = row 1
  const double g0 = a[0] * b2[0] + a[3] * b2[1] + a[6], g1 = a[1] * b2[0] + a[4] * b2[1] + a[7];
  const double g2 = a[0] * b1[0] + a[1] * b1[1] + a[2], g3 = a[3] * b1[0] + a[4] * b1[1] + a[5];
  const double Kg = fmax(fmax(g0, g1), fmax(g2, g3));
  const double u24 = 5.9604644775390625e-08;   // 2^-24
  o->Er = (float)(16.0 * u24 * Kr * 1.0001) ;
  const double Eg2 = 2.0 * 8.0 * u24 * Kg * 1.0001;
  o->c1 = (float)((1.0 + 1.9073486328125e-06) * (1.0 + 2.44140625e-04) * (1.0 + 1e-6));   // (1 + 2^-19)(1 + 2^-12), rounded up
  o->c2 = (float)(Eg2 * Eg2 * 4097.0 * 1.0001);
  o->winv = (float)((1.0 / w) * (1.0 - 7.62939453125e-06) * (1.0 - 1e-6));               // carries the (1 - 2^-17) of e_lo
}

DG_HD float f_filter_gain(const FFilter32& f, const Pt32& p) {
#if DG_DEVICE_PASS
#define DG_FMAF __fmaf_rn
#define DG_RCPF(x) __fdividef(1.0f, (x))
#else
#define DG_FMAF fmaf
#define DG_RCPF(x) (1.0f / (x))
#endif
  const float rxc = DG_FMAF(f.F[0], p.s, DG_FMAF(f.F[3], p.t, f.F[6]));
  const float ryc = DG_FMAF(f.F[1], p.s, DG_FMAF(f.F[4], p.t, f.F[7]));
  const float rwc = DG_FMAF(f.F[2], p.s, DG_FMAF(f.F[5], p.t, f.F[8]));
  const float r = DG_FMAF(p.u, rxc, DG_FMAF(p.v, ryc, rwc));
  const float rx = DG_FMAF(f.F[0], p.u, DG_FMAF(f.F[1], p.v, f.F[2]));
  const float ry = DG_FMAF(f.F[3], p.u, DG_FMAF(f.F[4], p.v, f.F[5]));
  const float rl = fmaxf(fabsf(r) - f.Er, 0.0f);
  const float num = rl * rl;
  float e_lo;
  if (f.sym) {
    const float a = DG_FMAF(rxc, rxc, ryc * ryc), b = DG_FMAF(rx, rx, ry * ry);
    e_lo = num * (DG_RCPF(DG_FMAF(a, f.c1, f.c2)) + DG_RCPF(DG_FMAF(b, f.c1, f.c2)));
  } else {
    const float den = DG_FMAF(rxc, rxc, DG_FMAF(ryc, ryc, DG_FMAF(rx, rx, ry * ry)));
    e_lo = num * DG_RCPF(DG_FMAF(den, f.c1, f.c2));
  }
#undef DG_FMAF
#undef DG_RCPF
  const float g = 1.0f - e_lo * f.winv;
  return g > 0.0f ? g : 0.0f;   // NaN (0/0) -> 0: such a model has a NaN FP64 score and can never be accepted
}

#if DG_DEVICE_PASS
// ---- packed pairs: Blackwell FFMA2 / FMUL2 / FADD2 (PTX fma.rn.f32x2 ...), operands are 64-bit register pairs
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }

struct FFilter32x2 {     // per-model constants broadcast into both halves
  f32x2 F[9];
  f32x2 c1, c2, nwinv, one;
  float Er;
  int sym;
};
__device__ __forceinline__ void f_filter_pack(const FFilter32& f, FFilter32x2* o) {
#pragma unroll
  for (int i = 0; i < 9; ++i) o->F[i] = pk2(f.F[i], f.F[i]);
  o->c1 = pk2(f.c1, f.c1); o->c2 = pk2(f.c2, f.c2); o->nwinv = pk2(-f.winv, -f.winv); o->one = pk2(1.0f, 1.0f);
  o->Er = f.Er; o->sym = f.sym;
}
// gains of the two correspondences of one tile pair {u0 u1 v0 v1} {s0 s1 t0 t1}; `hi_live` = the second one exists
__device__ __forceinline__ f32x2 f_filter_gain2(const FFilter32x2& f, const float4 A, const float4 B, bool hi_live) {
  const f32x2 u = pk2(A.x, A.y), v = pk2(A.z, A.w), s = pk2(B.x, B.y), t = pk2(B.z, B.w);
  const f32x2 rxc = fma2(f.F[0], s, fma2(f.F[3], t, f.F[6]));
  const f32x2 ryc = fma2(f.F[1], s, fma2(f.F[4], t, f.F[7]));
  const f32x2 rwc = fma2(f.F[2], s, fma2(f.F[5], t, f.F[8]));
  const f32x2 r = fma2(u, rxc, fma2(v, ryc, rwc));
  const f32x2 rx = fma2(f.F[0], u, fma2(f.F[1], v, f.F[2]));
  const f32x2 ry = fma2(f.F[3], u, fma2(f.F[4], v, f.F[5]));
  float r0, r1;
  upk2(r, r0, r1);
  const f32x2 rl = pk2(fmaxf(fabsf(r0) - f.Er, 0.0f), fmaxf(fabsf(r1) - f.Er, 0.0f));
  const f32x2 num = mul2(rl, rl);
  f32x2 e;
  if (f.sym) {
    const f32x2 a = fma2(rxc, rxc, mul2(ryc, ryc)), b = fma2(rx, rx, mul2(ry, ry));
    float a0, a1, b0, b1;
    upk2(fma2(a, f.c1, f.c2), a0, a1);
    upk2(fma2(b, f.c1, f.c2), b0, b1);
    e = mul2(num, pk2(__fdividef(1.0f, a0) + __fdividef(1.0f, b0), __fdividef(1.0f, a1) + __fdividef(1.0f, b1)));
  } else {
    const f32x2 den = fma2(rxc, rxc, fma2(ryc, ryc, fma2(rx, rx, mul2(ry, ry))));
    float d0, d1;
    upk2(fma2(den, f.c1, f.c2), d0, d1);
    e = mul2(num, pk2(__fdividef(1.0f, d0), __fdividef(1.0f, d1)));
  }
  float g0, g1;
  upk2(fma2(e, f.nwinv, f.one), g0, g1);
  g0 = fmaxf(g0, 0.0f);                      // NaN -> 0 (fmaxf returns the other operand)
  g1 = hi_live ? fmaxf(g1, 0.0f) : 0.0f;
  return pk2(g0, g1);
}
#endif

// ---------------------------------------------------------------------------------------------------------------
// The same idea for the HOMOGRAPHY wave with the Sampson metric (reference HDs + pinvJ, Htools.c:135-199).
// With r = (r1, r2) the linearised residual pair and J = [a b c 0; d e 0 c] its 2 x 4 Jacobian, HDs returns
// |J^+ r|^2 = r^T (J J^T)^-1 r  >=  |r|^2 / lambda_max(J J^T), and lambda_max has the closed form
// (A + D)/2 + sqrt(((A - D)/2)^2 + B^2) with A = a^2+b^2+c^2, D = d^2+e^2+c^2, B = ad+be.  For the models that matter
// (near-affine H: J J^T nearly isotropic) the inequality is nearly tight.  Both r and J are invariant under
// translations of the two images when H is conjugated accordingly (H' = T1^-1 H T2), so the FP32 evaluation runs on
// the centred tile of the pair, exactly as for F, with the same kind of rounding budgets:
//   |r^_k - r_k| <= Er = 16 2^-24 K_r,   |J^ - J|_F <= 2.5 Eg,  Eg = 8 2^-24 K_g,
//   e_lo = ((|r^_1| - Er)_+^2 + (|r^_2| - Er)_+^2) / (lambda^_max c1 + c2) (1 - 2^-17) <= e,   c2 = (2.5 Eg)^2 (1 + 2^12).
// ~22 FP32 instructions per (model, correspondence) instead of ~300 FP64 ones (HDs has 8 FP64 divisions).
// ---------------------------------------------------------------------------------------------------------------
struct HFilter32 {
  float H[9];       // centred, max-normalised, COLUMN-major like the engine's h (maps image 2 -> image 1)
  float Er, c1, c2, winv;
};
DG_HD void h_filter_setup(const double* h, const Tile32& T, double w, HFilter32* o) {
  // Hm[r][c] = h[r + 3 c];  H' = T1^-1 Hm T2  (T_k: translation by the centroid of image k)
  double G[9], Hp[9];
  for (int r = 0; r < 3; ++r) {
    G[3 * r] = h[r]; G[3 * r + 1] = h[r + 3];
    G[3 * r + 2] = h[r] * T.cen[2] + h[r + 3] * T.cen[3] + h[r + 6];
  }
  for (int cc = 0; cc < 3; ++cc) {
    Hp[cc] = G[cc] - T.cen[0] * G[6 + cc];
    Hp[3 + cc] = G[3 + cc] - T.cen[1] * G[6 + cc];
    Hp[6 + cc] = G[6 + cc];
  }
  double mx = 0.0;
  for (int i = 0; i < 9; ++i) mx = fmax(mx, fabs(Hp[i]));
  const double sc = (mx > 0.0 && mx < 1e300) ? 1.0 / mx : 1.0;
  double a[9];
  for (int r = 0; r < 3; ++r)
    for (int cc = 0; cc < 3; ++cc) { o->H[r + 3 * cc] = (float)(Hp[3 * r + cc] * sc); a[r + 3 * cc] = fabs((double)o->H[r + 3 * cc]); }
  const double b1x = T.bnd[0], b1y = T.bnd[1], b2x = T.bnd[2], b2y = T.bnd[3];
  const double wmag = a[2] * b2x + a[5] * b2y + a[8];
  const double Kr1 = a[0] * b2x + a[3] * b2y + a[6] + b1x * wmag;
  const double Kr2 = a[1] * b2x + a[4] * b2y + a[7] + b1y * wmag;
  const double Kg = fmax(fmax(fmax(a[0] + a[2] * b1x, a[3] + a[5] * b1x), fmax(a[1] + a[2] * b1y, a[4] + a[5] * b1y)), wmag);
  const double u24 = 5.9604644775390625e-08;   // 2^-24
  o->Er = (float)(16.0 * u24 * fmax(Kr1, Kr2) * 1.0001);
  const double Eg = 2.5 * 8.0 * u24 * Kg * 1.0001;
  o->c1 = (float)((1.0 + 3.814697265625e-06) * (1.0 + 2.44140625e-04) * (1.0 + 1e-6));   // (1 + 2^-18)(1 + 2^-12), rounded up
  o->c2 = (float)(Eg * Eg * 4097.0 * 1.0001);
  o->winv = (float)((1.0 / w) * (1.0 - 7.62939453125e-06) * (1.0 - 1e-6));
}
// 1 - e_lo / w WITHOUT the clamp at zero (h_filter_gain clamps): <= 0 means "the Sampson error is at least w".
DG_HD float h_filter_raw(const HFilter32& f, const Pt32& p) {
#if DG_DEVICE_PASS
#define DG_FMAF __fmaf_rn
#define DG_RCPF(x) __fdividef(1.0f, (x))
#define DG_SQRTF(x) __fsqrt_ru(x)
#else
#define DG_FMAF fmaf
#define DG_RCPF(x) (1.0f / (x))
#define DG_SQRTF(x) (sqrtf(x) * 1.0000002f)
#endif
  const float* H = f.H;
  const float nw = -DG_FMAF(H[2], p.s, DG_FMAF(H[5], p.t, H[8]));
  const float r1 = DG_FMAF(p.u, nw, DG_FMAF(H[0], p.s, DG_FMAF(H[3], p.t, H[6])));
  const float r2 = DG_FMAF(p.v, nw, DG_FMAF(H[1], p.s, DG_FMAF(H[4], p.t, H[7])));
  const float a = DG_FMAF(-H[2], p.u, H[0]), b = DG_FMAF(-H[5], p.u, H[3]);
  const float d = DG_FMAF(-H[2], p.v, H[1]), e = DG_FMAF(-H[5], p.v, H[4]);
  const float cc = nw * nw;
  const float A = DG_FMAF(a, a, DG_FMAF(b, b, cc)), D = DG_FMAF(d, d, DG_FMAF(e, e, cc)), B = DG_FMAF(a, d, b * e);
  const float hs = 0.5f * (A + D), hd = 0.5f * (A - D);
  const float lam = hs + DG_SQRTF(DG_FMAF(hd, hd, B * B));
  const float l1 = fmaxf(fabsf(r1) - f.Er, 0.0f), l2 = fmaxf(fabsf(r2) - f.Er, 0.0f);
  const float e_lo = DG_FMAF(l1, l1, l2 * l2) * DG_RCPF(DG_FMAF(lam, f.c1, f.c2));
#undef DG_FMAF
#undef DG_RCPF
#undef DG_SQRTF
  return 1.0f - e_lo * f.winv;
}
DG_HD float h_filter_gain(const HFilter32& f, const Pt32& p) {
  const float g = h_filter_raw(f, p);
  return g > 0.0f ? g : 0.0f;
}

#if DG_DEVICE_PASS
struct HFilter32x2 {
  f32x2 H0, H1, H3, H4, H6, H7, nH2, nH5, nH8;
  f32x2 c1, c2, nwinv, one, half, mone;
  float Er;
};
__device__ __forceinline__ void h_filter_pack(const HFilter32& f, HFilter32x2* o) {
  o->H0 = pk2(f.H[0], f.H[0]); o->H1 = pk2(f.H[1], f.H[1]); o->H3 = pk2(f.H[3], f.H[3]); o->H4 = pk2(f.H[4], f.H[4]);
  o->H6 = pk2(f.H[6], f.H[6]); o->H7 = pk2(f.H[7], f.H[7]);
  o->nH2 = pk2(-f.H[2], -f.H[2]); o->nH5 = pk2(-f.H[5], -f.H[5]); o->nH8 = pk2(-f.H[8], -f.H[8]);
  o->c1 = pk2(f.c1, f.c1); o->c2 = pk2(f.c2, f.c2); o->nwinv = pk2(-f.winv, -f.winv); o->one = pk2(1.0f, 1.0f);
  o->half = pk2(0.5f, 0.5f); o->mone = pk2(-1.0f, -1.0f);
  o->Er = f.Er;
}
__device__ __forceinline__ f32x2 h_filter_raw2(const HFilter32x2& f, const float4 A4, const float4 B4) {
  const f32x2 u = pk2(A4.x, A4.y), v = pk2(A4.z, A4.w), s = pk2(B4.x, B4.y), t = pk2(B4.z, B4.w);
  const f32x2 nw = fma2(f.nH2, s, fma2(f.nH5, t, f.nH8));
  const f32x2 r1 = fma2(u, nw, fma2(f.H0, s, fma2(f.H3, t, f.H6)));
  const f32x2 r2 = fma2(v, nw, fma2(f.H1, s, fma2(f.H4, t, f.H7)));
  const f32x2 a = fma2(f.nH2, u, f.H0), b = fma2(f.nH5, u, f.H3), d = fma2(f.nH2, v, f.H1), e = fma2(f.nH5, v, f.H4);
  const f32x2 cc = mul2(nw, nw);
  const f32x2 A = fma2(a, a, fma2(b, b, cc)), D = fma2(d, d, fma2(e, e, cc)), B = fma2(a, d, mul2(b, e));
  const f32x2 hs = mul2(add2(A, D), f.half), hd = mul2(fma2(D, f.mone, A), f.half);
  float q0, q1, h0, h1;
  upk2(fma2(hd, hd, mul2(B, B)), q0, q1);
  upk2(hs, h0, h1);
  const f32x2 lam = pk2(h0 + __fsqrt_ru(q0), h1 + __fsqrt_ru(q1));
  float x0, x1, y0, y1;
  upk2(r1, x0, x1);
  upk2(r2, y0, y1);
  const f32x2 l1 = pk2(fmaxf(fabsf(x0) - f.Er, 0.0f), fmaxf(fabsf(x1) - f.Er, 0.0f));
  const f32x2 l2 = pk2(fmaxf(fabsf(y0) - f.Er, 0.0f), fmaxf(fabsf(y1) - f.Er, 0.0f));
  float d0, d1;
  upk2(fma2(lam, f.c1, f.c2), d0, d1);
  const f32x2 el = mul2(fma2(l1, l1, mul2(l2, l2)), pk2(__fdividef(1.0f, d0), __fdividef(1.0f, d1)));
  return fma2(el, f.nwinv, f.one);
}
__device__ __forceinline__ f32x2 h_filter_gain2(const HFilter32x2& f, const float4 A4, const float4 B4, bool hi_live) {
  float g0, g1;
  upk2(h_filter_raw2(f, A4, B4), g0, g1);
  g0 = fmaxf(g0, 0.0f);
  g1 = hi_live ? fmaxf(g1, 0.0f) : 0.0f;
  return pk2(g0, g1);
}
#endif

}  // namespace dg
