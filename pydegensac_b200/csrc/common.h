// common.h -- portability layer for the B200 LO-RANSAC / DEGENSAC engine.
//
// The engine is written once as SPMD code for one CTA per image pair.  The same source
// also compiles with plain g++ as a ONE-THREAD "host emulation" (tid=0, nt=1, every
// barrier a no-op).  That build exists only so the control flow can be debugged against
// the reference in a container without a GPU (tests/ build it as a test helper); the
// Python package and the C-ABI library never link or load it -- the product path is the
// CUDA library only and fails loudly when it is missing.
#pragma once
#include <stdint.h>
#include <math.h>
#include <float.h>

#if defined(__CUDACC__)
#define DG_HD __host__ __device__ __forceinline__
#define DG_HDN __host__ __device__ __noinline__ inline   /* heavy leaf: one copy, keeps ptxas time sane */
#define DG_ENG __device__
#define DG_ENGN __device__ __noinline__ inline
#else
#define DG_HD inline
#define DG_HDN inline
#define DG_ENG
#define DG_ENGN inline
#endif

// One CTA owns one pair: DG_SYNC() is the CTA barrier (a no-op in the one-thread host emulation).
#if defined(__CUDA_ARCH__)
#define DG_DEVICE_PASS 1
#define DG_SYNC() __syncthreads()
#else
#define DG_DEVICE_PASS 0
#define DG_SYNC() ((void)0)
#endif

// Optional phase profiling (build with -DDG_PROF): thread 0 of every CTA accumulates clock64() deltas.
#if defined(DG_PROF) && DG_DEVICE_PASS
extern __device__ unsigned long long g_dg_prof[64];
#define DG_PROF_LEAD() (threadIdx.x == 0)
#define DG_PROF_BEGIN(id) long long prof_t_##id = DG_PROF_LEAD() ? clock64() : 0
#define DG_PROF_END(id) do { if (DG_PROF_LEAD()) atomicAdd(&g_dg_prof[id], (unsigned long long)(clock64() - prof_t_##id)); } while (0)
#define DG_PROF_COUNT(id, n) do { if (DG_PROF_LEAD()) atomicAdd(&g_dg_prof[id], (unsigned long long)(n)); } while (0)
#else
#define DG_PROF_BEGIN(id) ((void)0)
#define DG_PROF_END(id) ((void)0)
#define DG_PROF_COUNT(id, n) ((void)0)
#endif

namespace dg {

// Algorithm constants (reference: rtools.h:4-15, 31-41; Appendix B of SURVEY.md)
constexpr int kIterSam = 50;          // ITER_SAM: LO blocked for the first 50 samples
constexpr int kRanRep = 10;           // RAN_REP: inner LO samples
constexpr int kIlsqIters = 4;         // ILSQ_ITERS
constexpr double kTC = 4.0;           // TC
constexpr int kMWM = 2;               // MWM is (9/4) in INTEGER arithmetic == 2 (rtools.h:38)
constexpr int kMaxSamples = 1000000;  // MAX_SAMPLES
constexpr double kEps = 2.2204e-16;   // DEGENSAC_EPS

// RANSAC score (reference rtools.h:18-29); comparison is on J only (rtools.c:238-249)
struct Score {
  unsigned I;
  double J;
  unsigned Is;
  unsigned Ilafs;
};
DG_HD Score make_score() { Score s; s.I = 0; s.J = 0.0; s.Is = 0; s.Ilafs = 0; return s; }
DG_HD bool score_less(const Score& a, const Score& b) { return a.J < b.J; }

// error metric ids as the reference's binding layer numbers them (bindings.cpp:10-17)
enum FMetric { F_SAMPSON = 0, F_SYMM_EPI = 1 };
enum HMetric { H_SAMPSON = 0, H_SYMM_SQ_MAX = 1, H_SYMM_MAX = 2, H_SYMM_SQ_SUM = 3, H_SYMM_SUM = 4 };

}  // namespace dg
