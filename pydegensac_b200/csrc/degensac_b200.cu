// degensac_b200.cu -- sm_100a kernel + C ABI (include/degensac_b200.h) of the LO-RANSAC / DEGENSAC engine.
//
// One persistent CTA (256 threads, two per SM) processes one image pair at a time; pairs are claimed from an atomic
// work counter:
//   * the pair's correspondences are read ONCE from HBM (coalesced 16-byte loads of the [n][dim] rows) and
//     de-interleaved into a structure-of-arrays copy (4 x n doubles) in the CTA's slab of global memory -- L1/L2
//     resident; shared-memory residency measured slower, see the CTA shape below -- plus the centred FP32 tile of the
//     wave filter (pair-interleaved, 16 B per correspondence);
//   * engine_f.h / engine_h.h run the speculative hypothesis WAVES (two threads per 7-point sample / one per 4-point
//     sample, one warp per scored model, FP32 upper-bound filter with packed FFMA2) and the ordered REPLAY (LO, DEGENSAC,
//     termination) in exact FP64;
//   * residual rows, index lists, the hypothesis queue and the LO hash table live in the same slab; shared memory holds
//     only the block scratch (reductions, warp tiles of the small solves).
// Every launch in flight owns its slabs and work counter (pool keyed by stream): the device entry points are re-entrant.
// All FP64 arithmetic on the path is compiled with -fmad=false so residuals, scores and solves round exactly like the
// reference's x86-64 (no-FMA) build; there is no tensor-core work and no CPU fallback.
#include <cuda_runtime.h>
#include <mutex>
#include <vector>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/degensac_b200.h"
#include "engine_f.h"
#include "engine_h.h"
#include "engine_h2el.h"
#include "filter32.h"
#include "workspace.h"

#ifdef DG_PROF
__device__ unsigned long long g_dg_prof[64];
#endif

namespace {

// CTA shape.  256 threads x 2 CTAs per SM measured fastest on B200 (DESIGN.md sections 3.1 and 7): the waves and the
// O(N) passes of the replay want the 8 warps, while more, smaller CTAs per SM lose to instruction-cache misses (each
// CTA walks a different part of a ~300 KB code image).  Shared memory holds the block scratch only; the pair's FP64
// correspondences and FP32 filter tile live in the CTA's slab (L1/L2 resident), which measured faster than shared
// memory because the serial steps need that L1 capacity.
constexpr int kThreads = 256;
constexpr int kCtasPerSm = 2;
constexpr int kChunk = 512;   // iterations hypothesised per wave

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

// One batch as the caller passed it; the fields an entry point does not take keep these zeros.
struct Job {
  const double* x1y1 = nullptr;
  const double* x2y2 = nullptr;
  const int32_t* offsets = nullptr;   // ragged batches: pair p owns rows offsets[p] .. offsets[p+1] of the concatenated arrays; nullptr: n each
  int n_pairs = 0, n = 0, dim = 0;    // n: correspondences per pair (ragged: the largest, which sizes the slabs)
  double px_th = 0, conf = 0, laf_coef = 0;
  int max_iters = 0, metric = 0, sym_check = 0, degen = 0;
  unsigned flags = 0;                 // DGB200_FLAG_*
  const uint64_t* seeds = nullptr;
  double* model_out = nullptr;
  uint8_t* mask_out = nullptr;
  int32_t* stats_out = nullptr;
};

// A Job on the device plus what launch() derives for the kernel.
struct BatchArgs : Job {
  unsigned char* workspace;
  size_t ws_stride;
  int chunk;
  int* work_counter;
  int aligned16;        // both input pointers 16-byte aligned: dim == 2 rows are read as double2
  int filter32;         // FP32 upper-bound filter in the F wave (DGB200_FILTER32=0 scores the wave in FP64; same results)
  const int* ready;     // host-buffer flavour: number of leading pairs whose input has landed in HBM (nullptr: all)
  int* status;          // [0] = 1 once a CTA gave up waiting for its input, [1] = smallest pair index given up on
  long long wait_cycles;   // patience of that wait
};

template <int KIND>  // 0: fundamental matrix, 1: homography, 2: homography from elliptical features (rows u10, engine_h2el.h)
__global__ void __launch_bounds__(kThreads, kCtasPerSm) ransac_pairs_kernel(BatchArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = (int)threadIdx.x, nt = (int)blockDim.x;
  dg::BlockScratch* sc = reinterpret_cast<dg::BlockScratch*>(smem_raw);
  unsigned char* slab = a.workspace + (size_t)blockIdx.x * a.ws_stride;
  dg::Workspace W;
  double* soa;
  const bool use_laf = (a.laf_coef > 0) && (a.dim == 6);
  dg::workspace_carve(slab, a.n, a.chunk, use_laf, &W, &soa);
  const size_t row = dg::align_up(sizeof(double) * (size_t)a.n, 128) / sizeof(double);
  dg::Pt32* tile32 = reinterpret_cast<dg::Pt32*>(dg::workspace_tile32(slab, a.n, a.chunk, use_laf));
  dg::Tile32 t32;

  dg::Ctx c;
  c.tid = tid; c.nt = nt; c.lane = tid & 31; c.wid = tid >> 5; c.nw = nt >> 5;
  c.N = a.n;
  c.x1 = soa; c.y1 = soa + row; c.x2 = soa + 2 * row; c.y2 = soa + 3 * row;
  c.sc = sc;
  c.t32 = nullptr;
  for (int i = 0; i < 8; ++i) c.laf[i] = use_laf ? W.laf[i] : nullptr;

  for (;;) {
    DG_SYNC();
    if (tid == 0) sc->pair = atomicAdd(a.work_counter, 1);
    DG_SYNC();
    const int p = sc->pair;
    if (p >= a.n_pairs) break;
    if (a.ready) {
      // The host streams the batch in chunks on a copy stream while this kernel runs and bumps `ready` after each
      // chunk.  The wait is bounded: when copies cannot overlap the kernel (a profiler serialising the streams, a
      // stalled link) the CTA records the pair, raises the abort flag and retires; the host then runs the pairs from
      // the smallest recorded index on in a second, ordinary launch.  Nothing can hang.
      if (tid == 0) {
        int ok = (*reinterpret_cast<volatile int*>(a.status) == 0) ? 1 : 0;
        if (ok) {
          const long long t0 = clock64();
          while (*reinterpret_cast<const volatile int*>(a.ready) <= p) {
            __nanosleep(500);
            if (clock64() - t0 > a.wait_cycles || *reinterpret_cast<volatile int*>(a.status) != 0) { ok = 0; break; }
          }
        }
        if (!ok) { atomicMin(a.status + 1, p); atomicExch(a.status, 1); }
        sc->ok = ok;
      }
      DG_SYNC();
      if (!sc->ok) break;
    }
    // ---- stage the pair: HBM -> SoA tile (the only read of the pair from HBM)
    const size_t row0 = a.offsets ? (size_t)a.offsets[p] : (size_t)p * a.n;
    const int n = a.offsets ? a.offsets[p + 1] - a.offsets[p] : a.n;
    c.N = n;
    const double* g1 = a.x1y1 + row0 * a.dim;
    const double* g2 = (KIND == 2) ? g1 + 5 : a.x2y2 + row0 * a.dim;   // u10 rows: (x', y', a', b', c', x, y, a, b, c)
    if (a.dim == 2 && a.aligned16) {   // rows are 16 bytes, so every pair of a ragged batch starts aligned too
      const double2* v1 = reinterpret_cast<const double2*>(g1);
      const double2* v2 = reinterpret_cast<const double2*>(g2);
      for (int i = tid; i < n; i += nt) {
        const double2 q1 = __ldcg(v1 + i), q2 = __ldcg(v2 + i);   // L2 only: the chunk may have landed after this kernel started
        soa[i] = q1.x; soa[row + i] = q1.y; soa[2 * row + i] = q2.x; soa[3 * row + i] = q2.y;
      }
    } else {
      for (int i = tid; i < n; i += nt) {
        const double* q1 = g1 + (size_t)i * a.dim;
        const double* q2 = g2 + (size_t)i * a.dim;
        soa[i] = __ldcg(q1); soa[row + i] = __ldcg(q1 + 1);
        soa[2 * row + i] = __ldcg(q2); soa[3 * row + i] = __ldcg(q2 + 1);
        if (use_laf) {   // columns (x, y, a11, a12, a21, a22): p1 = x + (a12, a22), p2 = x + (a11, a21) (bindings.cpp:355-385)
          W.laf[0][i] = q1[0] + q1[3]; W.laf[1][i] = q1[1] + q1[5]; W.laf[2][i] = q2[0] + q2[3]; W.laf[3][i] = q2[1] + q2[5];
          W.laf[4][i] = q1[0] + q1[2]; W.laf[5][i] = q1[1] + q1[4]; W.laf[6][i] = q2[0] + q2[2]; W.laf[7][i] = q2[1] + q2[4];
        }
      }
    }
    DG_SYNC();
    const unsigned long long seed = a.seeds ? a.seeds[p] : (unsigned long long)p;
    double* model = a.model_out + (size_t)p * 9;
    unsigned char* mask = a.mask_out + row0;
    int* s_stats = sc->stats;
    if (KIND == 0) {
      c.t32 = nullptr;
      if (a.filter32) {
        dg::blk_prepare_tile32(c, tile32, &t32);
        c.t32 = &t32;
      }
      dg::FParams P;
      dg::f_thresholds(a.px_th, a.sym_check, &P.th, &P.sym_th);
      P.conf = a.conf; P.laf_coef = a.laf_coef; P.max_iters = a.max_iters; P.metric = a.metric; P.degen = a.degen;
      P.do_laf = use_laf ? 1 : 0; P.th_laf = a.laf_coef * P.th;
      P.do_sym = P.sym_th > 0; P.seed = seed; P.chunk = a.chunk;
      P.final_lsq = (a.flags & DGB200_FLAG_FINAL_LSQ) ? 1 : 0;
      dg::ransac_F_pair(c, P, W, model, mask, s_stats);
    } else if (KIND == 2) {
      c.t32 = nullptr;
      dg::H2Params P;
      P.th = a.px_th * a.px_th; P.conf = a.conf; P.max_iters = a.max_iters; P.seed = seed; P.chunk = a.chunk;
      dg::ransac_H2el_pair(c, P, W, g1, model, mask, s_stats);
    } else {
      c.t32 = nullptr;
      if (a.filter32 && a.metric == dg::H_SAMPSON) {   // FP32 upper-bound filter of the H wave (Sampson metric)
        dg::blk_prepare_tile32(c, tile32, &t32);
        c.t32 = &t32;
      }
      dg::HParams P;
      dg::h_thresholds(a.metric, a.px_th, a.sym_check, &P.th, &P.sym_th);
      P.conf = a.conf; P.laf_coef = a.laf_coef; P.max_iters = a.max_iters; P.metric = a.metric;
      P.do_laf = use_laf ? 1 : 0; P.th_laf = a.laf_coef * P.th;
      P.do_sym = P.sym_th > 0; P.seed = seed; P.chunk = a.chunk;
      P.final_lsq = (a.flags & DGB200_FLAG_FINAL_LSQ) ? 1 : 0;
      dg::ransac_H_pair(c, P, W, model, mask, s_stats);
    }
    DG_SYNC();
    // "no model" convention of the Python layer (utils.py:104-107, 143-145): zero model -> empty mask
    double asum = 0.0;
    for (int i = 0; i < 9; ++i) asum += fabs(model[i]);
    if (asum == 0.0)
      for (int i = tid; i < n; i += nt) mask[i] = 0;
    if (a.stats_out && tid < 4) a.stats_out[(size_t)p * 4 + tid] = s_stats[tid];
  }
}

// ------------------------------------------------------------------------------------ host side
// Device-wide state (created once per device) and a pool of launch contexts: a launch needs its own slab area and
// work counter, so two calls in flight on different streams never share scratch.  A context is reused by the stream
// that used it last (stream order serialises the two kernels) or by anybody once its last launch has completed.
struct LaunchCtx {
  unsigned char* ws = nullptr; size_t ws_bytes = 0;
  int* counter = nullptr;
  cudaEvent_t done = nullptr;
  cudaStream_t last_stream = nullptr;
  bool used = false;
};
struct Cache {
  int device = -1;
  int sm_count = 0;
  std::vector<LaunchCtx> ctxs;
  unsigned char* io = nullptr; size_t io_bytes = 0;   // staging for the host-buffer flavour
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_feed = nullptr;
  cudaStream_t s_run = nullptr, s_copy = nullptr;     // host-buffer flavour: kernel stream + input feed stream
  int* ready = nullptr;                               // device: pairs whose input has landed; status word follows
  int* h_ready = nullptr;                             // pinned: cumulative pair counts per chunk
};
constexpr int kMaxChunks = 16;
std::mutex g_mu;
Cache g_c;
thread_local char g_err[512] = "";
long long g_launches = 0;
double g_last_ms = 0.0;

int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
  if (e != cudaSuccess) snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  else snprintf(g_err, sizeof(g_err), "%s", what);
  return code;
}
#define CU(call)                                                     \
  do {                                                               \
    cudaError_t e__ = (call);                                        \
    if (e__ != cudaSuccess) return fail(DGB200_E_CUDA, #call, e__);  \
  } while (0)

void destroy_device_state() {   // with the owning device current
  for (LaunchCtx& x : g_c.ctxs) {
    if (x.ws) cudaFree(x.ws);
    if (x.counter) cudaFree(x.counter);
    if (x.done) cudaEventDestroy(x.done);
  }
  g_c.ctxs.clear();
  if (g_c.io) cudaFree(g_c.io);
  if (g_c.ready) cudaFree(g_c.ready);
  if (g_c.h_ready) cudaFreeHost(g_c.h_ready);
  if (g_c.ev0) cudaEventDestroy(g_c.ev0);
  if (g_c.ev1) cudaEventDestroy(g_c.ev1);
  if (g_c.ev_feed) cudaEventDestroy(g_c.ev_feed);
  if (g_c.s_run) cudaStreamDestroy(g_c.s_run);
  if (g_c.s_copy) cudaStreamDestroy(g_c.s_copy);
  g_c = Cache();
}

int ensure_device() {
  if (g_c.device >= 0) { CU(cudaSetDevice(g_c.device)); return 0; }
  int cnt = 0;
  cudaError_t e = cudaGetDeviceCount(&cnt);
  if (e != cudaSuccess || cnt <= 0) return fail(DGB200_E_CUDA, "no CUDA device: the B200 engine has no CPU fallback", e);
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, dev));
  Cache c;
  c.sm_count = prop.multiProcessorCount;
  cudaError_t err = cudaSuccess;
  auto step = [&](cudaError_t r) { if (err == cudaSuccess) err = r; };
  step(cudaEventCreate(&c.ev0));
  step(cudaEventCreate(&c.ev1));
  step(cudaEventCreateWithFlags(&c.ev_feed, cudaEventDisableTiming));
  step(cudaStreamCreateWithFlags(&c.s_run, cudaStreamNonBlocking));
  step(cudaStreamCreateWithFlags(&c.s_copy, cudaStreamNonBlocking));
  step(cudaMalloc(&c.ready, 4 * sizeof(int)));
  step(cudaHostAlloc(&c.h_ready, kMaxChunks * sizeof(int), cudaHostAllocDefault));
  if (err != cudaSuccess) {   // nothing half-initialised survives
    g_c = c; g_c.device = -1;
    destroy_device_state();
    return fail(DGB200_E_CUDA, "device state", err);
  }
  c.device = dev;
  g_c = c;
  return 0;
}

// a launch context whose scratch nobody can still be using on another stream
int acquire_ctx(cudaStream_t st, size_t need, LaunchCtx** out) {
  LaunchCtx* pick = nullptr;
  for (LaunchCtx& x : g_c.ctxs)
    if (x.used && x.last_stream == st) { pick = &x; break; }
  if (!pick)
    for (LaunchCtx& x : g_c.ctxs)
      if (!x.used || cudaEventQuery(x.done) == cudaSuccess) { pick = &x; break; }
  if (!pick) {
    g_c.ctxs.reserve(64);     // pointers handed out stay valid
    if (g_c.ctxs.size() >= 64) return fail(DGB200_E_CUDA, "too many launches in flight on distinct streams");
    g_c.ctxs.emplace_back();
    pick = &g_c.ctxs.back();
    CU(cudaEventCreateWithFlags(&pick->done, cudaEventDisableTiming));
    CU(cudaMalloc(&pick->counter, sizeof(int)));
  }
  if (need > pick->ws_bytes) {
    if (pick->ws) {
      if (pick->used) CU(cudaEventSynchronize(pick->done));   // same-stream reuse with a larger batch: wait before freeing
      cudaFree(pick->ws);
    }
    pick->ws = nullptr; pick->ws_bytes = 0;
    CU(cudaMalloc(&pick->ws, need));
    pick->ws_bytes = need;
  }
  *out = pick;
  return 0;
}

template <int KIND>
int launch(const Job& j, cudaStream_t st, const int* ready = nullptr, int* status = nullptr, long long wait_cycles = 0) {
  BatchArgs a;
  static_cast<Job&>(a) = j;
  a.ready = ready; a.status = status; a.wait_cycles = wait_cycles;
  a.chunk = kChunk;
  a.filter32 = (env_int("DGB200_FILTER32", 1) != 0 && (KIND == 0 || (KIND == 1 && j.metric == dg::H_SAMPSON))) ? 1 : 0;   // parity switch, read at every launch
  a.aligned16 = ((((uintptr_t)j.x1y1) | ((uintptr_t)j.x2y2)) & 15) == 0 ? 1 : 0;
  const size_t smem = dg::align_up(sizeof(dg::BlockScratch), 128);
  auto kern = ransac_pairs_kernel<KIND>;
  int per_sm = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem));
  if (per_sm < 1) return fail(DGB200_E_CUDA, "kernel does not fit on an SM");
  int grid = g_c.sm_count * per_sm;     // persistent CTAs: a whole number of CTAs per SM
  if (grid > j.n_pairs) grid = j.n_pairs;
  a.ws_stride = dg::align_up(dg::workspace_bytes(j.n, a.chunk, j.laf_coef > 0 && j.dim == 6), 256);
  LaunchCtx* lc = nullptr;
  const int rc = acquire_ctx(st, a.ws_stride * (size_t)grid, &lc);
  if (rc) return rc;
  a.workspace = lc->ws;
  a.work_counter = lc->counter;
  CU(cudaMemsetAsync(lc->counter, 0, sizeof(int), st));
  kern<<<grid, kThreads, smem, st>>>(a);
  CU(cudaGetLastError());
  CU(cudaEventRecord(lc->done, st));
  lc->used = true; lc->last_stream = st;
  ++g_launches;
  return 0;
}

int check_args(int kind, const void* p1, const void* p2, int n_pairs, int n, int dim, int metric, double laf_coef,
               const void* m, const void* k) {
  if (!p1 || !p2 || !m || !k) return fail(DGB200_E_ARG, "null buffer");
  if (n_pairs < 1) return fail(DGB200_E_ARG, "n_pairs must be >= 1");
  if (kind == 2) {
    if (dim != 10) return fail(DGB200_E_ARG, "u10 should be an array with dims [n,10]");
    if (n < 4) return fail(DGB200_E_ARG, "u10 should be an array with dims [n,10], n>=4");
    return 0;
  }
  if (dim != 2 && dim != 6) return fail(DGB200_E_ARG, "x1y1 should be an array with dims [n,2], [n,6]");
  if (kind == 0 && n < 8) return fail(DGB200_E_ARG, "x1y1 should be an array with dims [n,2], n>=8");
  if (kind == 1 && n < 4) return fail(DGB200_E_ARG, "x1y1 should be an array with dims [n,2], n>=4");
  if (kind == 0 && (metric < 0 || metric > 1)) return fail(DGB200_E_METRIC, "unknown fundamental-matrix error_type");
  if (kind == 1 && (metric < 0 || metric > 4)) return fail(DGB200_E_METRIC, "unknown homography error_type");
  if (laf_coef > 0 && dim != 6) return fail(DGB200_E_ARG, "laf_coef > 0 needs [n,6] inputs (x, y, a11, a12, a21, a22)");
  return 0;
}
// ragged batches: offsets[0] = 0, non-decreasing, every pair at least `min_n` rows; returns the largest pair in *n_max
int check_offsets(int kind, const int32_t* offsets, int n_pairs, int* n_max, long long* total) {
  if (!offsets) return fail(DGB200_E_ARG, "null offsets");
  if (offsets[0] != 0) return fail(DGB200_E_ARG, "offsets[0] must be 0");
  int mx = 0;
  const int min_n = kind == 0 ? 8 : 4;   // (kind 2, elliptical features: 4 as well)
  for (int p = 0; p < n_pairs; ++p) {
    const long long n = (long long)offsets[p + 1] - offsets[p];
    if (n < min_n) return fail(DGB200_E_ARG, kind == 0 ? "every pair needs n >= 8 correspondences" : "every pair needs n >= 4 correspondences");
    if (n > mx) mx = (int)n;
  }
  *n_max = mx;
  *total = offsets[n_pairs];
  return 0;
}

template <int KIND>
int run_host(const Job& h) {   // h: a batch in host memory
  std::lock_guard<std::mutex> lk(g_mu);
  const int32_t* offsets = h.offsets;
  const int n_pairs = h.n_pairs, dim = h.dim;
  int n = h.n;
  long long rows = (long long)n_pairs * n;
  if (offsets) {
    if (n_pairs < 1) return fail(DGB200_E_ARG, "n_pairs must be >= 1");
    const int rc0 = check_offsets(KIND, offsets, n_pairs, &n, &rows);
    if (rc0) return rc0;
  }
  int rc = check_args(KIND, h.x1y1, h.x2y2, n_pairs, n, dim, h.metric, h.laf_coef, h.model_out, h.mask_out);
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  const size_t in_b = dg::align_up(sizeof(double) * (size_t)rows * dim, 256);
  const size_t seed_b = dg::align_up(sizeof(uint64_t) * (size_t)n_pairs, 256);
  const size_t off_b = dg::align_up(sizeof(int32_t) * ((size_t)n_pairs + 1), 256);
  const size_t model_b = dg::align_up(sizeof(double) * 9 * (size_t)n_pairs, 256);
  const size_t mask_b = dg::align_up((size_t)rows, 256);
  const size_t stats_b = dg::align_up(sizeof(int) * 4 * (size_t)n_pairs, 256);
  const size_t need = 2 * in_b + seed_b + off_b + model_b + mask_b + stats_b;
  if (need > g_c.io_bytes) {
    if (g_c.io) cudaFree(g_c.io);
    g_c.io = nullptr; g_c.io_bytes = 0;
    CU(cudaMalloc(&g_c.io, need));
    g_c.io_bytes = need;
  }
  unsigned char* p = g_c.io;
  double* d1 = (double*)p; p += in_b;
  double* d2 = (double*)p; p += in_b;
  uint64_t* dseed = (uint64_t*)p; p += seed_b;
  int32_t* doff = (int32_t*)p; p += off_b;
  double* dmodel = (double*)p; p += model_b;
  unsigned char* dmask = p; p += mask_b;
  int* dstats = (int*)p;
  Job j = h;   // the same batch in the staging buffer
  j.x1y1 = d1; j.x2y2 = d2; j.offsets = offsets ? doff : nullptr; j.n = n; j.seeds = h.seeds ? dseed : nullptr;
  j.model_out = dmodel; j.mask_out = dmask; j.stats_out = dstats;
  // Input feed overlapped with the kernel: the batch is copied in chunks on a copy stream; after every chunk the
  // device-side `ready` count is bumped (a 4-byte copy from pinned memory, ordered behind the chunk) and the
  // persistent CTAs wait on it before staging a pair.  Chunk 0 covers the pairs the CTAs start with.
  cudaStream_t st = g_c.s_run, cs = g_c.s_copy;
  int nchunks = 8;
  int first = 2 * kCtasPerSm * g_c.sm_count;   // two pairs per resident CTA
  if (first > n_pairs) first = n_pairs;
  int rest = n_pairs - first;
  if (rest <= 0) nchunks = 1;
  const int per = (nchunks > 1) ? (rest + (nchunks - 2)) / (nchunks - 1) : 0;
  static const int k_init[4] = {0, 0, 0x7fffffff, 0};      // ready, abort flag, first pair given up on
  CU(cudaMemcpyAsync(g_c.ready, k_init, sizeof(k_init), cudaMemcpyHostToDevice, cs));
  // patience of a waiting CTA: the whole input at a pessimistic 4 GB/s plus 20 ms, in SM cycles (<= 2.1 GHz)
  const double feed_s = 2.0 * sizeof(double) * (double)rows * (double)dim / 4e9 + 0.020;
  long long wait_cycles = (long long)(feed_s * 2.1e9);
  if (const char* e = getenv("DGB200_FEED_WAIT_US")) wait_cycles = (long long)(atof(e) * 2.1e3);   // tests: force the fallback
  if (h.seeds) CU(cudaMemcpyAsync(dseed, h.seeds, sizeof(uint64_t) * (size_t)n_pairs, cudaMemcpyHostToDevice, cs));
  if (offsets) CU(cudaMemcpyAsync(doff, offsets, sizeof(int32_t) * ((size_t)n_pairs + 1), cudaMemcpyHostToDevice, cs));
  CU(cudaEventRecord(g_c.ev_feed, cs));
  CU(cudaStreamWaitEvent(st, g_c.ev_feed, 0));
  CU(cudaEventRecord(g_c.ev0, st));
  rc = launch<KIND>(j, st, g_c.ready, g_c.ready + 1, wait_cycles);
  if (rc) return rc;
  CU(cudaEventRecord(g_c.ev1, st));
  auto row_of = [&](int pair) -> size_t { return offsets ? (size_t)offsets[pair] : (size_t)pair * n; };
  int done = 0;
  for (int ci = 0; ci < nchunks && done < n_pairs; ++ci) {
    int cnt = (ci == 0) ? first : per;
    if (done + cnt > n_pairs) cnt = n_pairs - done;
    const size_t off = row_of(done) * dim;
    const size_t elems = (row_of(done + cnt) - row_of(done)) * dim;
    const cudaError_t e1 = cudaMemcpyAsync(d1 + off, h.x1y1 + off, sizeof(double) * elems, cudaMemcpyHostToDevice, cs);
    const cudaError_t e2 = (KIND == 2) ? cudaSuccess   // one array of u10 rows
                                       : cudaMemcpyAsync(d2 + off, h.x2y2 + off, sizeof(double) * elems, cudaMemcpyHostToDevice, cs);
    done += cnt;
    g_c.h_ready[ci] = (e1 == cudaSuccess && e2 == cudaSuccess) ? done : n_pairs + 1;   // on a failed copy release the CTAs anyway
    cudaMemcpyAsync(g_c.ready, &g_c.h_ready[ci], sizeof(int), cudaMemcpyHostToDevice, cs);
    if (e1 != cudaSuccess || e2 != cudaSuccess) {
      cudaStreamSynchronize(cs); cudaStreamSynchronize(st);
      return fail(DGB200_E_CUDA, "input copy failed", e1 != cudaSuccess ? e1 : e2);
    }
  }
  int h_status[4] = {0, 0, 0, 0};
  CU(cudaMemcpyAsync(h_status, g_c.ready, sizeof(h_status), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(cs));
  CU(cudaStreamSynchronize(st));
  if (h_status[1] != 0) {
    // The feed could not overlap the kernel and some CTAs stopped taking pairs.  Everything has landed by now: run
    // the pairs from the first abandoned index on in an ordinary launch (pairs before it were completed -- a CTA only
    // abandons the pair it was about to START; pairs it had in flight are finished before it exits).
    int from = h_status[2];
    if (from < 0) from = 0;
    if (from < n_pairs) {
      Job r = j;
      r.n_pairs = n_pairs - from;
      r.seeds = h.seeds ? dseed + from : nullptr;
      r.model_out = dmodel + (size_t)9 * from;
      r.stats_out = dstats + (size_t)4 * from;
      if (offsets) {
        // ragged: re-base the offsets of the remaining pairs (host copy, tiny)
        std::vector<int32_t> rebased((size_t)r.n_pairs + 1);
        for (int q = 0; q <= r.n_pairs; ++q) rebased[q] = offsets[from + q] - offsets[from];
        CU(cudaMemcpyAsync(doff, rebased.data(), sizeof(int32_t) * rebased.size(), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
      }
      const size_t off = row_of(from);
      r.x1y1 = d1 + off * dim; r.x2y2 = d2 + off * dim; r.mask_out = dmask + off;
      rc = launch<KIND>(r, st);
      if (rc) return rc;
      CU(cudaEventRecord(g_c.ev1, st));
    }
  }
  CU(cudaMemcpyAsync(h.model_out, dmodel, sizeof(double) * 9 * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(h.mask_out, dmask, (size_t)rows, cudaMemcpyDeviceToHost, st));
  if (h.stats_out) CU(cudaMemcpyAsync(h.stats_out, dstats, sizeof(int) * 4 * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0.f;
  CU(cudaEventElapsedTime(&ms, g_c.ev0, g_c.ev1));
  g_last_ms = ms;
  return 0;
}

template <int KIND>
int run_dev(const Job& j, void* stream) {   // j: a batch in device memory
  std::lock_guard<std::mutex> lk(g_mu);
  int rc = check_args(KIND, j.x1y1, j.x2y2, j.n_pairs, j.n, j.dim, j.metric, j.laf_coef, j.model_out, j.mask_out);
  if (rc) return rc;
  rc = ensure_device();
  if (rc) return rc;
  return launch<KIND>(j, (cudaStream_t)stream);
}

}  // namespace

extern "C" {

int dgb200_find_fundamental_batch_ex(const double* x1y1, const double* x2y2, int n_pairs, int n, int dim, double px_th,
                                     double conf, int max_iters, int error_type, int sym_check, double laf_coef,
                                     int degen_check, const uint64_t* seeds, double* F_out, uint8_t* mask_out,
                                     int32_t* stats_out, unsigned flags) {
  Job j;
  j.x1y1 = x1y1; j.x2y2 = x2y2; j.n_pairs = n_pairs; j.n = n; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = seeds;
  j.model_out = F_out; j.mask_out = mask_out; j.stats_out = stats_out;
  j.degen = degen_check; j.flags = flags;
  return run_host<0>(j);
}
int dgb200_find_homography_batch_ex(const double* x1y1, const double* x2y2, int n_pairs, int n, int dim, double px_th,
                                    double conf, int max_iters, int error_type, int sym_check, double laf_coef,
                                    const uint64_t* seeds, double* H_out, uint8_t* mask_out, int32_t* stats_out,
                                    unsigned flags) {
  Job j;
  j.x1y1 = x1y1; j.x2y2 = x2y2; j.n_pairs = n_pairs; j.n = n; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = seeds;
  j.model_out = H_out; j.mask_out = mask_out; j.stats_out = stats_out;
  j.flags = flags;
  return run_host<1>(j);
}
int dgb200_find_fundamental_batch(const double* x1y1, const double* x2y2, int n_pairs, int n, int dim, double px_th,
                                  double conf, int max_iters, int error_type, int sym_check, double laf_coef,
                                  int degen_check, const uint64_t* seeds, double* F_out, uint8_t* mask_out,
                                  int32_t* stats_out) {
  return dgb200_find_fundamental_batch_ex(x1y1, x2y2, n_pairs, n, dim, px_th, conf, max_iters, error_type, sym_check,
                                          laf_coef, degen_check, seeds, F_out, mask_out, stats_out, 0);
}
int dgb200_find_homography_batch(const double* x1y1, const double* x2y2, int n_pairs, int n, int dim, double px_th,
                                 double conf, int max_iters, int error_type, int sym_check, double laf_coef,
                                 const uint64_t* seeds, double* H_out, uint8_t* mask_out, int32_t* stats_out) {
  return dgb200_find_homography_batch_ex(x1y1, x2y2, n_pairs, n, dim, px_th, conf, max_iters, error_type, sym_check,
                                         laf_coef, seeds, H_out, mask_out, stats_out, 0);
}
int dgb200_find_fundamental_batch_dev_ex(const double* d_x1y1, const double* d_x2y2, int n_pairs, int n, int dim,
                                         double px_th, double conf, int max_iters, int error_type, int sym_check,
                                         double laf_coef, int degen_check, const uint64_t* d_seeds, double* d_F_out,
                                         uint8_t* d_mask_out, int32_t* d_stats_out, void* stream, unsigned flags) {
  Job j;
  j.x1y1 = d_x1y1; j.x2y2 = d_x2y2; j.n_pairs = n_pairs; j.n = n; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = d_seeds;
  j.model_out = d_F_out; j.mask_out = d_mask_out; j.stats_out = d_stats_out;
  j.degen = degen_check; j.flags = flags;
  return run_dev<0>(j, stream);
}
int dgb200_find_homography_batch_dev_ex(const double* d_x1y1, const double* d_x2y2, int n_pairs, int n, int dim,
                                        double px_th, double conf, int max_iters, int error_type, int sym_check,
                                        double laf_coef, const uint64_t* d_seeds, double* d_H_out, uint8_t* d_mask_out,
                                        int32_t* d_stats_out, void* stream, unsigned flags) {
  Job j;
  j.x1y1 = d_x1y1; j.x2y2 = d_x2y2; j.n_pairs = n_pairs; j.n = n; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = d_seeds;
  j.model_out = d_H_out; j.mask_out = d_mask_out; j.stats_out = d_stats_out;
  j.flags = flags;
  return run_dev<1>(j, stream);
}
int dgb200_find_fundamental_batch_dev(const double* d_x1y1, const double* d_x2y2, int n_pairs, int n, int dim,
                                      double px_th, double conf, int max_iters, int error_type, int sym_check,
                                      double laf_coef, int degen_check, const uint64_t* d_seeds, double* d_F_out,
                                      uint8_t* d_mask_out, int32_t* d_stats_out, void* stream) {
  return dgb200_find_fundamental_batch_dev_ex(d_x1y1, d_x2y2, n_pairs, n, dim, px_th, conf, max_iters, error_type,
                                              sym_check, laf_coef, degen_check, d_seeds, d_F_out, d_mask_out,
                                              d_stats_out, stream, 0);
}
int dgb200_find_homography_batch_dev(const double* d_x1y1, const double* d_x2y2, int n_pairs, int n, int dim,
                                     double px_th, double conf, int max_iters, int error_type, int sym_check,
                                     double laf_coef, const uint64_t* d_seeds, double* d_H_out, uint8_t* d_mask_out,
                                     int32_t* d_stats_out, void* stream) {
  return dgb200_find_homography_batch_dev_ex(d_x1y1, d_x2y2, n_pairs, n, dim, px_th, conf, max_iters, error_type,
                                             sym_check, laf_coef, d_seeds, d_H_out, d_mask_out, d_stats_out, stream, 0);
}
int dgb200_find_fundamental_ragged(const double* x1y1, const double* x2y2, const int32_t* offsets, int n_pairs, int dim,
                                   double px_th, double conf, int max_iters, int error_type, int sym_check,
                                   double laf_coef, int degen_check, const uint64_t* seeds, double* F_out,
                                   uint8_t* mask_out, int32_t* stats_out) {
  Job j;
  j.x1y1 = x1y1; j.x2y2 = x2y2; j.n_pairs = n_pairs; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = seeds;
  j.model_out = F_out; j.mask_out = mask_out; j.stats_out = stats_out;
  j.offsets = offsets; j.degen = degen_check;
  return run_host<0>(j);
}
int dgb200_find_homography_ragged(const double* x1y1, const double* x2y2, const int32_t* offsets, int n_pairs, int dim,
                                  double px_th, double conf, int max_iters, int error_type, int sym_check,
                                  double laf_coef, const uint64_t* seeds, double* H_out, uint8_t* mask_out,
                                  int32_t* stats_out) {
  Job j;
  j.x1y1 = x1y1; j.x2y2 = x2y2; j.n_pairs = n_pairs; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = seeds;
  j.model_out = H_out; j.mask_out = mask_out; j.stats_out = stats_out;
  j.offsets = offsets;
  return run_host<1>(j);
}
int dgb200_find_fundamental_ragged_dev(const double* d_x1y1, const double* d_x2y2, const int32_t* d_offsets, int n_pairs,
                                       int n_max, int dim, double px_th, double conf, int max_iters, int error_type,
                                       int sym_check, double laf_coef, int degen_check, const uint64_t* d_seeds,
                                       double* d_F_out, uint8_t* d_mask_out, int32_t* d_stats_out, void* stream) {
  if (!d_offsets) return fail(DGB200_E_ARG, "null offsets");
  Job j;
  j.x1y1 = d_x1y1; j.x2y2 = d_x2y2; j.n_pairs = n_pairs; j.n = n_max; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = d_seeds;
  j.model_out = d_F_out; j.mask_out = d_mask_out; j.stats_out = d_stats_out;
  j.offsets = d_offsets; j.degen = degen_check;
  return run_dev<0>(j, stream);
}
int dgb200_find_homography_ragged_dev(const double* d_x1y1, const double* d_x2y2, const int32_t* d_offsets, int n_pairs,
                                      int n_max, int dim, double px_th, double conf, int max_iters, int error_type,
                                      int sym_check, double laf_coef, const uint64_t* d_seeds, double* d_H_out,
                                      uint8_t* d_mask_out, int32_t* d_stats_out, void* stream) {
  if (!d_offsets) return fail(DGB200_E_ARG, "null offsets");
  Job j;
  j.x1y1 = d_x1y1; j.x2y2 = d_x2y2; j.n_pairs = n_pairs; j.n = n_max; j.dim = dim; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.metric = error_type; j.sym_check = sym_check; j.laf_coef = laf_coef; j.seeds = d_seeds;
  j.model_out = d_H_out; j.mask_out = d_mask_out; j.stats_out = d_stats_out;
  j.offsets = d_offsets;
  return run_dev<1>(j, stream);
}
int dgb200_find_fundamental(const double* x1y1, const double* x2y2, int n, int dim, double px_th, double conf,
                            int max_iters, int error_type, int sym_check, double laf_coef, int degen_check,
                            uint64_t seed, double* F_out, uint8_t* mask_out, int32_t* stats_out) {
  return dgb200_find_fundamental_batch(x1y1, x2y2, 1, n, dim, px_th, conf, max_iters, error_type, sym_check, laf_coef,
                                       degen_check, &seed, F_out, mask_out, stats_out);
}
int dgb200_find_homography(const double* x1y1, const double* x2y2, int n, int dim, double px_th, double conf,
                           int max_iters, int error_type, int sym_check, double laf_coef, uint64_t seed, double* H_out,
                           uint8_t* mask_out, int32_t* stats_out) {
  return dgb200_find_homography_batch(x1y1, x2y2, 1, n, dim, px_th, conf, max_iters, error_type, sym_check, laf_coef,
                                      &seed, H_out, mask_out, stats_out);
}

// u10 rows (x', y', a', b', c', x, y, a, b, c): both halves of a correspondence come from the one array
int dgb200_find_homography_2el_batch(const double* u10, int n_pairs, int n, double px_th, double conf, int max_iters,
                                     const uint64_t* seeds, double* H_out, uint8_t* mask_out, int32_t* stats_out) {
  Job j;
  j.x1y1 = u10; j.x2y2 = u10; j.n_pairs = n_pairs; j.n = n; j.dim = 10; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.seeds = seeds; j.model_out = H_out; j.mask_out = mask_out; j.stats_out = stats_out;
  return run_host<2>(j);
}
int dgb200_find_homography_2el_batch_dev(const double* d_u10, int n_pairs, int n, double px_th, double conf,
                                         int max_iters, const uint64_t* d_seeds, double* d_H_out, uint8_t* d_mask_out,
                                         int32_t* d_stats_out, void* stream) {
  Job j;
  j.x1y1 = d_u10; j.x2y2 = d_u10; j.n_pairs = n_pairs; j.n = n; j.dim = 10; j.px_th = px_th; j.conf = conf;
  j.max_iters = max_iters; j.seeds = d_seeds; j.model_out = d_H_out; j.mask_out = d_mask_out; j.stats_out = d_stats_out;
  return run_dev<2>(j, stream);
}

int dgb200_version(void) { return 2; }
int dgb200_device_count(void) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) return -1;
  return cnt;
}
int dgb200_set_device(int device) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_c.device >= 0 && g_c.device != device) {
    cudaSetDevice(g_c.device);      // free the old device's state with that device current
    cudaDeviceSynchronize();
    destroy_device_state();
  }
  CU(cudaSetDevice(device));
  return 0;
}
const char* dgb200_last_error(void) { return g_err; }
long long dgb200_kernel_launches(void) { return g_launches; }
double dgb200_last_kernel_ms(void) { return g_last_ms; }
#ifdef DG_PROF
void dgb200_prof_read(unsigned long long* out, int reset) {
  cudaMemcpyFromSymbol(out, g_dg_prof, sizeof(unsigned long long) * 64);
  if (reset) { unsigned long long z[64] = {0}; cudaMemcpyToSymbol(g_dg_prof, z, sizeof(z)); }
}
#endif
void dgb200_release(void) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_c.device < 0) return;
  cudaSetDevice(g_c.device);
  cudaDeviceSynchronize();
  for (LaunchCtx& x : g_c.ctxs) {
    if (x.ws) cudaFree(x.ws);
    x.ws = nullptr; x.ws_bytes = 0;
  }
  if (g_c.io) cudaFree(g_c.io);
  g_c.io = nullptr; g_c.io_bytes = 0;
}

}  // extern "C"
