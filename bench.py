#!/usr/bin/env python
"""bench.py -- image-pairs/sec of the B200 LO-RANSAC / DEGENSAC engine vs the reference on the host CPU.
One JSON line on stdout (rank 0).

    python bench.py --gpus 1 --steps 5 --warmup 3                       # headline: BASELINE config 2
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1      # the reference's own CPU path, same config
    python bench.py --config 3 | 4 | 5 | 1                              # the other BASELINE.json configs

Configs (BASELINE.json `configs`, SURVEY.md section 8(d)); a step = one pass of the hot path over one batch:
  2  findFundamentalMatrix, scene F(2000, 0.30, seed=s), px 1.0, conf 0.9999, 10k iters          (default, the metric)
  4  the same with a dominant plane (pi = 0.8): DEGENSAC's plane-and-parallax branch on every pair
  3  findHomography, 5000 correspondences (1500 inliers), px 3.0, conf 0.999, 10k iters
  5  config 2 as STRONG scaling: a fixed batch of 8192 pairs split over the N GPUs + the final gather
  1  single-call latency: findHomography on the frozen v_dogman tentatives (th 4.0, conf 0.99, 2000 iters),
     one call at a time through the public API; value = calls per second, config.ms_per_call the latency
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "image-pairs/sec (2000 corr, 10k iters) F-matrix"
CONFIGS = {
    2: dict(kind="F", n=2000, plane=0.0, px_th=1.0, conf=0.9999, max_iters=10000, pairs=16384, metric=METRIC,
            workload="findFundamentalMatrix batch: scene F(2000,0.30,seed=s) per pair, px_th 1.0, conf 0.9999, "
                     "max_iters 10000, sampson, sym check on, degeneracy check on",
            flop_per_pair=1.44e8),           # SURVEY.md section 8(d): 1 940 residual passes x 2000 x 37
    4: dict(kind="F", n=2000, plane=0.8, px_th=1.0, conf=0.9999, max_iters=10000, pairs=4096,
            metric="image-pairs/sec (2000 corr, 10k iters) F-matrix, dominant-plane scene",
            workload="findFundamentalMatrix batch: scene F(2000,0.30,seed=s,plane 0.8), px_th 1.0, conf 0.9999, "
                     "max_iters 10000, sampson, sym check on, degeneracy check on", flop_per_pair=None),
    3: dict(kind="H", n=5000, n_in=1500, px_th=3.0, conf=0.999, max_iters=10000, pairs=4096,
            metric="image-pairs/sec (5000 corr, 10k iters) homography",
            workload="findHomography batch: 5000 correspondences (1500 inliers, H_GT), px_th 3.0, conf 0.999, "
                     "max_iters 10000, sampson, sym check on, LO on", flop_per_pair=None),
    5: dict(kind="F", n=2000, plane=0.0, px_th=1.0, conf=0.9999, max_iters=10000, total_pairs=8192, metric=METRIC,
            workload="findFundamentalMatrix: FIXED batch of 8192 pairs (scene F(2000,0.30,seed=s)) sharded over the "
                     "GPUs, px_th 1.0, conf 0.9999, max_iters 10000, final gather of (F, stats, mask)",
            flop_per_pair=1.44e8),
    1: dict(kind="H1", n=811, px_th=4.0, conf=0.99, max_iters=2000, pairs=32,
            metric="findHomography calls/sec, one call at a time (v_dogman tentatives, 811 corr, 2000 iters)",
            workload="pydegensac.findHomography(src, dst, 4.0, 0.99, 2000) on tests/golden/dogman_v1.npz, sequential "
                     "single calls", flop_per_pair=None),
}


def algo_bytes(cfg):
    """SURVEY.md section 8(d): one read of the pair (x1,y1,x2,y2 FP64) + F/H (72 B) + mask (N B) + stats (16 B)."""
    return cfg["n"] * 4 * 8 + 72 + cfg["n"] + 16


def gen_batch(cfg, n_pairs, seed0):
    from pydegensac_b200.scenes import batch_F, scene_H
    if cfg["kind"] == "F":
        return batch_F(n_pairs, cfg["n"], 0.30, seed0, cfg["plane"])
    p1 = np.empty((n_pairs, cfg["n"], 2)); p2 = np.empty((n_pairs, cfg["n"], 2))
    for i in range(n_pairs):
        a, b, _ = scene_H(cfg["n"], cfg["n_in"], seed0 + i)
        p1[i], p2[i] = a, b
    return p1, p2


def dogman():
    d = np.load(os.path.join(ROOT, "tests", "golden", "dogman_v1.npz"))
    return np.ascontiguousarray(d["src"], dtype=np.float64), np.ascontiguousarray(d["dst"], dtype=np.float64)


DUMP_MASK_BYTES = 48 << 20


def dump_outputs(dirname, model, mask, stats=None):
    """Writes what a caller of the timed path receives for its last step, as DIR/<name>.npy, so that two builds can be
    compared output for output: every pair's model (and stats), its inlier count, and the inlier masks of a fixed,
    seeded sample of pairs (all of them when they fit in DUMP_MASK_BYTES as float32)."""
    os.makedirs(dirname, exist_ok=True)
    P, N = mask.shape
    k = min(P, DUMP_MASK_BYTES // (4 * N))
    rows = np.arange(P) if k == P else np.sort(np.random.default_rng(0).choice(P, k, replace=False))
    out = {"model": model.reshape(P, 3, 3).astype(np.float64), "inliers": mask.sum(1).astype(np.float64),
           "mask": mask[rows].astype(np.float32), "mask_rows": rows.astype(np.float64)}
    if stats is not None:
        out["stats"] = stats.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


# ----------------------------------------------------------------------------- CPU reference arm
def _cpu_worker(args):
    cfg_id, seed0, count = args
    cfg = CONFIGS[cfg_id]
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    from oracle import ref
    if cfg["kind"] == "H1":
        src, dst = dogman()
        ref.find_homography_raw(src, dst, cfg["px_th"], cfg["conf"], 100, seed=1, rng=ref.RNG_GLIBC)
        t = time.perf_counter()
        for i in range(count):
            ref.find_homography(src, dst, cfg["px_th"], cfg["conf"], cfg["max_iters"], seed=seed0 + i, rng=ref.RNG_GLIBC)
        return time.perf_counter() - t, 0
    p1, p2 = gen_batch(cfg, count, seed0)
    if cfg["kind"] == "F":
        ref.find_fundamental(p1[0], p2[0], cfg["px_th"], cfg["conf"], 100, seed=1, rng=ref.RNG_GLIBC)   # load / warm
    else:
        ref.find_homography_raw(p1[0], p2[0], cfg["px_th"], cfg["conf"], 100, seed=1, rng=ref.RNG_GLIBC)
    t = time.perf_counter()
    inl = 0
    for i in range(count):
        if cfg["kind"] == "F":
            F, m, st = ref.find_fundamental(p1[i], p2[i], cfg["px_th"], cfg["conf"], cfg["max_iters"], degen_check=True,
                                            seed=seed0 + i, rng=ref.RNG_GLIBC)
        else:
            F, m, st = ref.find_homography_raw(p1[i], p2[i], cfg["px_th"], cfg["conf"], cfg["max_iters"], seed=seed0 + i,
                                               rng=ref.RNG_GLIBC)
        inl += int(m.sum())
    return time.perf_counter() - t, inl


def cpu_reference_rate(cfg_id, pairs_per_proc, procs, seed0=100000):
    """Unmodified reference (oracle/_ref, its own glibc RNG) on `procs` processes, one per core (the library is not
    thread-safe: global hash table + libc RNG).  Returns (pairs/s over the pool, single-process pairs/s, wall s)."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    jobs = [(cfg_id, seed0 + i * pairs_per_proc, pairs_per_proc) for i in range(procs)]
    with ctx.Pool(procs) as pool:
        pool.map(_cpu_worker, [(cfg_id, seed0, 1)] * procs)          # spawn + import + warm-up, untimed
        t = time.perf_counter()
        res = pool.map(_cpu_worker, jobs, chunksize=1)
        wall = time.perf_counter() - t
    busy = [r[0] for r in res]
    total = pairs_per_proc * procs
    return total / max(max(busy), 1e-9), pairs_per_proc / (sum(busy) / len(busy)), wall


def host_cores():
    """Cores this process may actually use: CPU affinity capped by the cgroup CPU quota (a container that sees
    128 logical CPUs but has cpu.max = 16 CPUs gets 16 worker processes, not 128 oversubscribed ones)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return n


def cpu_pairs_per_core(cfg_id, args):
    """Bounded sample: ~10-30 s of CPU work per step whatever the config (a config-2 pair costs ~45 ms of one core,
    a dominant-plane pair ~190 ms, a 5000-point homography ~25 ms, a dogman call ~12 ms)."""
    if args.cpu_pairs_per_core > 0:
        return args.cpu_pairs_per_core
    return {2: 16, 5: 16, 4: 6, 3: 32, 1: 64}[cfg_id]


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref
    cfg = CONFIGS[args.config]
    cores = host_cores()
    if not ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libdegensac_ref.so not built"}))
        return
    procs = 1 if cfg["kind"] == "H1" else cores      # single-call latency is a one-core measurement
    per = cpu_pairs_per_core(args.config, args)
    vals = []
    for s in range(args.warmup + args.steps):
        rate, single, wall = cpu_reference_rate(args.config, per, procs, seed0=100000 + s * per * procs)
        if s >= args.warmup:
            vals.append((rate, single, wall))
    rate = float(np.mean([v[0] for v in vals]))
    single = float(np.mean([v[1] for v in vals]))
    ms = float(np.mean([v[2] for v in vals])) * 1e3
    conf = {"workload": cfg["workload"], "config_id": args.config, "pairs_per_step": per * procs}
    if cfg["kind"] == "H1":
        conf["ms_per_call"] = 1e3 / rate
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": rate, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if args.config == 5 else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic" if cfg["kind"] != "H1" else "frozen AKAZE tentatives (tests/golden)",
        "config": conf,
        "cpu_baseline": {"value": rate, "unit": "pairs/s", "cores": procs, "kind": "reference",
                         "sample": "%d pairs per process x %d processes (one per core), unmodified reference C core "
                                   "with its own glibc RNG; single-process rate %.1f pairs/s" % (per, procs, single)},
        "e2e": {"value": rate, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in o.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nme, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.2)


def rooflines(cfg, P, kernel_ms):
    """Structured roofline objects of the dominant kernel: the HBM one the contract asks for (irrelevant by design:
    the pair is read once and re-used ~2-25k times on chip) and the FP64 one that actually bounds the path."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    achieved = algo_bytes(cfg) * P / (kernel_ms / 1e3) / 1e9
    traffic = None
    cid = [k for k, v in CONFIGS.items() if v is cfg][0]
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if cid in (2, 5) and os.path.exists(tf):      # dram bytes per pair from the committed ncu capture of config 2
        try:
            traffic = json.load(open(tf)).get("per_pair_bytes") * P
        except Exception:
            traffic = None
    hbm = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
           "traffic": traffic, "peak_source": peak_src,
           "kernel": "ransac_pairs_kernel<%s>" % ("F" if cfg["kind"] == "F" else "H"), "kernel_ms": kernel_ms,
           "algorithmic_bytes_per_pair": algo_bytes(cfg),
           "note": "the path is FP64-issue / latency bound, not HBM bound (SURVEY.md section 8(d)): see roofline_fp64"}
    fp64 = None
    if cfg.get("flop_per_pair"):
        try:
            pk = json.load(open(os.path.join(ROOT, "profiles", "fp64_peak.json")))
            flops = cfg["flop_per_pair"] * P / (kernel_ms / 1e3) / 1e12
            fp64 = {"bound": "fp64", "achieved": flops, "unit": "TFLOP/s",
                    "peak": pk["dmul_dadd_tflops"], "frac": flops / pk["dmul_dadd_tflops"],
                    "peak_dfma": pk["dfma_tflops"], "frac_of_dfma_peak": flops / pk["dfma_tflops"],
                    "peak_source": "measured on this pool's B200 (tools/fp64_peak.cu -> profiles/fp64_peak.json): "
                                   "DMUL+DADD pairs, the ceiling of a -fmad=false build; DFMA peak beside it",
                    "work": "reference-equivalent FP64 work: %.3g flop per pair (SURVEY.md section 8(d): the O(N) "
                            "residual passes the reference itself executes)" % cfg["flop_per_pair"]}
        except Exception:
            fp64 = None
    return hbm, fp64


def run_gpu_arm(args):
    import torch
    from pydegensac_b200 import _cabi
    from pydegensac_b200.parallel import ShardedBatch, pin_to_gpu_numa
    import pydegensac_b200 as pdg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    numa_cpus = pin_to_gpu_numa(local_rank) if world > 1 else 0      # pinned-memory copies stay on the GPU's socket
    _cabi.lib().dgb200_set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    cfg = CONFIGS[args.config]
    if cfg["kind"] == "H1":
        return run_latency(args, cfg, dev, rank)

    if args.config == 5:
        P = cfg["total_pairs"] // world
        scaling = "strong"
    else:
        P = args.pairs_per_gpu if args.pairs_per_gpu > 0 else cfg["pairs"]
        scaling = "weak"
    N = cfg["n"]
    kind = "F" if cfg["kind"] == "F" else "H"
    p1, p2 = gen_batch(cfg, P, seed0=rank * P)
    seeds = (np.arange(P, dtype=np.uint64) + np.uint64(rank * P))
    params = dict(px_th=cfg["px_th"], conf=cfg["conf"], max_iters=cfg["max_iters"], degen=True)
    sb = ShardedBatch(kind, P, N, 2, params, dev, dist)
    hp1 = torch.from_numpy(p1).pin_memory()
    hp2 = torch.from_numpy(p2).pin_memory()
    hseed = torch.from_numpy(seeds.view(np.int64).copy()).pin_memory()
    sb.d1.copy_(hp1); sb.d2.copy_(hp2); sb.dseed.copy_(hseed)          # device-resident inputs for `value`
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    stream = torch.cuda.current_stream()

    def step_device():
        sb.launch(stream.cuda_stream)
        if world > 1:
            sb.gather()                     # the path's only collective: records of all ranks on rank 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = _cabi.kernel_launches()
    times = []
    barrier()
    for _ in range(args.steps):
        flush.fill_(1)                       # evict L2 between timed iterations (not timed)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step_device()
        e1.record(stream)
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    barrier()
    launches = _cabi.kernel_launches() - launches0
    dumped = None
    if args.dump_outputs and rank == 0:     # the last timed step's results, before the legs below run the batch again
        if world > 1:
            from pydegensac_b200.parallel import unpack_records
            dumped = unpack_records(sb.gathered.view(world * P, sb.stride).cpu().numpy())
        else:
            dumped = (sb.model.cpu().numpy(), sb.mask.cpu().numpy().astype(bool), sb.stats.cpu().numpy())
    sampler.stop_flag = True        # (its nvidia-smi forks would perturb the host-side e2e leg below)
    sampler.join(2.0)
    total_ms = float(sum(times))
    tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    value = world * P * args.steps / (total_ms / 1e3)
    # kernel-only time of the dominant (only) kernel, rank 0: events around the launch alone
    kt = []
    for _ in range(max(3, args.steps)):
        flush.fill_(1)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        sb.launch(stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        kt.append(e0.elapsed_time(e1))
    kernel_ms = float(np.mean(kt))

    # e2e: HOST buffers in, records out, copies inside the timed region.
    #   1 GPU : the public batched API (pydegensac_b200.find*Batch) with pinned host arrays
    #   N GPUs: pydegensac_b200.parallel.ShardedBatch.step -- each rank's H2D + kernel + ONE gather, rank 0 D2H
    hn1, hn2 = hp1.numpy(), hp2.numpy()
    api = pdg.findFundamentalMatrixBatch if kind == "F" else pdg.findHomographyBatch
    if world == 1:
        api(hn1, hn2, cfg["px_th"], cfg["conf"], cfg["max_iters"], seeds=seeds)    # untimed warm-up step (sizes the staging buffers)
    else:
        sb.step(hp1, hp2, hseed)
    barrier()
    t0 = time.perf_counter()
    mean_inl = None
    for _ in range(args.steps):
        if world == 1:
            M_h, mask_h = api(hn1, hn2, cfg["px_th"], cfg["conf"], cfg["max_iters"], seeds=seeds)
        else:
            rec = sb.step(hp1, hp2, hseed)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * P * args.steps / float(te.item())

    # the gathered records are what a caller gets: rank 0 recomputes a sample of every rank's block and compares
    gather_check = None
    if world > 1:
        if rank == 0:
            from pydegensac_b200.parallel import unpack_records
            gather_check = True
            for r in range(world):
                q1, q2 = gen_batch(cfg, 2, seed0=r * P)
                sd = np.arange(2, dtype=np.uint64) + np.uint64(r * P)
                if kind == "F":
                    Mr, mr, sr = _cabi.fundamental_batch(q1, q2, cfg["px_th"], cfg["conf"], cfg["max_iters"], 0, True, 0.0, True, sd)
                else:
                    Mr, mr, sr = _cabi.homography_batch(q1, q2, cfg["px_th"], cfg["conf"], cfg["max_iters"], 0, True, 0.0, sd)
                Mg, mg, sg = unpack_records(rec[r * P:r * P + 2])
                gather_check = gather_check and bool(np.array_equal(Mg, Mr) and np.array_equal(mg, mr) and np.array_equal(sg, sr))
            mean_inl = float(rec[:, 88:].sum(1).mean())
    else:
        mean_inl = float(mask_h.sum(1).mean())

    if rank == 0:
        hbm, fp64 = rooflines(cfg, P, kernel_ms)
        cpu = None
        if not args.no_cpu_baseline:
            try:
                from oracle import ref
                if ref.available():
                    # timed in a FRESH interpreter (the reference arm with one step): forking 16 workers out of
                    # this process -- CUDA context, pinned staging buffers, sampler thread -- halves their speed
                    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--gpus", "1",
                                          "--steps", "1", "--warmup", "1", "--config", str(args.config),
                                          "--cpu-pairs-per-core", str(args.cpu_pairs_per_core)],
                                         capture_output=True, text=True, timeout=900,
                                         env={k: v for k, v in os.environ.items()
                                              if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")})
                    ref_line = json.loads(out.stdout.strip().splitlines()[-1])
                    cpu = ref_line["cpu_baseline"]
                    cpu["sample"] += " (separate process, 1 timed step after 1 warm-up step)"
            except Exception as ex:  # pragma: no cover
                cpu = {"value": None, "unit": "pairs/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
        sm = sorted(sampler.samples)
        stride = 72 + 16 + N
        line = {
            "metric": cfg["metric"], "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "config_id": args.config,
                       "pairs_per_gpu": P, "global_pairs": world * P,
                       "parallelism": "pairs sharded x%d, one final gather of (model, stats, mask) records" % world,
                       "l2": "256 MB flush write between timed iterations", "mean_inliers": mean_inl,
                       "numa_pinned_cpus": numa_cpus, "gathered_records_verified": gather_check},
            "e2e": {"value": e2e_value, "unit": "pairs/s",
                    "h2d_bytes_per_step": int(world * (2 * P * N * 2 * 8 + P * 8)),
                    "d2h_bytes_per_step": int(world * P * stride) if world > 1 else int(P * (72 + N + 16)),
                    "api": "pydegensac_b200.find%sBatch (host arrays)" % ("FundamentalMatrix" if kind == "F" else "Homography")
                           if world == 1 else "pydegensac_b200.parallel.ShardedBatch.step (pinned host blocks -> records on rank 0)"},
            "gpu_launches": int(launches),
            "roofline": hbm,
            "roofline_fp64": fp64,
            "cpu_baseline": cpu,
            "clocks": {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": sampler.max_mhz,
                       "reasons": sorted(sampler.reasons)},
        }
        print(json.dumps(line))
        if dumped is not None:
            dump_outputs(args.dump_outputs, *dumped)
    if world > 1:
        dist.destroy_process_group()


def run_latency(args, cfg, dev, rank):
    """BASELINE config 1: one findHomography call at a time (what a pydegensac user does today)."""
    import torch
    import pydegensac_b200 as pdg
    from pydegensac_b200 import _cabi
    if rank != 0:
        return
    src, dst = dogman()
    calls = args.pairs_per_gpu if args.pairs_per_gpu > 0 else cfg["pairs"]
    for i in range(max(3, args.warmup)):
        pdg.findHomography(src, dst, cfg["px_th"], cfg["conf"], cfg["max_iters"], seed=i)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    launches0 = _cabi.kernel_launches()
    t0 = time.perf_counter()
    kms = []
    for s in range(args.steps):
        last = []
        for i in range(calls):
            H, mask = pdg.findHomography(src, dst, cfg["px_th"], cfg["conf"], cfg["max_iters"], seed=1000 + s * calls + i)
            kms.append(_cabi.last_kernel_ms())
            last.append((H, mask))
    wall = time.perf_counter() - t0
    launches = _cabi.kernel_launches() - launches0
    sampler.stop_flag = True
    n_calls = args.steps * calls
    e2e_rate = n_calls / wall
    kernel_ms = float(np.mean(kms))
    cpu = None
    if not args.no_cpu_baseline:
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--gpus", "1", "--steps", "1",
                                  "--warmup", "1", "--config", "1"], capture_output=True, text=True, timeout=600,
                                 env={k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")})
            ref_line = json.loads(out.stdout.strip().splitlines()[-1])
            cpu = ref_line["cpu_baseline"]
            cpu["ms_per_call"] = 1e3 / cpu["value"]
        except Exception as ex:  # pragma: no cover
            cpu = {"value": None, "unit": "pairs/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
    hbm, _ = rooflines(cfg, 1, kernel_ms)
    sm = sorted(sampler.samples)
    line = {"metric": cfg["metric"], "value": 1e3 / kernel_ms, "unit": "pairs/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "frozen AKAZE tentatives (tests/golden/dogman_v1.npz)",
            "config": {"workload": cfg["workload"], "config_id": 1, "calls_per_step": calls,
                       "ms_per_call_kernel": kernel_ms, "ms_per_call_e2e": 1e3 / e2e_rate, "mean_inliers": float(np.sum(mask))},
            "e2e": {"value": e2e_rate, "unit": "pairs/s", "h2d_bytes_per_step": int(calls * (2 * 811 * 2 * 8 + 8)),
                    "d2h_bytes_per_step": int(calls * (72 + 811 + 16)), "api": "pydegensac_b200.findHomography"},
            "gpu_launches": int(launches), "roofline": hbm, "roofline_fp64": None, "cpu_baseline": cpu,
            "clocks": {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": sampler.max_mhz, "reasons": sorted(sampler.reasons)}}
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, np.stack([h for h, _ in last]), np.stack([np.asarray(m, bool) for _, m in last]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--pairs-per-gpu", type=int, default=0, help="0 = the config's default")
    ap.add_argument("--cpu-pairs-per-core", type=int, default=0, help="0 = sized per config for ~10-30 s per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
