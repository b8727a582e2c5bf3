"""One-thread host emulation of the engine (same headers as the CUDA kernels) against the compiled reference on
seeded inputs: identical masks, models within 1e-6, same sample / LO counts.  CPU only."""
import numpy as np
import pytest

from tests.conftest import norm_model
from pydegensac_b200.scenes import scene_F, scene_H


def _cmp(a, b, what):
    if np.abs(a[0]).sum() == 0 and np.abs(b[0]).sum() == 0:
        return
    assert np.array_equal(a[1], b[1]), "mask differs: " + what
    assert np.linalg.norm(norm_model(a[0]) - norm_model(b[0])) < 1e-6, what
    assert a[2][0] == b[2][0] and a[2][1] == b[2][1], what


@pytest.mark.parametrize("plane", [0.0, 0.8])
@pytest.mark.parametrize("degen", [False, True])
def test_F_config2_and_4(ref_oracle, plane, degen):
    from tests.hostemu import emu
    p1, p2, _ = scene_F(2000, 0.3, 0, plane)
    for seed in range(3):
        a = ref_oracle.find_fundamental(p1, p2, 1.0, 0.9999, 10000, degen_check=degen, seed=seed)
        b = emu.find_fundamental(p1, p2, 1.0, 0.9999, 10000, degen_check=degen, seed=seed)
        _cmp(a, b, "F plane=%s degen=%s seed=%d" % (plane, degen, seed))
        assert b[2][2] == a[2][2]   # plane inlier count found by DEGENSAC


@pytest.mark.parametrize("et", range(5))
def test_H_config3_all_metrics(ref_oracle, et):
    from tests.hostemu import emu
    p1, p2, _ = scene_H()
    for seed in range(2):
        a = ref_oracle.find_homography_raw(p1, p2, 3.0, 0.999, 10000, error_type=et, seed=seed)
        b = emu.find_homography_raw(p1, p2, 3.0, 0.999, 10000, error_type=et, seed=seed)
        _cmp(a, b, "H metric=%d seed=%d" % (et, seed))


def test_randomised_configs(ref_oracle):
    """Ragged sizes, thresholds, confidence, tiny max_iters (ITER_SAM edge), gates on/off, chunk sizes."""
    from tests.hostemu import emu
    rng = np.random.default_rng(2024)
    for case in range(60):
        kind = rng.choice(["F", "H"])
        n = int(rng.choice([8, 9, 12, 20, 50, 100, 300, 1000]))
        ratio = float(rng.choice([0.1, 0.3, 0.5, 0.8, 1.0]))
        px = float(rng.choice([0.25, 0.5, 1.0, 3.0]))
        conf = float(rng.choice([0.9, 0.99, 0.9999]))
        mi = int(rng.choice([10, 49, 50, 51, 100, 1000, 3000]))
        sym = bool(rng.integers(2)); seed = int(rng.integers(1 << 30)); sc = int(rng.integers(1000))
        chunk = int(rng.choice([64, 512]))
        if kind == "F":
            plane = float(rng.choice([0, 0, 0.5, 0.9])); et = int(rng.integers(2)); dg = bool(rng.integers(2))
            p1, p2, _ = scene_F(n, ratio, sc, plane)
            a = ref_oracle.find_fundamental(p1, p2, px, conf, mi, error_type=et, sym_check=sym, degen_check=dg, seed=seed)
            b = emu.find_fundamental(p1, p2, px, conf, mi, error_type=et, sym_check=sym, degen_check=dg, seed=seed, chunk=chunk)
            if mi < 50 and dg and a[2][2] > 0:
                continue   # post-loop DEGENSAC branch reads a stale loop index in the reference (DESIGN.md, deviations)
        else:
            et = int(rng.integers(5))
            p1, p2, _ = scene_H(n, int(n * ratio), sc)
            a = ref_oracle.find_homography_raw(p1, p2, px, conf, mi, error_type=et, sym_check=sym, seed=seed)
            b = emu.find_homography_raw(p1, p2, px, conf, mi, error_type=et, sym_check=sym, seed=seed, chunk=chunk)
            if a[2][3] <= 4 or a[2][2] >= a[2][0] or np.abs(b[0]).sum() == 0:
                continue   # no consensus beyond the minimal sample / no valid hypothesis at all: the reference's
                #            post-loop LO then runs on uninitialised heap memory (exp_ranH.c:527, :794) and is not reproducible
        _cmp(a, b, "case %d %s n=%d" % (case, kind, n))


def test_leaves_against_reference_leaves(ref_oracle):
    """Known-answer checks of leaves against the reference's own exported C leaves (bit-exact where the arithmetic
    order is shared, tolerance where the algorithm differs)."""
    import ctypes
    from tests.hostemu import emu
    E = emu.lib()
    dp = ctypes.POINTER(ctypes.c_double)
    rng = np.random.default_rng(0)
    # Sampson residual of F: bit-exact
    E.emu_f_resid.restype = ctypes.c_double
    E.emu_f_resid.argtypes = [ctypes.c_int, dp] + [ctypes.c_double] * 4
    p1, p2, _ = scene_F(50, 0.5, 1)
    F = rng.normal(size=9)
    u = np.ones((50, 6)); u[:, 0:2] = p1; u[:, 3:5] = p2
    out = ref_oracle.fds(u, F)
    mine = np.array([E.emu_f_resid(0, F.ctypes.data_as(dp), *p1[i], *p2[i]) for i in range(50)])
    assert np.array_equal(out, mine)
    # 9x9 null space: bit-exact (same elimination order)
    E.emu_nullspace9.argtypes = [dp, dp]
    for _ in range(20):
        M = np.zeros((9, 9)); M[:7] = rng.normal(size=(7, 9)) * 100
        b = M.copy(); nb = np.zeros(81)
        ka, na = ref_oracle.nullspace(M)
        kb = E.emu_nullspace9(b.ctypes.data_as(dp), nb.ctypes.data_as(dp))
        assert ka == kb == 2 and np.array_equal(na[:18], nb[:18])
    # SuperFastHash of an index list: bit-exact
    E.emu_hash.argtypes = [ctypes.POINTER(ctypes.c_int), ctypes.c_int]; E.emu_hash.restype = ctypes.c_uint32
    for n in (1, 2, 7, 600):
        idx = np.sort(rng.choice(5000, n, replace=False)).astype(np.int32)
        assert ref_oracle.superfasthash(idx) == E.emu_hash(idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), n)
    # nsamples
    E.emu_nsamples.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double]
    for ni, n_, s, cf in [(600, 2000, 7, 0.9999), (1500, 5000, 4, 0.999), (8, 2000, 7, 0.99), (2000, 2000, 7, 0.9)]:
        assert ref_oracle.nsamples(ni, n_, s, cf) == E.emu_nsamples(ni, n_, s, cf)
    # third right singular vector in CCMATH's (unsorted) order: bit-exact
    E.emu_gkr_v3.argtypes = [dp, dp]
    for t in range(200):
        A = rng.normal(size=(3, 3))
        if t % 2 == 0:
            U, s, Vt = np.linalg.svd(A); s[2] = 0; A = (U * s) @ Vt
        A = np.ascontiguousarray(A)
        ve = np.zeros(3)
        E.emu_gkr_v3(A.ctypes.data_as(dp), ve.ctypes.data_as(dp))
        vr = ref_oracle.svd_v(A)[:, 2]
        assert min(np.abs(vr - ve).max(), np.abs(vr + ve).max()) == 0.0


def test_philox_stream_contract(ref_oracle):
    """The harness' restatement of the sampling stream and the engine's rng.h agree (value31 and the stateless sample)."""
    import ctypes
    from tests.hostemu import emu
    E = emu.lib()
    E.emu_value31.restype = ctypes.c_uint32
    E.emu_value31.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32]
    for seed in (0, 1, 2**40 + 17):
        for k in (0, 1, 50, 9999):
            for j in range(12):
                assert ref_oracle.value31(seed, k, j) == E.emu_value31(seed, k, j)
            for N, m in ((2000, 7), (5000, 4), (8, 7), (4, 4)):
                b = (ctypes.c_int * 8)()
                a = ref_oracle.stateless_sample(seed, k, N, m)
                E.emu_minimal_sample(ctypes.c_uint64(seed), k, N, m, b)
                assert list(a) == list(b)[:m]
                assert len(set(list(b)[:m])) == m


def test_F_laf_gate_vs_reference(ref_oracle):
    """LAF-consistency gate (laf_consistensy_coef > 0 with [N,6] inputs, SURVEY.md section 8(f).1): randomised scenes,
    emulation identical to the compiled reference; the gate must actually change at least one result."""
    from tests.hostemu import emu
    from pydegensac_b200.scenes import scene_F_laf
    rng = np.random.default_rng(5)
    checked = changed = 0
    for case in range(36):
        n = int(rng.choice([100, 300, 600, 1000])); ratio = float(rng.choice([0.4, 0.6, 0.8])); seed = int(rng.integers(1 << 20))
        jitter = float(rng.choice([0.2, 0.6, 1.5])); laf = float(rng.choice([0.5, 1.0, 2.0, 5.0])); et = int(rng.integers(2))
        sym = bool(rng.integers(2)); mi = int(rng.choice([200, 1000, 3000])); plane = float(rng.choice([0, 0, 0.6]))
        x1, x2, _ = scene_F_laf(n, ratio, seed, jitter, plane)
        a = ref_oracle.find_fundamental(x1, x2, 1.0, 0.999, mi, error_type=et, sym_check=sym, laf_coef=laf, degen_check=True, seed=seed)
        if a[2][3] <= 4 or a[2][2] >= a[2][0]:
            continue    # reference ran on uninitialised memory (no valid hypothesis): not comparable
        b = emu.find_fundamental(x1, x2, 1.0, 0.999, mi, et, sym, laf, True, seed)
        _cmp(a, b, "F LAF case %d (n=%d laf=%g metric=%d)" % (case, n, laf, et))
        a0 = ref_oracle.find_fundamental(x1, x2, 1.0, 0.999, mi, error_type=et, sym_check=sym, laf_coef=0.0, degen_check=True, seed=seed)
        changed += int(not np.array_equal(a[1], a0[1]))
        checked += 1
    assert checked >= 25
    assert changed >= 1, "the LAF gate never changed a result: the test scenes do not exercise it"


def test_H_laf_gate_vs_reference(ref_oracle):
    """LAF gate of the homography driver, all five metrics: the reference's quirks (Sampson variant mixing the main
    correspondence's linearised rows with the helper point's Jacobian, `p1_inliers` accumulating over the whole run,
    the final prune) must be reproduced for identical masks."""
    from tests.hostemu import emu
    from pydegensac_b200.scenes import scene_H_laf
    rng = np.random.default_rng(9)
    checked = changed = 0
    for case in range(40):
        n = int(rng.choice([100, 300, 800])); nin = int(n * float(rng.choice([0.4, 0.6, 0.8]))); seed = int(rng.integers(1 << 20))
        jitter = float(rng.choice([0.2, 0.6, 1.5])); laf = float(rng.choice([0.5, 1.0, 2.0, 5.0, 20.0])); et = int(rng.integers(5))
        sym = bool(rng.integers(2)); mi = int(rng.choice([200, 1000, 3000])); px = float(rng.choice([1.0, 3.0]))
        x1, x2, _ = scene_H_laf(n, nin, seed, jitter)
        a = ref_oracle.find_homography_raw(x1, x2, px, 0.999, mi, error_type=et, sym_check=sym, laf_coef=laf, seed=seed)
        b = emu.find_homography_raw(x1, x2, px, 0.999, mi, et, sym, laf, seed)
        _cmp(a, b, "H LAF case %d (n=%d laf=%g metric=%d)" % (case, n, laf, et))
        a0 = ref_oracle.find_homography_raw(x1, x2, px, 0.999, mi, error_type=et, sym_check=sym, laf_coef=0.0, seed=seed)
        changed += int(not np.array_equal(a[1], a0[1]))
        checked += 1
    assert changed >= 5, "the LAF gate hardly changed a result: the test scenes do not exercise it"
