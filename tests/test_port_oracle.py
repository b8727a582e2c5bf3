"""Pins the plain-C restatement (oracle/port) against the golden vectors produced by the unmodified reference and
against the reference's recorded answers on randomised inputs."""
import json
import os

import numpy as np
import pytest

from tests.conftest import norm_model
from pydegensac_b200.scenes import scene_F, scene_H

HERE = os.path.dirname(os.path.abspath(__file__))
G = np.load(os.path.join(HERE, "golden", "golden_v1.npz"))
META = json.loads(str(G["meta"]))


@pytest.mark.parametrize("i", range(len(META)))
def test_port_matches_golden(i):
    from oracle import port
    m = META[i]
    if m["kind"] == "F":
        p1, p2, _ = scene_F(**m["scene"])
        M, mask, st = port.find_fundamental(p1, p2, **m["call"])
    else:
        p1, p2, _ = scene_H(**m["scene"])
        M, mask, st = port.find_homography_raw(p1, p2, **m["call"])
    gm = G["model_%d" % i]
    if np.abs(gm).sum() == 0:
        assert np.abs(M).sum() == 0
        return
    assert np.array_equal(mask, G["mask_%d" % i])
    assert np.linalg.norm(norm_model(M) - norm_model(gm)) < 1e-6
    assert list(st[:2]) == list(G["stats_%d" % i][:2])


def test_port_vs_reference_randomised(ref_oracle):
    from oracle import port
    rng = np.random.default_rng(99)
    for case in range(40):
        kind = rng.choice(["F", "H"])
        n = int(rng.choice([8, 12, 20, 50, 100, 300, 1000]))
        ratio = float(rng.choice([0.3, 0.5, 0.8, 1.0]))
        px = float(rng.choice([0.5, 1.0, 3.0])); conf = float(rng.choice([0.9, 0.99, 0.9999]))
        mi = int(rng.choice([50, 51, 100, 1000, 3000]))
        sym = bool(rng.integers(2)); seed = int(rng.integers(1 << 30)); sc = int(rng.integers(1000))
        if kind == "F":
            plane = float(rng.choice([0, 0, 0.5, 0.9])); et = int(rng.integers(2)); dg = bool(rng.integers(2))
            p1, p2, _ = scene_F(n, ratio, sc, plane)
            a = ref_oracle.find_fundamental(p1, p2, px, conf, mi, error_type=et, sym_check=sym, degen_check=dg, seed=seed)
            b = port.find_fundamental(p1, p2, px, conf, mi, error_type=et, sym_check=sym, degen_check=dg, seed=seed)
        else:
            et = int(rng.integers(5))
            p1, p2, _ = scene_H(n, int(n * ratio), sc)
            a = ref_oracle.find_homography_raw(p1, p2, px, conf, mi, error_type=et, sym_check=sym, seed=seed)
            if a[2][3] <= 4 or a[2][2] >= a[2][0]:   # no consensus / every sample rejected: reference runs on uninitialised memory
                continue
            b = port.find_homography_raw(p1, p2, px, conf, mi, error_type=et, sym_check=sym, seed=seed)
        if np.abs(a[0]).sum() == 0 and np.abs(b[0]).sum() == 0:
            continue
        assert np.array_equal(a[1], b[1]), "case %d %s" % (case, kind)
        assert np.linalg.norm(norm_model(a[0]) - norm_model(b[0])) < 1e-6


def test_port_laf_gate_matches_golden_laf():
    """The plain-C restatement reproduces the LAF-gate golden vectors (produced by the unmodified reference)."""
    import json
    import os
    from oracle import port
    from pydegensac_b200.scenes import scene_F_laf, scene_H_laf
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_laf_v1.npz"))
    meta = json.loads(str(G["meta"]))
    for i, m in enumerate(meta):
        p1, p2 = (scene_F_laf if m["kind"] == "F" else scene_H_laf)(**m["scene"])[:2]
        out = (port.find_fundamental if m["kind"] == "F" else port.find_homography_raw)(p1, p2, **m["call"])
        assert np.array_equal(out[1], G["mask_%d" % i].astype(bool)), "mask differs (LAF case %d)" % i
        assert np.linalg.norm(norm_model(out[0]) - norm_model(G["model_%d" % i])) < 1e-6
        assert int(out[2][0]) == int(G["stats_%d" % i][0]) and int(out[2][1]) == int(G["stats_%d" % i][1])
