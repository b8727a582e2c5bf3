"""C-ABI surface and Python API validation layer (no GPU needed: no compute calls succeed here)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "pydegensac_b200", "libdegensac_b200.so")


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "degensac_b200.h")).read()
    return sorted(set(re.findall(r"\b(dgb200_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    if not os.path.exists(LIB):
        pytest.skip("libdegensac_b200.so not built (python -m pydegensac_b200.build)")
    lib = ctypes.CDLL(LIB)
    syms = _declared_symbols()
    assert len(syms) >= 12
    for s in syms:
        assert hasattr(lib, s), "missing export " + s
    assert lib.dgb200_version() == 2


def test_argument_errors_before_any_cuda_call():
    if not os.path.exists(LIB):
        pytest.skip("libdegensac_b200.so not built")
    from pydegensac_b200 import _cabi
    p = np.zeros((1, 5, 2))
    with pytest.raises(ValueError):   # F needs n >= 8 (bindings.cpp:270)
        _cabi.fundamental_batch(p, p, 1.0, 0.99, 10, 0, True, 0.0, True, None)
    p = np.zeros((1, 3, 2))
    with pytest.raises(ValueError):   # H needs n >= 4
        _cabi.homography_batch(p, p, 1.0, 0.99, 10, 0, True, 0.0, None)
    p = np.zeros((1, 10, 2))
    with pytest.raises(ValueError):   # unknown metric
        _cabi.homography_batch(p, p, 1.0, 0.99, 10, 7, True, 0.0, None)
    with pytest.raises(ValueError):   # LAF gate needs the [n,6] layout (homography too)
        _cabi.homography_batch(np.zeros((1, 10, 2)), np.zeros((1, 10, 2)), 1.0, 0.99, 10, 0, True, 3.0, None)
    with pytest.raises(ValueError):   # LAF gate needs the [n,6] layout
        _cabi.fundamental_batch(np.zeros((1, 10, 2)), np.zeros((1, 10, 2)), 1.0, 0.99, 10, 0, True, 3.0, True, None)


def test_no_cpu_fallback_without_gpu():
    """Without a CUDA device every compute entry point must fail loudly (checked in a child process that sees no
    device, so that it runs on GPU machines too)."""
    if not os.path.exists(LIB):
        pytest.skip("libdegensac_b200.so not built")
    code = """if True:
        import pytest, torch
        assert not torch.cuda.is_available()
        import pydegensac_b200 as pdg
        from pydegensac_b200.scenes import scene_F
        p1, p2, _ = scene_F(50, 0.5, 0)
        with pytest.raises(RuntimeError):
            pdg.findFundamentalMatrix(p1, p2, 1.0, 0.99, 100, seed=1)
        with pytest.raises(RuntimeError):
            pdg.findHomography(p1, p2, 1.0, 0.99, 100, seed=1)
        with pytest.raises(RuntimeError):
            pdg.findFundamentalMatrixBatch(p1[None], p2[None], 1.0, 0.99, 100)
    """
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]


def test_python_validation_matches_reference_layer():
    import pydegensac_b200 as pdg
    a = np.zeros((10, 2))
    with pytest.raises(ValueError):
        pdg.findHomography(np.zeros((10, 3)), np.zeros((10, 3)))
    with pytest.raises(ValueError):
        pdg.findHomography(np.zeros((3, 2)), np.zeros((3, 2)))
    with pytest.raises(ValueError):
        pdg.findHomography("nope", a)
    with pytest.raises(ValueError):
        pdg.findHomography(a, a, error_type="not_a_metric")
    with pytest.raises(ValueError):
        pdg.findFundamentalMatrix(a, a, error_type="symm_max")   # an H metric, not an F metric
    with pytest.raises(AssertionError):
        pdg.findFundamentalMatrix(np.zeros((10, 2)), np.zeros((11, 2)))
    assert pdg.error_type_dict_homography == {"sampson": 0, "symm_sq_max": 1, "symm_max": 2, "symm_sq_sum": 3, "symm_sum": 4}
    assert pdg.error_type_dict_fundamental == {"sampson": 0, "symm_epipolar": 1}


def test_convert_cv2_kpts():
    cv2 = pytest.importorskip("cv2")
    import pydegensac_b200 as pdg
    kps = [cv2.KeyPoint(10.0, 20.0, 4.0, 90.0), cv2.KeyPoint(1.5, 2.5, 2.0, 0.0)]
    out = pdg.convert_cv2_kpts_to_xyA(kps)
    assert out.shape == (2, 6)
    assert np.allclose(out[0], [10, 20, 0, 4, -4, 0], atol=1e-12)
    assert np.allclose(out[1], [1.5, 2.5, 2, 0, 0, 2], atol=1e-12)
