"""ctypes loader for oracle/_ref/libdegensac_ref.so -- TEST INFRASTRUCTURE ONLY.

The shared object is the UNMODIFIED reference C core (compiled where it lies under
/root/reference by oracle/build_ref.sh) plus oracle/ref_harness.c, which interposes the
libc RNG so the reference can be driven by the engine's Philox sampling stream.
Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this.
"""
import ctypes
import hashlib
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_ref", "libdegensac_ref.so")
_SO_LSQ = os.path.join(_HERE, "_ref", "libdegensac_ref_lsq.so")   # the same sources compiled with -D__FINAL_LSQ__
_lib = None
_lib_lsq = None

RNG_GLIBC = 0   # reference's own rand()/random(), seeded from the (settable) time
RNG_PHILOX = 1  # replay of the engine's counter-based stream


def available():
    return os.path.exists(_SO)


def available_final_lsq():
    return os.path.exists(_SO_LSQ)


def lib(final_lsq=False):
    global _lib, _lib_lsq
    if final_lsq:
        if _lib_lsq is None:
            os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
            _lib_lsq = _declare(ctypes.CDLL(_SO_LSQ))
        return _lib_lsq
    if _lib is None:
        os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
        _lib = _declare(ctypes.CDLL(_SO))
    return _lib


def _declare(_lib):
    if True:   # (same exports in both flavours)
        dp = ctypes.POINTER(ctypes.c_double)
        _lib.ref_find_fundamental.argtypes = [dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int,
                                              ctypes.c_int, ctypes.c_uint64, dp, ctypes.POINTER(ctypes.c_ubyte),
                                              ctypes.POINTER(ctypes.c_int)]
        _lib.ref_find_fundamental.restype = ctypes.c_int
        _lib.ref_find_homography.argtypes = [dp, dp, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                             ctypes.c_int, ctypes.c_uint64, dp, ctypes.POINTER(ctypes.c_ubyte),
                                             ctypes.POINTER(ctypes.c_int)]
        _lib.ref_find_homography.restype = ctypes.c_int
        _lib.ref_value31.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32]
        _lib.ref_value31.restype = ctypes.c_uint32
        _lib.ref_stateless_sample.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_int,
                                              ctypes.POINTER(ctypes.c_int)]
        _lib.FDs.argtypes = [dp, dp, dp, ctypes.c_int]
        _lib.nullspace.argtypes = [dp, dp, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        _lib.nullspace.restype = ctypes.c_int
        _lib.SuperFastHash.argtypes = [ctypes.c_char_p, ctypes.c_int]
        _lib.SuperFastHash.restype = ctypes.c_uint32
        _lib.nsamples.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double]
        _lib.svduv.argtypes = [dp, dp, dp, ctypes.c_int, dp, ctypes.c_int]
        _lib.ref_minv3.argtypes = [dp]
        _lib.ref_minv3.restype = ctypes.c_int
        if hasattr(_lib, "ref_find_homography_2el"):
            _lib.ref_find_homography_2el.argtypes = [dp, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                                     ctypes.c_int, ctypes.c_uint64, dp, ctypes.POINTER(ctypes.c_ubyte),
                                                     ctypes.POINTER(ctypes.c_int)]
            _lib.ref_find_homography_2el.restype = ctypes.c_int
            _lib.ref_h_from_2el.argtypes = [dp, dp, dp]
            _lib.ref_h_from_2el.restype = ctypes.c_int
    return _lib


def _dptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def find_fundamental(pts1, pts2, px_th=0.5, conf=0.9999, max_iters=100000, error_type=0, sym_check=True,
                     laf_coef=0.0, degen_check=True, seed=0, rng=RNG_PHILOX, final_lsq=False):
    """Reference exp_ransacFcustomLAF behind the binding-layer conventions. Returns (F 3x3, mask bool[N], stats[4]).
    (final_lsq is accepted for symmetry but the reference's F text under __FINAL_LSQ__ does not compile,
    exp_ranF.c:1702; the F polish is pinned by oracle/port instead.)"""
    if final_lsq:
        raise ValueError("the reference has no compilable F driver with __FINAL_LSQ__")
    p1 = np.ascontiguousarray(pts1, dtype=np.float64)
    p2 = np.ascontiguousarray(pts2, dtype=np.float64)
    n, dim = p1.shape
    F = np.zeros(9, dtype=np.float64)
    mask = np.zeros(n, dtype=np.uint8)
    stats = np.zeros(4, dtype=np.int32)
    rc = lib(final_lsq).ref_find_fundamental(_dptr(p1), _dptr(p2), n, dim, px_th, conf, int(max_iters), int(error_type),
                                    int(bool(sym_check)), float(max(0.0, laf_coef)), int(bool(degen_check)), int(rng),
                                    ctypes.c_uint64(int(seed)), _dptr(F),
                                    mask.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)),
                                    stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int)))
    if rc != 0:
        raise ValueError("reference rejected the input (rc=%d)" % rc)
    return F.reshape(3, 3), mask.astype(bool), stats


def find_homography_raw(pts1, pts2, px_th=1.0, conf=0.999, max_iters=50000, error_type=0, sym_check=True,
                        laf_coef=0.0, seed=0, rng=RNG_PHILOX, final_lsq=False):
    """Reference exp_ransacHcustomLAF; returns the RAW core output (9 doubles, column-major, maps image2->image1)."""
    p1 = np.ascontiguousarray(pts1, dtype=np.float64)
    p2 = np.ascontiguousarray(pts2, dtype=np.float64)
    n, dim = p1.shape
    H = np.zeros(9, dtype=np.float64)
    mask = np.zeros(n, dtype=np.uint8)
    stats = np.zeros(4, dtype=np.int32)
    rc = lib(final_lsq).ref_find_homography(_dptr(p1), _dptr(p2), n, dim, px_th, conf, int(max_iters), int(error_type),
                                   int(bool(sym_check)), float(max(0.0, laf_coef)), int(rng),
                                   ctypes.c_uint64(int(seed)), _dptr(H),
                                   mask.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)),
                                   stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int)))
    if rc != 0:
        raise ValueError("reference rejected the input (rc=%d)" % rc)
    return H.reshape(3, 3), mask.astype(bool), stats


def find_homography(*a, **k):
    """As the reference's Python layer: zero model -> all-False; else H_out = inv(H.T) (utils.py:104-109)."""
    H, mask, stats = find_homography_raw(*a, **k)
    if np.abs(H).sum() == 0:
        return H, np.zeros_like(mask), stats
    return np.linalg.inv(H.T), mask, stats


def find_homography_2el_raw(u10, px_th=1.0, conf=0.999, max_iters=50000, seed=0, rng=RNG_PHILOX):
    """Reference ransacH2el (ranH2el.c:19) on rows (x', y', a', b', c', x, y, a, b, c); th = px_th^2. RAW output."""
    u = np.ascontiguousarray(u10, dtype=np.float64)
    n = u.shape[0]
    assert u.shape[1] == 10
    H = np.zeros(9, dtype=np.float64)
    mask = np.zeros(n, dtype=np.uint8)
    stats = np.zeros(4, dtype=np.int32)
    rc = lib().ref_find_homography_2el(_dptr(u), n, px_th, conf, int(max_iters), int(rng), ctypes.c_uint64(int(seed)),
                                       _dptr(H), mask.ctypes.data_as(ctypes.POINTER(ctypes.c_ubyte)),
                                       stats.ctypes.data_as(ctypes.POINTER(ctypes.c_int)))
    if rc != 0:
        raise ValueError("reference rejected the input (rc=%d)" % rc)
    return H.reshape(3, 3), mask.astype(bool), stats


def h_from_2el(ua, ub):
    """Reference A2toRH (ranH2el.c:233) on two rows; returns (ok, h[9])."""
    ua = np.ascontiguousarray(ua, dtype=np.float64); ub = np.ascontiguousarray(ub, dtype=np.float64)
    h = np.zeros(9)
    ok = lib().ref_h_from_2el(_dptr(ua), _dptr(ub), _dptr(h))
    return bool(ok), h


# ---- single leaves of the reference, for known-answer tests of the engine's restatements of them
def fds(u6, F):
    """FDs (Ftools.c): Sampson residuals of F[9] on rows (x1, y1, 1, x2, y2, 1)."""
    u = np.ascontiguousarray(u6, dtype=np.float64); F = np.ascontiguousarray(F, dtype=np.float64)
    out = np.zeros(len(u))
    lib().FDs(_dptr(u), _dptr(F), _dptr(out), len(u))
    return out


def nullspace(M):
    """nullspace (utools.c) of a 9x9 matrix; returns (dimension, the 81 doubles it writes)."""
    a = np.ascontiguousarray(M, dtype=np.float64).copy()
    out = np.zeros(81)
    buf = (ctypes.c_int * 18)()
    k = lib().nullspace(_dptr(a), _dptr(out), 9, buf)
    return k, out


def superfasthash(idx):
    """SuperFastHash (hash.c) of an int32 index list, as the reference hashes its samples."""
    b = np.ascontiguousarray(idx, dtype=np.int32).tobytes()
    return lib().SuperFastHash(b, len(b))


def nsamples(ni, n, s, conf):
    """nsamples (rtools.c): iterations needed for confidence conf with ni inliers of n, samples of size s."""
    return lib().nsamples(ni, n, s, conf)


def svd_v(A):
    """svduv (CCMATH) of a 3x3 matrix: the right singular vectors as columns, in CCMATH's (unsorted) order."""
    a = np.ascontiguousarray(A, dtype=np.float64).copy()
    d = np.zeros(3); u = np.zeros(9); v = np.zeros(9)
    lib().svduv(_dptr(d), _dptr(a), _dptr(u), 3, _dptr(v), 3)
    return v.reshape(3, 3)


def value31(seed, k, j):
    """The harness' Philox stream: 31-bit value j of iteration k."""
    return lib().ref_value31(seed, k, j)


def stateless_sample(seed, k, N, m):
    """The harness' stateless minimal sample of iteration k: m distinct indices of N."""
    sel = (ctypes.c_int * 8)()
    lib().ref_stateless_sample(ctypes.c_uint64(seed), k, N, m, sel)
    return np.array(list(sel)[:m], dtype=np.int32)


def row_digests(a):
    """8-byte digest of each row of a [K, M] float64 array, NaNs canonicalised (all NaNs compare equal)."""
    a = np.where(np.isnan(a), np.nan, a)
    return np.array([int.from_bytes(hashlib.sha1(r.tobytes()).digest()[:8], "little") for r in a], dtype=np.uint64)


def minv3_digests(mats):
    """CCMATH minv (matutls/minv.c) on each row of mats [K, 9] taken as a 3x3 matrix, in place.  Returns the return
    codes and the row_digests of the matrices it leaves: a bit-for-bit record small enough to store."""
    out = np.ascontiguousarray(mats, dtype=np.float64).copy()
    rc = np.array([lib().ref_minv3(_dptr(row)) for row in out], dtype=np.int32)
    return rc, row_digests(out)
