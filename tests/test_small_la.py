"""Small linear algebra that replaces LAPACK / CCMATH on the path (host build of the engine headers):
the SVD-free rank-2 projection (dominant eigenvector of adj(F)^T adj(F) by repeated squaring) against numpy's SVD and
against the Jacobi route it falls back to."""
import ctypes

import numpy as np
import pytest

from tests.hostemu import emu


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _rank2_numpy(F):
    U, s, Vt = np.linalg.svd(F)
    s[2] = 0.0
    return U @ np.diag(s) @ Vt


@pytest.mark.parametrize("kind", ["random", "unnormalised", "near_rank2", "clustered"])
def test_rank2_projection_matches_svd(kind):
    L = emu.lib()
    rng = np.random.default_rng(11)
    worst = 0.0
    fast = 0
    for t in range(400):
        F = rng.uniform(-0.5, 0.5, (3, 3))
        if kind == "unnormalised":          # entries spanning 12 orders of magnitude, as an un-normalised 8-point F
            sc = np.array([1e-6, 1e-3, 1.0])
            F = F * sc[:, None] * sc[None, :]
        elif kind == "near_rank2":
            U, s, Vt = np.linalg.svd(F)
            s[2] *= 1e-7
            F = U @ np.diag(s) @ Vt
        elif kind == "clustered":           # two smallest singular values within 5 %: the fast path must decline
            U, s, Vt = np.linalg.svd(F)
            s[2] = 0.97 * s[1]
            F = U @ np.diag(s) @ Vt
        F = np.ascontiguousarray(F)
        v = np.zeros(3)
        fast += L.emu_smallest_right_sv3_fast(_dp(F.copy()), _dp(v))
        A = F.copy()
        L.emu_enforce_rank2(_dp(A))
        B = F.copy()
        L.emu_enforce_rank2_slow(_dp(B))
        ref = _rank2_numpy(F)
        n = np.linalg.norm(ref)
        worst = max(worst, np.linalg.norm(A - ref) / n, np.linalg.norm(B - ref) / n)
        assert np.linalg.matrix_rank(A, tol=1e-9 * n) <= 2
    # clustered case: the projection itself is ill-conditioned (eps / relative gap), everything else is ~1e-14
    assert worst < (2e-10 if kind == "clustered" else 5e-12), worst
    if kind == "clustered":
        assert fast < 400          # some of them must have taken the Jacobi fallback
    else:
        assert fast > 380          # the SVD-free path handles (nearly) all ordinary matrices


def test_minv3_is_ccmath_minv_bit_for_bit(ref_oracle):
    """The engine's 3x3 inverse restates CCMATH minv operation for operation: the symmetric-transfer metrics push every
    correspondence through it, and when exact four-point fits compete with MSAC scores 4 - O(1e-13) the rounding noise
    of THIS routine decides which sample counts as the new best (i.e. whether the reference schedules one more LO)."""
    from oracle.ref import row_digests
    E = emu.lib()
    rng = np.random.default_rng(0)
    mats = []
    for t in range(5000):
        A = rng.normal(size=(3, 3)) * 10 ** rng.uniform(-3, 3)
        if t % 5 == 0:
            A[2] = A[0] * 2 + A[1] * 1e-13 * rng.normal()   # nearly singular (the -1 exit leaves the matrix half-processed)
        if t % 7 == 0:
            A[:, 0] *= 1e-9
        mats.append(A.ravel())
    ra, da = ref_oracle.minv3_digests(np.array(mats))   # return codes and digests of the matrices minv leaves
    b = np.array(mats)
    rb = np.array([E.emu_minv3(_dp(row)) for row in b])
    bad = np.flatnonzero((ra != rb) | (da != row_digests(b)))
    assert not bad.size, "matrices whose inverse differs from CCMATH minv: %s" % bad[:20]


def test_symmetric_max_metric_follows_the_reference_through_noise_level_ties(ref_oracle):
    """Scenes whose best sample is supported by its own four points only, metric symm_max: the LO schedule of the
    reference depends on which exact fit has the smaller rounding noise.  (These five configurations came out of the
    randomised GPU sweep with one LO run more or less than the reference before minv was restated exactly.)"""
    from pydegensac_b200.scenes import scene_H
    cases = [(20, 0.3, 2.0, 0.999, 3000, False, 198095051, 75908), (20, 0.3, 1.0, 0.95, 10000, True, 517737514, 26308),
             (50, 0.2, 2.0, 0.999, 1000, False, 633781542, 57556), (200, 0.2, 3.0, 0.9999, 10000, True, 1388931049, 35015),
             (100, 0.3, 0.5, 0.999, 10000, False, 1334272533, 66883)]
    for n, ratio, px, conf, iters, sym, seed, scene in cases:
        p1, p2, _ = scene_H(n, max(4, int(n * ratio)), scene)
        a = ref_oracle.find_homography_raw(p1, p2, px, conf, iters, error_type=2, sym_check=sym, seed=seed)
        b = emu.find_homography_raw(p1, p2, px, conf, iters, error_type=2, sym_check=sym, seed=seed)
        assert np.array_equal(a[1], b[1]) and a[2][0] == b[2][0] and a[2][1] == b[2][1]
