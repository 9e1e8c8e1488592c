"""Oracle groundwork for the second half of SURVEY §8f row N4 (relpose_8pt / essential_matrix_8pt,
solvers/relpose_8pt.cc:52-95) — the device kernel is not built yet (DESIGN.md §0).  The oracle restatement (a) recovers
the ground truth on noise-free data, exactly 8 points and over-determined, (b) returns a matrix with singular values
(s, s, 0), and (c) equals the reference's own source file run on mini-Eigen bit for bit (logic pin; the symmetric
eigen-solver is iterative in Eigen, so parity with a real PoseLib build is to tolerance by construction)."""
import os
import sys

import numpy as np
import plo_py as P
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from ref_store import RefStore  # noqa: E402

REF = RefStore("ref_8pt", P.ref2_available())  # the reference's results, stored in tests/golden/ref_8pt/


@pytest.fixture(autouse=True, scope="module")
def _save_store():
    yield
    REF.save()


@pytest.fixture(autouse=True)
def _store_key(request):
    REF.begin(request.node)
    yield
    REF.end()


def _scene(n, seed, noise=0.0):
    rng = np.random.default_rng(seed)
    X = np.c_[rng.uniform(-1, 1, (n, 2)), rng.uniform(3, 6, n)]
    R = np.linalg.qr(np.eye(3) + 0.2 * rng.normal(size=(3, 3)))[0]
    R *= np.sign(np.linalg.det(R))
    t = rng.normal(size=3)
    t /= np.linalg.norm(t)
    Y = X @ R.T + t + noise * rng.normal(size=(n, 3))
    return X / np.linalg.norm(X, axis=1)[:, None], Y / np.linalg.norm(Y, axis=1)[:, None], R, t


def _skew(t):
    return np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])


@pytest.mark.parametrize("n", [8, 9, 20, 200])
def test_essential_matrix_8pt_recovers_ground_truth(n):
    for seed in range(20):
        x1, x2, R, t = _scene(n, seed)
        E = P.essential_matrix_8pt(x1, x2)
        Eg = _skew(t) @ R
        En, Eg = E / np.linalg.norm(E), Eg / np.linalg.norm(Eg)
        assert min(np.abs(En - Eg).max(), np.abs(En + Eg).max()) < 1e-9
        s = np.linalg.svd(E, compute_uv=False)
        assert abs(s[0] - s[1]) < 1e-12 * s[0] and s[2] < 1e-12 * s[0]  # relpose_8pt.cc:74-81
        poses = P.relpose_8pt(x1, x2)
        assert len(poses) >= 1  # the true pose passes the cheirality test of motion_from_essential
        q = poses[:, :4]
        Rs = [np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                        [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                        [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]]) for w, x, y, z in q]
        assert min(np.abs(Rk - R).max() + np.abs(p[4:] - t).max() for Rk, p in zip(Rs, poses)) < 1e-8


def _reference_8pt(x1, x2):
    with P.reference_sources():
        return P.essential_matrix_8pt(x1, x2), P.relpose_8pt(x1, x2)


def test_8pt_equals_the_reference_source_on_mini_eigen():
    """The reference's side: oracle/_ref/libplref2.so, or without it its results stored in tests/golden/ref_8pt/."""
    for n in (8, 9, 12, 50, 300):
        for seed in range(30):
            x1, x2, _, _ = _scene(n, 1000 * n + seed, noise=0.002 if seed % 2 else 0.0)
            a, pa = P.essential_matrix_8pt(x1, x2), P.relpose_8pt(x1, x2)
            b, pb = REF(lambda: _reference_8pt(x1, x2))
            assert np.array_equal(a, b) and pa.shape == pb.shape and np.array_equal(pa, pb), (n, seed)
