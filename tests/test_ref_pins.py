"""CPU-only: the parts of the
UNMODIFIED reference that compile without Eigen — robust/sampling.cc and the loop templates of robust/ransac_impl.h —
pin (1) the sampler of the oracle AND of the engine bit for bit, (2) the dynamic-iteration arithmetic, (3) the
control flow of the oracle's ransac<> / score_models<> restatement: the reference's loop drives the oracle's estimators
and must arrive at exactly the oracle loop's result.
The reference's side is oracle/_ref/libplref.so (`make -C oracle ref`, where the reference's sources are) or, without
it, that library's results stored in tests/golden/ref_pins/ (tests/golden/ref_store.py)."""
import math
import os
import sys

import numpy as np
import plo_py as P
import pytest

from poselib_b200 import cabi
from poselib_b200 import problem_generator as G

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from ref_store import RefStore  # noqa: E402

REF = RefStore("ref_pins", P.ref_available())  # the reference's results, stored in tests/golden/ref_pins/


@pytest.fixture(autouse=True, scope="module")
def _save_store():
    yield
    REF.save()


@pytest.fixture(autouse=True)
def _store_key(request):
    REF.begin(request.node)
    yield
    REF.end()


def test_random_int_stream_and_known_answer():
    r = REF(lambda: P.ref_random_ints(0, 6))
    assert r.tolist() == [2065550767, -1581685260, -2146876081, 1917616620, 1369994395, 1954456298]  # SURVEY App. A.1
    for seed in (0, 1, 99, 2**40 + 3):
        assert REF.same(lambda: P.ref_random_ints(seed, 4000), P.random_ints(seed, 4000))


@pytest.mark.parametrize("n,k", [(10000, 5), (200, 3), (5000, 7), (20000, 4), (7, 7), (6, 5), (33, 4)])
@pytest.mark.parametrize("seed", [0, 7, 2**33 + 1])
def test_reference_sampler_pins_oracle_and_engine(n, k, seed):
    oracle = P.sample_table(n, k, P.RansacOpt(seed=seed), 4000)
    assert REF.same(lambda: P.ref_sample_table(n, k, P.RansacOpt(seed=seed), 4000), oracle)
    assert np.array_equal(oracle, cabi.host_sample_table(n, k, cabi.RansacOpt(seed=seed), 4000))


@pytest.mark.parametrize("n,k,budget", [(5000, 7, 100000), (400, 5, 300), (50, 4, 40), (64, 3, 100000), (9, 4, 5)])
def test_reference_prosac_sampler_pins_oracle_and_engine(n, k, budget):
    kw = dict(seed=5, progressive_sampling=True, max_prosac_iterations=budget)
    oracle = P.sample_table(n, k, P.RansacOpt(**kw), 3000)
    assert REF.same(lambda: P.ref_sample_table(n, k, P.RansacOpt(**kw), 3000), oracle)
    assert np.array_equal(oracle, cabi.host_sample_table(n, k, cabi.RansacOpt(**kw), 3000))


def test_reference_iteration_arithmetic_pins_oracle_and_engine():
    rng = np.random.default_rng(1)
    for _ in range(500):
        nd = int(rng.integers(1, 30000))
        ni = int(rng.integers(0, nd + 1))
        k = int(rng.choice([0, 3, 4, 5, 7]))
        assert REF(lambda: P.ref_all_inlier_sample_probability(ni, nd, k)) == P.all_inlier_sample_probability(ni, nd, k)
        sp = float(rng.choice([0.99, 0.9999]))
        mult, mn, mx = float(rng.choice([1.0, 3.0])), int(rng.integers(0, 2000)), int(rng.integers(1, 200000))
        ref = REF(lambda: P.ref_compute_dynamic_max_iter(ni, nd, max(k, 1), math.log(1 - sp), mult, mn, mx))
        assert ref == P.compute_dynamic_max_iter(ni, nd, max(k, 1), math.log(1 - sp), mult, mn, mx)
        if nd >= max(k, 1):
            assert ref == cabi.host_dynamic_max_iter(ni, nd, max(k, 1), sp, mult, mn, mx)


def test_reference_loop_with_the_mock_estimator_of_the_reference_tests():
    # tests/ransac_test.cc:71-122: exact stop iterations of ransac<MockEstimator, int>
    for nd, k, inl, kw in [(100, 5, 80, {}), (100, 5, 80, dict(min_iterations=50, max_iterations=1000)),
                           (100, 7, 10, dict(min_iterations=10, max_iterations=333)), (10, 5, 10, {}), (4, 5, 4, {})]:
        r, o = REF(lambda: P.ref_ransac_mock(nd, k, inl, P.RansacOpt(**kw)).as_dict()), P.ransac_mock(nd, k, inl, P.RansacOpt(**kw))
        assert r == o.as_dict()


CASES = [
    ("pnp", lambda: G.abspose_problem(300, 0.5, 71, 0), dict(max_iterations=600, min_iterations=100, seed=1), 12.0),
    ("pnp", lambda: G.abspose_problem(60, 0.3, 71, 1), dict(max_iterations=300, min_iterations=400, seed=2), 8.0),
    ("relpose", lambda: G.relpose_problem(400, 0.4, 72, 0), dict(max_iterations=1500, min_iterations=100, seed=3), 1.5),
    ("relpose", lambda: G.relpose_problem(5, 1.0, 72, 1), dict(max_iterations=20, min_iterations=5, seed=4), 1.5),
    ("fundamental", lambda: G.relpose_problem(400, 0.5, 73, 0, prosac_sorted=True),
     dict(max_iterations=800, min_iterations=100, seed=5, progressive_sampling=True, max_prosac_iterations=300), 1.5),
    ("homography", lambda: G.homography_problem(2500, 0.5, 41, 5), dict(max_iterations=3000, min_iterations=200, seed=15), 1.5),
    ("homography", lambda: G.homography_problem(3, 1.0, 74, 0), dict(max_iterations=50, min_iterations=5, seed=6), 1.5),
]


@pytest.mark.parametrize("kind,gen,kw,me", CASES)
@pytest.mark.parametrize("with_initial_model", [False, True])
def test_reference_loop_drives_oracle_estimators_to_the_oracle_loop_result(kind, gen, kw, me, with_initial_model):
    p = gen()
    a, b = (p["x"] / G.FOCAL, p["X"]) if kind == "pnp" else (p["x1"] / G.FOCAL, p["x2"] / G.FOCAL)
    init = None
    if with_initial_model:
        kw = dict(kw, score_initial_model=True)
        if kind in ("pnp", "relpose"):
            init = np.r_[p["q_gt"], p["t_gt"]] + 0.01
            init[:4] /= np.linalg.norm(init[:4])
        else:
            init = np.eye(3) + 0.01
    rfc = kind == "fundamental"
    r = REF(lambda: P.ref_ransac(kind, a, b, P.RansacOpt(**kw), me / G.FOCAL, init=init, rfc=rfc))
    o = P.ransac(kind, a, b, P.RansacOpt(**kw), me / G.FOCAL, init=init, rfc=rfc)
    assert r["stats"] == o["stats"]
    assert np.array_equal(r["inliers"], o["inliers"])
    assert np.array_equal(np.asarray(r["model"]), np.asarray(o["model"]), equal_nan=True)


def _roots(n, roots):
    return n, roots[:max(n, 0)]


def test_reference_univariate_solvers_pin_the_oracle_bitwise():
    """misc/univariate.cc compiled from the reference: the oracle's cubic / quadratic solvers (used by p3p, relpose_7pt
    and homography_4pt) must return the same number of roots and the same bits."""
    rng = np.random.default_rng(2)
    for i in range(4000):
        scale = 10.0 ** rng.integers(-3, 4)
        a, b, c = rng.normal(0, scale, 3)
        if i % 7 == 0:
            c = b * b / (4 * a)            # double root
        for name, args, k in (("solve_quadratic_real", (a, b, c), 2), ("solve_cubic_single_real", (a, b, c), 1),
                              ("solve_cubic_real", (a, b, c), 3)):
            no, ro = getattr(P, name)(*args)
            assert REF.same(lambda: _roots(*getattr(P, name)(*args, ref=True)), _roots(no, ro)), (name, args, no, ro)


def test_reference_sturm_root_isolation_pins_the_oracle_bitwise():
    """misc/sturm.h bisect_sturm<10> compiled from the reference vs the oracle's restatement: random degree-10
    polynomials, polynomials with known roots (clustered / multiple), and the determinant polynomials of real 5-point
    problems (captured through the oracle's solver)."""
    rng = np.random.default_rng(3)
    polys = [rng.normal(size=11) for _ in range(1500)]
    for _ in range(800):                         # prescribed real roots, some clustered, some complex pairs
        nreal = int(rng.integers(0, 11))
        nreal -= (10 - nreal) % 2
        roots = list(rng.uniform(-3, 3, max(nreal, 0)))
        if len(roots) >= 2 and rng.random() < 0.3:
            roots[1] = roots[0] + 10.0 ** rng.integers(-9, -2)
        p = np.poly1d([1.0])
        for r in roots:
            p = p * np.poly1d([1.0, -r])
        for _ in range((10 - len(roots)) // 2):
            re, im = rng.normal(), abs(rng.normal()) + 0.1
            p = p * np.poly1d([1.0, -2 * re, re * re + im * im])
        polys.append(p.coeffs[::-1] * rng.uniform(0.1, 10))
    polys.append(np.r_[rng.normal(size=10), 0.0])    # leading coefficient zero: no roots by definition (sturm.h:234)
    exact = 0
    for c in polys:
        c = np.ascontiguousarray(c, dtype=np.float64)
        assert len(c) == 11
        o = P.bisect_sturm10(c)
        assert REF.same(lambda: P.ref_bisect_sturm10(c), o), (c, o)
        exact += 1
    assert exact == len(polys)


def test_reference_p3p_scalar_helpers_pin_the_oracle_bitwise():
    """solvers/p3p_common.h root2real / refine_lambda (the scalar part of Ding's P3P) compiled from the reference."""
    rng = np.random.default_rng(4)
    for i in range(3000):
        b, c = rng.normal(0, 3, 2)
        if i % 5 == 0:
            c = b * b / 4 + rng.choice([0.0, 1e-13, -1e-13, 5e-13])   # around the THRESHOLD branches
        assert REF.same(lambda: P.p3p_root2real(b, c, ref=True), P.p3p_root2real(b, c)), (b, c)
    for _ in range(2000):
        # a consistent instance: three unit bearings, true depths perturbed as the solver's initial estimate would be
        x = rng.normal(size=(3, 3))
        x /= np.linalg.norm(x, axis=1, keepdims=True)
        lam = rng.uniform(0.5, 5.0, 3)
        X = x * lam[:, None]
        a12, a13, a23 = (np.sum((X[0] - X[1]) ** 2), np.sum((X[0] - X[2]) ** 2), np.sum((X[1] - X[2]) ** 2))
        b12, b13, b23 = x[0] @ x[1], x[0] @ x[2], x[1] @ x[2]
        l0 = lam * (1 + rng.normal(0, 1e-3, 3))
        ro = P.p3p_refine_lambda(l0, a12, a13, a23, b12, b13, b23)
        assert REF.same(lambda: P.p3p_refine_lambda(l0, a12, a13, a23, b12, b13, b23, ref=True), ro)


@pytest.mark.parametrize("kind", ["fundamental", "homography"])
def test_reference_scorers_and_masks_pin_the_oracle_bitwise(kind):
    """robust/utils.cc compiled from the reference: compute_sampson_msac_score(F) / get_inliers(F) and
    compute_homography_msac_score / get_homography_inliers are element-access + scalar code, so they run as the
    reference wrote them.  Score bits, inlier counts and masks of the oracle must be identical — for good models,
    perturbed models, random and degenerate (rank-deficient, zero) models, on normalised and pixel-scale coordinates."""
    rng = np.random.default_rng(5)
    for idx in range(6):
        n = [50, 333, 1000, 2500, 5000, 8][idx]
        p = G.homography_problem(n, 0.5, 81, idx) if kind == "homography" else G.relpose_problem(n, 0.4, 81, idx)
        for scale, thr in ((1.0 / G.FOCAL, 1.5 / G.FOCAL), (1.0, 2.0)):
            x1, x2 = p["x1"] * scale, p["x2"] * scale
            if kind == "homography":
                gt = p["H_gt"]  # exact for the normalised coordinates, merely "some model" for the pixel-scale ones
            else:
                t = p["t_gt"]
                gt = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ p["R_gt"]
            models = [gt, gt + rng.normal(0, 1e-3, (3, 3)), rng.normal(size=(3, 3)), np.zeros((3, 3)),
                      np.outer(rng.normal(size=3), rng.normal(size=3)), np.eye(3)]
            for M in models:
                sr, cr, mr = REF(lambda: P.ref_score(kind, M, x1, x2, thr * thr, want_inliers=True))
                so, co = P.score(kind, M, x1, x2, thr * thr)
                mo = P.inliers(kind, M, x1, x2, thr * thr)
                assert cr == co
                assert (sr == so) or (np.isnan(sr) and np.isnan(so)), (sr, so)
                assert np.array_equal(mr, mo)


def test_reference_real_focal_check_pins_the_oracle():
    rng = np.random.default_rng(6)
    agree = 0
    for i in range(3000):
        if i % 3 == 0:
            p = G.relpose_problem(8, 1.0, 82, i)
            t = p["t_gt"]
            f1, f2 = rng.uniform(0.5, 3.0, 2)
            E = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ p["R_gt"]
            F = np.diag([1 / f2, 1 / f2, 1.0]) @ E @ np.diag([1 / f1, 1 / f1, 1.0]) + rng.normal(0, 1e-4, (3, 3)) * (i % 2)
        else:
            F = rng.normal(size=(3, 3))
        assert REF(lambda: P.ref_calculate_RFC(F)) == bool(P.calculate_RFC(F))
        agree += 1
    assert agree == 3000


REF_CAMERAS = [  # tests/example_cameras.h of the reference (the models whose projection is element-access code)
    ("SIMPLE_RADIAL", [2425.85, 932.383, 628.265, -0.0397695]),
    ("PINHOLE", [3425.62, 3426.29, 3118.41, 2069.07]),
    ("SIMPLE_PINHOLE", [3425.62, 3118.41, 2069.07]),
    ("OPENCV", [2575.94, 2608.29, 1599.26, 1257.13, 0.141865, -0.465301, 0, 0]),
    ("OPENCV", [868.993378, 866.063001, 525.942323, 420.042529, -0.399431, 0.188924, 0.000153, 0.000571]),
]


def test_reference_camera_scalar_code_pins_the_oracle_bitwise():
    """misc/camera_models.cc compiled from the reference: Newton undistortion (undistort_poly1/2), the OpenCV distortion
    and its Jacobian, Camera::focal / rescale, and the projections (+ pinhole projection Jacobians) that are pure
    element-access code."""
    rng = np.random.default_rng(8)
    for _ in range(3000):
        k1, k2, rd = rng.normal(0, 0.2), rng.normal(0, 0.05), abs(rng.normal(0, 0.6))
        for two in (0, 1):
            assert REF.same(lambda: P.undistort_poly(k1, k2, two, rd, ref=True), P.undistort_poly(k1, k2, two, rd))
        d4, x2 = rng.normal(0, [0.3, 0.2, 1e-3, 1e-3]), rng.normal(0, 0.5, 2)
        assert REF.same(lambda: P.opencv_distortion(d4, x2, ref=True), P.opencv_distortion(d4, x2))
        assert REF.same(lambda: P.opencv_distortion(d4, x2, True, ref=True), P.opencv_distortion(d4, x2, True))
    X = np.c_[rng.uniform(-0.6, 0.6, (500, 2)), np.ones(500)] * rng.uniform(0.5, 9.0, (500, 1))
    for cam in REF_CAMERAS:
        assert REF.same(lambda: P.ref_camera_focal(cam), P.camera_focal(cam))
        assert REF.same(lambda: P.camera_rescale(cam, 1.0 / 1234.5, ref=True), P.camera_rescale(cam, 1.0 / 1234.5))
        xp_jac, J, xp = P.camera_project_with_jac(cam, X)
        assert REF.same(lambda: P.ref_camera_project(cam, X), xp)
        if cam[0] in ("PINHOLE", "SIMPLE_PINHOLE"):
            assert REF.same(lambda: P.ref_camera_project(cam, X, with_jac=True), (xp_jac, J))
