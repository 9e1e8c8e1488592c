"""CPU-only: the reference's
OWN sources for the whole hot path — robust.cc, robust/ransac.cc + ransac_impl.h, robust/estimators/*.cc,
robust/bundle.cc + optim/*.h, robust/utils.cc, solvers/{p3p,relpose_5pt,relpose_7pt,homography_4pt}.cc,
misc/{essential,camera_models,univariate}.cc — compiled UNMODIFIED on top of mini-Eigen (oracle/ref/mini), which
implements every Eigen operation with the oracle's restatement of it (oracle/plo_math.h).

`reference sources on mini-Eigen == oracle` therefore pins the oracle's transcription of PoseLib's LOGIC (formulas,
branches, loop structure, call order, sign conventions) against the reference's own text; it does not pin Eigen's
arithmetic itself (summation order inside 3-/4-term reductions, the decompositions), which both sides share here.

Result of the comparison (asserted below):
  * bit-identical: p3p, homography_4pt, every scorer and inlier mask (pose / F / H / tangent), every LM refiner
    (absolute pose, relative pose, fundamental, homography; all four loss types), all five camera models
    (project / unproject with Jacobians, Newton undistortion), and END TO END ransac_pnp / ransac_homography /
    estimate_absolute_pose / estimate_homography (RANSAC loop + LO + final bundle), PROSAC included.
  * relpose_5pt / relpose_7pt: the oracle restates the generated polynomial expansions of the reference structurally
    (table-driven monomial products, polynomial multiplication for the determinant; mixed determinants for the
    7-point cubic) instead of copying ~200 lines of generated expressions, so the operation ORDER differs: same
    solution count, solutions equal up to the conditioning of the minimal problem (median 1e-15, worst 1e-7 over
    the sample).  End to end, ransac_relpose / ransac_fundamental / estimate_* return the same iteration count,
    refinement count, inlier count and inlier mask; the model agrees to 1e-9 (relative poses up to the |t| gauge) and the
    MSAC score to 1e-12 relative.
    Switched to the reference's operation order (test hook plo_set_reference_order; the 480-term determinant order is
    parsed from the reference's source at run time, nothing of it is stored here) the oracle is BIT-IDENTICAL to the
    reference's sources on the whole path, degenerate inputs included (last four tests of this file).
  * FixCameraRelativePoseRefiner (tangent Sampson): the oracle models Vector4d::norm() with the SSE2 packet order
    (a0²+a2²)+(a1²+a3²) in that one place; mini-Eigen sums left to right.  Agreement 1e-9.
The reference's side is oracle/_ref/libplref2.so (`make -C oracle ref2`, where the reference's sources are) or, without
it, that library's results stored in tests/golden/ref_sources/ (tests/golden/ref_store.py).  The tests that need
the reference's source text itself (the operation-order table) or its alternative build run only where it is.
"""
import os
import sys

import numpy as np
import plo_py as P
import pytest

from poselib_b200 import problem_generator as G

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from ref_store import RefStore  # noqa: E402

REF = RefStore("ref_sources", P.ref2_available())  # the reference's results, stored in tests/golden/ref_sources/


@pytest.fixture(autouse=True, scope="module")
def _save_store():
    yield
    REF.save()


@pytest.fixture(autouse=True)
def _store_key(request):
    REF.begin(request.node, stored="reference_order" not in request.fixturenames)  # runs only with the reference
    yield
    REF.end()

CAMT = (G.FOCAL, G.FOCAL, 0.0, 0.0)
CAMERAS = [("SIMPLE_PINHOLE", [1000.0, 3.0, -4.0]), ("PINHOLE", [1000.0, 1010.0, 3.0, -4.0]),
           ("SIMPLE_RADIAL", [1000.0, 3.0, -4.0, -0.03]), ("RADIAL", [1050.0, -15.0, 25.0, -0.04012, 0.00123]),
           ("OPENCV", [900.0, 901.0, 3.0, 4.0, 0.01, -0.02, 1e-4, 2e-4])]


def both(f):
    """(oracle result, reference-sources result) of the same wrapper call."""
    return f(), REF(lambda: reference(f))


def reference(f):
    with P.reference_sources():
        return f()


def same_as_reference(f):
    """Bitwise: the oracle's result of the wrapper call equals the reference sources' result."""
    return REF.same(lambda: reference(f), f())


def same(a, b):
    if isinstance(a, dict):
        return all(same(a[k], b[k]) for k in a if k != "counters")
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return np.array_equal(np.asarray(a), np.asarray(b))


def maxdiff(a, b):
    if isinstance(a, (tuple, list)):
        return max(maxdiff(x, y) for x, y in zip(a, b))
    return float(np.abs(np.asarray(a, dtype=float) - np.asarray(b, dtype=float)).max())


# ---- minimal solvers ---------------------------------------------------------------------------------------------
def test_p3p_lambdatwist_is_bit_identical_and_finds_the_pose():
    """solvers/p3p_lambdatwist.cc (SURVEY row N2's alternative P3P) compiled from the reference on mini-Eigen == the
    oracle restatement, bit for bit (libm is the same on both sides); the true pose is among the solutions."""
    found = 0
    for s in range(400):
        x, X, R, t = G.minimal_abspose(s)
        a = P.p3p_lambdatwist(x, X)
        assert REF.same(lambda: reference(lambda: P.p3p_lambdatwist(x, X)), a), s
        for p in a:
            q = p[:4]
            Rq = np.array([[1 - 2 * (q[2]**2 + q[3]**2), 2 * (q[1] * q[2] - q[0] * q[3]), 2 * (q[1] * q[3] + q[0] * q[2])],
                           [2 * (q[1] * q[2] + q[0] * q[3]), 1 - 2 * (q[1]**2 + q[3]**2), 2 * (q[2] * q[3] - q[0] * q[1])],
                           [2 * (q[1] * q[3] - q[0] * q[2]), 2 * (q[2] * q[3] + q[0] * q[1]), 1 - 2 * (q[1]**2 + q[2]**2)]])
            if np.abs(p[4:] - t).max() < 1e-6 and np.abs(Rq - R).max() < 1e-6:
                found += 1
                break
    assert found >= 396, found


def test_p3p_and_homography_4pt_are_bit_identical():
    for s in range(300):
        x, X, _, _ = G.minimal_abspose(s)
        assert same_as_reference(lambda: P.p3p(x, X)), s
        x1, x2, _ = G.minimal_homography(s)
        for cheir in (True, False):
            assert same_as_reference(lambda: P.homography_4pt(x1, x2, cheir)), s
    # degenerate input: three collinear points, and a cheirality violation
    x1, x2, _ = G.minimal_homography(0)
    x1c = x1.copy()
    x1c[2] = 0.5 * (x1c[0] + x1c[1])
    assert same_as_reference(lambda: P.homography_4pt(x1c, x2, False))
    x2f = x2.copy()
    x2f[3] = -x2f[3]
    (na, _), (nb, _) = both(lambda: P.homography_4pt(x1, x2f, True))
    assert na == nb


def test_relpose_5pt_and_7pt_agree_up_to_conditioning():
    d5, d7, count_mismatch = [], [], 0
    for s in range(300):
        x1, x2, _, _ = G.minimal_relpose(s, 5)
        a, b = both(lambda: P.relpose_5pt_E(x1, x2))
        if a.shape != b.shape:
            count_mismatch += 1  # a real root at the edge of existence; must stay exceptional
        else:
            d5.append(maxdiff(a, b) if a.size else 0.0)
        pa, pb = both(lambda: P.relpose_5pt(x1, x2))
        if pa.shape == pb.shape and pa.size:
            d5.append(maxdiff(pa, pb))
        x1, x2, _, _ = G.minimal_relpose(s, 7)
        a, b = both(lambda: P.relpose_7pt(x1, x2))
        assert a.shape == b.shape, s
        d7.append(maxdiff(a, b) if a.size else 0.0)
    assert count_mismatch <= 1
    assert np.median(d5) < 1e-12 and np.percentile(d5, 99) < 1e-6 and max(d5) < 1e-4
    assert max(d7) < 1e-11


# ---- scorers, masks, refiners ------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_scorers_masks_and_refiners_are_bit_identical(seed):
    p = G.relpose_problem(800, 0.5, 2, seed)
    x1n, x2n = p["x1"] / G.FOCAL, p["x2"] / G.FOCAL
    thr = (1.0 / G.FOCAL) ** 2
    pose = P.ransac("relpose", x1n, x2n, P.RansacOpt(max_iterations=300, min_iterations=50, seed=seed), 1.0 / G.FOCAL)["model"]
    F = P.ransac("fundamental", p["x1"], p["x2"], P.RansacOpt(max_iterations=300, min_iterations=50, seed=seed), 1.0)["model"]
    h = G.homography_problem(800, 0.5, 4, seed)
    H = P.ransac("homography", h["x1"], h["x2"], P.RansacOpt(max_iterations=300, min_iterations=50, seed=seed), 1.0)["model"]
    q = G.config_c1(seed)
    xn = q["x"] / G.FOCAL
    apose = P.ransac("pnp", xn, q["X"], P.RansacOpt(**q["ransac"]), 12.0 / G.FOCAL)["model"]
    cases = [("relpose", pose, x1n, x2n, thr), ("fundamental", F, p["x1"], p["x2"], 1.0),
             ("homography", H, h["x1"], h["x2"], 1.0), ("pnp", apose, xn, q["X"], (12.0 / G.FOCAL) ** 2)]
    for kind, model, a, b, t in cases:
        for scale in (1.0, 0.25, 16.0):  # thresholds that move points across the inlier boundary
            assert same(*both(lambda: P.score(kind, model, a, b, t * scale))), kind
            assert same(*both(lambda: P.inliers(kind, model, a, b, t * scale))), kind
        pert = np.array(model, dtype=float).copy()
        if kind in ("relpose", "pnp"):
            pert[4:] += 0.01
        else:
            pert = pert * 1.001 + 1e-7
        for loss in ("TRIVIAL", "TRUNCATED", "HUBER", "CAUCHY"):
            bo = P.BundleOpt(loss_type=loss, loss_scale=0.5 * np.sqrt(t), max_iterations=25)
            ra, rb = both(lambda: P.refine(kind, pert, a, b, bo))
            assert same(ra, rb), (kind, loss, maxdiff(ra, rb))


# ---- camera models -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cam", CAMERAS, ids=[c[0] for c in CAMERAS])
def test_camera_models_are_bit_identical(cam):
    rng = np.random.default_rng(0)
    X = np.c_[rng.uniform(-0.4, 0.4, (300, 2)), np.ones(300)]
    X /= np.linalg.norm(X, axis=1)[:, None]
    assert same_as_reference(lambda: P.camera_project_with_jac(cam, X))
    xp = P.camera_project_with_jac(cam, X)[2]
    assert same_as_reference(lambda: P.camera_unproject_with_jac(cam, xp))
    assert same_as_reference(lambda: P.camera_unproject2(cam, xp))
    assert same_as_reference(lambda: P.camera_focal(cam))


# ---- RANSAC and estimate_*, end to end ---------------------------------------------------------------------------
def _close_runs(a, b, sign_free=False, tol=1e-9):
    sa, sb = a["stats"], b["stats"]
    assert (sa["iterations"], sa["refinements"], sa["num_inliers"]) == (sb["iterations"], sb["refinements"], sb["num_inliers"])
    assert np.array_equal(a["inliers"], b["inliers"])
    assert abs(sa["model_score"] - sb["model_score"]) <= 1e-12 * abs(sa["model_score"])
    am, bm = np.asarray(a["model"], dtype=float), np.asarray(b["model"], dtype=float)
    if am.ndim == 1 and not sign_free:
        # 7-vectors here are relative poses: |t| is a gauge freedom the refiner never renormalises (relative.h:152-157), and
        # it is the one quantity that drifts (up to 1e-5) between two last-bit-different runs; compare the direction
        am = np.r_[am[:4], am[4:] / max(np.linalg.norm(am[4:]), 1e-300)]
        bm = np.r_[bm[:4], bm[4:] / max(np.linalg.norm(bm[4:]), 1e-300)]
    d = maxdiff(am, bm)
    if sign_free:
        d = min(d, maxdiff(am, -bm))
    assert d < tol


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_pnp_and_homography_pipelines_are_bit_identical_end_to_end(seed):
    q = G.config_c1(seed)
    ro = P.RansacOpt(seed=seed, **q["ransac"])
    assert same(*both(lambda: P.ransac("pnp", q["x"] / G.FOCAL, q["X"], ro, 12.0 / G.FOCAL)))
    assert same(*both(lambda: P.estimate("pnp", q["x"], q["X"], ro, P.BundleOpt(), 12.0, CAMT)))
    h = G.homography_problem(1000, 0.5, 4, seed)
    for prosac in (False, True):
        ro = P.RansacOpt(max_iterations=2000, min_iterations=100, seed=seed, progressive_sampling=prosac)
        assert same(*both(lambda: P.ransac("homography", h["x1"], h["x2"], ro, 1.0)))
        a, b = both(lambda: P.estimate("homography", h["x1"], h["x2"], ro, P.BundleOpt(), 1.0))
        assert same(a, b) and a["stats"]["num_inliers"] > 200


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_relpose_and_fundamental_pipelines_agree_end_to_end(seed):
    p = G.relpose_problem(1000, 0.4, 2, seed)
    ro = P.RansacOpt(max_iterations=2000, min_iterations=100, seed=seed)
    _close_runs(*both(lambda: P.ransac("relpose", p["x1"] / G.FOCAL, p["x2"] / G.FOCAL, ro, 1.0 / G.FOCAL)))
    a, b = both(lambda: P.estimate("relpose", p["x1"], p["x2"], ro, P.BundleOpt(), 1.0, CAMT, CAMT))
    _close_runs(a, b)
    assert a["stats"]["num_inliers"] > 300
    for rfc in (False, True):
        _close_runs(*both(lambda: P.ransac("fundamental", p["x1"], p["x2"], ro, 1.0, rfc=rfc)), sign_free=True)
        _close_runs(*both(lambda: P.estimate("fundamental", p["x1"], p["x2"], ro, P.BundleOpt(), 1.0, rfc=rfc)), sign_free=True)


def test_initial_model_and_prosac_on_relpose():
    p = G.relpose_problem(1500, 0.4, 2, 9, prosac_sorted=True)
    ro = P.RansacOpt(max_iterations=3000, min_iterations=100, seed=4, progressive_sampling=True)
    a, b = both(lambda: P.estimate("relpose", p["x1"], p["x2"], ro, P.BundleOpt(), 1.0, CAMT, CAMT))
    _close_runs(a, b)
    ro2 = P.RansacOpt(max_iterations=500, min_iterations=50, seed=4, score_initial_model=True)
    _close_runs(*both(lambda: P.estimate("relpose", p["x1"], p["x2"], ro2, P.BundleOpt(), 1.0, CAMT, CAMT, init=a["model"])))


def test_headline_configuration_c2_agrees():
    c = G.config_c2(0)
    ro = P.RansacOpt(seed=0, **c["ransac"])
    a, b = both(lambda: P.estimate("relpose", c["x1"], c["x2"], ro, P.BundleOpt(), c["max_error"], CAMT, CAMT))
    _close_runs(a, b)
    assert a["stats"]["num_inliers"] > 2500


# ---- distorted cameras and the tangent Sampson path ----------------------------------------------------------------
def test_distorted_cameras_and_tangent_sampson_path():
    cam = CAMERAS[3]
    p = G.relpose_problem(1500, 0.5, 2, 5)
    X1 = np.c_[p["x1"] / G.FOCAL, np.ones(len(p["x1"]))]
    X2 = np.c_[p["x2"] / G.FOCAL, np.ones(len(p["x2"]))]
    d1, d2 = P.camera_project_with_jac(cam, X1)[2], P.camera_project_with_jac(cam, X2)[2]
    ro = P.RansacOpt(max_iterations=1000, min_iterations=100, seed=3)
    a, b = both(lambda: P.ransac_relpose_cameras(d1, d2, cam, cam, ro, 1.5))
    _close_runs(a, b)
    pose = a["model"]
    u1, M1 = P.camera_unproject_with_jac(cam, d1)
    u2, M2 = P.camera_unproject_with_jac(cam, d2)
    for thr in (0.5, 2.25, 30.0):
        assert same(*both(lambda: P.score_tangent(pose, u1, u2, M1, M2, thr, True)))
    pert = pose.copy()
    pert[4:] += 0.01
    ra, rb = both(lambda: P.refine_relpose_tangent(pert, u1, u2, M1, M2, P.BundleOpt()))
    assert maxdiff(ra, rb) < 1e-9  # Vector4d::norm() order, see the module docstring
    for ts in (False, True):
        _close_runs(*both(lambda: P.estimate("relpose", d1, d2, ro, P.BundleOpt(), 1.5, cam, cam, tangent_sampson=ts)))
    q = G.config_c1(1)
    xd = P.camera_project_with_jac(cam, np.c_[q["x"] / G.FOCAL, np.ones(len(q["x"]))])[2]
    for c in (cam, CAMERAS[4]):
        xd = P.camera_project_with_jac(c, np.c_[q["x"] / G.FOCAL, np.ones(len(q["x"]))])[2]
        a, b = both(lambda: P.estimate("pnp", xd, q["X"], P.RansacOpt(**q["ransac"]), P.BundleOpt(), 12.0, c))
        assert same(a, b) and a["stats"]["num_inliers"] >= 90


# ---- edge sizes -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["relpose", "fundamental", "homography", "pnp"])
def test_edge_sizes_agree_in_all_discrete_outputs(kind):
    """Fewer points than the sample size, exactly the sample size, all inliers, all outliers, max < min iterations:
    the reference's sources and the oracle take the same path (iterations, refinements, inlier count, mask)."""
    for n in (2, 3, 4, 5, 6, 7, 8, 9, 12, 30):
        for ratio in (1.0, 0.5, 0.0):
            if kind == "pnp":
                q = G.abspose_problem(max(n, 10), ratio, 1, n)
                a1, a2, thr, kw = q["x"][:n], q["X"][:n], 12.0, dict(cam1=CAMT)
            elif kind == "homography":
                h = G.homography_problem(max(n, 10), ratio, 4, n)
                a1, a2, thr, kw = h["x1"][:n], h["x2"][:n], 1.0, {}
            else:
                p = G.relpose_problem(max(n, 10), ratio, 2, n)
                a1, a2, thr = p["x1"][:n], p["x2"][:n], 1.0
                kw = dict(cam1=CAMT, cam2=CAMT) if kind == "relpose" else {}
            for ro in (P.RansacOpt(max_iterations=200, min_iterations=20, seed=n),
                       P.RansacOpt(max_iterations=10, min_iterations=50, seed=n)):
                a, b = both(lambda: P.estimate(kind, a1, a2, ro, P.BundleOpt(), thr, **kw))
                sa, sb = a["stats"], b["stats"]
                assert (sa["iterations"], sa["refinements"], sa["num_inliers"]) == \
                       (sb["iterations"], sb["refinements"], sb["num_inliers"]), (kind, n, ratio)
                assert np.array_equal(a["inliers"], b["inliers"]), (kind, n, ratio)


# ---- sensitivity to Eigen's internal summation order ----------------------------------------------------------------
@pytest.mark.skipif(not P.ref2_available(variant="alt"), reason="oracle/_ref/libplref2_alt.so not built")
def test_outcome_does_not_depend_on_eigens_summation_order():
    """The one thing this image cannot pin is the order in which real Eigen adds up 3- and 4-term reductions.  The same
    reference sources are therefore also built with mini-Eigen's reductions in the order Eigen 3.4 is recalled to use in an
    SSE2 build (2-wide packets combined as a tree: (x0+x2)+(x1+x3); tree-shaped inner sums in coefficient-based products:
    x0+(x1+x2)) — `make -C oracle ref2alt`.  On every fixture case (tests/golden/reference_cases.py: all RANSAC and
    estimate_* cases of the GPU parity suite) both orders give the same iterations, refinements, inlier counts and inlier
    masks; the MSAC scores agree to 1e-13 and the models to 1e-9 (relative poses compared up to the |t| gauge, which
    is the one quantity that drifts, by up to 1e-5)."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import reference_cases as RC
    worst_model = []
    for name in sorted(RC.CASES):
        case = RC.CASES[name]()
        with P.reference_sources():
            a = RC.run(P, case)
        with P.reference_sources(alt=True):
            b = RC.run(P, case)
        sa, sb = a["stats"], b["stats"]
        assert (sa["iterations"], sa["refinements"], sa["num_inliers"]) == (sb["iterations"], sb["refinements"], sb["num_inliers"]), name
        assert np.array_equal(a["inliers"], b["inliers"]), name
        assert abs(sa["model_score"] - sb["model_score"]) <= 1e-13 * abs(sa["model_score"]), name
        am, bm = np.asarray(a["model"], dtype=float), np.asarray(b["model"], dtype=float)
        if case["kind"] == "relpose":  # |t| is a gauge freedom (see _close_runs): it drifts by up to 1e-5, the direction does not
            am = np.r_[am[:4], am[4:] / np.linalg.norm(am[4:])]
            bm = np.r_[bm[:4], bm[4:] / np.linalg.norm(bm[4:])]
        d = np.abs(am - bm).max()
        if am.ndim == 2:
            d = min(d, np.abs(am + bm).max())
        worst_model.append(d / np.abs(am).max())
    assert max(worst_model) < 1e-9 and np.median(worst_model) < 1e-12


# ---- the operation order of the generated expansions is the ONLY difference ---------------------------------------
REF_5PT = "/root/reference/PoseLib/solvers/relpose_5pt.cc"


def _parse_reference_det_terms():
    """The term order of the degree-10 determinant expansion (relpose_5pt.cc:191-352), read from the reference's source at
    run time: rows (k, sign, r0, c0, r1, c1, r2, c2).  Nothing of it is stored in this repository."""
    import re
    src = open(REF_5PT).read()
    i = src.index("double c[11];")
    j = src.index("bisect_sturm", i)
    rows = []
    for m in re.finditer(r"c\[(\d+)\]\s*=\s*(.*?);", src[i:j], re.S):
        k, expr = int(m.group(1)), re.sub(r"\s+", " ", m.group(2))
        for sg, t in re.findall(r"([+-]?)\s*(A\(\d+, \d+\) \* A\(\d+, \d+\) \* A\(\d+, \d+\))", expr):
            f = [int(v) for ab in re.findall(r"A\((\d+), (\d+)\)", t) for v in ab]
            rows.append([k, -1 if sg == "-" else 1] + f)
    return rows


@pytest.fixture
def reference_order():
    import os
    if not os.path.exists(REF_5PT):
        pytest.skip("needs the reference's source file to read the term order from")
    P.set_reference_order(True, _parse_reference_det_terms())
    try:
        yield
    finally:
        P.set_reference_order(False)


def test_incomplete_order_tables_are_rejected():
    import os
    if not os.path.exists(REF_5PT):
        pytest.skip("needs the reference's source file")
    rows = _parse_reference_det_terms()
    assert len(rows) == 480
    try:
        with pytest.raises(ValueError):
            P.set_reference_order(True, rows[:-1])  # one term missing
        bad = [r[:] for r in rows]
        bad[7][1] = -bad[7][1]  # one sign flipped
        with pytest.raises(ValueError):
            P.set_reference_order(True, bad)
    finally:
        P.set_reference_order(False)


def test_with_the_reference_operation_order_the_solvers_are_bit_identical(reference_order):
    """relpose_5pt (trace constraints by rule, determinant expansion in the injected order) and relpose_7pt (cubic by
    rule) — the two places where the oracle's default order differs — equal the reference's sources bit for bit."""
    for s in range(300):
        x1, x2, _, _ = G.minimal_relpose(s, 5)
        a, b = both(lambda: P.relpose_5pt_E(x1, x2))
        assert a.shape == b.shape and np.array_equal(a, b), s
        a, b = both(lambda: P.relpose_5pt(x1, x2))
        assert a.shape == b.shape and np.array_equal(a, b), s
        x1, x2, _, _ = G.minimal_relpose(s, 7)
        a, b = both(lambda: P.relpose_7pt(x1, x2))
        assert a.shape == b.shape and np.array_equal(a, b), s


def test_with_the_reference_operation_order_the_whole_path_is_bit_identical(reference_order):
    """estimate_* for all four kinds on 240 random problems — sizes 8..800, inlier ratios 0.1..1, all four losses, PROSAC
    on/off, and DEGENERATE data (identical views + noise, duplicated points, pure zoom, planar 3D points, collinear image
    points) where the default order's last-bit differences decide ties: stats, masks, scores and models all identical."""
    rng = np.random.default_rng(123)
    for it in range(240):
        kind = ["relpose", "fundamental", "homography", "pnp"][it % 4]
        n = int(rng.choice([8, 15, 40, 100, 300, 800]))
        ratio = float(rng.choice([0.1, 0.3, 0.6, 0.9, 1.0]))
        mode = int(rng.integers(0, 5))
        if kind == "pnp":
            p = G.abspose_problem(n, ratio, 1, it)
            a1, a2, thr, kw = p["x"].copy(), p["X"].copy(), float(rng.choice([2.0, 12.0])), dict(cam1=CAMT)
            if mode == 1:
                a2[:, 2] = a2[:, 2].mean()
            if mode == 2:
                a1[:n // 2], a2[:n // 2] = a1[0], a2[0]
        elif kind == "homography":
            p = G.homography_problem(n, ratio, 4, it)
            a1, a2, thr, kw = p["x1"].copy(), p["x2"].copy(), float(rng.choice([0.5, 3.0])), {}
            if mode == 2:
                a1[:n // 2], a2[:n // 2] = a1[0], a2[0]
            if mode == 3:
                a1[:, 1] = a1[:, 0] * 0.5 + 3
        else:
            p = G.relpose_problem(n, ratio, 2, it)
            a1, a2, thr = p["x1"].copy(), p["x2"].copy(), float(rng.choice([0.5, 3.0]))
            kw = dict(cam1=CAMT, cam2=CAMT) if kind == "relpose" else {}
            if mode == 1:
                a2 = a1 + rng.normal(0, 0.3, a1.shape)
            if mode == 2:
                a1[:n // 2], a2[:n // 2] = a1[0], a2[0]
            if mode == 3:
                a2 = a1 * 1.1
        ro = P.RansacOpt(max_iterations=int(rng.choice([50, 500, 3000])), min_iterations=int(rng.choice([10, 100])),
                         seed=int(rng.integers(0, 1 << 30)), progressive_sampling=bool(rng.integers(0, 2)))
        bo = P.BundleOpt(loss_type=str(rng.choice(["TRIVIAL", "TRUNCATED", "HUBER", "CAUCHY"])))
        a, b = both(lambda: P.estimate(kind, a1, a2, ro, bo, thr, **kw))
        assert a["stats"] == b["stats"], (it, kind, n, ratio, mode, a["stats"], b["stats"])
        assert np.array_equal(a["inliers"], b["inliers"]), (it, kind)
        assert np.array_equal(a["model"], b["model"], equal_nan=True), (it, kind)


def test_with_the_reference_operation_order_the_fixture_cases_are_bit_identical(reference_order):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import reference_cases as RC
    for name in sorted(RC.CASES):
        case = RC.CASES[name]()
        a, b = both(lambda: RC.run(P, case))
        assert a["stats"] == b["stats"] and np.array_equal(a["inliers"], b["inliers"]), name
        assert np.array_equal(a["model"], b["model"]), name


def test_with_the_reference_operation_order_the_tangent_sampson_path_is_bit_identical(reference_order):
    """Distorted cameras: ransac_relpose(cameras), the tangent-Sampson refiner (Vector4d::norm() left to right, the oracle's
    own convention, instead of the packet order it models by default in that one place) and estimate_relative_pose with
    and without tangent_sampson."""
    for cam, seed in ((CAMERAS[3], 5), (CAMERAS[4], 6), (CAMERAS[2], 7)):
        p = G.relpose_problem(1200, 0.5, 2, seed)
        X1 = np.c_[p["x1"] / G.FOCAL, np.ones(len(p["x1"]))]
        X2 = np.c_[p["x2"] / G.FOCAL, np.ones(len(p["x2"]))]
        d1, d2 = P.camera_project_with_jac(cam, X1)[2], P.camera_project_with_jac(cam, X2)[2]
        ro = P.RansacOpt(max_iterations=1000, min_iterations=100, seed=seed)
        a, b = both(lambda: P.ransac_relpose_cameras(d1, d2, cam, cam, ro, 1.5))
        assert same(a, b)
        u1, M1 = P.camera_unproject_with_jac(cam, d1)
        u2, M2 = P.camera_unproject_with_jac(cam, d2)
        pert = a["model"].copy()
        pert[4:] += 0.01
        for loss in ("TRIVIAL", "TRUNCATED", "HUBER", "CAUCHY"):
            bo = P.BundleOpt(loss_type=loss, loss_scale=1.0)
            assert same(*both(lambda: P.refine_relpose_tangent(pert, u1, u2, M1, M2, bo))), loss
        for ts in (False, True):
            assert same(*both(lambda: P.estimate("relpose", d1, d2, ro, P.BundleOpt(), 1.5, cam, cam, tangent_sampson=ts)))
