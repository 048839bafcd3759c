"""Independent pins of the pieces of the oracle that restate THIRD-PARTY code absent from the reference tree
(Ceres 2.0 trust region / dogleg, Open3D KDTreeFlann) -- the reference holds no tests or golden vectors, so these are
the strongest checks available in this image (VERDICT r1, "pin what can be pinned"):

  * min_on_boundary_2d (our bracketing + bisection) against the roots of the QUARTIC Ceres solves
    (dogleg_strategy.cc MakePolynomialForBoundaryConstrainedProblem / FindMinimumOnTrustRegionBoundary), via numpy.roots;
  * the converged pose of a fixed-correspondence, plane-only problem against scipy.optimize.least_squares(loss='cauchy')
    (same objective: 1/2 sum log(1 + r_i^2), 1-D residual blocks) and first-order optimality by finite differences;
  * exact kNN against FLANN (cv2.flann, exhaustive checks; answers recorded in tests/golden/opencv_pins.npz) besides cKDTree;
  * the trust-region bookkeeping under a SMALL initial radius (dogleg boundary steps, rejected steps, radius updates):
    invariants that hold for Ceres' DoglegStrategy whatever the problem.
"""
import os

import numpy as np
import pytest
import scipy.optimize
from scipy.linalg import expm

from tloam_b200 import synth

BIG = 10 ** 9
CAPS = dict(edge_maxnum=BIG, sphere_maxnum=BIG, planar_maxnum=BIG, ground_maxnum=BIG)


def hat(w):
    return np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])


def exp_se3(a):
    M = np.zeros((4, 4))
    M[:3, :3] = hat(a[3:])
    M[:3, 3] = a[:3]
    return expm(M)


from tests_helpers_quartic import boundary_min_quartic  # noqa: E402


def test_min_on_boundary_2d_against_the_quartic_roots(oracle):
    rng = np.random.default_rng(3)
    for trial in range(300):
        A = rng.normal(size=(2, 2))
        B = A @ A.T * 10 ** rng.uniform(-3, 3) + np.eye(2) * 10 ** rng.uniform(-6, 0)     # SPD like the subspace model
        if trial % 7 == 0:
            B = A + A.T                                                                    # and indefinite ones
        g = rng.normal(size=2) * 10 ** rng.uniform(-3, 3)
        r = 10 ** rng.uniform(-4, 2)
        y = oracle.min_on_boundary_2d(B, g, r)
        yq, fq = boundary_min_quartic(B, g, r)
        Bs = 0.5 * (B + B.T)
        fy = 0.5 * y @ Bs @ y + g @ y
        scale = abs(fq) + r * np.linalg.norm(g) + r * r * np.abs(Bs).max()
        assert abs(np.linalg.norm(y) - r) <= 1e-12 * r
        assert fy <= fq + 1e-9 * scale, (trial, fy, fq)         # at least as good as the best quartic root ...
        assert fy >= fq - 1e-9 * scale, (trial, fy, fq)         # ... and not better than the global minimum
        if np.linalg.norm(y - yq) > 1e-5 * r:                   # different point: only legitimate on a (near) tie
            assert abs(fy - fq) <= 1e-9 * scale


def plane_problem(seed=11, scale=0.03):
    cfg = synth.scaled(scale, seed=seed)
    T_gt = synth.se3_exp([1.0, -0.5, 0.0, 0.01, -0.02, 0.25])
    mp, scan = synth.make_map(cfg, T_gt), synth.make_scan(cfg, T_gt, 1)
    predict = T_gt @ synth.se3_exp(np.asarray(synth.CONFIG1_PERTURB) * 0.5)
    return mp, scan, predict


def test_fixed_correspondence_solve_against_scipy_cauchy_least_squares(oracle):
    """ONE outer iteration = one Ceres solve over fixed correspondences.  Plane factors are 1-D residual blocks, so
    Ceres' CauchyLoss(1.0) objective 1/2 sum log(1 + r_i^2) is exactly scipy's loss='cauchy', f_scale=1."""
    mp, scan, predict = plane_problem()
    cfg = dict(factor_num=2, max_iterations=1, ceres_max_num_iterations=8, **CAPS)
    o = oracle.Oracle(**cfg)
    o.set_input_target(mp)
    o.set_input_source(scan)
    x0 = oracle.se3_log(predict)
    P, N, D = [], [], []
    for cloud in (2, 3):
        valid, prim = o.build_factors(cloud, x0)
        m = valid.astype(bool)
        P.append(scan[cloud][m]); N.append(prim[m, :3]); D.append(prim[m, 3])
    P, N, D = np.concatenate(P), np.concatenate(N), np.concatenate(D)
    assert len(P) > 300
    rc, T, st = o.scan_matching(predict)
    assert rc == 0 and st.n_outer == 1 and sum(st.outer[0].n_factors) == len(P)

    def resid(a):                      # PointToPlaneErr (ref: registration.cpp:96-117), weight 1
        M = exp_se3(a)
        return np.einsum("ij,ij->i", P @ M[:3, :3].T + M[:3, 3], N) + D

    def cost(a):
        return 0.5 * np.sum(np.log1p(resid(a) ** 2))

    assert np.isclose(st.outer[0].initial_cost, cost(x0), rtol=1e-12)
    sol = scipy.optimize.least_squares(resid, x0, loss="cauchy", f_scale=1.0, method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15,
                                       x_scale=1.0, max_nfev=400)
    x_or = np.array(st.x_final)
    # the restated trust-region loop stops on Ceres' function tolerance (1e-6 relative), scipy runs to 1e-15:
    d = np.linalg.inv(exp_se3(sol.x)) @ T
    dt, dr = np.linalg.norm(d[:3, 3]), np.arccos(np.clip((np.trace(d[:3, :3]) - 1) / 2, -1, 1))
    assert dt < 2e-5 and dr < 2e-6, (dt, dr)
    assert cost(x_or) <= cost(sol.x) * (1 + 1e-6)
    assert np.isclose(st.outer[0].final_cost, cost(x_or), rtol=1e-10)
    # first-order optimality of the oracle's answer by central differences through the left perturbation
    g0 = np.zeros(6); g1 = np.zeros(6)
    for k in range(6):
        e = np.zeros(6); e[k] = 1e-6
        for gvec, xx in ((g0, x0), (g1, x_or)):
            M = exp_se3(xx)
            fp = 0.5 * np.sum(np.log1p((np.einsum("ij,ij->i", P @ (exp_se3(e) @ M)[:3, :3].T + (exp_se3(e) @ M)[:3, 3], N) + D) ** 2))
            fm = 0.5 * np.sum(np.log1p((np.einsum("ij,ij->i", P @ (exp_se3(-e) @ M)[:3, :3].T + (exp_se3(-e) @ M)[:3, 3], N) + D) ** 2))
            gvec[k] = (fp - fm) / 2e-6
    assert np.linalg.norm(g1) < 2e-3 * np.linalg.norm(g0), (np.linalg.norm(g0), np.linalg.norm(g1))


def test_knn_against_flann_exhaustive(oracle):
    # FLANN_INDEX_KDTREE_SINGLE (= flann::KDTreeSingleIndexParams, the exact tree Open3D's KDTreeFlann builds), exhaustive
    # checks, through OpenCV: its answers are recorded in tests/golden/opencv_pins.npz (tools/make_golden.py opencv)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "opencv_pins.npz"))
    pts, qs, idx_f, d2_f = g["knn_points"], g["knn_queries"], g["flann_idx"], g["flann_d2"]
    r = 3.0
    idx, d2, cnt = oracle.knn(pts.astype(np.float64), qs.astype(np.float64), r, 5)
    for i in range(len(qs)):
        inside = d2_f[i] < np.float32(r * r)
        k = int(inside.sum())
        # FLANN works in float32: compare the neighbour SETS where float32 leaves no doubt (gap to the radius / next one)
        if np.any(np.abs(d2_f[i] - r * r) < 1e-3):
            continue
        assert cnt[i] == k
        assert set(idx[i, :k]) == set(idx_f[i, :k]) or np.min(np.diff(np.sort(d2_f[i]))) < 1e-4


@pytest.mark.parametrize("radius", [1e-3, 1e-2, 1e-1])
def test_small_trust_region_radius_drives_the_dogleg_branches(oracle, radius):
    """initial_trust_region_radius << |Gauss-Newton step|: every first step is a dogleg step ON the boundary
    (|step| = radius, used_gauss_newton = 0), accepted steps with rho > 0.75 grow the radius to max(radius, 3 |step|),
    rejected steps halve it, the cost never increases -- DoglegStrategy / TrustRegionMinimizer invariants."""
    mp, scan, predict = plane_problem(seed=12)
    o = oracle.Oracle(initial_trust_region_radius=radius, ceres_max_num_iterations=8, **CAPS)
    o.set_input_target(mp)
    o.set_input_source(scan)
    rc, T, st = o.scan_matching(predict)
    assert rc == 0
    boundary = 0
    for oi in range(st.n_outer):
        ot = st.outer[oi]
        rad = radius
        cost = ot.initial_cost
        for ii in range(min(ot.n_inner, 8)):
            it = ot.inner[ii]
            assert np.isclose(it.radius, rad, rtol=1e-12), (oi, ii, it.radius, rad)
            if not it.used_gauss_newton:
                boundary += 1
                assert np.isclose(it.step_norm_scaled, it.radius, rtol=1e-9)
            else:
                assert it.step_norm_scaled <= it.radius * (1 + 1e-12)
            if it.accepted == 1:
                assert it.model_cost_change > 0 and it.relative_decrease > 1e-3
                assert it.candidate_cost < cost
                cost = it.candidate_cost
                if it.relative_decrease < 0.25:
                    rad *= 0.5
                if it.relative_decrease > 0.75:
                    rad = max(rad, 3.0 * it.step_norm_scaled)
            elif it.accepted == 0:
                assert it.relative_decrease <= 1e-3
                rad *= 0.5
        assert ot.final_cost <= ot.initial_cost * (1 + 1e-12)
    assert boundary >= 2           # the boundary branch really ran (never with the default radius 1e4)
