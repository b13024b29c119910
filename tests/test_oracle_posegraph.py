"""Pose-graph terms of the BundleGraph (SURVEY.md section 8f-3: GSLAM::SE3Edge / GPSEdge, Optimizer.h:127-148) in the BA oracle
(oracle/ba_ref.c).  PARITY UNPINNED by reference tests (the reference has no optimiser); pinned here: the SE3 logarithm and product
against the reference's own SE3 class (tests/golden/reference_se3.npz), the edge conventions against the reference's comments (SE3_12 = SE3_1^-1 SE3_2:
zero residual on consistent measurements), the gradient against central differences of the cost, and the optimum against an
independent scipy least-squares on the stacked residuals."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from gslam_b200 import synth


def retract_wc(pose_wc, d):
    """T_cw <- Exp(d) T_cw expressed on the T_wc the problem stores."""
    out = pose_wc.copy()
    L = O.lib()
    for i in range(pose_wc.shape[0]):
        cw = np.zeros(7); new = np.zeros(7); back = np.zeros(7)
        L.orc_se3_inverse(pose_wc[i].ctypes.data, cw.ctypes.data)
        L.orc_se3_retract(cw.ctypes.data, np.ascontiguousarray(d[i]).ctypes.data, new.ctypes.data)
        L.orc_se3_inverse(new.ctypes.data, back.ctypes.data)
        out[i] = back
    return out


def test_se3_log_and_product_equal_the_reference_class():
    rng = np.random.default_rng(0)
    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_se3.npz"))   # written through oracle/_ref
    for k in range(200):
        scale = [1e-12, 1e-6, 0.3, 2.5][k % 4]
        a = synth._small_se3(rng, 1, 1.0, scale)[0]; b = synth._small_se3(rng, 1, 2.0, 1.0)[0]
        if k % 7 == 0:
            a[:4] = -a[:4]                                     # the other quaternion of the same rotation
        want = ref["se3_log"][k]
        assert np.allclose(O.se3_log(a), want, rtol=0, atol=1e-14)
        wm = ref["se3_mul"][k]
        assert np.allclose(O.se3_mul(a, b), wm, rtol=0, atol=1e-14)
        assert np.allclose(synth.se3_mul(a, b), wm, rtol=0, atol=1e-13)     # the generator's numpy algebra too


def test_consistent_measurements_have_zero_residual():
    """Optimizer.h:127-148: SE3_12 := SE3_1^-1 * SE3_2 and SE3_gps := SE3_frame -- at the ground truth with noise-free measurements the
    pose-graph cost vanishes and the estimate is a fixed point."""
    pb = synth.synth_ba(12, 0, n_fixed=1, seed=2)
    pb.cam_pose_wc[...] = pb.gt_pose_wc
    pe = synth.synth_pose_edges(pb, seed=1, n_loops=6, gps_every=3, sigma_t=0.0, sigma_r=0.0, with_info=True)
    assert O.ba_cost(pb, 0.01, pe) < 1e-24
    r = O.ba_solve(pb, pe, max_iterations=3, function_tolerance=0.0)
    assert r.final_cost < 1e-24 and np.allclose(pb.cam_pose_wc, pb.gt_pose_wc, atol=1e-12)


@pytest.mark.parametrize("with_info", [False, True])
def test_gradient_matches_central_differences(with_info):
    pb = synth.synth_ba(8, 40, obs_per_point=3, n_fixed=0, seed=5, pose_sigma_t=0.1, pose_sigma_deg=3.0)
    pe = synth.synth_pose_edges(pb, seed=3, n_loops=4, gps_every=2, with_info=with_info)
    lin = O.ba_linearize(pb, 0.0, pe)      # (Huber off: the cost is smooth)
    only_obs = O.ba_linearize(pb, 0.0)
    g_pose = lin["gc"] - only_obs["gc"]     # the pose-graph part of -gradient
    assert np.abs(g_pose).max() > 0
    h = 1e-6
    for i in range(pb.n_cams):
        for a in range(6):
            d = np.zeros((pb.n_cams, 6)); d[i, a] = h
            plus = pb.copy(); plus.cam_pose_wc = retract_wc(pb.cam_pose_wc, d)
            minus = pb.copy(); minus.cam_pose_wc = retract_wc(pb.cam_pose_wc, -d)
            pose_cost = lambda q: O.ba_cost(q, 0.0, pe) - O.ba_cost(q, 0.0)
            num = (pose_cost(plus) - pose_cost(minus)) / (2 * h)
            assert abs(-num - g_pose[i, a]) <= 1e-6 * np.abs(g_pose).max() + 1e-9, (i, a, num, g_pose[i, a])
    # the Hessian blocks are symmetric positive semi-definite and the off-diagonal coupling reaches the reduced system
    S, gt, dc, it = O.ba_reduced_system(pb, 0.0, 0.0, 1, 1e-10, pe)
    S0, _, _, _ = O.ba_reduced_system(pb, 0.0, 0.0, 1, 1e-10)
    D = S - S0
    assert np.allclose(D, D.T, atol=1e-9) and np.linalg.eigvalsh(D).min() > -1e-8
    i, j = int(pe.se3_first[0]), int(pe.se3_second[0])
    assert np.abs(D[6 * i:6 * i + 6, 6 * j:6 * j + 6]).max() > 0


def test_pose_graph_optimum_equals_an_independent_least_squares():
    """A pure pose graph (no landmarks): the oracle's LM against scipy.optimize.least_squares on the stacked whitened residuals
    L' Log(Z^-1 T_1^-1 T_2) (numerical Jacobian: nothing of the oracle's linearisation is shared)."""
    scipy_opt = pytest.importorskip("scipy.optimize")
    pb = synth.synth_ba(10, 0, n_fixed=1, seed=7, pose_sigma_t=0.05, pose_sigma_deg=0.5)
    pe = synth.synth_pose_edges(pb, seed=2, n_loops=5, gps_every=0, with_info=True)
    a = pb.copy()
    r = O.ba_solve(a, pe, max_iterations=60, function_tolerance=0.0, pcg_max_iters=500, pcg_tol=1e-14)
    assert r.final_cost < r.initial_cost
    chol = [np.linalg.cholesky(0.5 * (M.reshape(6, 6) + M.reshape(6, 6).T)) for M in pe.se3_info]
    base = pb.cam_pose_wc.copy()

    def residuals(x):
        d = np.zeros((pb.n_cams, 6)); d[1:] = x.reshape(-1, 6)
        T = retract_wc(base, d)
        out = []
        for k in range(pe.n_se3):
            E = O.se3_mul(synth.se3_inv(pe.se3_meas[k]), O.se3_mul(synth.se3_inv(T[pe.se3_first[k]]), T[pe.se3_second[k]]))
            out.append(chol[k].T @ O.se3_log(E))
        return np.concatenate(out)
    sol = scipy_opt.least_squares(residuals, np.zeros(6 * (pb.n_cams - 1)), xtol=1e-14, ftol=1e-14, gtol=1e-14)
    assert abs(sol.cost - r.final_cost) <= 1e-9 * max(sol.cost, 1e-12) + 1e-12, (sol.cost, r.final_cost)


def test_mixed_graph_solves_and_respects_fixed_frames():
    pb = synth.synth_ba(20, 300, obs_per_point=4, n_fixed=2, seed=3)
    pe = synth.synth_pose_edges(pb, seed=1, n_loops=5, gps_every=4, with_info=True)
    a = pb.copy()
    r = O.ba_solve(a, pe, max_iterations=15, function_tolerance=0.0, pcg_max_iters=300, pcg_tol=1e-12)
    assert r.final_cost < 0.05 * r.initial_cost and r.accepted >= 10
    assert np.allclose(a.cam_pose_wc[:2], pb.cam_pose_wc[:2], atol=1e-12)
    assert abs(O.ba_cost(a, 0.01, pe) - r.final_cost) <= 1e-12 * r.final_cost
    # invalid edges are refused
    bad = synth.synth_pose_edges(pb, seed=1); bad.se3_second[0] = pb.n_cams
    with pytest.raises(Exception):
        O.ba_solve(pb.copy(), bad, max_iterations=1)
