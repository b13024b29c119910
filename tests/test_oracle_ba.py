"""Pins oracle/ba_ref.c: pose conventions against the reference's own SE3 class (tests/golden/reference_se3.npz), Jacobians against finite
differences, the optimum against scipy.optimize.least_squares (tests/golden/ba_golden.npz), plus known answers
(SURVEY.md §8c KAT-B).  The reference ships no BA implementation or test, so beyond these the parity is unpinned."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
from gslam_b200 import synth
from gslam_b200.synth import BAProblem

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "ba_golden.npz"))
REF = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_se3.npz"))   # written through oracle/_ref


def golden_problem() -> BAProblem:
    return BAProblem(cam_pose_wc=G["cam_pose_wc"].copy(), cam_dof=G["cam_dof"].copy(), points=G["points"].copy(),
                     point_free=G["point_free"].copy(), obs_cam=G["obs_cam"].copy(), obs_point=G["obs_point"].copy(),
                     obs_xyz=G["obs_xyz"].copy())


def rand_pose(rng):
    q = rng.standard_normal(4); q /= np.linalg.norm(q)
    return np.concatenate([q, rng.standard_normal(3)])


def test_layout_sizes_match_reference():
    want = {"KeyPoint": 28, "SE3": 56, "SIM3": 64, "Point3d": 24, "BundleEdge": 48, "KeyFrameEstimzation": 72,
            "MapPointEstimation": 32, "GImage": 32}
    sizes = dict(zip(REF["sizeof_names"].tolist(), REF["sizeof"].tolist()))
    for k, v in want.items():
        assert sizes[k] == v, k
    offs = REF["keypoint_offsets"].tolist()
    assert offs == [0, 4, 8, 12, 16, 20, 24]  # == gb_keypoint / KP_DTYPE
    from gslam_b200.capi import KP_DTYPE
    assert [KP_DTYPE.fields[n][1] for n in KP_DTYPE.names] == offs
    # SIM3 raw memory = pose7 + scale: what the plugin memcpy's into gb_ba_problem.cam_pose_wc
    p = rand_pose(np.random.default_rng(0)); raw = REF["sim3_raw"]
    assert np.array_equal(raw[:7], p) and raw[7] == 2.5


def test_se3_conventions_match_reference():
    rng = np.random.default_rng(1)
    L = oracle.lib()
    for i in range(200):
        T = rand_pose(rng); p = rng.standard_normal(3)
        inv_ref = REF["se3_inverse"][i]; inv_orc = np.zeros(7)
        L.orc_se3_inverse(T.ctypes.data, inv_orc.ctypes.data)
        assert np.allclose(inv_ref, inv_orc, atol=1e-14)
        # camera-frame point q = T_wc^-1 * p  (SE3.h:100-103,129-131) is what the residual uses
        q_ref = REF["se3_transform"][i]
        Rm = synth._quat_to_R(inv_orc[:4])
        assert np.allclose(q_ref, Rm @ p + inv_orc[4:], atol=1e-13)
        # retraction Exp([v,w]) * T equals the reference's exp()*T away from w=0 (where the reference is NaN)
        d = 0.3 * rng.standard_normal(6)
        want = REF["se3_exp_mul"][i].copy()
        got = np.zeros(7); L.orc_se3_retract(T.ctypes.data, d.ctypes.data, got.ctypes.data)
        if want[3] * got[3] < 0: want[:4] = -want[:4]
        assert np.allclose(want, got, atol=1e-12)
    # small-angle: finite where the reference's exp is not (SE3.h:284-285)
    d = np.array([0.1, 0.2, 0.3, 0, 0, 0.0]); T = rand_pose(rng); got = np.zeros(7)
    L.orc_se3_retract(T.ctypes.data, d.ctypes.data, got.ctypes.data)
    assert np.isfinite(got).all() and np.allclose(got[:4], T[:4]) and np.allclose(got[4:], T[4:] + d[:3])


def test_gradient_matches_finite_differences():
    pb = synth.synth_ba(6, 40, obs_per_point=4, n_fixed=1, seed=3)
    delta = 0.01
    lin = oracle.ba_linearize(pb, delta)
    c0 = lin["cost"]
    assert abs(c0 - oracle.ba_cost(pb, delta)) < 1e-15
    eps = 1e-6
    L = oracle.lib()
    # cameras: perturb T_cw on the left, gradient g_c = -J'r  => dcost/dxi = -g_c
    for i in [1, 3, 5]:
        for a in range(6):
            vals = []
            for s in (+1, -1):
                q = pb.copy()
                cw = np.zeros(7); L.orc_se3_inverse(q.cam_pose_wc[i].ctypes.data, cw.ctypes.data)
                d = np.zeros(6); d[a] = s * eps
                out = np.zeros(7); L.orc_se3_retract(cw.ctypes.data, d.ctypes.data, out.ctypes.data)
                wc = np.zeros(7); L.orc_se3_inverse(out.ctypes.data, wc.ctypes.data)
                q.cam_pose_wc[i] = wc
                vals.append(oracle.ba_cost(q, delta))
            fd = (vals[0] - vals[1]) / (2 * eps)
            assert abs(fd + lin["gc"][i, a]) < 1e-6 * max(1.0, abs(fd)), (i, a, fd, lin["gc"][i, a])
    for j in [0, 7, 39]:
        for a in range(3):
            vals = []
            for s in (+1, -1):
                q = pb.copy(); q.points[j, a] += s * eps
                vals.append(oracle.ba_cost(q, delta))
            fd = (vals[0] - vals[1]) / (2 * eps)
            assert abs(fd + lin["gp"][j, a]) < 1e-6 * max(1.0, abs(fd))
    # fixed camera contributes no gradient
    assert np.all(lin["gc"][0] == 0) and np.all(lin["U"][0] == 0)


def test_noise_free_known_answer():
    pb = synth.synth_ba(10, 200, all_visible=True, n_fixed=2, pixel_sigma=0.0, seed=7)
    r = oracle.ba_solve(pb, max_iterations=50, function_tolerance=0.0, pcg_max_iters=200, pcg_tol=1e-14)
    assert r.final_cost < 1e-20
    assert np.abs(pb.points - pb.gt_points).max() < 1e-6
    a = pb.cam_pose_wc.copy(); b = pb.gt_pose_wc
    s = np.sign(np.sum(a[:, :4] * b[:, :4], axis=1))[:, None]
    assert np.abs(a[:, :4] * s - b[:, :4]).max() < 1e-8 and np.abs(a[:, 4:] - b[:, 4:]).max() < 1e-7


def test_optimum_matches_scipy_golden():
    pb = golden_problem()
    r = oracle.ba_solve(pb, huber_delta=0.0, max_iterations=200, function_tolerance=1e-14, pcg_max_iters=300, pcg_tol=1e-13)
    want = float(G["scipy_cost_nohuber"])
    assert abs(r.final_cost - want) / want < 1e-6, (r.final_cost, want)


def test_fixed_everything_is_a_noop():
    pb = synth.synth_ba(5, 30, obs_per_point=3, seed=2)
    pb.cam_dof[:] = 0; pb.point_free[:] = 0
    before = pb.copy()
    r = oracle.ba_solve(pb, max_iterations=3)
    assert np.array_equal(pb.points, before.points)
    assert np.allclose(pb.cam_pose_wc, before.cam_pose_wc, atol=1e-15)
    assert r.accepted == 0


def test_pnp_recovers_pose():
    rng = np.random.default_rng(5)
    pose = rand_pose(rng); pose[4:] *= 0.1
    cw = np.zeros(7); oracle.lib().orc_se3_inverse(pose.ctypes.data, cw.ctypes.data)
    Rm = synth._quat_to_R(cw[:4])
    pc = np.stack([rng.uniform(-2, 2, 100), rng.uniform(-2, 2, 100), rng.uniform(4, 10, 100)], axis=1)
    xyz = (pc - cw[4:]) @ Rm  # p_w = R^T (p_c - t)
    xy1 = np.concatenate([pc[:, :2] / pc[:, 2:3], np.ones((100, 1))], axis=1)
    init = pose.copy(); init[4:] += 0.05; init[:4] += 0.01; init[:4] /= np.linalg.norm(init[:4])
    out, r, info = oracle.ba_pnp(xyz, xy1, init, want_info=True, max_iterations=30, function_tolerance=0.0)
    if out[3] * pose[3] < 0: out[:4] = -out[:4]
    assert np.allclose(out, pose, atol=1e-9) and r.final_cost < 1e-20
    assert np.allclose(info, info.T) and np.all(np.linalg.eigvalsh(info) > 0)


def test_invalid_indices_rejected():
    pb = synth.synth_ba(4, 10, obs_per_point=2, seed=1)
    pb.obs_cam[0] = 99
    with pytest.raises(RuntimeError):
        oracle.ba_solve(pb, max_iterations=1)


@pytest.mark.parametrize("shape", [dict(nc=500, np_=100000, lo=8, hi=12, split=1), dict(nc=60, np_=5000, lo=1, hi=6, split=1),
                                   dict(nc=300, np_=300, lo=0, hi=300, split=2), dict(nc=7, np_=3, lo=200, hi=400, split=4)])
def test_large_graph_sweep_plan_covers_everything_once_and_is_balanced(shape):
    """Host logic of csrc/ba_sweep.cu (no device): the items dealt to the teams cover every camera slice and every landmark exactly
    once, landmark groups hold <= 128 observations / <= 32 landmarks (or are one long landmark), and the teams' costs are balanced."""
    import ctypes as C
    from gslam_b200 import capi
    rng = np.random.default_rng(shape["nc"])
    nc, npts, split = shape["nc"], shape["np_"], shape["split"]
    per_pt = rng.integers(shape["lo"], shape["hi"] + 1, npts)
    pt_off = np.concatenate([[0], np.cumsum(per_pt)]).astype(np.int32)
    no = int(pt_off[-1])
    cam_of = rng.integers(0, nc, no)
    cam_off = np.concatenate([[0], np.cumsum(np.bincount(cam_of, minlength=nc))]).astype(np.int32)
    n_teams = 592
    items = np.zeros((npts + nc * split + 8, 4), np.int32); team_off = np.zeros(n_teams + 1, np.int32); n = C.c_int(0)
    rc = capi.lib().gb_dbg_ba_sweep_plan(nc, npts, split, cam_off.ctypes.data, pt_off.ctypes.data, n_teams, items.ctypes.data, items.shape[0],
                                         team_off.ctypes.data, C.byref(n))
    assert rc == 0
    items = items[:n.value]
    assert team_off[0] == 0 and team_off[-1] == n.value and np.all(np.diff(team_off) >= 0)
    cams = items[items[:, 0] < 0]; grps = items[items[:, 0] >= 0]
    seen = sorted((int(-1 - a), int(b)) for a, b, _, _ in cams)
    assert seen == [(i, s) for i in range(nc) for s in range(split)]
    for a, b, s0, s1 in cams:                                  # the slices of a camera tile its observation range
        i = -1 - a
        assert cam_off[i] <= s0 <= s1 <= cam_off[i + 1]
    assert sum(int(s1 - s0) for _, _, s0, s1 in cams) == no
    order = np.argsort(grps[:, 0], kind="stable"); g = grps[order]
    assert g[0, 0] == 0 and g[-1, 1] == npts and np.array_equal(g[1:, 0], g[:-1, 1])     # landmarks: a partition, in order
    assert np.array_equal(g[:, 2], pt_off[g[:, 0]]) and np.array_equal(g[:, 3], pt_off[g[:, 1]])
    L = g[:, 1] - g[:, 0]; obs = g[:, 3] - g[:, 2]
    assert np.all(L <= 32) and np.all((obs <= 128) | (L == 1))
    cost = np.zeros(n_teams)
    for k in range(n_teams):
        for a, b, c, d in items[team_off[k]:team_off[k + 1]]:
            cost[k] += (0.4 * (d - c) + 150.0) if a < 0 else ((d - c) + 40.0)
    if n.value > 4 * n_teams:
        assert cost.max() < 1.25 * cost.mean() + 700.0


def test_multithreaded_oracle_equals_the_sequential_one():
    """bench.py's reference arm runs the BA port with OpenMP threads (orc_ba_set_threads); the regrouped loops must give the sequential
    sums (blocks bit for bit where only the loop nest changed, the cost and the Schur complement to rounding) and the same solve."""
    pb = synth.synth_ba(50, 2000, obs_per_point=5, n_fixed=2, seed=42)
    seq = oracle.ba_linearize(pb, 0.01)
    a = pb.copy(); r1 = oracle.ba_solve(a, max_iterations=6, function_tolerance=0.0)
    S1, g1, d1, _ = oracle.ba_reduced_system(pb, 0.01, 1e-4, 50, 1e-10)
    try:
        oracle.ba_set_threads(4)
        par = oracle.ba_linearize(pb, 0.01)
        for k in ("U", "gc", "V", "gp", "W"):
            assert np.array_equal(par[k], seq[k]), k
        assert abs(par["cost"] - seq["cost"]) <= 1e-14 * seq["cost"]
        S4, g4, d4, _ = oracle.ba_reduced_system(pb, 0.01, 1e-4, 50, 1e-10)
        assert np.abs(S4 - S1).max() <= 1e-12 * np.abs(S1).max() and np.abs(g4 - g1).max() <= 1e-12 * np.abs(g1).max()
        b = pb.copy(); r4 = oracle.ba_solve(b, max_iterations=6, function_tolerance=0.0)
    finally:
        oracle.ba_set_threads(1)
    assert r4.accepted == r1.accepted and abs(r4.final_cost - r1.final_cost) <= 1e-9 * r1.final_cost
    assert np.abs(b.cam_pose_wc - a.cam_pose_wc).max() < 1e-8
