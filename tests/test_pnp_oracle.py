"""CPU tests of the PnP oracle (oracle/pnp.py), the NumPy restatement of csrc/pnp.cu: exact scenes, the P3P
solution set against cv2.solveP3P, the degenerate samples, the Levenberg-Marquardt result against scipy's,
the fp32 inlier test against a plain float32 evaluation, the accuracy against the true motion, the
F RANSAC -> pose -> point_map -> PnP chain (whose bounds the GPU tests reuse), synth.two_view_bank's points,
geometry.point_map and geometry.rows_with_points."""

import cv2
import numpy as np
import pytest
import torch
from scipy.optimize import least_squares

from oracle import fundamental as of
from oracle import pnp as op
from oracle import pose as opose
from parity import record
from sslam_b200 import geometry, synth

KP = 2600
# Bounds of the chain on seeds 0-5 (largest oracle errors: 0.50 deg, 6.8 %), and of PnP alone against exact
# points (largest: 0.19 deg, 21 mm, seed 1: the refinement is not kept there because it loses one row).
CHAIN_ROT_DEG, CHAIN_T_REL = 0.6, 0.08
ALONE_ROT_DEG, ALONE_T_MM = 0.25, 25.0


def cam_of(K):
    return (K[0, 0], K[1, 1], K[0, 2], K[1, 2])


def rot_err_deg(Ra, Rb):
    return float(np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0))))


def exact_rows(seed, n=4):
    """Float64 (X in camera 1, exact pixel in camera 2) of n synth points, and the true (R, t), K."""
    bank, _, Rs, ts, K, Xs = synth.two_view_bank(2, max(n, 8), seed=seed, poses=True, points=True)
    p = Xs[1][:n] @ K.T
    return np.concatenate([Xs[0][:n], p[:, :2] / p[:, 2:]], 1), Rs[0], ts[0], K


def noisy_rows(seed):
    """Exact points of camera 1 against camera-2 keypoints with 0.3 px noise, 30 % outlier rows."""
    bank, _, Rs, ts, K, Xs = synth.two_view_bank(2, KP, seed=20 + seed, noise=0.3, poses=True, points=True)
    pairs, _, _, _ = synth.two_view_lists([2048], 2048, KP, inlier_frac=0.7, seed=30 + seed)
    r = pairs[0]
    return np.concatenate([Xs[0][r[:, 0]], bank[1][r[:, 1]]], 1).astype(np.float32), Rs[0], ts[0], K


@pytest.mark.parametrize("seed", range(8))
def test_exact_scene_p3p_has_true_pose(seed):
    q, R, t, K = exact_rows(seed)
    y = op.bearings(q[None, :3, 3:], cam_of(K))
    Rs, ts, valid = op.p3p(y, q[None, :3, :3])
    err = min(max(np.abs(Rs[0, i].reshape(3, 3) - R).max(), np.abs(ts[0, i] - t).max())
              for i in range(4) if valid[0, i])
    assert err < 1e-9
    # the fourth row picks the true pose
    Rp, tp, ok = op.sample_poses(q.astype(np.float32), cam_of(K), [0], seed=0)
    assert ok[0] and np.abs(Rp[0].reshape(3, 3) - R).max() < 1e-5


@pytest.mark.parametrize("seed", range(8))
def test_solution_set_equals_cv2_solve_p3p(seed):
    rng = np.random.default_rng(seed)
    K = np.array([[525.0, 0, 319.5], [0, 525.0, 239.5], [0, 0, 1]])
    total = 0
    for _ in range(50):
        X = rng.uniform([-3, -2, 4], [3, 2, 10], (3, 3))
        uv = (X @ K.T)[:, :2] / X[:, 2:]
        Rs, ts, valid = op.p3p(op.bearings(uv[None], cam_of(K)), X[None])
        mine = [(Rs[0, i].reshape(3, 3), ts[0, i]) for i in range(4) if valid[0, i]]
        n, cR, cT = cv2.solveP3P(X, uv, K, None, flags=cv2.SOLVEPNP_P3P)
        assert len(mine) == n
        for rv, tv in zip(cR, cT):
            Rc = cv2.Rodrigues(rv)[0]
            assert any(np.abs(Rc - a).max() < 1e-6 and np.abs(tv[:, 0] - b).max() < 1e-6 for a, b in mine)
        total += n
    record(f"pnp_p3p_vs_cv2_seed{seed}", {"samples": 50, "solutions": total})


def test_degenerate_samples():
    q, R, t, K = exact_rows(0, n=8)
    cam = cam_of(K)
    rows = q[:4].astype(np.float32)
    assert op.sample_poses(rows, cam, np.arange(8), 0)[2].all()
    # collinear and coincident solver points (rows 0-2 of every sample are these)
    for X in (np.array([[0.0, 0, 5], [1, 1, 6], [2, 2, 7], [3, 3, 8]]), np.array([[0.0, 0, 5]] * 3 + [[1, 0, 6]])):
        bad = rows.copy()
        bad[:, :3] = X
        assert not op.sample_poses(bad, cam, np.arange(16), 0)[2].any()
    # every point behind the camera
    back = rows.copy()
    back[:, :3] = -rows[:, :3]
    back[:, 3:] = rows[:, 3:]
    Rb, tb, ok = op.sample_poses(back, cam, np.arange(16), 0)
    for s in np.flatnonzero(ok):
        assert ((back[:, :3].astype(np.float64) @ Rb[s].reshape(3, 3).T + tb[s])[:, 2] > 0).all()
    # n < 4, and a NaN row
    assert not op.sample_poses(rows[:3], cam, np.arange(4), 0)[2].any()
    nanr = rows.copy()
    nanr[2, 0] = np.nan
    assert not op.sample_poses(nanr, cam, np.arange(16), 0)[2].any()
    o = op.ransac_pnp(rows[:3], cam, iters=16)
    assert o["best"] == -1 and not o["R"].any() and (o["hyp_count"] == -1).all()
    # a best sample without any inlier is no model either (t^2 = 1e-60 rounds to 0 in fp32: no row passes)
    o = op.ransac_pnp(rows, cam, iters=16, threshold=1e-30)
    assert o["best"] == 0 and (o["hyp_count"] == 0).all() and not o["R"].any() and not o["rms"].any()


@pytest.mark.parametrize("seed", range(4))
def test_lm_equals_scipy_least_squares(seed):
    rows, _, _, K = noisy_rows(seed)
    cam = cam_of(K)
    o = op.ransac_pnp(rows, cam, refine_iters=0)
    R0, t0 = o["R"], o["t"]
    inl = rows[o["hyp_mask"]]

    def res(x):
        return op.residuals(op.exp_so3(x[:3]) @ R0, t0 + x[3:], inl, cam)
    sol = least_squares(res, np.zeros(6), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000)
    Rs, ts = op.exp_so3(sol.x[:3]) @ R0, t0 + sol.x[3:]
    R, t, c0, c1, _ = op.refine(R0, t0, inl, cam, 100)
    assert np.abs(R - Rs).max() < 1e-9 and np.abs(t - ts).max() < 1e-9
    assert abs(c1 - float(np.sum(sol.fun ** 2))) <= 1e-9 * c1 and c1 < c0
    # the analytic Jacobian against central differences
    J = op.jacobian(R0, t0, inl[:50], cam)
    Jn = np.empty_like(J)
    for j in range(6):
        e = np.zeros(6)
        e[j] = 1e-6
        f = (lambda x: op.residuals(op.exp_so3(x[:3]) @ R0, t0 + x[3:], inl[:50], cam))
        Jn[:, j] = (f(e) - f(-e)) / 2e-6
    assert np.abs(J - Jn).max() <= 1e-4 * np.abs(J).max()


def test_fp32_inlier_test_equals_float32_numpy():
    rows, R, t, K = noisy_rows(0)
    cam = cam_of(K)
    h = op.to32(R, t)[0]
    X = rows[:, :3]
    Xc = np.stack([(X[:, 0] * h[3 * i] + X[:, 1] * h[3 * i + 1]) + X[:, 2] * h[3 * i + 2] + h[9 + i]
                   for i in range(3)], 1).astype(np.float32)
    fx, fy, cx, cy = (np.float32(v) for v in cam)
    iz = (np.float32(1) / Xc[:, 2]).astype(np.float32)
    e = ((fx * Xc[:, 0]) * iz + cx - rows[:, 3]) ** 2 + ((fy * Xc[:, 1]) * iz + cy - rows[:, 4]) ** 2
    assert e.dtype == np.float32
    ref = (Xc[:, 2] > 0) & (e < np.float32(9.0))
    assert np.array_equal(op.inliers(R, t, rows, cam, 3.0), ref)
    # and with a double evaluation away from the threshold
    e64 = op.residuals(R, t, rows, cam).reshape(2, -1)
    e64 = (e64 ** 2).sum(0)
    far = np.abs(e64 - 9.0) > 1e-3
    assert np.array_equal(ref[far], (e64 < 9.0)[far])


@pytest.mark.parametrize("seed", range(4))
def test_accuracy_against_true_motion(seed):
    rows, R, t, K = noisy_rows(seed)
    o = op.ransac_pnp(rows, cam_of(K))
    rot, tmm = rot_err_deg(o["R"], R), 1000.0 * float(np.linalg.norm(o["t"] - t))
    assert rot < ALONE_ROT_DEG and tmm < ALONE_T_MM, (rot, tmm)
    assert o["rms"][1] <= o["rms"][0]
    record(f"pnp_oracle_accuracy_seed{seed}", {"rot_deg": rot, "t_mm": tmm, "inliers": int(o["mask"].sum()),
                                               "refit_used": bool(o["refit_used"])})


def chain_inputs(seed):
    """Three-set bank and two lists: (0, 1) for the initialisation, (1, 2) for the tracking."""
    bank, _, Rs, ts, K, _ = synth.two_view_bank(3, KP, seed=40 + seed, noise=0.3, poses=True, points=True)
    pairs, scores, counts, _ = synth.two_view_lists([2048, 2048], 2048, KP, inlier_frac=0.7, seed=50 + seed)
    return bank, Rs, ts, K, pairs, scores, counts


def chain_errors(R, t, Rs, ts):
    s = ts[1] / np.linalg.norm(ts[0])
    return rot_err_deg(R, Rs[1]), float(np.linalg.norm(t - s) / np.linalg.norm(s))


def oracle_chain(seed):
    bank, Rs, ts, K, pairs, _, _ = chain_inputs(seed)
    cam = cam_of(K)
    r = pairs[0]
    pts = np.concatenate([bank[0][r[:, 0]], bank[1][r[:, 1]]], 1)
    f = of.verify_fundamental(pts, 1024, 3.0, 0)
    vr = r[f["mask"]]
    po = opose.recover_pose(pts[f["mask"]], K.T @ f["H"].reshape(3, 3) @ K, cam, refine_iters=10)
    M = np.full((KP, 3), np.nan)
    X2 = po["points"] @ po["R"].T + po["t"]
    for k in range(len(vr) - 1, -1, -1):                  # lowest row wins
        if po["mask"][k]:
            M[vr[k, 1]] = X2[k]
    r2 = pairs[1]
    rows = np.concatenate([M[r2[:, 0]], bank[2][r2[:, 1]]], 1).astype(np.float32)
    o = op.ransac_pnp(rows[np.isfinite(rows).all(1)], cam)
    return chain_errors(o["R"], o["t"], Rs, ts)


@pytest.mark.parametrize("seed", range(6))
def test_chain_against_true_motion(seed):
    rot, trel = oracle_chain(seed)
    assert rot < CHAIN_ROT_DEG and trel < CHAIN_T_REL, (rot, trel)
    record(f"pnp_oracle_chain_seed{seed}", {"rot_deg": rot, "t_rel": trel})


def test_two_view_bank_points():
    for seed, sets in ((0, 2), (3, 4)):
        bank, F = synth.two_view_bank(sets, 300, seed=seed, noise=0.3)
        out = synth.two_view_bank(sets, 300, seed=seed, noise=0.3, poses=True, points=True)
        assert len(out) == 6 and bank.tobytes() == out[0].tobytes() and F.tobytes() == out[1].tobytes()
        _, _, Rs, ts, K, Xs = out
        assert Xs.shape == (sets, 300, 3) and Xs.dtype == np.float64
        exact, _, Xe = synth.two_view_bank(sets, 300, seed=seed, points=True)
        for s in range(sets):
            p = Xe[s] @ K.T
            assert np.abs(p[:, :2] / p[:, 2:] - exact[s]).max() < 1e-3
            if s:
                assert np.abs(Xs[s - 1] @ Rs[s - 1].T + ts[s - 1] - Xs[s]).max() < 1e-12


def test_point_map_lowest_row_and_transform():
    pairs = torch.tensor([[[0, 2], [1, 2], [2, 5], [3, 0], [4, 1], [5, 3]]], dtype=torch.int32)
    pts = torch.arange(18.0).reshape(1, 6, 3)
    mask = torch.tensor([[0, 1, 1, 1, 1, 1]], dtype=torch.uint8)
    m = geometry.point_map(pairs, torch.tensor([5]), pts, mask, 4)
    assert m.shape == (1, 4, 3) and m.dtype == torch.float32
    assert torch.equal(m[0, 0], pts[0, 3]) and torch.equal(m[0, 1], pts[0, 4]) and torch.equal(m[0, 2], pts[0, 1])
    assert torch.isnan(m[0, 3]).all()                    # row 5 is beyond the count
    R = torch.tensor([[[0.0, -1, 0], [1, 0, 0], [0, 0, 1]]], dtype=torch.float64)
    t = torch.tensor([[1.0, 2.0, 3.0]], dtype=torch.float64)
    mt = geometry.point_map(pairs, torch.tensor([5]), pts, mask, 4, R, t)
    assert torch.allclose(mt[0, 2].double(), R[0] @ pts[0, 1].double() + t[0])
    assert torch.isnan(mt[0, 3]).all()


def test_rows_with_points_keeps_order():
    pairs = torch.tensor([[[0, 2], [1, 2], [2, 5], [3, 0], [9, 1], [0, 4]]], dtype=torch.int32)
    maps = torch.tensor([[[1.0, 2, 3], [float("nan"), 0, 0], [1, 1, 1], [2, 2, 2]]])
    rows, sc, n = geometry.rows_with_points(pairs, torch.arange(6.0)[None], torch.tensor([5]), maps)
    assert n.tolist() == [3] and rows.dtype == torch.int32
    assert rows[0, :3].tolist() == [[0, 2], [2, 5], [3, 0]] and (rows[0, 3:] == -1).all()
    assert sc[0].tolist() == [0.0, 2.0, 3.0, 0.0, 0.0, 0.0]
