"""CPU tests of the relative-pose oracle (oracle/pose.py), the NumPy restatement of csrc/pose.cu: exact
two-view scenes, the candidate set against cv2.decomposeEssentialMat, the chosen pose and mask against
cv2.recoverPose, the Levenberg-Marquardt result against scipy's, the no-pose cases, and the true motions
synth.two_view_bank returns."""

import cv2
import numpy as np
import pytest
from scipy.optimize import least_squares

from oracle import pose as op
from parity import record
from sslam_b200 import synth


def cam_of(K):
    return (K[0, 0], K[1, 1], K[0, 2], K[1, 2])


def exact_scene(seed, n=500):
    """Exact float64 projections of n points (depth 4-10 m) under the true motion of two_view_bank(seed)."""
    _, _, Rs, ts, K = synth.two_view_bank(2, 8, seed=seed, poses=True)
    rng = np.random.default_rng(100 + seed)
    pix = rng.uniform([0.0, 0.0], [639.0, 479.0], (n, 2))
    X = (np.concatenate([pix, np.ones((n, 1))], 1) @ np.linalg.inv(K).T) * rng.uniform(4.0, 10.0, (n, 1))
    Y = X @ Rs[0].T + ts[0]
    p2 = Y @ K.T
    pts = np.concatenate([pix, p2[:, :2] / p2[:, 2:]], 1)
    return pts, X, Rs[0], ts[0], K


def noisy_lists(seed):
    """A general-motion list (0.3 px noise, 30 % outliers) verified by cv2's F RANSAC -> (pts, E, K, R, t)."""
    bank, _, Rs, ts, K = synth.two_view_bank(2, 2600, seed=5 + seed, noise=0.3, poses=True)
    pairs, _, _, _ = synth.two_view_lists([2048], 2048, 2600, inlier_frac=0.7, seed=6 + seed)
    r = pairs[0]
    pts = np.concatenate([bank[0][r[:, 0]], bank[1][r[:, 1]]], 1).astype(np.float64)
    F, m = cv2.findFundamentalMat(pts[:, :2], pts[:, 2:], cv2.FM_RANSAC, 3.0, 0.99, 1024)
    return pts[m[:, 0].astype(bool)], K.T @ F @ K, K, Rs[0], ts[0]


def rot_err_deg(Ra, Rb):
    return float(np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0))))


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_exact_scene_recovers_true_pose(seed):
    pts, X, R, t, K = exact_scene(seed)
    E = op.skew(t) @ R
    tn = t / np.linalg.norm(t)
    o = op.recover_pose(pts, E, cam_of(K), distance_thresh=1e3, refine_iters=0)
    assert o["have"]
    assert np.abs(o["R"] - R).max() < 1e-9 and np.abs(o["t"] - tn).max() < 1e-9
    assert o["mask"].all() and o["cand_good"][o["best"]] == len(pts)
    assert (o["cand_good"] < len(pts)).sum() == 3
    rel = np.abs(o["points"] - X / np.linalg.norm(t)) / np.linalg.norm(X / np.linalg.norm(t), axis=1, keepdims=True)
    assert rel.max() < 1e-6
    r = op.recover_pose(pts, E, cam_of(K), distance_thresh=1e3, refine_iters=10)
    assert np.abs(r["R"] - R).max() < 1e-9 and np.abs(r["t"] - tn).max() < 1e-9
    assert r["rms"][1] <= r["rms"][0] < 1e-6


@pytest.mark.parametrize("seed", range(8))
def test_candidates_equal_cv2_decomposition(seed):
    _, E, _, _, _ = noisy_lists(seed)
    R1, R2, t = cv2.decomposeEssentialMat(E)
    cands = op.candidates(E)
    mine = {(np.round(R, 9).tobytes(), np.round(tt, 9).tobytes()) for R, tt in cands}
    ref = {(np.round(R, 9).tobytes(), np.round(s * t[:, 0], 9).tobytes()) for R in (R1, R2) for s in (1, -1)}
    assert mine == ref
    assert len(mine) == 4


def cv2_depths(Q, R, t):
    X = Q[:3] / Q[3]
    return X[2], (R @ X + t.reshape(3, 1))[2]


@pytest.mark.parametrize("seed", range(8))
def test_unrefined_pose_equals_cv2_recover_pose(seed):
    """refine_iters = 0 is cv2.recoverPose: the same candidate to 1e-6.  Its mask comes from a linear
    (DLT) triangulation, ours from the rays' midpoint, so on noisy rows the two depths differ slightly: a
    row may be kept on one side only when a bound (0 or distance_thresh, on either camera) lies between
    the two depths, or when it sits in the 1e-6 band of a bound or of den's limit.  Both are counted."""
    pts, E, K, _, _ = noisy_lists(seed)
    dist = 50.0
    o = op.recover_pose(pts, E, cam_of(K), distance_thresh=dist, refine_iters=0)
    ret, R, t, mask, Q = cv2.recoverPose(E, pts[:, :2], pts[:, 2:], K, distanceThresh=dist)
    assert o["have"]
    assert np.abs(o["R"] - R).max() < 1e-6 and np.abs(o["t"] - t[:, 0]).max() < 1e-6
    d = mask[:, 0].astype(bool) != o["mask"]
    f1, f2, _ = op.rays(pts, cam_of(K))
    _, _, info = op.triangulate(o["R"], o["t"], f1, f2, dist)
    c1, c2 = cv2_depths(Q, R, t)
    straddle = np.zeros(len(pts), bool)
    for ours, theirs in ((info["z1"], c1), (info["z2"], c2)):
        for bound in (0.0, dist):
            straddle |= (ours - bound) * (theirs - bound) <= 0.0
    assert (straddle | o["band"])[d].all()
    assert d.sum() <= 0.05 * len(pts)
    record(f"pose_cv2_recover_pose_seed{seed}", {"rows": len(pts), "good": int(o["mask"].sum()), "cv2_good": int(ret),
                                                 "mask_rows_differing": int(d.sum()),
                                                 "differing_in_1e-6_band": int((d & o["band"]).sum())})


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_lm_equals_scipy_least_squares(seed):
    pts, E, K, _, _ = noisy_lists(seed)
    cam = cam_of(K)
    o = op.recover_pose(pts, E, cam, refine_iters=0)
    R0, t0 = o["R"], o["t"]
    f1, f2, usable = op.rays(pts, cam)
    f1, f2 = f1[usable], f2[usable]
    B = np.stack(op.basis(t0))

    def res(x):
        R, t = op.apply_step(R0, t0, B, x)
        return op.sampson(op.skew(t) @ R, f1, f2, cam)[0]
    sol = least_squares(res, np.zeros(5), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000)
    Rs, ts = op.apply_step(R0, t0, B, sol.x)
    R, t, c0, c1, acc = op.refine(R0, t0, f1, f2, cam, 100)
    assert np.abs(R - Rs).max() < 1e-6 and np.abs(t - ts).max() < 1e-6
    assert abs(c1 - float(np.sum(sol.fun ** 2))) <= 1e-6 * c1
    assert c1 < c0


def test_no_pose_cases():
    pts, X, R, t, K = exact_scene(0, n=50)
    cam = cam_of(K)
    E = op.skew(t) @ R
    for bad in (np.zeros((3, 3)), np.outer([1.0, 2.0, 3.0], [0.5, -1.0, 2.0]), np.full((3, 3), np.nan),
                np.where(np.eye(3) > 0, np.inf, 0.0)):
        o = op.recover_pose(pts, bad, cam)
        assert not o["have"] and not o["R"].any() and not o["cand_good"].any() and not o["mask"].any()
    o = op.recover_pose(pts[:0], E, cam)
    assert not o["have"] and not o["cand_good"].any()
    # points at infinity (a purely rotating camera): the rays are parallel under every candidate
    p2 = np.concatenate([pts[:, :2], np.ones((50, 1))], 1) @ (K @ R @ np.linalg.inv(K)).T
    inf_pts = np.concatenate([pts[:, :2], p2[:, :2] / p2[:, 2:]], 1)
    o = op.recover_pose(inf_pts, E, cam)
    assert not o["have"] and not o["cand_good"].any()
    # every point beyond distance_thresh (depths are 13-50 |t| here)
    o = op.recover_pose(pts, E, cam, distance_thresh=1.0)
    assert not o["have"] and not o["cand_good"].any() and not o["points"].any()
    # a row whose keypoint index is out of range is NaN in the list: never good, not refined
    pn = pts.copy()
    pn[3] = np.nan
    o = op.recover_pose(pn, E, cam, distance_thresh=1e3)
    assert o["have"] and not o["mask"][3] and o["mask"].sum() == 49 and o["cand_good"].max() == 49


def test_two_view_bank_poses():
    for seed, sets in ((0, 2), (3, 4)):
        bank, F = synth.two_view_bank(sets, 300, seed=seed, noise=0.3)
        bank2, F2, Rs, ts, K = synth.two_view_bank(sets, 300, seed=seed, noise=0.3, poses=True)
        assert bank.tobytes() == bank2.tobytes() and F.tobytes() == F2.tobytes()
        assert Rs.shape == (sets - 1, 3, 3) and ts.shape == (sets - 1, 3) and K.shape == (3, 3)
        Ki = np.linalg.inv(K)
        for s in range(sets - 1):
            assert np.abs(Rs[s] @ Rs[s].T - np.eye(3)).max() < 1e-12 and np.linalg.det(Rs[s]) > 0
            Fm = Ki.T @ op.skew(ts[s]) @ Rs[s] @ Ki
            Fm /= np.linalg.norm(Fm)
            assert min(np.abs(Fm - F[s]).max(), np.abs(Fm + F[s]).max()) < 1e-12
