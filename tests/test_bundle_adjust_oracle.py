"""CPU tests of the window bookkeeping (geometry.window_tracks / window_map in torch against the loop oracle)
and of the bundle-adjustment oracle (oracle/bundle_adjust.py, the NumPy restatement of csrc/bundle_adjust.cu):
exact scenes, the least-squares optimum against scipy, the robust optimum with gross outliers, and the
12-frame chain with a sliding-window adjustment after every tracking step."""

import numpy as np
import pytest
import torch
from scipy.optimize import least_squares, minimize

from oracle import bundle_adjust as oba
from oracle import triangulate as otri
from parity import record
from sslam_b200 import geometry, synth
from test_triangulate_oracle import FRAMES, cam_of, chain12_inputs, init_map, rot_err_deg


# ---------------------------------------------------------------------------- window bookkeeping
def hand_window():
    """W = 4, K = 6: carried chains, a born keypoint whose frame-a keypoint has no track (claimed, by the lowest
    of two), one whose frame-a keypoint has a track, two keypoints inheriting one track, a broken link."""
    W, K = 4, 6
    rng = np.random.default_rng(0)
    maps = np.full((W, K, 3), np.nan, np.float32)
    fin = [[0, 1, 2, 4], [0, 1, 2, 3, 5], [0, 1, 3, 4, 5], [1, 2, 3]]
    for w, js in enumerate(fin):
        maps[w, js] = rng.uniform(1.0, 5.0, (len(js), 3)).astype(np.float32)
    links = np.full((W - 1, K), -1, np.int32)
    born = np.zeros((W - 1, K), bool)
    links[0, [0, 1, 2, 3, 5]] = [0, 1, 1, 3, 2]             # 1 and 2 inherit track of (0, 1); 3 born claims (0, 3)
    born[0, 3] = True
    links[0, 5] = 5                                         # (1, 5): a link to a keypoint without a track
    links[1, [0, 1, 3, 4, 5]] = [0, 1, 4, 4, 2]             # 3 and 4 born with link 4 (no track): 3 claims
    born[1, [3, 4]] = True
    links[1, 5] = 2
    born[1, 5] = True                                       # born, but (1, 2) has a track: no claim
    links[2, [1, 2, 3]] = [1, 9, 3]                         # (3, 2): link out of range
    Rs = np.stack([np.eye(3)] + [synth._rotation(np.array([0.01, -0.02, 0.03]) * w) for w in range(1, W)])
    ts = np.stack([np.array([0.1, 0.0, -0.05]) * w for w in range(W)])
    return maps, links, born, Rs, ts


def test_window_tracks_and_map_equal_the_loop_oracle():
    maps, links, born, Rs, ts = hand_window()
    W, K = maps.shape[:2]
    ref = oba.window_tracks(maps, links, born, Rs, ts)
    obs, pts, cnt, tr = geometry.window_tracks(torch.as_tensor(maps)[None], torch.as_tensor(links)[None],
                                               torch.as_tensor(born)[None], torch.as_tensor(Rs)[None],
                                               torch.as_tensor(ts)[None])
    assert int(cnt[0]) == ref["count"]
    assert np.array_equal(tr[0].numpy(), ref["track_of"])
    assert np.array_equal(obs[0].numpy(), ref["obs"])
    assert np.array_equal(np.isnan(pts[0].numpy()), np.isnan(ref["points"]))
    assert np.array_equal(np.nan_to_num(pts[0].numpy()), np.nan_to_num(ref["points"]))
    o = ref["obs"]
    assert (o[ref["count"]:] == -1).all() and np.isnan(ref["points"][ref["count"]:]).all()   # padding
    t01 = ref["track_of"][0, 1]
    assert ref["track_of"][1, 1] == t01 and ref["track_of"][1, 2] == t01 and o[t01, 1] == 1  # lowest j observes
    t13 = ref["track_of"][1, 3]
    assert o[t13, 0] == 3 and ref["track_of"][0, 3] == -1                                      # claimed
    t23, t24 = ref["track_of"][2, 3], ref["track_of"][2, 4]
    assert o[t23, 1] == 4 and o[t24, 1] == -1                                                 # lowest j claims
    assert o[ref["track_of"][2, 5], 1] == -1                                                  # has a track: no claim
    assert ref["track_of"][3, 2] != ref["track_of"][2, 2]                                     # broken link
    # window_map without and with a mask
    Xr = ref["points"].copy()
    for mk in (None, (np.random.default_rng(1).random(o.shape) < 0.7) & (o >= 0)):
        got = geometry.window_map(tr, pts, torch.as_tensor(Rs)[None], torch.as_tensor(ts)[None],
                                  obs=None if mk is None else obs,
                                  mask=None if mk is None else torch.as_tensor(mk.astype(np.uint8))[None])[0].numpy()
        exp = oba.window_map(ref["track_of"], Xr, Rs, ts, obs=o, mask=mk)
        assert np.array_equal(np.isnan(got), np.isnan(exp)) and np.array_equal(np.nan_to_num(got), np.nan_to_num(exp))
    # frame 0's keypoints root their tracks: their points map back onto them
    back = oba.window_map(ref["track_of"], Xr, Rs, ts)
    assert np.abs(np.nan_to_num(back[0]) - np.nan_to_num(maps[0])).max() < 1e-5


# ---------------------------------------------------------------------------- scenes
def absolute(Rs, ts, W):
    """Relative motions X_{s+1} = R[s] X_s + t[s] -> absolute poses of W frames in frame 0's coordinates."""
    R, t = [np.eye(3)], [np.zeros(3)]
    for s in range(W - 1):
        R.append(Rs[s] @ R[-1])
        t.append(Rs[s] @ t[-1] + ts[s])
    return np.stack(R), np.stack(t)


def scene(W, n, seed, noise=0.0):
    bank, _, Rs, ts, K, Xs = synth.two_view_bank(W, n, seed=seed, noise=noise, poses=True, points=True)
    R, t = absolute(Rs, ts, W)
    obs = np.tile(np.arange(n, dtype=np.int32)[:, None], (1, W))
    return bank, R, t, Xs[0], obs, cam_of(K)


def perturb(R, t, X, fixed, seed, rot=2e-3, trans=2e-2, pts=2e-2):
    rng = np.random.default_rng(seed)
    R, t = R.copy(), t.copy()
    for w in range(fixed, len(R)):
        R[w] = synth._rotation(rng.normal(0, rot, 3)) @ R[w]
        t[w] = t[w] + rng.normal(0, trans, 3)
    return R, t, (X + rng.normal(0, pts, X.shape)).astype(np.float32)


@pytest.mark.parametrize("W", [2, 5, 8])
def test_exact_scene_returns_the_truth(W):
    bank, R, t, X, obs, cam = scene(W, 200, seed=W)
    fixed = 2
    R0, t0, X0 = perturb(R, t, X, fixed, seed=W)
    o = oba.bundle_adjust(bank, np.arange(W), obs, X0, len(X), R0, t0, cam, fixed=fixed, huber=float("inf"),
                          refine_iters=50)
    assert np.array_equal(o["R"][:fixed], R0[:fixed]) and np.array_equal(o["t"][:fixed], t0[:fixed])
    eR = max(np.abs(o["R"][w] - R[w]).max() for w in range(W))
    et = max(np.abs(o["t"][w] - t[w]).max() for w in range(W))
    eX = np.abs(o["points"] - X).max() / np.abs(X).max()
    # The bank holds fp32 pixels (rounded by up to 3e-5 px), which moves the optimum off the truth: poses agree
    # to 1e-6, points to 5e-6 of their magnitude (1.7e-6 measured at W = 2, where only points are free).
    assert eR < 1e-6 and et < 1e-6 and eX < 5e-6, (eR, et, eX)
    assert o["rms"][1] < 1e-4 < o["rms"][0] and o["accepted"] > 0 and o["mask"].all()


def flat_cost(theta, bank, R0, t0, obs, cam, fixed, n, huber):
    """The kernel's cost at pose increments (R = Exp(w) R0, t = t0 + d) and points theta[6 nf:]."""
    W = len(R0)
    nf = W - fixed
    P = np.concatenate([R0.reshape(W, 9), t0], 1).copy()
    for f in range(nf):
        w = fixed + f
        P[w, :9] = (synth._rotation(theta[6 * f:6 * f + 3]) @ R0[w]).reshape(9)
        P[w, 9:] = t0[w] + theta[6 * f + 3:6 * f + 6]
    X = theta[6 * nf:].reshape(n, 3)
    uv = bank[np.arange(W)[None].repeat(n, 0), obs].astype(np.float64)
    res, _ = oba._project(P, X, uv, cam)
    return res


@pytest.mark.parametrize("seed", range(2))
def test_least_squares_optimum_equals_scipy(seed):
    W, n, fixed = 4, 120, 2
    bank, R, t, X, obs, cam = scene(W, n, seed=20 + seed, noise=0.3)
    R0, t0, X0 = perturb(R, t, X, fixed, seed=seed)
    o = oba.bundle_adjust(bank, np.arange(W), obs, X0, n, R0, t0, cam, fixed=fixed, huber=float("inf"),
                          refine_iters=60)
    nf = W - fixed
    th0 = np.concatenate([np.zeros(6 * nf), X0.astype(np.float64).reshape(-1)])
    s = least_squares(lambda th: flat_cost(th, bank, R0, t0, obs, cam, fixed, n, None).reshape(-1), th0,
                      method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    cs = float(np.sum(s.fun ** 2))
    rel = abs(o["cost"] - cs) / cs
    assert rel < 1e-9, (o["cost"], cs)
    assert o["rms"][1] <= o["rms"][0]
    record(f"ba_oracle_vs_scipy_seed{seed}", {"cost": o["cost"], "scipy": cs, "rel": rel, "accepted": o["accepted"]})


def test_robust_optimum_with_gross_outliers():
    W, n, fixed, d = 3, 60, 2, 2.0
    bank, R, t, X, obs, cam = scene(W, n, seed=31, noise=0.3)
    rng = np.random.default_rng(3)
    bad = rng.choice(n, 6, replace=False)
    bank = bank.copy()
    bank[2, bad] += rng.uniform(20.0, 40.0, (6, 2)).astype(np.float32)           # gross outliers in frame 2
    R0, t0, X0 = perturb(R, t, X, fixed, seed=4)
    o = oba.bundle_adjust(bank, np.arange(W), obs, X0, n, R0, t0, cam, fixed=fixed, huber=d, refine_iters=60)
    assert o["rms"][1] <= o["rms"][0] and not o["mask"][bad, 2].any()
    nf = W - fixed

    def robust(th):
        r = flat_cost(th, bank, o["R"], o["t"], obs, cam, fixed, n, d)
        s = (r * r).sum(-1)
        return float(np.where(s <= d * d, s, 2.0 * d * np.sqrt(s) - d * d).sum())
    th = np.concatenate([np.zeros(6 * nf), o["points"].astype(np.float64).reshape(-1)])
    c0 = robust(th)
    m = minimize(robust, th, method="BFGS", options=dict(gtol=1e-12, maxiter=200))
    drop = (c0 - m.fun) / c0
    assert drop <= 1e-9, drop
    assert abs(c0 - o["cost"]) <= 1e-6 * c0                        # the fp32 points of the output
    record("ba_oracle_robust", {"cost": o["cost"], "minimize": float(m.fun), "rel_drop": drop})


# ---------------------------------------------------------------------------- the 12-frame chain
BA_WINDOW = 5
# Bounds of the adjusted 12-frame chain on seeds 0-5 (largest errors over frames 2-11: 0.75 deg of absolute
# rotation and 0.78 first baselines of camera centre, both on seed 2; without adjustment 1.50 deg and 0.72).
CHAIN_BA_ROT_DEG, CHAIN_BA_POS = 0.9, 0.9


def centre(R, t):
    return -R.T @ t


def oracle_chain_ba(seed, ba=True):
    """Frames 0, 1 initialise; every step k = 1..10 tracks frame k + 1 (track_and_map), then, with ``ba``,
    adjusts the last min(k + 1, 5) frames with the first two held and replaces their maps by window_map's.
    -> per frame 2..11: dict(rot (deg, absolute), pos (camera centre error in units of the first baseline),
    model)."""
    bank, Rs, ts, K, pairs, _, _ = chain12_inputs(seed)
    cam = cam_of(K)
    maps = {1: init_map(bank, pairs, K)}
    poses = {1: (np.eye(3), np.zeros(3))}
    links = {}
    Rt, tt = absolute(Rs[1:], ts[1:], FRAMES - 1)                  # true poses of frames 1..11 in frame 1's coordinates
    s0 = np.linalg.norm(ts[0])
    out = []
    for k in range(1, FRAMES - 1):
        o = otri.track_and_map(maps[k], bank[k], bank[k + 1], pairs[k], cam)
        model = bool(o["R"].any())
        if not model:
            out.append(dict(rot=float("nan"), pos=float("nan"), model=False))
            break
        Ra, ta = poses[k]
        poses[k + 1] = (o["R"] @ Ra, o["R"] @ ta + o["t"])
        maps[k + 1], links[k + 1] = o["next_map"], oba.track_links(maps[k], pairs[k], o)
        if ba:
            fr = list(range(max(1, k + 2 - BA_WINDOW), k + 2))
            W = len(fr)
            Rw = np.stack([poses[f][0] for f in fr])
            tw = np.stack([poses[f][1] for f in fr])
            trk = oba.window_tracks(np.stack([maps[f] for f in fr]), np.stack([links[f][0] for f in fr[1:]]),
                                    np.stack([links[f][1] for f in fr[1:]]), Rw, tw)
            b = oba.bundle_adjust(bank, np.array(fr), trk["obs"], trk["points"], trk["count"], Rw, tw, cam,
                                  fixed=min(2, W), huber=3.0, refine_iters=10)
            new = oba.window_map(trk["track_of"], b["points"], b["R"], b["t"], obs=trk["obs"], mask=b["mask"])
            for i, f in enumerate(fr):
                poses[f] = (b["R"][i], b["t"][i])
                maps[f] = new[i]
        R, t = poses[k + 1]
        out.append(dict(rot=rot_err_deg(R, Rt[k]), pos=float(np.linalg.norm(centre(R, t) - centre(Rt[k], tt[k]) / s0)),
                        model=True))
    return out


@pytest.mark.parametrize("seed", range(6))
def test_chain_with_window_adjustment(seed):
    with_ba, without = oracle_chain_ba(seed), oracle_chain_ba(seed, ba=False)
    assert len(with_ba) == FRAMES - 2 and all(s["model"] for s in with_ba)
    record(f"ba_oracle_chain12_seed{seed}", {"rot_deg": [s["rot"] for s in with_ba], "pos": [s["pos"] for s in with_ba],
                                            "rot_deg_without": [s["rot"] for s in without],
                                            "pos_without": [s["pos"] for s in without]})
    assert max(s["rot"] for s in with_ba) < CHAIN_BA_ROT_DEG and max(s["pos"] for s in with_ba) < CHAIN_BA_POS



def test_window_adjustment_lowers_the_last_frames_drift():
    last = [(oracle_chain_ba(s)[-1]["pos"], oracle_chain_ba(s, ba=False)[-1]["pos"]) for s in range(6)]
    a, b = float(np.mean([x for x, _ in last])), float(np.mean([y for _, y in last]))
    record("ba_oracle_chain12_last_pos", {"with": a, "without": b, "per_seed": last})
    assert a < b, (a, b)
