"""GPU tests of the sliding-window bundle adjustment (csrc/bundle_adjust.cu, geometry.bundle_adjust_device,
FrameStore.bundle_adjust) and of the window bookkeeping on the device: parity with oracle/bundle_adjust.py on
ragged, aliased batches, batch independence and determinism, CUDA-graph replay of one full window step, the
12-frame chain against the oracle chain, track_and_map's provenance outputs and argument errors."""

import ctypes

import numpy as np
import pytest
import torch

from oracle import bundle_adjust as oba
from parity import record
from sslam_b200 import synth
from test_bundle_adjust_oracle import BA_WINDOW, absolute, oracle_chain_ba, perturb
from test_triangulate_oracle import FRAMES, cam_of, chain12_inputs, rot_err_deg

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def T(x, dev):
    return torch.as_tensor(np.ascontiguousarray(x)).to(dev)


def batch(W, fixed, n=160, F=8, seed=0):
    """Windows over one 8-frame bank (slots aliased between windows): 0 clean, 1 with a few gross outliers,
    2 without tracks, 3 with single-observation tracks, an out-of-range keypoint, a NaN point and a point
    behind a camera, 4 without a pose."""
    bank, _, Rs, ts, K, Xs = synth.two_view_bank(F, n, seed=seed, noise=0.3, poses=True, points=True)
    Ra, ta = absolute(Rs, ts, F)
    rng = np.random.default_rng(seed)
    P = 5
    fi = np.stack([np.arange(s, s + W) % F for s in (0, 1, 0, 2, 3)]).astype(np.int32)
    N = W * n
    obs = np.full((P, N, W), -1, np.int32)
    pts = np.full((P, N, 3), np.nan, np.float32)
    cnt = np.zeros(P, np.int32)
    R = np.zeros((P, W, 3, 3))
    t = np.zeros((P, W, 3))
    for p in range(P):
        f0 = fi[p, 0]
        X = Xs[0] @ Ra[f0].T + ta[f0]                     # the points in window frame 0's camera = world
        Rw = np.stack([Ra[f] @ Ra[f0].T for f in fi[p]])
        tw = np.stack([ta[f] - Rw[i] @ ta[f0] for i, f in enumerate(fi[p])])
        Rw, tw, X0 = perturb(Rw, tw, X, fixed, seed=seed + p, rot=1e-3, trans=1e-2, pts=1e-2)
        R[p], t[p] = Rw, tw
        cnt[p] = n
        obs[p, :n] = np.arange(n)[:, None]
        pts[p, :n] = X0
    bank = bank.copy()
    bank[fi[1, -1], rng.choice(n, 8, replace=False)] += 30.0          # gross outliers (aliased into window 3)
    cnt[2] = 0
    obs[3, :10, 1:] = -1                                                # one observation
    obs[3, 12, 0] = n + 7                                               # out of range
    pts[3, 13] = np.nan                                                 # a NaN point
    pts[3, 14] = -pts[3, 14]                                            # behind the cameras
    R[4] = 0.0                                                          # no pose
    return bank, fi, obs, pts, cnt, R, t, cam_of(K)


def run(dev, bank, fi, obs, pts, cnt, R, t, cam, **kw):
    from sslam_b200 import geometry
    out = geometry.bundle_adjust_device(T(bank, dev), T(fi, dev), T(obs, dev), T(pts, dev), T(cnt, dev), T(R, dev),
                                        T(t, dev), cam, want_mask=True, **kw)
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out]


CASES = [(W, fixed, huber, iters) for W in (2, 3, 5, 8) for fixed in sorted({1, 2, W}) for huber in (3.0, float("inf"))
         for iters in (0, 10)]


@pytest.mark.parametrize("W,fixed,huber,iters", CASES)
def test_oracle_parity_ragged_aliased(dev, W, fixed, huber, iters):
    bank, fi, obs, pts, cnt, R, t, cam = batch(W, fixed)
    Ro, to, Xo, rms, acc, mask = run(dev, bank, fi, obs, pts, cnt, R, t, cam, fixed=fixed, huber=huber,
                                     refine_iters=iters)
    near, worst = 0, [0.0, 0.0, 0.0]
    for p in range(len(fi)):
        ref = oba.bundle_adjust(bank, fi[p], obs[p], pts[p], cnt[p], R[p], t[p], cam, fixed=fixed, huber=huber,
                                refine_iters=iters)
        assert acc[p] == ref["accepted"], (p, acc[p], ref["accepted"])
        assert np.abs(Ro[p] - ref["R"]).max() < 1e-8 and np.abs(to[p] - ref["t"]).max() < 1e-8, p
        assert np.array_equal(Ro[p, :fixed], R[p, :fixed]) and np.array_equal(to[p, :fixed], t[p, :fixed])
        fin = np.isfinite(ref["points"])
        assert np.array_equal(fin, np.isfinite(Xo[p]))
        e = np.abs(Xo[p][fin] - ref["points"][fin]).max() / max(np.abs(ref["points"][fin]).max(), 1.0) if fin.any() else 0.0
        assert e < 1e-6, (p, e)
        er = np.abs(rms[p] - ref["rms"]).max() / max(np.abs(ref["rms"]).max(), 1e-300)
        assert er < 1e-8 or not ref["rms"].any() and not rms[p].any(), (p, rms[p], ref["rms"])
        d = mask[p].astype(bool) != ref["mask"]
        if d.any():
            assert (np.abs(ref["s"][d] - 9.0) <= 1e-6 * 9.0).all(), p
            near += int(d.sum())
        worst = [max(worst[0], float(np.abs(Ro[p] - ref["R"]).max())), max(worst[1], float(e)), max(worst[2], float(er))]
    assert acc[2] == 0 and acc[4] == 0 and not rms[2].any() and not rms[4].any()
    assert np.array_equal(Ro[4], R[4]) and np.array_equal(np.isnan(Xo[4]), np.isnan(pts[4]))
    assert not mask[3, :10].any() and not mask[3, 12, 0] and not mask[3, 13].any() and not mask[3, 14].any()
    if iters:
        assert (rms[:, 1] <= rms[:, 0] + 1e-12).all() and acc[0] > 0
    record(f"ba_oracle_parity_W{W}_fixed{fixed}_huber{huber}_iters{iters}",
           {"accepted": [int(a) for a in acc], "near_threshold_mask_rows": near, "max_abs_R": worst[0],
            "max_rel_point": worst[1], "max_rel_rms": worst[2]})


def test_batch_independence_and_determinism(dev):
    bank, fi, obs, pts, cnt, R, t, cam = batch(5, 2, seed=3)
    rep = 7
    big = [np.concatenate([x] * rep) for x in (fi, obs, pts, cnt, R, t)]
    a = run(dev, bank, *big, cam)
    b = run(dev, bank, *big, cam)
    alone = run(dev, bank, fi[1:2], obs[1:2], pts[1:2], cnt[1:2], R[1:2], t[1:2], cam)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    for k in range(rep):
        for x, y in zip(a, alone):
            assert x[5 * k + 1:5 * k + 2].tobytes() == y.tobytes()


# ---------------------------------------------------------------------------- the chain on the device
def device_chain(seed, dev, ba=True):
    from sslam_b200 import geometry
    from test_gpu_triangulate import device_init
    bank, Rs, ts, K, pairs, scores, counts = chain12_inputs(seed)
    b, pr, sc, cn = T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev)
    maps = {1: device_init(b, pr, sc, cn, K, dev)}
    I = torch.eye(3, dtype=torch.float64, device=dev)[None]
    poses = {1: (I, torch.zeros(1, 3, dtype=torch.float64, device=dev))}
    links = {}
    Rt, tt = absolute(Rs[1:], ts[1:], FRAMES - 1)
    s0 = np.linalg.norm(ts[0])
    out = []
    for k in range(1, FRAMES - 1):
        pidx = T(np.array([[k, k + 1]], np.int32), dev)
        R, t, _, _, _, nxt, lk, bn = geometry.track_and_map(maps[k], b, b, pr[k:k + 1], sc[k:k + 1], cn[k:k + 1], K,
                                                            pidx, want_links=True)
        Ra, ta = poses[k]
        poses[k + 1] = (R @ Ra, (R @ ta[..., None])[..., 0] + t)
        maps[k + 1], links[k + 1] = nxt, (lk, bn)
        if ba:
            fr = list(range(max(1, k + 2 - BA_WINDOW), k + 2))
            Rw = torch.stack([poses[f][0] for f in fr], 1)
            tw = torch.stack([poses[f][1] for f in fr], 1)
            obs, X, cnt, tr = geometry.window_tracks(torch.stack([maps[f] for f in fr], 1),
                                                     torch.stack([links[f][0] for f in fr[1:]], 1),
                                                     torch.stack([links[f][1] for f in fr[1:]], 1), Rw, tw)
            Rb, tb, Xb, _, _, mask = geometry.bundle_adjust_device(b, T(np.array([fr], np.int32), dev), obs, X, cnt, Rw,
                                                                   tw, K, fixed=min(2, len(fr)), want_mask=True)
            new = geometry.window_map(tr, Xb, Rb, tb, obs=obs, mask=mask)
            for i, f in enumerate(fr):
                poses[f] = (Rb[:, i], tb[:, i])
                maps[f] = new[:, i]
        Rn, tn = poses[k + 1][0][0].cpu().numpy(), poses[k + 1][1][0].cpu().numpy()
        out.append(dict(rot=rot_err_deg(Rn, Rt[k]), pos=float(np.linalg.norm(-Rn.T @ tn + Rt[k].T @ tt[k] / s0))))
    return out


@pytest.mark.parametrize("seed", range(2))
def test_chain12_with_window_adjustment_against_oracle(dev, seed):
    got, ref = device_chain(seed, dev), oracle_chain_ba(seed)
    drot = max(abs(g["rot"] - r["rot"]) for g, r in zip(got, ref))
    dpos = max(abs(g["pos"] - r["pos"]) for g, r in zip(got, ref))
    record(f"ba_chain12_seed{seed}", {"rot_deg": [g["rot"] for g in got], "pos": [g["pos"] for g in got],
                                      "max_abs_diff_rot_deg": drot, "max_abs_diff_pos": dpos})
    assert len(got) == len(ref) and drot < 1e-3 and dpos < 1e-3, (drot, dpos)


def window_step(b, maps_prev, pr, sc, cn, K, k, pidx, fi, Rw, tw, prev_links):
    """One full sliding-window step: track_and_map into frame k + 1, the window's tracks, the adjustment and the
    refined maps."""
    from sslam_b200 import geometry
    R, t, _, _, _, nxt, lk, bn = geometry.track_and_map(maps_prev[-1], b, b, pr[k:k + 1], sc[k:k + 1], cn[k:k + 1], K,
                                                        pidx, want_links=True)
    Rn = R @ Rw[:, -1]
    tn = (R @ tw[:, -1, :, None])[..., 0] + t
    obs, X, cnt, tr = geometry.window_tracks(torch.stack(maps_prev + [nxt], 1),
                                             torch.stack([x[0] for x in prev_links] + [lk], 1),
                                             torch.stack([x[1] for x in prev_links] + [bn], 1),
                                             torch.cat([Rw, Rn[:, None]], 1), torch.cat([tw, tn[:, None]], 1))
    Rb, tb, Xb, rms, acc, mask = geometry.bundle_adjust_device(b, fi, obs, X, cnt, torch.cat([Rw, Rn[:, None]], 1),
                                                               torch.cat([tw, tn[:, None]], 1), K, want_mask=True)
    return Rb, tb, rms, acc, geometry.window_map(tr, Xb, Rb, tb, obs=obs, mask=mask)


def test_window_step_graph_replay_and_links(dev):
    from sslam_b200 import geometry
    from test_gpu_triangulate import device_init
    bank, _, _, K, pairs, scores, counts = chain12_inputs(0)
    b, pr, sc, cn = T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev)
    m1 = device_init(b, pr, sc, cn, K, dev)
    p1 = T(np.array([[1, 2]], np.int32), dev)
    plain = geometry.track_and_map(m1, b, b, pr[1:2], sc[1:2], cn[1:2], K, p1)
    linked = geometry.track_and_map(m1, b, b, pr[1:2], sc[1:2], cn[1:2], K, p1, want_links=True)
    for x, y in zip(plain, linked[:6]):                                   # the first six outputs are unchanged
        assert torch.equal(x.nan_to_num(), y.nan_to_num()) and torch.equal(x.isnan(), y.isnan())
    lk, bn = linked[6], linked[7]
    fin = torch.isfinite(linked[5]).all(-1)
    assert torch.equal(lk >= 0, fin) and not (bn & ~fin).any() and bn.any() and (~bn & fin).any()
    R2 = linked[0]
    I = torch.eye(3, dtype=torch.float64, device=dev)[None, None]
    Rw = torch.cat([I, R2[:, None]], 1)
    tw = torch.cat([torch.zeros(1, 1, 3, dtype=torch.float64, device=dev), linked[1][:, None]], 1)
    fi = T(np.array([[1, 2, 3]], np.int32), dev)
    pidx = T(np.array([[2, 3]], np.int32), dev)
    args = (b, [m1, linked[5]], pr, sc, cn, K, 2, pidx, fi, Rw, tw, [(lk, bn)])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = [x.clone() for x in window_step(*args)]
        window_step(*args)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = window_step(*args)
    for x in out:
        x.zero_()
    g.replay()
    torch.cuda.synchronize()
    for x, y in zip(out, eager):
        assert torch.equal(x.nan_to_num(), y.nan_to_num()) and torch.equal(x.isnan(), y.isnan())
    assert int(eager[3][0]) > 0 and float(eager[2][0, 1]) <= float(eager[2][0, 0])


def test_frame_store_bundle_adjust(dev):
    from sslam_b200 import geometry
    from sslam_b200.framestore import FrameStore

    class FE:                                                           # the store only needs keypoints here
        grid, patch = "pixel", 1
    bank, fi, obs, pts, cnt, R, t, cam = batch(3, 2)
    store = FrameStore.__new__(FrameStore)
    store.fe = FE()
    store.capacity = 8
    store.bank = {"keypoints": T(bank, dev)}
    store.slot_of = lambda f: f % 8
    store.holds = lambda f: True
    windows = [[int(x) for x in row] for row in fi]
    got = store.bundle_adjust(windows, T(obs, dev), T(pts, dev), T(cnt, dev), T(R, dev), T(t, dev), cam, want_mask=True)
    ref = geometry.bundle_adjust_device(T(bank, dev), T(fi, dev), T(obs, dev), T(pts, dev), T(cnt, dev), T(R, dev),
                                        T(t, dev), cam, want_mask=True)
    for x, y in zip(got, ref):
        assert torch.equal(x.nan_to_num(), y.nan_to_num())


def test_bad_arguments(dev):
    from sslam_b200 import _lib, ops
    lib = _lib.load()
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)
    p, z = ctypes.c_void_p(buf.data_ptr()), ctypes.c_void_p(0)

    def call(W=3, N=8, fixed=2, huber=3.0, thr=3.0, refine=10, ws=p, wsb=1 << 20, kp=p, fx=500.0):
        return lib.sslam_bundle_adjust(kp, 1, 8, p, 1, W, N, p, p, p, p, p, fx, 500.0, 320.0, 240.0, fixed, huber,
                                       thr, refine, p, p, p, p, z, z, ws, wsb, z)
    assert call() == 0
    assert call(W=9) == -2 and call(W=1) == -1 and call(N=65537) == -2
    assert call(fixed=0) == -1 and call(fixed=4) == -1 and call(fixed=3) == 0
    assert call(huber=0.0) == -1 and call(huber=float("nan")) == -1 and call(huber=float("inf")) == 0
    assert call(thr=0.0) == -1 and call(refine=101) == -1 and call(refine=-1) == -1
    assert call(kp=z) == -1 and call(ws=z) == -1 and call(wsb=16) == -3 and call(fx=0.0) == -1
    torch.cuda.synchronize()
    kp = torch.zeros(1, 8, 2, device=dev)
    fi = torch.zeros(1, 3, dtype=torch.int32, device=dev)
    ob = torch.zeros(1, 4, 3, dtype=torch.int32, device=dev)
    X = torch.zeros(1, 4, 3, device=dev)
    c = torch.ones(1, dtype=torch.int32, device=dev)
    R = torch.eye(3, dtype=torch.float64, device=dev).expand(1, 3, 3, 3)
    t = torch.zeros(1, 3, 3, dtype=torch.float64, device=dev)
    ops.bundle_adjust(kp, fi, ob, X, c, R, t, 500.0, 500.0, 320.0, 240.0)
    with pytest.raises(RuntimeError):
        ops.bundle_adjust(kp, fi, ob[:, :, :2], X, c, R, t, 500.0, 500.0, 320.0, 240.0)     # obs W differs
    with pytest.raises(RuntimeError):
        ops.bundle_adjust(kp, fi, ob, X[:, :3], c, R, t, 500.0, 500.0, 320.0, 240.0)        # points N differs
    with pytest.raises(RuntimeError):
        ops.bundle_adjust(kp, fi, ob, X, c, R[:, :2], t, 500.0, 500.0, 320.0, 240.0)        # R W differs
    with pytest.raises(_lib.SslamError):
        ops.bundle_adjust(kp, fi, ob, X, c, R, t, 500.0, 500.0, 320.0, 240.0, fixed=5)
    fi9 = torch.zeros(1, 9, dtype=torch.int32, device=dev)
    with pytest.raises(_lib.SslamError):
        ops.bundle_adjust(kp, fi9, torch.zeros(1, 4, 9, dtype=torch.int32, device=dev), X, c,
                          torch.eye(3, dtype=torch.float64, device=dev).expand(1, 9, 3, 3),
                          torch.zeros(1, 9, 3, dtype=torch.float64, device=dev), 500.0, 500.0, 320.0, 240.0)
    torch.cuda.synchronize()
