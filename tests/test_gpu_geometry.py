"""GPU tests of the RANSAC homography (csrc/ransac.cu, sslam_b200/geometry.py): bit parity of the
hypotheses, counts and best index with oracle/geometry.py, batch independence and determinism, the
ground truth of the synthetic sequences (a pure translation of 16 px every 8 frames), the frame store,
CUDA-graph capture and the cv2-shaped host API."""

import ctypes

import numpy as np
import pytest
import torch

from oracle import geometry as og
from parity import record

pytestmark = pytest.mark.gpu

H_TRUE = np.array([[1.02, 0.03, 12.5], [-0.02, 0.98, -7.25], [2e-5, -1e-5, 1.0]])
CORNERS = np.array([[0, 0], [639, 0], [639, 479], [0, 479]], dtype=np.float64)
T_PX = 3.0


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def warp(H, xy):
    p = np.concatenate([xy, np.ones((xy.shape[0], 1))], 1) @ np.asarray(H, dtype=np.float64).reshape(3, 3).T
    return p[:, :2] / p[:, 2:3]


def gt_shift(a, b):
    return -16.0 * (b // 8 - a // 8)


def keypoint_bank(F=3, K=2600, seed=0):
    """F keypoint sets where set s+1 is set s under H_TRUE (0.3 px noise) with 30 % of points replaced."""
    rng = np.random.default_rng(seed)
    bank = np.empty((F, K, 2))
    bank[0] = rng.uniform([0, 0], [640, 480], size=(K, 2))
    for s in range(1, F):
        bank[s] = warp(H_TRUE, bank[s - 1]) + rng.normal(0, 0.3, size=(K, 2))
        out = rng.random(K) < 0.3
        bank[s][out] = rng.uniform([0, 0], [640, 480], size=(int(out.sum()), 2))
    return bank.astype(np.float32)


def match_lists(ns, L, K, seed=1):
    """Padded lists of ns[p] rows (ascending i): j = i for 60 % of the rows, random otherwise."""
    rng = np.random.default_rng(seed)
    P = len(ns)
    pairs = np.full((P, L, 2), -1, dtype=np.int32)
    scores = np.zeros((P, L), dtype=np.float32)
    for p, n in enumerate(ns):
        i = np.sort(rng.choice(K, size=n, replace=False))
        j = np.where(rng.random(n) < 0.6, i, rng.integers(0, K, size=n))
        pairs[p, :n, 0], pairs[p, :n, 1] = i, j
        scores[p, :n] = rng.random(n).astype(np.float32)
    return pairs, scores, np.asarray(ns, dtype=np.int32)


def corr(k1, k2, pairs, n, a, b):
    r = pairs[:n]
    return np.concatenate([k1[a][r[:, 0]], k2[b][r[:, 1]]], 1).astype(np.float32)


def run(dev, k1, k2, pairs, scores, counts, pair_index=None, iters=1024, seed=0, threshold=T_PX):
    from sslam_b200 import ops
    P, L = pairs.shape[:2]
    ws = torch.empty(ops._lib.load().sslam_ransac_workspace_bytes(P, L, iters), dtype=torch.uint8, device=dev)
    t = lambda x: torch.as_tensor(x).to(dev)                                   # noqa: E731
    out = ops.ransac_homography(t(k1), t(k2), t(pairs), t(scores), t(counts),
                                pair_index=None if pair_index is None else t(pair_index),
                                threshold=threshold, iters=iters, seed=seed, want_mask=True, workspace=ws)
    torch.cuda.synchronize()
    hc, best, hm = ops.ransac_workspace_views(ws, P, L, iters)
    return [x.cpu().numpy() for x in out], hc.cpu().numpy(), best.cpu().numpy(), hm.cpu().numpy()


@pytest.mark.parametrize("iters", [1, 64, 1024])
def test_oracle_parity_ragged_aliased(dev, iters):
    ns = [0, 1, 3, 4, 5, 100, 2048]
    L, K = 2100, 2600
    bank = keypoint_bank(K=K)
    pairs, scores, counts = match_lists(ns, L, K)
    pidx = np.array([[0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [2, 2], [0, 1]], dtype=np.int32)
    (H, op, osc, oc, mask), hc, best, hm = run(dev, bank, bank, pairs, scores, counts, pidx, iters=iters, seed=11)
    t2 = og.t2_of(T_PX)
    boundary = refit_flips = 0
    for p, n in enumerate(ns):
        a, b = pidx[p]
        pts = corr(bank, bank, pairs[p], n, a, b)
        ref = og.verify(pts, iters=iters, threshold=T_PX, seed=11)
        assert np.array_equal(hc[p], ref["hyp_count"]), p
        assert best[p] == ref["best"], p
        assert np.array_equal(hm[p, :n].astype(bool), ref["hyp_mask"]), p
        assert not hm[p, n:].any()
        Hg = H[p].reshape(9)
        if ref["best"] < 0:
            assert not Hg.any() and oc[p] == 0 and not mask[p].any()
        else:
            assert Hg[8] == 1.0
            if np.abs(Hg - ref["H"]).max() > 1e-9 * np.abs(ref["H"]).max():
                # the refit was accepted on one side only: its count differs in a row at the threshold
                e_ref = og.sq_errors(ref["H"].astype(np.float32)[None], pts)[0]
                assert (np.abs(e_ref - t2) <= 1e-6 * t2).any(), (p, Hg, ref["H"])
                refit_flips += 1
                continue
            got = mask[p, :n].astype(bool)
            if not np.array_equal(got, ref["mask"]):
                e_ref = og.sq_errors(ref["H"].astype(np.float32)[None], pts)[0]
                d = got != ref["mask"]
                assert (np.abs(e_ref[d] - t2) <= 1e-6 * t2).all(), p
                boundary += int(d.sum())
        keep = mask[p, :n].astype(bool)
        assert oc[p] == keep.sum()
        assert np.array_equal(op[p, :oc[p]], pairs[p, :n][keep])
        assert np.array_equal(osc[p, :oc[p]], scores[p, :n][keep])
        assert (op[p, oc[p]:] == -1).all() and (osc[p, oc[p]:] == 0).all() and not mask[p, n:].any()
    record(f"ransac_oracle_parity_iters{iters}", {"pairs": len(ns), "threshold_rows": boundary,
                                                  "refit_acceptance_flips": refit_flips})


def test_batch_independence_and_determinism(dev):
    K, L = 2600, 600
    bank = keypoint_bank(K=K, seed=4)
    rng = np.random.default_rng(5)
    ns = rng.integers(0, 600, size=64)
    ns[37] = 500
    pairs, scores, counts = match_lists(list(ns), L, K, seed=6)
    pidx = np.tile(np.array([[0, 1]], np.int32), (64, 1))
    batch, *_ = run(dev, bank, bank, pairs, scores, counts, pidx, seed=3)
    again, *_ = run(dev, bank, bank, pairs, scores, counts, pidx, seed=3)
    alone, *_ = run(dev, bank, bank, pairs[37:38], scores[37:38], counts[37:38], pidx[37:38], seed=3)
    for x, y in zip(batch, again):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(batch, alone):
        assert x[37:38].tobytes() == y.tobytes()
    # outlier-free lists: every seed finds the same inlier set
    clean = keypoint_bank(F=2, K=K, seed=8)
    cp = np.full((1, 800, 2), -1, np.int32)
    i = np.sort(rng.choice(K, size=800, replace=False))
    clean[1][i] = (warp(H_TRUE, clean[0][i].astype(np.float64)) + rng.normal(0, 0.3, (800, 2))).astype(np.float32)
    cp[0, :, 0] = cp[0, :, 1] = i
    cs, cc = np.zeros((1, 800), np.float32), np.array([800], np.int32)
    m0 = run(dev, clean, clean, cp, cs, cc, np.array([[0, 1]], np.int32), seed=0)[0][4]
    m1 = run(dev, clean, clean, cp, cs, cc, np.array([[0, 1]], np.int32), seed=12345)[0][4]
    assert m0.all() and np.array_equal(m0, m1)


@pytest.fixture(scope="module")
def sequence(dev):
    from models.descriptor_refiner import DescriptorRefiner
    from sslam_b200 import matchers, synth
    from sslam_b200.pipeline import FrontEnd
    torch.manual_seed(0)
    refiner = DescriptorRefiner(384, 384, 128, 4).to(dev)
    sal, feat = synth.make_sequence(24, seq_id=0, device=dev)
    fe = FrontEnd(refiner, num_keypoints=2048, grid="pixel")
    feats, pairs, pscores, counts = fe.run_sequence(sal, feat, matchers.M1)
    return fe, sal, feat, feats, pairs, pscores, counts


# Keypoints are integer pixels, so a correspondence is either exactly translated (error 0) or off by at
# least 1 px.  At T_GT = 0.5 px only the exact ones are inliers and the refit on them is exact up to
# rounding.  At an integer threshold the fp32 transfer error of a 1-, 2- or 3-px miss lands on either side
# of t^2, and at the default 3 px matches to a neighbouring keypoint 1-2 px away are inliers as well and
# pull the least-squares fit off the pure translation; that deviation is recorded, not bounded.
T_GT = 0.5


def test_sequence_end_to_end(dev, sequence):
    from sslam_b200 import evaluation, geometry, ops
    fe, sal, feat, feats, pairs, pscores, counts = sequence
    kp = feats["keypoints_pixel"]
    H3, _, _, vc3 = geometry.verify_homography_device(kp, kp[1:], pairs, pscores, counts, num_pairs=23)
    H, vp, vs, vc, mask = geometry.verify_homography_device(kp, kp[1:], pairs, pscores, counts, num_pairs=23,
                                                            threshold=T_GT, want_mask=True)
    Hn, kpn = H.cpu().numpy(), kp.cpu().numpy().astype(np.float64)
    pn, cn, vpn, vcn, mn = (x.cpu().numpy() for x in (pairs, counts, vp, vc, mask))
    Hgt = np.zeros((23, 3, 3))
    err_hist = {}
    for p in range(23):
        Hgt[p] = [[1, 0, gt_shift(p, p + 1)], [0, 1, 0], [0, 0, 1]]
        d = np.linalg.norm(warp(Hn[p], CORNERS) - warp(Hgt[p], CORNERS), axis=1)
        assert d.max() < 0.05, (p, d)
        n = int(cn[p])
        keep = mn[p, :n].astype(bool)
        assert vcn[p] == keep.sum() and np.array_equal(vpn[p, :vcn[p]], pn[p, :n][keep])
        r = pn[p, :n]
        e = np.linalg.norm(kpn[p + 1][r[:, 1]] - (kpn[p][r[:, 0]] + [gt_shift(p, p + 1), 0]), axis=1)
        assert keep[e <= T_GT - 0.05].all() and not keep[e > T_GT + 0.05].any()
        err_hist[p] = [int((e == 0).sum()), int(((e > 0) & (e < T_PX)).sum()), int((e >= T_PX).sum())]
    dev3 = [float(np.linalg.norm(warp(H3.cpu().numpy()[p], CORNERS) - warp(Hgt[p], CORNERS), axis=1).max())
            for p in range(23)]
    gt_est = evaluation.ground_truth_matches_device(kp, kp[1:], H, num_pairs=23)
    gt_ref = evaluation.ground_truth_matches_device(kp, kp[1:], torch.as_tensor(Hgt).to(dev), num_pairs=23)
    md_ref, _ = ops.nn_points(kp, kp[1:], H=torch.as_tensor(Hgt).to(dev), num_pairs=23)
    md_ref = md_ref.cpu().numpy()
    near = 0
    for p in range(23):
        a = {tuple(x) for x in gt_est[0][p, :int(gt_est[1][p])].cpu().numpy().tolist()}
        b = {tuple(x) for x in gt_ref[0][p, :int(gt_ref[1][p])].cpu().numpy().tolist()}
        for i in {i for i, _ in a ^ b}:
            # a row at the threshold, or one whose nearest keypoint is tied (two at the same integer distance)
            d = np.sort(np.linalg.norm(kpn[p + 1] - (kpn[p][i] + [gt_shift(p, p + 1), 0]), axis=1))
            assert abs(md_ref[p, i] - T_PX) < 1e-6 or d[1] - d[0] < 1e-6, (p, i, d[:2])
            near += 1
    record("ransac_sequence_gt_lists", {"pairs": 23, "threshold_or_tie_rows": near, "threshold_px": T_GT,
                                        "kept": int(vcn.sum()), "input": int(cn.sum()),
                                        "kept_at_3px": int(vc3.sum()),
                                        "max_corner_dev_px_at_3px": max(dev3),
                                        "gt_error_exact_near_far_pair0": err_hist[0]})


def test_frame_store_spacings(dev, sequence):
    from sslam_b200 import matchers
    from sslam_b200.framestore import FrameStore
    fe, sal, feat = sequence[:3]
    store = FrameStore(fe, capacity=24)
    frames = store.push(sal, feat)
    fp, pairs, scores, counts = store.match_spacings(frames, spacings=(1, 5, 10), variant=matchers.M1)
    H, _, _, vc = store.verify_pairs(fp, pairs, scores, counts, threshold=T_GT)
    Hn = H.cpu().numpy()
    assert (vc.cpu().numpy() > 0).all()
    for p, (a, b) in enumerate(fp):
        assert abs(Hn[p, 0, 2] - gt_shift(a, b)) < 0.05 and abs(Hn[p, 1, 2]) < 0.05, (a, b, Hn[p])
        assert np.abs(Hn[p] - np.array([[1, 0, Hn[p, 0, 2]], [0, 1, Hn[p, 1, 2]], [0, 0, 1]])).max() < 1e-4


def test_graph_capture_with_sequence(dev, sequence):
    from sslam_b200 import geometry, matchers
    fe, sal, feat = sequence[:3]

    def step():
        feats, pairs, pscores, counts = fe.run_sequence(sal, feat, matchers.M1)
        kp = feats["keypoints_pixel"]
        return geometry.verify_homography_device(kp, kp[1:], pairs, pscores, counts, want_mask=True)

    eager = [x.clone() for x in step()]
    replay, out = fe.capture(step)
    for x in out:
        x.zero_()
    replay()
    torch.cuda.synchronize()
    for x, y in zip(out, eager):
        assert torch.equal(x, y)


def test_host_api_matches_oracle(dev):
    from sslam_b200 import geometry
    rng = np.random.default_rng(3)
    src = rng.uniform([0, 0], [640, 480], size=(500, 2))
    dst = warp(H_TRUE, src) + rng.normal(0, 0.3, size=(500, 2))
    out = rng.random(500) < 0.4
    dst[out] = rng.uniform([0, 0], [640, 480], size=(int(out.sum()), 2))
    pts = np.concatenate([src, dst], 1).astype(np.float32)
    H, mask = geometry.find_homography(pts[:, :2], pts[:, 2:], 3.0, 1024, 0)
    ref = og.verify(pts, iters=1024, threshold=3.0, seed=0)
    assert H.shape == (3, 3) and H.dtype == np.float64 and mask.shape == (500, 1) and mask.dtype == np.uint8
    assert np.abs(H.reshape(9) - ref["H"]).max() <= 1e-9 * np.abs(ref["H"]).max()
    assert np.array_equal(mask[:, 0].astype(bool), ref["mask"])
    for n in (0, 3):
        H, mask = geometry.find_homography(pts[:n, :2], pts[:n, 2:])
        assert H is None and mask.shape == (n, 1) and not mask.any()


def test_bad_arguments(dev):
    from sslam_b200 import _lib
    lib = _lib.load()
    t = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
    p, z = ctypes.c_void_p(t.data_ptr()), ctypes.c_void_p(0)

    def call(kp=p, iters=16, thr=3.0, L=8, ws=p):
        return lib.sslam_ransac_homography(kp, 1, p, 1, z, 1, 8, 8, p, p, p, L, iters, thr, 0, z, p, p, p, z, ws,
                                           1 << 16, z)
    assert call() == 0
    assert call(kp=z) == -1 and call(iters=0) == -1 and call(thr=0.0) == -1 and call(L=16385) == -1
    assert call(ws=z) == -1
    torch.cuda.synchronize()
