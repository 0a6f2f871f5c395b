"""GPU tests of the RANSAC fundamental matrix (csrc/ransac.cu FModel, sslam_b200/geometry.py): bit parity of
the per-slot counts, best slot and pre-refit mask with oracle/fundamental.py, batch independence and
determinism, general-motion two-view scenes (synth.two_view_bank) against the true F and against the
homography, the synthetic sequences through the frame store, CUDA-graph capture and the cv2-shaped host
API."""

import ctypes

import numpy as np
import pytest
import torch

from oracle import fundamental as of
from parity import record
from sslam_b200 import synth

pytestmark = pytest.mark.gpu

T_PX = 3.0
BAND = 1e-3            # relative band around t^2 inside which fp32 last-bit differences may flip a row


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def corr(k1, k2, pairs, n, a, b):
    r = pairs[:n]
    return np.concatenate([k1[a][r[:, 0]], k2[b][r[:, 1]]], 1).astype(np.float32)


def run(dev, k1, k2, pairs, scores, counts, pair_index=None, iters=1024, seed=0, threshold=T_PX, model="fundamental"):
    from sslam_b200 import ops
    P, L = pairs.shape[:2]
    ws = torch.empty(ops.ransac_workspace_bytes(P, L, iters, model=model), dtype=torch.uint8, device=dev)
    t = lambda x: torch.as_tensor(x).to(dev)                                   # noqa: E731
    fn = ops.ransac_fundamental if model == "fundamental" else ops.ransac_homography
    out = fn(t(k1), t(k2), t(pairs), t(scores), t(counts), pair_index=None if pair_index is None else t(pair_index),
             threshold=threshold, iters=iters, seed=seed, want_mask=True, workspace=ws)
    torch.cuda.synchronize()
    hc, best, hm = ops.ransac_workspace_views(ws, P, L, iters, model=model)
    return [x.cpu().numpy() for x in out], hc.cpu().numpy(), best.cpu().numpy(), hm.cpu().numpy()


def near_threshold(F64, pts, t2):
    e1, e2 = of.sq_errors(np.asarray(F64).reshape(1, 9).astype(np.float32), pts)
    return (np.abs(e1[0] - t2) <= BAND * t2) | (np.abs(e2[0] - t2) <= BAND * t2)


def parity_bank(K=2600):
    """Sets 0-2: one general-motion scene (0.3 px noise); sets 3, 4: integer pixels and an exact affine
    image of them (every 7-point sample of a list over (3, 4) is degenerate)."""
    bank, _ = synth.two_view_bank(3, K, seed=0, noise=0.3)
    rng = np.random.default_rng(9)
    p1 = np.round(rng.uniform([0, 0], [640, 480], (K, 2)))
    p2 = np.stack([p1[:, 0] + 0.25 * p1[:, 1] + 12, -0.5 * p1[:, 0] + p1[:, 1] - 7], 1)
    return np.concatenate([bank, p1[None].astype(np.float32), p2[None].astype(np.float32)], 0)


@pytest.mark.parametrize("iters", [1, 64, 1024])
def test_oracle_parity_ragged_aliased(dev, iters):
    ns = [0, 1, 6, 7, 8, 100, 2048, 300]
    L, K = 2100, 2600
    bank = parity_bank(K)
    pairs, scores, counts, _ = synth.two_view_lists(ns, L, K, inlier_frac=0.6, seed=1)
    pairs[7, :300, 1] = pairs[7, :300, 0]                              # the planar list: true matches only
    pidx = np.array([[0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [3, 4]], dtype=np.int32)
    (F, op, osc, oc, mask), hc, best, hm = run(dev, bank, bank, pairs, scores, counts, pidx, iters=iters, seed=11)
    t2 = of.t2_of(T_PX)
    assert hc.shape == (len(ns), 3 * iters)
    boundary = refit_flips = 0
    for p, n in enumerate(ns):
        a, b = pidx[p]
        pts = corr(bank, bank, pairs[p], n, a, b)
        ref = of.verify_fundamental(pts, iters=iters, threshold=T_PX, seed=11)
        assert np.array_equal(hc[p], ref["hyp_count"]), p
        assert best[p] == ref["best"], p
        assert np.array_equal(hm[p, :n].astype(bool), ref["hyp_mask"]), p
        assert not hm[p, n:].any()
        Fg = F[p].reshape(9)
        if ref["best"] < 0:
            assert not Fg.any() and oc[p] == 0 and not mask[p].any(), p
            continue
        assert abs(np.linalg.norm(Fg) - 1.0) < 1e-12
        keep = mask[p, :n].astype(bool)
        dg, dr = of.epipolar_distance(Fg, pts), of.epipolar_distance(ref["H"], pts)
        if np.abs(dg - dr)[ref["mask"]].max() > 1e-3:
            # the refit was accepted on one side only: its count sits at the best hypothesis's
            m = int(ref["hyp_mask"].sum())
            Fr = of.refit(pts, ref["hyp_mask"])
            assert Fr is not None and abs(int(of.inliers(Fr, pts, T_PX).sum()) - m) <= 2, p
            refit_flips += 1
        elif not np.array_equal(keep, ref["mask"]):
            d = keep != ref["mask"]
            assert near_threshold(ref["H"], pts, t2)[d].all(), p
            boundary += int(d.sum())
        assert oc[p] == keep.sum()
        assert np.array_equal(op[p, :oc[p]], pairs[p, :n][keep])
        assert np.array_equal(osc[p, :oc[p]], scores[p, :n][keep])
        assert (op[p, oc[p]:] == -1).all() and (osc[p, oc[p]:] == 0).all() and not mask[p, n:].any()
    assert best[7] == -1 and oc[7] == 0                                 # the exactly planar list has no F
    record(f"fundamental_oracle_parity_iters{iters}", {"pairs": len(ns), "threshold_rows": boundary,
                                                       "refit_acceptance_flips": refit_flips})


def test_batch_independence_and_determinism(dev):
    K, L = 2600, 600
    bank, _ = synth.two_view_bank(2, K, seed=4, noise=0.3)
    rng = np.random.default_rng(5)
    ns = rng.integers(0, 600, size=64)
    ns[37] = 500
    pairs, scores, counts, _ = synth.two_view_lists(list(ns), L, K, seed=6)
    pidx = np.tile(np.array([[0, 1]], np.int32), (64, 1))
    batch, *_ = run(dev, bank, bank, pairs, scores, counts, pidx, seed=3)
    again, *_ = run(dev, bank, bank, pairs, scores, counts, pidx, seed=3)
    alone, *_ = run(dev, bank, bank, pairs[37:38], scores[37:38], counts[37:38], pidx[37:38], seed=3)
    for x, y in zip(batch, again):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(batch, alone):
        assert x[37:38].tobytes() == y.tobytes()
    # outlier-free lists: every seed finds the same inlier set (all of it)
    cp, cs, cc, _ = synth.two_view_lists([800], 800, K, inlier_frac=1.0, seed=7)
    one = np.array([[0, 1]], np.int32)
    masks = [run(dev, bank, bank, cp, cs, cc, one, seed=s)[0][4] for s in (0, 12345, 2 ** 63 + 5)]
    assert masks[0].all() and all(np.array_equal(masks[0], m) for m in masks[1:])


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_general_motion_against_true_model_and_homography(dev, seed):
    """The motivating case: a translating camera in a 3-D scene, 0.3 px noise, 30 % outliers.  The F path
    keeps the true correspondences; homography RANSAC on the same lists keeps only those near one plane."""
    K = 2600
    bank, Ft = synth.two_view_bank(2, K, seed=5 + seed, noise=0.3)
    pairs, scores, counts, true = synth.two_view_lists([2048], 2048, K, inlier_frac=0.7, seed=6 + seed)
    one = np.array([[0, 1]], np.int32)
    (F, _, _, oc, mask), *_ = run(dev, bank, bank, pairs, scores, counts, one)
    (H, _, _, hoc, hmask), *_ = run(dev, bank, bank, pairs, scores, counts, one, model="homography")
    true = true[0]
    pts = corr(bank, bank, pairs[0], 2048, 0, 1)
    d = of.epipolar_distance(Ft[0], pts)
    keep, hkeep = mask[0].astype(bool), hmask[0].astype(bool)
    far = (keep != (d < T_PX)) & (np.abs(d - T_PX) > 0.5)
    assert (far & true).sum() <= 0.002 * true.sum()
    assert (far & ~true).sum() <= 0.03 * (~true).sum()
    ref = of.verify_fundamental(pts, iters=1024, threshold=T_PX, seed=0)
    de = np.abs(of.epipolar_distance(F[0].reshape(9), pts) - of.epipolar_distance(ref["H"], pts))[ref["mask"]]
    record(f"fundamental_general_motion_seed{seed}", {
        "rows": 2048, "true": int(true.sum()), "true_kept_F": int((keep & true).sum()),
        "true_kept_H": int((hkeep & true).sum()), "outliers_kept_F": int((keep & ~true).sum()),
        "rows_off_true_mask_beyond_0.5px": int(far.sum()), "kept_F": int(oc[0]), "kept_H": int(hoc[0]),
        "max_epipolar_dev_from_oracle_px": float(de.max())})


@pytest.fixture(scope="module")
def sequence(dev):
    from models.descriptor_refiner import DescriptorRefiner
    from sslam_b200 import synth as sy
    from sslam_b200.pipeline import FrontEnd
    torch.manual_seed(0)
    refiner = DescriptorRefiner(384, 384, 128, 4).to(dev)
    sal, feat = sy.make_sequence(24, seq_id=0, device=dev)
    fe = FrontEnd(refiner, num_keypoints=2048, grid="pixel")
    return fe, sal, feat


def gt_shift(a, b):
    return -16.0 * (b // 8 - a // 8)


def test_frame_store_spacings(dev, sequence):
    """The synthetic sequences translate a flat canvas, so F is not identifiable there: every sample of 7
    exact correspondences is degenerate, and every F a sample with a 1-2 px neighbour match yields keeps
    all exact correspondences.  At the default 3 px every exact correspondence is kept."""
    from sslam_b200 import matchers
    from sslam_b200.framestore import FrameStore
    fe, sal, feat = sequence
    store = FrameStore(fe, capacity=24)
    frames = store.push(sal, feat)
    fp, pairs, scores, counts = store.match_spacings(frames, spacings=(1, 5, 10), variant=matchers.M1)
    F, vp, _, vc, mask = store.verify_pairs(fp, pairs, scores, counts, model="fundamental", want_mask=True)
    H, *_ = store.verify_pairs(fp, pairs, scores, counts)                      # the default is the homography
    assert torch.equal(H[:, 2, 2].cpu(), torch.ones(len(fp), dtype=torch.float64))
    kp = store.bank["keypoints"].cpu().numpy().astype(np.float64)
    slots = store.pair_index(fp).cpu().numpy()
    pn, cn, mn, vcn = pairs.cpu().numpy(), counts.cpu().numpy(), mask.cpu().numpy(), vc.cpu().numpy()
    exact_total = kept_total = 0
    for p, (a, b) in enumerate(fp):
        n = int(cn[p])
        r = pn[p, :n]
        sa, sb = slots[p]
        e = np.linalg.norm(kp[sb][r[:, 1]] - (kp[sa][r[:, 0]] + [gt_shift(a, b), 0]), axis=1)
        exact = e == 0
        keep = mn[p, :n].astype(bool)
        assert keep[exact].all(), (a, b, int(exact.sum()), int(keep[exact].sum()))
        assert vcn[p] == keep.sum()
        exact_total += int(exact.sum())
        kept_total += int(keep.sum())
    record("fundamental_frame_store_spacings", {"pairs": len(fp), "input": int(cn.sum()), "exact": exact_total,
                                                "kept": kept_total, "threshold_px": T_PX})


def test_graph_capture_with_sequence(dev, sequence):
    from sslam_b200 import geometry, matchers
    fe, sal, feat = sequence

    def step():
        feats, pairs, pscores, counts = fe.run_sequence(sal, feat, matchers.M1)
        kp = feats["keypoints_pixel"]
        return geometry.verify_fundamental_device(kp, kp[1:], pairs, pscores, counts, want_mask=True)

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
    bank, _ = synth.two_view_bank(2, 500, seed=3, noise=0.3)
    rng = np.random.default_rng(3)
    pts = np.concatenate([bank[0], bank[1]], 1)
    out = rng.random(500) < 0.4
    pts[out, 2:] = rng.uniform([0, 0], [640, 480], size=(int(out.sum()), 2)).astype(np.float32)
    F, mask = geometry.find_fundamental(pts[:, :2], pts[:, 2:], 3.0, 1024, 0)
    ref = of.verify_fundamental(pts, iters=1024, threshold=3.0, seed=0)
    assert F.shape == (3, 3) and F.dtype == np.float64 and mask.shape == (500, 1) and mask.dtype == np.uint8
    Fr = ref["H"].reshape(3, 3)
    assert abs(Fr[2, 2]) > np.finfo(np.float32).eps and F[2, 2] == 1.0
    dg, dr = of.epipolar_distance(F, pts), of.epipolar_distance(Fr, pts)
    assert np.abs(dg - dr)[ref["mask"]].max() < 1e-3
    d = mask[:, 0].astype(bool) != ref["mask"]
    assert near_threshold(ref["H"], pts, of.t2_of(3.0))[d].all()
    for n in (0, 6):
        F, mask = geometry.find_fundamental(pts[:n, :2], pts[:n, 2:])
        assert F is None and mask.shape == (n, 1) and not mask.any()


def test_bad_arguments(dev):
    from sslam_b200 import _lib
    lib = _lib.load()
    t = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
    p, z = ctypes.c_void_p(t.data_ptr()), ctypes.c_void_p(0)
    assert lib.sslam_ransac_fundamental_workspace_bytes(1, 8, 16) <= 1 << 16

    def call(kp=p, iters=16, thr=3.0, L=8, ws=p):
        return lib.sslam_ransac_fundamental(kp, 1, p, 1, z, 1, 8, 8, p, p, p, L, iters, thr, 0, z, p, p, p, z, ws,
                                            1 << 16, z)
    assert call() == 0
    assert call(kp=z) == -1 and call(iters=0) == -1 and call(thr=0.0) == -1 and call(L=16385) == -1
    assert call(ws=z) == -1
    torch.cuda.synchronize()
