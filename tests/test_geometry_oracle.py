"""CPU: the RANSAC homography oracle (oracle/geometry.py) against known answers — the published
splitmix64 outputs, the ground truth of a synthetic planar scene and OpenCV's least-squares
homography on the same inliers — and its "no model" cases."""

import numpy as np
import pytest

from oracle import geometry as og

H_TRUE = np.array([[1.02, 0.03, 12.5], [-0.02, 0.98, -7.25], [2e-5, -1e-5, 1.0]])
CORNERS = np.array([[0, 0], [639, 0], [639, 479], [0, 479]], dtype=np.float64)


def warp(H, xy):
    p = np.concatenate([xy, np.ones((xy.shape[0], 1))], 1) @ np.asarray(H).reshape(3, 3).T
    return p[:, :2] / p[:, 2:3]


def planar_scene(n=500, outlier_frac=0.4, sigma=0.3, seed=3):
    """(n,4) float32 correspondences under H_TRUE: inliers with sigma px noise, the rest uniform."""
    rng = np.random.default_rng(seed)
    src = rng.uniform([0, 0], [640, 480], size=(n, 2))
    dst = warp(H_TRUE, src) + rng.normal(0, sigma, size=(n, 2))
    out = rng.random(n) < outlier_frac
    dst[out] = rng.uniform([0, 0], [640, 480], size=(int(out.sum()), 2))
    pts = np.concatenate([src, dst], 1).astype(np.float32)
    true_err = np.linalg.norm(warp(H_TRUE, pts[:, :2].astype(np.float64)) - pts[:, 2:], axis=1)
    return pts, true_err


def test_splitmix64_published_outputs_and_sampler():
    assert int(og.splitmix64(0, 0)) == 0xE220A8397B1DCDAF
    assert int(og.splitmix64(0, 1)) == 0x6E789E6AA1B965F4
    for n in (4, 5, 17, 2048):
        idx, ok = og.sample4(7, n, np.arange(4096))
        assert ok.mean() > 0.99
        good = idx[ok]
        assert ((good >= 0) & (good < n)).all()
        assert all(len(set(r)) == 4 for r in good.tolist())
    # the samples of hypothesis h depend on (seed, h, n) only
    a, _ = og.sample4(7, 100, np.arange(10, 20))
    b, _ = og.sample4(7, 100, np.arange(0, 64))
    assert np.array_equal(a, b[10:20])


def test_planar_scene_mask_matches_truth():
    t = 3.0
    pts, err = planar_scene()
    res = og.verify(pts, iters=1024, threshold=t, seed=0)
    truth = err < t
    near = np.abs(err - t) < 0.1
    diff = res["mask"] != truth
    assert not (diff & ~near).any(), np.nonzero(diff & ~near)
    assert int(diff.sum()) <= int(near.sum())
    assert res["refit_used"]
    assert res["H"][8] == 1.0


def test_refit_agrees_with_opencv_least_squares():
    cv2 = pytest.importorskip("cv2")
    pts, _ = planar_scene()
    res = og.verify(pts, iters=1024, threshold=3.0, seed=0)
    m = res["mask"]
    Hcv, _ = cv2.findHomography(pts[m, :2].astype(np.float64), pts[m, 2:].astype(np.float64), 0)
    d = np.linalg.norm(warp(res["H"], CORNERS) - warp(Hcv, CORNERS), axis=1)
    assert d.max() < 0.05, d


@pytest.mark.parametrize("case", ["n0", "n3", "collinear", "identical"])
def test_no_model(case):
    if case == "n0":
        pts = np.zeros((0, 4), np.float32)
    elif case == "n3":
        pts = np.array([[0, 0, 1, 1], [10, 0, 11, 1], [0, 10, 1, 11]], np.float32)
    elif case == "collinear":
        k = np.arange(50, dtype=np.float32)
        pts = np.stack([k, 2 * k + 1, 3 * k - 4, k + 7], 1)
    else:
        pts = np.tile(np.array([[5, 6, 7, 8]], np.float32), (40, 1))
    res = og.verify(pts, iters=256, threshold=3.0, seed=1)
    assert res["best"] == -1 and (res["hyp_count"] == -1).all()
    assert not res["H"].any() and not res["mask"].any()
