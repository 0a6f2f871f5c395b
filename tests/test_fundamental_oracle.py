"""CPU: the RANSAC fundamental-matrix oracle (oracle/fundamental.py) against known answers — the sampler's
properties, the true F of noise-free two-view scenes (synth.two_view_bank), cubics with known roots,
OpenCV's 8-point fit on the same inliers — and its "no model" cases, including exactly planar lists."""

import numpy as np
import pytest

from oracle import fundamental as of
from oracle import geometry as og
from sslam_b200 import synth


def two_view_pts(n=2048, noise=0.0, seed=0):
    bank, Ft = synth.two_view_bank(2, n, seed=seed, noise=noise)
    return np.concatenate([bank[0], bank[1]], 1), Ft[0]


def planar_pts(n=200, seed=0):
    """Integer pixels under an affine map with dyadic coefficients: exact in fp32, one homography."""
    rng = np.random.default_rng(seed)
    p1 = np.round(rng.uniform([0, 0], [640, 480], (n, 2)))
    p2 = np.stack([p1[:, 0] + 0.25 * p1[:, 1] + 12, -0.5 * p1[:, 0] + p1[:, 1] - 7], 1)
    return np.concatenate([p1, p2], 1).astype(np.float32)


def lam_roots(c3, c2, c1, c0):
    """Roots of c3 l^3 + c2 l^2 + c1 l + c0 as the 7-point solve takes them: l in [-1, 1], then 1/mu."""
    a = [np.array([v], dtype=np.float64) for v in (c3, c2, c1, c0)]
    lam, okl = of.cubic_roots(*a, closed=True)
    mu, okm = of.cubic_roots(*a[::-1], closed=False)
    with np.errstate(divide="ignore"):
        return list(lam[0][okl[0]]) + list(1.0 / mu[0][okm[0]])


def test_sampler_properties_and_batch_independence():
    for n in (7, 8, 17, 2048):
        idx, ok = of.sample_rows(7, n, np.arange(4096))
        assert ok.mean() > (0.9 if n == 7 else 0.99)
        good = idx[ok]
        assert ((good >= 0) & (good < n)).all()
        assert all(len(set(r)) == 7 for r in good.tolist())
    a, _ = of.sample_rows(7, 100, np.arange(10, 20))
    b, _ = of.sample_rows(7, 100, np.arange(0, 64))
    assert np.array_equal(a, b[10:20])
    # the 4-row instantiation is the homography's sampler
    for n in (4, 5, 100):
        i4, ok4 = og.sample4(3, n, np.arange(512))
        iR, okR = of.sample_rows(3, n, np.arange(512), R=4)
        assert np.array_equal(i4, iR) and np.array_equal(ok4, okR)
    # n = 6: no 7 distinct rows exist
    assert not of.sample_rows(0, 6, np.arange(64))[1].any()


def test_true_model_among_roots_noise_free():
    pts, Ft = two_view_pts()
    assert of.epipolar_distance(Ft, pts).max() < 1e-3                   # the generator's F is the truth
    F, ok = of.hypotheses(pts, 50, seed=0)
    worst = []
    for s in range(50):
        d = [of.epipolar_distance(F[3 * s + k], pts).max() for k in range(3) if ok[3 * s + k]]
        assert d, s
        worst.append(min(d))
    assert max(worst) < 0.05, max(worst)


@pytest.mark.parametrize("coeffs,roots", [
    ((1.0, -1.0, 0.0625, 0.09375), [-0.25, 0.5, 0.75]),        # three roots in [-1, 1]
    ((0.0, 2.0, 0.0, -0.5), [-0.5, 0.5, np.inf]),              # c3 = 0: mu = 0 is the root at infinity
    ((1.0, -0.25, -1.0, 0.25), [-1.0, 0.25, 1.0]),             # roots at -1 and +1
    ((1.0, -0.75, 0.0, 0.0625), [-0.25, 0.5]),                 # double root at 0.5
    ((1.0, -1.0, 1.0, -1.0), [1.0]),                           # one real root (x^2 + 1)(x - 1)
    ((1.0, 0.5, -6.5, 3.0), [-3.0, 0.5, 2.0]),                 # |lam| > 1 through q(mu)
])
def test_cubic_roots_known(coeffs, roots):
    # mu = 0 is bisected to within 2^-64 of 0: lam beyond 1e15 is the root at infinity (F = F1 - F2)
    got = [np.inf if abs(g) > 1e15 else g for g in lam_roots(*coeffs)]
    assert len(got) == len(roots), got
    for g, r in zip(sorted(got), sorted(roots)):
        assert g == r if np.isinf(r) else abs(g - r) < 1e-12, (got, roots)


def test_homography_related_sample_is_degenerate():
    pts = planar_pts()
    _, ok = of.hypotheses(pts, 256, seed=0)
    assert not ok.any()
    trans = pts.copy()
    trans[:, 2:] = trans[:, :2] + np.float32([16, 0])                   # the synthetic sequences' motion
    assert not of.hypotheses(trans, 256, seed=0)[1].any()


def test_refit_agrees_with_opencv_8point():
    cv2 = pytest.importorskip("cv2")
    pts, _ = two_view_pts(n=1000, noise=0.3, seed=2)
    rng = np.random.default_rng(3)
    out = rng.random(1000) < 0.3
    pts[out, 2:] = rng.uniform([0, 0], [640, 480], (int(out.sum()), 2)).astype(np.float32)
    res = of.verify_fundamental(pts, iters=1024, threshold=3.0, seed=0)
    m = res["hyp_mask"]
    Fr = of.refit(pts, m)
    Fcv, _ = cv2.findFundamentalMat(pts[m, :2].astype(np.float64), pts[m, 2:].astype(np.float64), cv2.FM_8POINT)
    d_ours, d_cv = of.epipolar_distance(Fr, pts[m]), of.epipolar_distance(Fcv, pts[m])
    assert np.abs(d_ours - d_cv).max() < 0.01, np.abs(d_ours - d_cv).max()
    assert abs(np.linalg.norm(Fr) - 1.0) < 1e-12 and abs(np.linalg.det(Fr.reshape(3, 3))) < 1e-12


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_motivating_case_mask_matches_true_model(seed):
    """General motion, 0.3 px noise, 30 % outliers.  Away from the threshold (0.5 px) the mask differs from the
    true F's on a few random matches that fall within t of one model's epipolar lines but not the other's:
    the most-inliers hypothesis collects some, and its refit is kept only when it has as many inliers.
    For the same reason it may drop a true correspondence that lies near the threshold of its own model."""
    t = 3.0
    bank, Ft = synth.two_view_bank(2, 2600, seed=5 + seed, noise=0.3)
    pairs, _, counts, true = synth.two_view_lists([2048], 2048, 2600, inlier_frac=0.7, seed=6 + seed)
    r, true = pairs[0], true[0]
    pts = np.concatenate([bank[0][r[:, 0]], bank[1][r[:, 1]]], 1)
    res = of.verify_fundamental(pts, iters=1024, threshold=t, seed=0)
    d = of.epipolar_distance(Ft[0], pts)
    far = (res["mask"] != (d < t)) & (np.abs(d - t) > 0.5)
    assert (far & true).sum() <= 0.002 * true.sum()
    assert (far & ~true).sum() <= 0.03 * (~true).sum()


@pytest.mark.parametrize("case", ["n0", "n6", "identical", "planar"])
def test_no_model(case):
    if case == "n0":
        pts = np.zeros((0, 4), np.float32)
    elif case == "n6":
        pts = two_view_pts()[0][:6]
    elif case == "identical":
        pts = np.tile(np.array([[5, 6, 7, 8]], np.float32), (40, 1))
    else:
        pts = planar_pts()
    res = of.verify_fundamental(pts, iters=256, threshold=3.0, seed=1)
    assert res["hyp_count"].shape == (3 * 256,)
    assert res["best"] == -1 and (res["hyp_count"] == -1).all()
    assert not res["H"].any() and not res["mask"].any()
