"""GPU tests of the relative pose (csrc/pose.cu, sslam_b200/geometry.py): parity with oracle/pose.py on a
ragged, aliased batch, batch independence and determinism, the F RANSAC -> E -> pose chain on general-motion
scenes against the true motion, the frame store and CUDA-graph capture, the cv2-shaped host API and
argument errors."""

import ctypes

import cv2
import numpy as np
import pytest
import torch

from oracle import pose as op
from parity import record
from sslam_b200 import synth

pytestmark = pytest.mark.gpu

KP = 2600


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def cam_of(K):
    return (K[0, 0], K[1, 1], K[0, 2], K[1, 2])


def corr(k1, k2, rows, a, b):
    """(n,4) float32 correspondences of list rows; NaN where an index is out of range (as the kernel)."""
    out = np.full((len(rows), 4), np.nan, np.float32)
    ok = (rows[:, 0] >= 0) & (rows[:, 0] < k1.shape[1]) & (rows[:, 1] >= 0) & (rows[:, 1] < k2.shape[1])
    out[ok] = np.concatenate([k1[a][rows[ok, 0]], k2[b][rows[ok, 1]]], 1)
    return out


def run(dev, k1, k2, E, pairs, scores, counts, pidx, K, dist=50.0, refine=10):
    from sslam_b200 import geometry
    t = lambda x: torch.as_tensor(x).to(dev)                                   # noqa: E731
    out = geometry.recover_pose_device(t(k1), t(k2), t(E), t(pairs), t(scores), t(counts), K,
                                       pair_index=None if pidx is None else t(pidx), distance_thresh=dist,
                                       refine_iters=refine, want_mask=True, want_points=True)
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out]


def rot_err_deg(Ra, Rb):
    return float(np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0))))


def t_err_deg(ta, tb):
    return float(np.degrees(np.arccos(np.clip(ta @ tb / np.linalg.norm(ta) / np.linalg.norm(tb), -1.0, 1.0))))


def library_f(dev, k1, k2, pairs, scores, counts, pidx):
    from sslam_b200 import geometry
    t = lambda x: torch.as_tensor(x).to(dev)                                   # noqa: E731
    out = geometry.verify_fundamental_device(t(k1), t(k2), t(pairs), t(scores), t(counts), pair_index=t(pidx))
    return [x.cpu().numpy() for x in out]


@pytest.mark.parametrize("refine", [0, 10])
def test_oracle_parity_ragged_aliased(dev, refine):
    bank, Ft, Rs, ts, K = synth.two_view_bank(3, KP, seed=0, noise=0.3, poses=True)
    ns = [0, 1, 4, 5, 6, 100, 2048, 100, 100]
    L = 2100
    pairs, scores, counts, _ = synth.two_view_lists(ns, L, KP, inlier_frac=0.9, seed=2)
    pairs[8, 3, 1] = KP + 5                                                  # an out-of-range index
    pidx = np.array([[0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [0, 1], [1, 2]], np.int32)
    Et = np.stack([K.T @ Ft[a] @ K for a, _ in pidx])
    Flib = library_f(dev, bank, bank, pairs[6:7], scores[6:7], counts[6:7], pidx[6:7])[0][0]
    E = Et.copy()
    E[6] = K.T @ Flib @ K                                                    # E from the library's F
    E[7] = 0.0                                                               # the F RANSAC's "no model"
    R, t, op_, osc, oc, cand, rms, mask, pts3 = run(dev, bank, bank, E, pairs, scores, counts, pidx, K,
                                                     refine=refine)
    band_rows = 0
    for p, n in enumerate(ns):
        a, b = pidx[p]
        q = corr(bank, bank, pairs[p, :n], a, b)
        ref = op.recover_pose(q, E[p], cam_of(K), refine_iters=refine)
        dc = np.abs(cand[p].astype(np.int64) - ref["cand_good"])
        assert (dc <= ref["cand_band"].sum()).all(), p
        if not ref["have"]:
            assert not R[p].any() and not t[p].any() and not rms[p].any() and oc[p] == 0, p
            assert not mask[p].any() and not pts3[p].any() and (op_[p] == -1).all(), p
            continue
        assert np.abs(R[p] - ref["R"]).max() < 1e-8 and np.abs(t[p] - ref["t"]).max() < 1e-8, p
        # 1e-8 relative; a list of 5 rows fits the 5 DOF exactly, and its refined rms is rounding noise
        assert np.allclose(rms[p], ref["rms"], rtol=1e-8, atol=1e-12), (p, rms[p], ref["rms"])
        keep = mask[p, :n].astype(bool)
        d = keep != ref["mask"]
        assert (d <= ref["band"]).all(), p
        band_rows += int(d.sum())
        both = keep & ref["mask"]
        X, Xr = pts3[p, :n][both].astype(np.float64), ref["points"][both]
        assert (np.linalg.norm(X - Xr, axis=1) <= 1e-5 * np.linalg.norm(Xr, axis=1)).all(), p
        assert not pts3[p, :n][~keep].any() and not mask[p, n:].any() and not pts3[p, n:].any()
        assert oc[p] == keep.sum()
        assert np.array_equal(op_[p, :oc[p]], pairs[p, :n][keep])
        assert np.array_equal(osc[p, :oc[p]], scores[p, :n][keep])
        assert (op_[p, oc[p]:] == -1).all() and (osc[p, oc[p]:] == 0).all()
    assert oc[0] == 0 and oc[7] == 0 and not R[7].any()
    assert rms[2, 0] == rms[2, 1]                                            # 4 rows: no refinement
    assert not mask[8, 3]
    record(f"pose_oracle_parity_refine{refine}", {"pairs": len(ns), "band_rows": band_rows})


def test_batch_independence_and_determinism(dev):
    bank, Ft, _, _, K = synth.two_view_bank(2, KP, seed=4, noise=0.3, poses=True)
    rng = np.random.default_rng(5)
    ns = rng.integers(0, 600, size=64)
    ns[37] = 500
    pairs, scores, counts, _ = synth.two_view_lists(list(ns), 600, KP, inlier_frac=0.8, seed=6)
    pidx = np.tile(np.array([[0, 1]], np.int32), (64, 1))
    E = np.tile((K.T @ Ft[0] @ K)[None], (64, 1, 1))
    batch = run(dev, bank, bank, E, pairs, scores, counts, pidx, K)
    again = run(dev, bank, bank, E, pairs, scores, counts, pidx, K)
    alone = run(dev, bank, bank, E[37:38], pairs[37:38], scores[37:38], counts[37:38], pidx[37:38], K)
    for x, y in zip(batch, again):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(batch, alone):
        assert x[37:38].tobytes() == y.tobytes()
    assert batch[4][37] > 0


@pytest.mark.parametrize("seed", range(8))
def test_pose_chain_against_true_motion(dev, seed):
    """F RANSAC -> E -> pose on general-motion lists (0.3 px noise, 30 % outliers).  The bounds, 0.5 deg in
    rotation and 8 deg in translation direction, hold for the oracle on the same inputs (largest over seeds
    0-7: 0.28 deg and 6.5 deg after the refinement)."""
    from sslam_b200 import geometry
    bank, _, Rs, ts, K = synth.two_view_bank(2, KP, seed=5 + seed, noise=0.3, poses=True)
    pairs, scores, counts, _ = synth.two_view_lists([2048], 2048, KP, inlier_frac=0.7, seed=6 + seed)
    t = lambda x: torch.as_tensor(x).to(dev)                                   # noqa: E731
    b1, b2 = t(bank[0:1]), t(bank[1:2])
    F, vp, vs, vc = geometry.verify_fundamental_device(b1, b2, t(pairs), t(scores), t(counts))
    E = geometry.essential_from_fundamental(F, K)
    out = {}
    for refine in (0, 10):
        R, tt, _, _, oc, _, rms = geometry.recover_pose_device(b1, b2, E, vp, vs, vc, K, refine_iters=refine)
        out[refine] = (R[0].cpu().numpy(), tt[0].cpu().numpy(), rms[0].cpu().numpy(), int(oc[0]))
    R0, t0, rms0, _ = out[0]
    R1, t1, rms1, good = out[10]
    assert rms1[1] <= rms0[1] and rms0[0] == rms1[0]
    n = int(vc[0])
    q = corr(bank, bank, vp[0, :n].cpu().numpy(), 0, 1)
    ref = op.recover_pose(q, E[0].cpu().numpy(), cam_of(K), refine_iters=10)
    errs = {"rot_unrefined": rot_err_deg(R0, Rs[0]), "rot_refined": rot_err_deg(R1, Rs[0]),
            "t_unrefined": t_err_deg(t0, ts[0]), "t_refined": t_err_deg(t1, ts[0]),
            "oracle_rot_refined": rot_err_deg(ref["R"], Rs[0]), "oracle_t_refined": t_err_deg(ref["t"], ts[0])}
    assert errs["rot_refined"] < 0.5 and errs["t_refined"] < 8.0, errs
    assert errs["oracle_rot_refined"] < 0.5 and errs["oracle_t_refined"] < 8.0, errs
    record(f"pose_chain_seed{seed}", dict(errs, f_inliers=n, good=good, rms_before=float(rms1[0]),
                                          rms_after=float(rms1[1])))


@pytest.fixture(scope="module")
def sequence(dev):
    from models.descriptor_refiner import DescriptorRefiner
    from sslam_b200.pipeline import FrontEnd
    torch.manual_seed(0)
    refiner = DescriptorRefiner(384, 384, 128, 4).to(dev)
    sal, feat = synth.make_sequence(24, seq_id=0, device=dev)
    fe = FrontEnd(refiner, num_keypoints=2048, grid="pixel")
    return fe, sal, feat


CAMERA = (525.0, 525.0, 319.5, 239.5)


def test_frame_store_relative_poses(dev, sequence):
    """The synthetic sequences translate a flat canvas, so the true F is not identifiable there and any F
    (and pose) comes from samples with near-miss matches: the outputs keep their format, a pair without a
    pose has zeros and an empty list, and every pose list is a subset of its F inlier list."""
    from sslam_b200 import matchers
    from sslam_b200.framestore import FrameStore
    fe, sal, feat = sequence
    store = FrameStore(fe, capacity=24)
    frames = store.push(sal, feat)
    fp, pairs, scores, counts = store.match_spacings(frames, spacings=(1, 5, 10), variant=matchers.M1)
    R, t, F, pp, ps, pc, mask, X = store.relative_poses(fp, pairs, scores, counts, CAMERA, want_mask=True,
                                                        want_points=True)
    F2, vp, _, vc = store.verify_pairs(fp, pairs, scores, counts, model="fundamental")
    P, L = pairs.shape[:2]
    assert R.shape == (P, 3, 3) and t.shape == (P, 3) and F.shape == (P, 3, 3) and pp.shape == (P, L, 2)
    assert ps.shape == (P, L) and pc.shape == (P,) and mask.shape == (P, L) and X.shape == (P, L, 3)
    assert torch.equal(F, F2)
    Rn, tn, ppn, pcn, vpn, vcn = (x.cpu().numpy() for x in (R, t, pp, pc, vp, vc))
    have = np.abs(tn).sum(1) > 0
    for p in range(P):
        assert pcn[p] <= vcn[p]
        sub = {tuple(r) for r in ppn[p, :pcn[p]]}
        assert sub <= {tuple(r) for r in vpn[p, :vcn[p]]}
        if have[p]:
            assert abs(np.linalg.norm(tn[p]) - 1) < 1e-12 and abs(np.linalg.det(Rn[p]) - 1) < 1e-9
        else:
            assert not Rn[p].any() and pcn[p] == 0
    record("pose_frame_store", {"pairs": P, "with_pose": int(have.sum()), "f_rows": int(vcn.sum()),
                                "pose_rows": int(pcn.sum())})


def test_graph_capture_with_sequence(dev, sequence):
    from sslam_b200 import geometry, matchers
    fe, sal, feat = sequence

    def step():
        feats, pairs, pscores, counts = fe.run_sequence(sal, feat, matchers.M1)
        kp = feats["keypoints_pixel"]
        F, vp, vs, vc = geometry.verify_fundamental_device(kp, kp[1:], pairs, pscores, counts)
        E = geometry.essential_from_fundamental(F, CAMERA)
        return (F,) + geometry.recover_pose_device(kp, kp[1:], E, vp, vs, vc, CAMERA, want_mask=True,
                                                   want_points=True)

    eager = [x.clone() for x in step()]
    replay, out = fe.capture(step)
    for x in out:
        x.zero_()
    replay()
    torch.cuda.synchronize()
    for x, y in zip(out, eager):
        assert torch.equal(x, y)


def test_host_api_against_cv2(dev):
    from sslam_b200 import geometry
    bank, Ft, _, _, K = synth.two_view_bank(2, 800, seed=3, noise=0.3, poses=True)
    pts1, pts2 = bank[0].astype(np.float64), bank[1].astype(np.float64)
    F, m = cv2.findFundamentalMat(pts1, pts2, cv2.FM_RANSAC, 3.0, 0.99, 1024)
    E = K.T @ F @ K
    ret, R, t, mask, X = geometry.recover_pose(E, pts1, pts2, K, 50.0, mask=m, refine_iters=0)
    cret, cR, ct, cmask, _ = cv2.recoverPose(E, pts1, pts2, K, distanceThresh=50.0, mask=m.copy())
    assert R.shape == (3, 3) and t.shape == (3, 1) and mask.shape == (800, 1) and mask.dtype == np.uint8
    assert X.shape == (4, 800) and (X[3] == 1.0).all()
    assert np.abs(R - cR).max() < 1e-6 and np.abs(t - ct).max() < 1e-6
    assert ret == int(mask.sum()) and abs(ret - cret) <= 0.02 * cret
    assert not mask[m[:, 0] == 0].any() and not X[:3, mask[:, 0] == 0].any()
    ret10, R10, t10, _, _ = geometry.recover_pose(E, pts1, pts2, K, mask=m)
    assert ret10 > 0 and abs(np.linalg.det(R10) - 1) < 1e-9
    ret0, R0, t0, mask0, X0 = geometry.recover_pose(E, pts1[:0], pts2[:0], K)
    assert ret0 == 0 and not R0.any() and mask0.shape == (0, 1) and X0.shape == (4, 0)
    with pytest.raises(ValueError):
        geometry.recover_pose(E, pts1, pts2, np.array([[525.0, 1.0, 320.0], [0.0, 525.0, 240.0], [0, 0, 1]]))


def test_bad_arguments(dev):
    from sslam_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
    p, z = ctypes.c_void_p(buf.data_ptr()), ctypes.c_void_p(0)

    def call(kp=p, E=p, L=8, refine=10, dist=50.0, fx=500.0, out=p):
        return lib.sslam_recover_pose(kp, 1, p, 1, z, 1, 8, 8, E, p, p, p, L, fx, 500.0, 320.0, 240.0, dist,
                                      refine, p, p, z, z, z, out, p, p, z, z)
    assert call() == 0
    assert call(kp=z) == -1 and call(E=z) == -1 and call(out=z) == -1
    assert call(L=16385) == -1 and call(refine=-1) == -1 and call(refine=101) == -1
    assert call(dist=0.0) == -1 and call(dist=float("inf")) == -1
    assert call(fx=0.0) == -1 and call(fx=float("nan")) == -1
    torch.cuda.synchronize()
