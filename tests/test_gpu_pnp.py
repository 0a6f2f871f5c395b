"""GPU tests of the PnP RANSAC (csrc/pnp.cu, sslam_b200/geometry.py, FrameStore.track_poses): bit parity with
oracle/pnp.py on a ragged, aliased batch, the refined pose against the oracle, batch independence and
determinism, accuracy against the true motion, the F RANSAC -> E -> pose -> point_map -> PnP chain and its
CUDA-graph replay, the frame store, the cv2-shaped host API and argument errors."""

import ctypes

import cv2
import numpy as np
import pytest
import torch

from oracle import pnp as op
from parity import record
from sslam_b200 import synth
from test_pnp_oracle import (ALONE_ROT_DEG, ALONE_T_MM, CHAIN_ROT_DEG, CHAIN_T_REL, KP, cam_of, chain_errors,
                             chain_inputs, noisy_rows, oracle_chain, rot_err_deg)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def T(x, dev):
    return torch.as_tensor(x).to(dev)


def rows5(pts, kp, rows, a, b):
    """(n,5) float32 rows (X, Y, Z, u, v) of list rows; NaN where an index is out of range (as the kernel)."""
    out = np.full((len(rows), 5), np.nan, np.float32)
    ok = (rows[:, 0] >= 0) & (rows[:, 0] < pts.shape[1]) & (rows[:, 1] >= 0) & (rows[:, 1] < kp.shape[1])
    out[ok] = np.concatenate([pts[a][rows[ok, 0]], kp[b][rows[ok, 1]]], 1)
    return out


def run(dev, pts, kp, pairs, scores, counts, pidx, cam, iters=1024, refine=10, seed=0):
    from sslam_b200 import ops
    P, L = pairs.shape[:2]
    ws = torch.empty(ops.ransac_workspace_bytes(P, L, iters, model="pnp"), dtype=torch.uint8, device=dev)
    out = ops.ransac_pnp(T(pts, dev), T(kp, dev), T(pairs, dev), T(scores, dev), T(counts, dev), *cam,
                         pair_index=None if pidx is None else T(pidx, dev), iters=iters, seed=seed,
                         refine_iters=refine, want_mask=True, workspace=ws)
    views = ops.ransac_workspace_views(ws, P, L, iters, model="pnp")
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out], [v.cpu().numpy() for v in views]


def parity_batch():
    """Ragged, aliased lists over a 3-set bank plus a set of collinear points."""
    bank, _, _, _, K, Xs = synth.two_view_bank(3, KP, seed=0, noise=0.3, poses=True, points=True)
    pts = np.concatenate([Xs, np.zeros((1, KP, 3))]).astype(np.float32)
    s = np.arange(KP) * 2.0 ** -7                                       # exact in fp32
    pts[3] = np.stack([s, 0.5 * s, 5.0 + s], 1)                          # set 3: exactly on one line
    ns = [0, 1, 3, 4, 5, 100, 2048, 100, 100, 100]
    pairs, scores, counts, _ = synth.two_view_lists(ns, 2100, KP, inlier_frac=0.7, seed=2)
    pidx = np.array([[0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [3, 1], [0, 1], [1, 2]], np.int32)
    pts[0][pairs[8, 7, 0]] = np.nan                                      # a row without a point
    pairs[9, 3, 1] = KP + 5                                              # an index out of range
    return pts, bank, pairs, scores, counts, pidx, cam_of(K), ns


@pytest.mark.parametrize("iters", [1, 64, 1024])
def test_oracle_parity_ragged_aliased(dev, iters):
    pts, bank, pairs, scores, counts, pidx, cam, ns = parity_batch()
    (R, t, op_, osc, oc, rms, mask), (hc, best, hmask) = run(dev, pts, bank, pairs, scores, counts, pidx, cam,
                                                             iters=iters)
    band_rows = 0
    for p, n in enumerate(ns):
        a, b = pidx[p]
        q = rows5(pts, bank, pairs[p, :n], a, b)
        ref = op.ransac_pnp(q, cam, iters=iters)
        assert np.array_equal(hc[p], ref["hyp_count"]), p
        assert best[p] == ref["best"], p
        assert np.array_equal(hmask[p, :n].astype(bool), ref["hyp_mask"]) and not hmask[p, n:].any(), p
        if ref["best"] < 0:
            assert not R[p].any() and not t[p].any() and not rms[p].any() and oc[p] == 0, p
            assert not mask[p].any() and (op_[p] == -1).all(), p
            continue
        assert np.abs(R[p] - ref["R"]).max() < 1e-8 and np.abs(t[p] - ref["t"]).max() < 1e-8, p
        assert np.allclose(rms[p], ref["rms"], rtol=1e-8, atol=1e-12), (p, rms[p], ref["rms"])
        keep = mask[p, :n].astype(bool)
        d = keep != ref["mask"]
        assert (d <= ref["band"]).all(), p
        band_rows += int(d.sum())
        assert oc[p] == keep.sum() and not mask[p, n:].any()
        assert np.array_equal(op_[p, :oc[p]], pairs[p, :n][keep])
        assert np.array_equal(osc[p, :oc[p]], scores[p, :n][keep])
        assert (op_[p, oc[p]:] == -1).all() and (osc[p, oc[p]:] == 0).all()
    assert (hc[:3] == -1).all() and (hc[7] == -1).all() and oc[7] == 0     # n < 4, collinear points
    assert not mask[8, 7] and not mask[9, 3]
    if iters == 1024:
        assert oc[6] > 1000 and oc[5] > 50
    record(f"pnp_oracle_parity_iters{iters}", {"lists": len(ns), "band_rows": band_rows,
                                                "with_model": int((best >= 0).sum())})


def test_batch_independence_and_determinism(dev):
    bank, _, _, _, K, Xs = synth.two_view_bank(2, KP, seed=4, noise=0.3, poses=True, points=True)
    pts = Xs.astype(np.float32)
    rng = np.random.default_rng(5)
    ns = rng.integers(0, 600, size=64)
    ns[37] = 500
    pairs, scores, counts, _ = synth.two_view_lists(list(ns), 600, KP, inlier_frac=0.7, seed=6)
    pidx = np.tile(np.array([[0, 1]], np.int32), (64, 1))
    batch, _ = run(dev, pts, bank, pairs, scores, counts, pidx, cam_of(K))
    again, _ = run(dev, pts, bank, pairs, scores, counts, pidx, cam_of(K))
    alone, _ = run(dev, pts, bank, pairs[37:38], scores[37:38], counts[37:38], pidx[37:38], cam_of(K))
    for x, y in zip(batch, again):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(batch, alone):
        assert x[37:38].tobytes() == y.tobytes()
    assert batch[4][37] > 0


@pytest.mark.parametrize("seed", range(4))
def test_accuracy_against_true_motion(dev, seed):
    """Exact points, 0.3 px keypoint noise, 30 % outlier rows; the bounds are the oracle's (test_pnp_oracle)."""
    rows, R, t, K = noisy_rows(seed)
    n = len(rows)
    pairs = np.stack([np.arange(n), np.arange(n)], 1).astype(np.int32)[None]
    (Rg, tg, _, _, oc, rms, _), _ = run(dev, rows[None, :, :3], rows[None, :, 3:], pairs, np.zeros((1, n), np.float32),
                                        np.array([n], np.int32), None, cam_of(K))
    rot, tmm = rot_err_deg(Rg[0], R), 1000.0 * float(np.linalg.norm(tg[0] - t))
    assert rot < ALONE_ROT_DEG and tmm < ALONE_T_MM, (rot, tmm)
    assert rms[0, 1] <= rms[0, 0]
    record(f"pnp_accuracy_seed{seed}", {"rot_deg": rot, "t_mm": tmm, "inliers": int(oc[0])})


def chain(b, pairs, scores, counts, K, pidx_f, pidx_pnp):
    """F RANSAC -> E -> pose -> point_map -> PnP on the device bank b."""
    from sslam_b200 import geometry
    F, vp, vs, vc = geometry.verify_fundamental_device(b, b, pairs[0:1], scores[0:1], counts[0:1], pair_index=pidx_f)
    E = geometry.essential_from_fundamental(F, K)
    R, t, _, _, _, _, _, mask, X = geometry.recover_pose_device(b, b, E, vp, vs, vc, K, pair_index=pidx_f,
                                                                want_mask=True, want_points=True)
    maps = geometry.point_map(vp, vc, X, mask, KP, R, t)
    rows, sc, n = geometry.rows_with_points(pairs[1:2], scores[1:2], counts[1:2], maps)
    return geometry.solve_pnp_device(maps, b, rows, sc, n, K, pair_index=pidx_pnp)


@pytest.mark.parametrize("seed", range(6))
def test_chain_against_true_motion(dev, seed):
    """Frames 0, 1 initialise (unit |t|), frame 2 is tracked against their points: its rotation is Rs[1] and
    its translation ts[1] / |ts[0]|, the scale check.  Bounds: the oracle's over the same seeds."""
    bank, Rs, ts, K, pairs, scores, counts = chain_inputs(seed)
    R, t, _, _, oc, rms = chain(T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev), K,
                                T(np.array([[0, 1]], np.int32), dev), T(np.array([[0, 2]], np.int32), dev))
    rot, trel = chain_errors(R[0].cpu().numpy(), t[0].cpu().numpy(), Rs, ts)
    orot, otrel = oracle_chain(seed)
    assert rot < CHAIN_ROT_DEG and trel < CHAIN_T_REL, (rot, trel)
    record(f"pnp_chain_seed{seed}", {"rot_deg": rot, "t_rel": trel, "oracle_rot_deg": orot, "oracle_t_rel": otrel,
                                     "pnp_inliers": int(oc[0]), "rms_px": rms[0].cpu().tolist()})


def test_chain_graph_replay(dev):
    bank, _, _, K, pairs, scores, counts = chain_inputs(0)
    args = (T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev), K, T(np.array([[0, 1]], np.int32), dev),
            T(np.array([[0, 2]], np.int32), dev))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = [x.clone() for x in chain(*args)]
        chain(*args)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = chain(*args)
    for x in out:
        x.zero_()
    g.replay()
    torch.cuda.synchronize()
    for x, y in zip(out, eager):
        assert torch.equal(x, y)
    assert int(eager[4][0]) > 0


@pytest.fixture(scope="module")
def sequence(dev):
    from models.descriptor_refiner import DescriptorRefiner
    from sslam_b200.pipeline import FrontEnd
    torch.manual_seed(0)
    refiner = DescriptorRefiner(384, 384, 128, 4).to(dev)
    sal, feat = synth.make_sequence(8, seq_id=0, device=dev)
    fe = FrontEnd(refiner, num_keypoints=2048, grid="pixel")
    return fe, sal, feat


CAMERA = (525.0, 525.0, 319.5, 239.5)


def test_frame_store_track_poses(dev, sequence):
    """The synthetic sequences translate a flat canvas, so the points any two-view initialisation gives are
    not a true scene: the outputs keep their format, a list without a model has zeros and an empty list,
    and every PnP list is a subsequence of its input list."""
    from sslam_b200 import geometry, matchers
    from sslam_b200.framestore import FrameStore
    fe, sal, feat = sequence
    store = FrameStore(fe, capacity=8)
    store.push(sal, feat)
    init = [(0, 1), (1, 2), (2, 3), (3, 4)]
    p1, s1, c1 = store.match_pairs(init, matchers.M1)
    R, t, _, _, _, _, mask, X = store.relative_poses(init, p1, s1, c1, CAMERA, want_mask=True, want_points=True)
    _, vp, _, vc = store.verify_pairs(init, p1, s1, c1, model="fundamental")
    K = store.bank["keypoints"].shape[1]
    maps = geometry.point_map(vp, vc, X, mask, K, R, t)
    maps[3] = float("nan")                                             # a list without any point
    track = [(1, 2), (2, 3), (3, 4), (4, 5)]
    p2, s2, c2 = store.match_pairs(track, matchers.M1)
    Rt, tt, pp, ps, pc = store.track_poses(track, p2, s2, c2, maps, CAMERA)
    P, L = p2.shape[:2]
    assert Rt.shape == (P, 3, 3) and tt.shape == (P, 3) and pp.shape == (P, L, 2) and ps.shape == (P, L)
    assert pc.shape == (P,) and Rt.dtype == torch.float64
    Rn, tn, ppn, pcn, p2n, c2n = (x.cpu().numpy() for x in (Rt, tt, pp, pc, p2, c2))
    have = np.abs(Rn).sum((1, 2)) > 0
    assert not have[3] and pcn[3] == 0
    for p in range(P):
        src = [tuple(r) for r in p2n[p, :c2n[p]]]
        it = iter(src)
        assert all(tuple(r) in it for r in ppn[p, :pcn[p]])           # a subsequence, in input order
        assert (ppn[p, pcn[p]:] == -1).all()
        if have[p]:
            assert abs(np.linalg.det(Rn[p]) - 1) < 1e-6
        else:
            assert not tn[p].any() and pcn[p] == 0
    record("pnp_frame_store", {"lists": P, "with_model": int(have.sum()), "rows_in": int(c2n.sum()),
                               "rows_kept": int(pcn.sum())})


def test_host_api_against_cv2(dev):
    from sslam_b200 import geometry
    bank, _, Rs, ts, K, Xs = synth.two_view_bank(2, 800, seed=3, noise=0.3, poses=True, points=True)
    rng = np.random.default_rng(9)
    X = Xs[0].astype(np.float32).astype(np.float64)
    uv = bank[1].astype(np.float64)
    out = rng.random(800) < 0.3
    uv[out] = rng.uniform([0, 0], [639, 479], (int(out.sum()), 2))
    ok, rvec, tvec, inl = geometry.solve_pnp_ransac(X, uv, K, iterations_count=1024, reprojection_error=3.0)
    cok, crvec, ctvec, cinl = cv2.solvePnPRansac(X, uv, K, None, iterationsCount=1024, reprojectionError=3.0,
                                                  flags=cv2.SOLVEPNP_P3P)
    assert ok and cok and rvec.shape == (3, 1) and tvec.shape == (3, 1) and inl.dtype == np.int32
    R = cv2.Rodrigues(rvec)[0]
    ref = op.ransac_pnp(np.concatenate([X, uv], 1).astype(np.float32), cam_of(K))
    assert np.abs(R - ref["R"]).max() < 1e-8 and np.abs(tvec[:, 0] - ref["t"]).max() < 1e-8
    d = np.zeros(800, bool)
    d[inl[:, 0]] = True
    assert ((d != ref["mask"]) <= ref["band"]).all()
    # Against cv2: the library is the oracle to 1e-8, so its distance to cv2's pose can differ from the
    # oracle's only by its distance to the oracle (triangle inequality of the Frobenius norm on R and of the
    # Euclidean norm on t), and its inlier set from cv2's only by the oracle's threshold-band rows.
    Rc, tc = cv2.Rodrigues(crvec)[0], ctvec[:, 0]
    nR, nR_o, nR_lo = (float(np.linalg.norm(a - b)) for a, b in ((R, Rc), (ref["R"], Rc), (R, ref["R"])))
    nt, nt_o, nt_lo = (float(np.linalg.norm(a - b)) for a, b in ((tvec[:, 0], tc), (ref["t"], tc),
                                                                  (tvec[:, 0], ref["t"])))
    assert abs(nR - nR_o) <= nR_lo + 1e-15 and abs(nt - nt_o) <= nt_lo + 1e-15, (nR, nR_o, nt, nt_o)
    rot, tmm = rot_err_deg(R, Rc), 1000.0 * nt
    c = np.zeros(800, bool)
    c[cinl[:, 0]] = True
    assert (d != c).sum() <= (ref["mask"] != c).sum() + ref["band"].sum()
    record("pnp_host_api_vs_cv2", {"rot_deg": rot, "t_mm": tmm, "oracle_t_mm": 1000.0 * nt_o,
                                   "inliers": int(inl.shape[0]), "cv2_inliers": int(cinl.shape[0]),
                                   "differing_rows": int((d != c).sum())})
    ok0, r0, t0, i0 = geometry.solve_pnp_ransac(X[:3], uv[:3], K)
    assert not ok0 and not r0.any() and not t0.any() and i0 is None
    with pytest.raises(ValueError):
        geometry.solve_pnp_ransac(X, uv, K, dist_coeffs=np.array([0.1, 0, 0, 0]))


def test_best_sample_without_inliers_is_no_model(dev):
    """At a 1e-30 px threshold t^2 rounds to 0 in fp32, so no row passes: every sample has 0 inliers, the best
    is sample 0, and the list has no model."""
    rows, _, _, K = noisy_rows(0)
    n = 64
    pairs = np.stack([np.arange(n), np.arange(n)], 1).astype(np.int32)[None]
    from sslam_b200 import ops
    ws = torch.empty(ops.ransac_workspace_bytes(1, n, 16, model="pnp"), dtype=torch.uint8, device=dev)
    R, t, pp, _, oc, rms = ops.ransac_pnp(T(rows[None, :n, :3], dev), T(rows[None, :n, 3:], dev), T(pairs, dev),
                                          torch.zeros(1, n, device=dev), torch.tensor([n], dtype=torch.int32,
                                                                                      device=dev),
                                          *cam_of(K), threshold=1e-30, iters=16, workspace=ws)
    hc, best, _ = ops.ransac_workspace_views(ws, 1, n, 16, model="pnp")
    ref = op.ransac_pnp(rows[:n], cam_of(K), iters=16, threshold=1e-30)
    assert (ref["hyp_count"] == 0).all() and ref["best"] == 0 and not ref["R"].any()
    assert np.array_equal(hc[0].cpu().numpy(), ref["hyp_count"]) and int(best[0]) == 0
    assert not R.any() and not t.any() and not rms.any() and int(oc[0]) == 0 and (pp == -1).all()


def test_bad_arguments(dev):
    from sslam_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
    p, z = ctypes.c_void_p(buf.data_ptr()), ctypes.c_void_p(0)

    def call(pts=p, L=8, iters=16, thr=3.0, refine=10, fx=500.0, out=p, ws=p, wsb=1 << 16):
        return lib.sslam_ransac_pnp(pts, 1, p, 1, z, 1, 8, 8, p, p, p, L, fx, 500.0, 320.0, 240.0, iters, thr, 0,
                                    refine, p, p, z, out, p, p, z, ws, wsb, z)
    assert call() == 0
    assert call(pts=z) == -1 and call(out=z) == -1 and call(ws=z) == -1 and call(wsb=16) == -3
    assert call(L=16385) == -1 and call(iters=0) == -1 and call(iters=65537) == -1
    assert call(refine=-1) == -1 and call(refine=101) == -1
    assert call(thr=0.0) == -1 and call(thr=float("nan")) == -1 and call(fx=0.0) == -1 and call(fx=float("inf")) == -1
    torch.cuda.synchronize()
