"""GPU tests of the triangulation under a known pose and of the tracking step with map growth
(csrc/triangulate.cu, geometry.triangulate_device / track_and_map, FrameStore.track_and_map): parity with
oracle/triangulate.py on a ragged, aliased batch, batch independence and determinism, the 12-frame chain
against the oracle chain and the true motion, CUDA-graph replay of one step, the frame store and argument
errors."""

import ctypes

import numpy as np
import pytest
import torch

from oracle import triangulate as otri
from parity import record
from sslam_b200 import synth
from test_triangulate_oracle import (CHAIN_MIN_ROWS, CHAIN_ROT_DEG, CHAIN_T_REL, FRAMES, KP, cam_of, chain12_inputs,
                                     oracle_chain12, step_errors)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def T(x, dev):
    return torch.as_tensor(x).to(dev)


def run(dev, bank, pairs, scores, counts, pidx, R, t, cam, refine=10):
    from sslam_b200 import ops
    out = ops.triangulate(T(bank, dev), T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev), T(R, dev),
                          T(t, dev), *cam, pair_index=None if pidx is None else T(pidx, dev), refine_iters=refine,
                          want_mask=True)
    torch.cuda.synchronize()
    return [x.cpu().numpy() for x in out]


def parity_batch():
    """Ragged lists aliasing a 3-set bank: sizes 0, 1, 5, 100, 2048, then a list without a pose, one with
    t = 0, one with an index out of range and one with a non-finite keypoint."""
    bank, _, Rs, ts, K, _ = synth.two_view_bank(3, KP, seed=0, noise=0.3, poses=True, points=True)
    ns = [0, 1, 5, 100, 2048, 100, 100, 100, 100]
    pairs, scores, counts, _ = synth.two_view_lists(ns, 2100, KP, inlier_frac=0.7, seed=2)
    pidx = np.array([[0, 1], [1, 2], [0, 1], [1, 2], [0, 1], [0, 1], [1, 2], [1, 2], [0, 1]], np.int32)
    R = np.stack([Rs[a] for a, _ in pidx]).reshape(-1, 9)
    t = np.stack([ts[a] for a, _ in pidx])
    R[5] = 0.0                                                           # no pose
    t[6] = 0.0                                                           # zero baseline
    pairs[7, 3, 1] = KP + 5                                              # an index out of range
    bank[0][pairs[8, 7, 0]] = np.nan                                     # a non-finite keypoint
    return bank, pairs, scores, counts, pidx, R, t, cam_of(K), ns


@pytest.mark.parametrize("refine", [0, 10])
def test_oracle_parity_ragged_aliased(dev, refine):
    bank, pairs, scores, counts, pidx, R, t, cam, ns = parity_batch()
    X, op_, osc, oc, mask = run(dev, bank, pairs, scores, counts, pidx, R, t, cam, refine)
    band_rows, worst = 0, 0.0
    for p, n in enumerate(ns):
        a, b = pidx[p]
        ref = otri.triangulate(otri.list_points(bank[a], bank[b], pairs[p, :n]), R[p].reshape(3, 3), t[p], cam,
                               refine_iters=refine)
        keep = mask[p, :n].astype(bool)
        d = keep != ref["mask"]
        assert (d <= ref["band"]).all(), p
        band_rows += int(d.sum())
        assert not mask[p, n:].any() and not X[p, n:].any()
        both = keep & ref["mask"]
        if both.any():
            e = np.abs(X[p, :n][both] - ref["points"][both]).max() / np.abs(ref["points"][both]).max()
            assert e < 1e-6, (p, e)
            worst = max(worst, float(e))
        assert not X[p, :n][~keep].any()
        assert oc[p] == keep.sum()
        assert np.array_equal(op_[p, :oc[p]], pairs[p, :n][keep])     # a subsequence in input order
        assert np.array_equal(osc[p, :oc[p]], scores[p, :n][keep])
        assert (op_[p, oc[p]:] == -1).all() and (osc[p, oc[p]:] == 0).all()
    assert oc[0] == 0 and oc[5] == 0 and oc[6] == 0 and oc[4] > 1000
    assert not mask[7, 3] and not mask[8, 7]
    record(f"tri_oracle_parity_refine{refine}", {"lists": len(ns), "band_rows": band_rows, "max_rel_point": worst,
                                                 "kept": [int(c) for c in oc]})


def test_batch_independence_and_determinism(dev):
    bank, _, Rs, ts, K, _ = synth.two_view_bank(2, KP, seed=4, noise=0.3, poses=True, points=True)
    rng = np.random.default_rng(5)
    ns = rng.integers(0, 600, size=64)
    ns[37] = 500
    pairs, scores, counts, _ = synth.two_view_lists(list(ns), 600, KP, inlier_frac=0.7, seed=6)
    pidx = np.tile(np.array([[0, 1]], np.int32), (64, 1))
    R, t = np.tile(Rs[0].reshape(1, 9), (64, 1)), np.tile(ts[0], (64, 1))
    batch = run(dev, bank, pairs, scores, counts, pidx, R, t, cam_of(K))
    again = run(dev, bank, pairs, scores, counts, pidx, R, t, cam_of(K))
    alone = run(dev, bank, pairs[37:38], scores[37:38], counts[37:38], pidx[37:38], R[37:38], t[37:38], cam_of(K))
    for x, y in zip(batch, again):
        assert x.tobytes() == y.tobytes()
    for x, y in zip(batch, alone):
        assert x[37:38].tobytes() == y.tobytes()
    assert batch[3][37] > 0


def device_init(b, pairs, scores, counts, K, dev):
    """F RANSAC -> E -> pose on list (0, 1) -> the point map of frame 1 (1, KP, 3)."""
    from sslam_b200 import geometry
    pidx = T(np.array([[0, 1]], np.int32), dev)
    F, vp, vs, vc = geometry.verify_fundamental_device(b, b, pairs[0:1], scores[0:1], counts[0:1], pair_index=pidx)
    E = geometry.essential_from_fundamental(F, K)
    R, t, _, _, _, _, _, mask, X = geometry.recover_pose_device(b, b, E, vp, vs, vc, K, pair_index=pidx,
                                                                want_mask=True, want_points=True)
    return geometry.point_map(vp, vc, X, mask, KP, R, t)


def step(b, maps, pairs, scores, counts, K, k, pidx):
    """track_and_map on list k, pidx = [[k, k + 1]] on the device."""
    from sslam_b200 import geometry
    return geometry.track_and_map(maps, b, b, pairs[k:k + 1], scores[k:k + 1], counts[k:k + 1], K, pidx)


@pytest.mark.parametrize("seed", range(6))
def test_chain12_against_oracle_and_true_motion(dev, seed):
    """Frames 0, 1 initialise (unit |t|), frames 2-11 are tracked and mapped one step at a time; step k's
    rotation is Rs[k] and its translation ts[k] / |ts[0]|.  Bounds: the oracle chain's (test_triangulate_oracle)."""
    from sslam_b200 import geometry
    bank, Rs, ts, K, pairs, scores, counts = chain12_inputs(seed)
    b, pr, sc, cn = T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev)
    maps = device_init(b, pr, sc, cn, K, dev)
    ref = oracle_chain12(seed)
    rots, trels, rows, dev_rot, dev_trel = [], [], [], 0.0, 0.0
    for k in range(1, FRAMES - 1):
        n = int(geometry.rows_with_points(pr[k:k + 1], sc[k:k + 1], cn[k:k + 1], maps)[2][0])
        R, t, _, _, pc, maps = step(b, maps, pr, sc, cn, K, k, T(np.array([[k, k + 1]], np.int32), dev))
        Rn, tn = R[0].cpu().numpy(), t[0].cpu().numpy()
        assert Rn.any() and int(pc[0]) > 0, k
        rot, trel = step_errors(Rn, tn, Rs, ts, k)
        o = ref[k - 1]
        # The pose and PnP refinements sum in a fixed tree order on the device and in NumPy's order in the
        # oracle, so each step's pose agrees to rounding and ten chained steps let that grow: the largest
        # difference measured on seeds 0-5 is 1.4e-5 deg (seed 5, last step).  The rows with a point that
        # enter each step's PnP are the oracle's exactly.
        assert n == o["rows"], (k, n, o["rows"])
        assert abs(rot - o["rot"]) < 1e-4 and abs(trel - o["trel"]) < 1e-4, (k, rot, o["rot"], trel, o["trel"])
        dev_rot, dev_trel = max(dev_rot, abs(rot - o["rot"])), max(dev_trel, abs(trel - o["trel"]))
        assert rot < CHAIN_ROT_DEG and trel < CHAIN_T_REL and n > CHAIN_MIN_ROWS, (k, rot, trel, n)
        rots.append(rot)
        trels.append(trel)
        rows.append(n)
    record(f"tri_chain12_seed{seed}", {"rot_deg": rots, "t_rel": trels, "rows_with_point": rows,
                                       "oracle_rows_with_point": [s["rows"] for s in ref],
                                       "max_abs_diff_rot_deg": dev_rot, "max_abs_diff_t_rel": dev_trel})


def test_track_and_map_graph_replay(dev):
    bank, _, _, K, pairs, scores, counts = chain12_inputs(0)
    b, pr, sc, cn = T(bank, dev), T(pairs, dev), T(scores, dev), T(counts, dev)
    maps = device_init(b, pr, sc, cn, K, dev)
    pidx = T(np.array([[1, 2]], np.int32), dev)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = [x.clone() for x in step(b, maps, pr, sc, cn, K, 1, pidx)]
        step(b, maps, pr, sc, cn, K, 1, pidx)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        out = step(b, maps, pr, sc, cn, K, 1, pidx)
    for x in out:
        x.zero_()
    g.replay()
    torch.cuda.synchronize()
    for x, y in zip(out, eager):
        assert torch.equal(x.nan_to_num(), y.nan_to_num()) and torch.equal(x.isnan(), y.isnan())
    assert int(eager[4][0]) > 0 and torch.isfinite(eager[5]).all(-1).sum() > int(eager[4][0])


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


def test_frame_store_track_and_map(dev, sequence):
    """The synthetic sequences translate a flat canvas, so the points are not a true scene: the outputs keep
    their format, every PnP list is a subsequence of its input list, and a lost list has zeros and an
    all-NaN map.  triangulate_pairs under the tracked poses gives the points the step adds."""
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
    Rt, tt, pp, ps, pc, nxt = store.track_and_map(track, p2, s2, c2, maps, CAMERA)
    P, L = p2.shape[:2]
    assert Rt.shape == (P, 3, 3) and tt.shape == (P, 3) and pp.shape == (P, L, 2) and ps.shape == (P, L)
    assert pc.shape == (P,) and nxt.shape == (P, K, 3) and nxt.dtype == torch.float32
    ref = store.track_poses(track, p2, s2, c2, maps, CAMERA)
    for x, y in zip((Rt, tt, pp, ps, pc), ref):
        assert torch.equal(x, y)
    pts, tp, ts_, tc = store.triangulate_pairs(track, p2, s2, c2, Rt, tt, CAMERA)
    Rn, pcn, ppn, p2n, c2n, tcn = (x.cpu().numpy() for x in (Rt, pc, pp, p2, c2, tc))
    have = np.abs(Rn).sum((1, 2)) > 0
    assert not have[3] and pcn[3] == 0 and tcn[3] == 0 and torch.isnan(nxt[3]).all()
    for p in range(P):
        src = [tuple(r) for r in p2n[p, :c2n[p]]]
        it = iter(src)
        assert all(tuple(r) in it for r in ppn[p, :pcn[p]])
        if not have[p]:
            assert torch.isnan(nxt[p]).all()
    record("tri_frame_store", {"lists": P, "with_model": int(have.sum()), "pnp_rows": int(pcn.sum()),
                               "triangulated_rows": int(tcn.sum()),
                               "keypoints_with_point": int(torch.isfinite(nxt).all(-1).sum())})


def test_bad_arguments(dev):
    from sslam_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
    p, z = ctypes.c_void_p(buf.data_ptr()), ctypes.c_void_p(0)

    def call(k1=p, L=8, thr=3.0, cos=0.99, dist=50.0, refine=10, fx=500.0, R=p, out=p):
        return lib.sslam_triangulate(k1, 1, p, 1, z, 1, 8, 8, p, p, p, L, R, p, fx, 500.0, 320.0, 240.0, thr, cos,
                                     dist, refine, z, out, p, p, z, z)
    assert call() == 0
    assert call(k1=z) == -1 and call(R=z) == -1 and call(out=z) == -1
    assert call(L=16385) == -1 and call(refine=-1) == -1 and call(refine=101) == -1
    assert call(thr=0.0) == -1 and call(thr=float("nan")) == -1 and call(thr=float("inf")) == -1
    assert call(cos=-0.1) == -1 and call(cos=1.5) == -1 and call(cos=float("nan")) == -1
    assert call(dist=0.0) == -1 and call(dist=-1.0) == -1 and call(fx=0.0) == -1
    torch.cuda.synchronize()
