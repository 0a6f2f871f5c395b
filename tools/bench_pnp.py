"""PnP RANSAC (csrc/pnp.cu) timed on 2D-3D match lists:

  c2  599 lists, one per consecutive pair of a 600-frame run
  c4  32 640 lists, as many as all pairs of 256 keyframes
  Both over 599 general-motion scenes (synth.two_view_bank, 2048 keypoints, 0.3 px noise; c4's list p reads
  scene p mod 599 through pair_index): list p pairs the exact 3-D points of camera 0 with the keypoints of
  camera 1, 2048 rows, 30 % outlier rows (synth.two_view_lists).

sslam_ransac_pnp runs WARMUP + REPS times per workload at iters = 1024 samples, 3 px, refine_iters 0 and 10,
timed with CUDA events around each call; then F RANSAC + E + pose + point_map + PnP is timed as one chain on c2
(frames 0, 1 of each scene initialise, frame 2 is tracked against their points, the rows without a point
dropped first).  Reports ms per batch (median, min, max), the per-kernel ms of one profiled call, the score
kernel's evaluations (lists x samples x rows) per second, and the GPU's name, power limit and max SM clock
read in the same run; for the chain also the rows that enter the PnP (those with a point) and the rows it
keeps.  Prints one JSON line; with OUT=<path> in the environment the result is also written there
(indented)."""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "semantic-slam-master_b200")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
from sslam_b200 import geometry, ops, synth  # noqa: E402

ITERS, THRESH, KPTS, SCENES = 1024, 3.0, 2048, 599
WARMUP, REPS = int(os.environ.get("WARMUP", 3)), int(os.environ.get("REPS", 20))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def timed(call):
    for _ in range(WARMUP):
        call()
    torch.cuda.synchronize()
    ms = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ops.profile_enable(True)
    call()
    torch.cuda.synchronize()
    kinds = {k: round(v[0], 4) for k, v in ops.profile_read().items()}
    ops.profile_enable(False)
    return out, dict(ms_median=round(statistics.median(ms), 4), ms_min=round(min(ms), 4), ms_max=round(max(ms), 4),
                     kernel_ms=kinds)


def scenes(dev):
    """Keypoints (3*SCENES, KPTS, 2): sets 3p, 3p+1, 3p+2 are cameras 0-2 of scene p; points (SCENES, KPTS, 3)
    of camera 0."""
    kp = np.empty((3 * SCENES, KPTS, 2), np.float32)
    pts = np.empty((SCENES, KPTS, 3), np.float32)
    K = None
    for p in range(SCENES):
        bank, _, _, _, K, Xs = synth.two_view_bank(3, KPTS, seed=1000 + p, noise=0.3, poses=True, points=True)
        kp[3 * p:3 * p + 3], pts[p] = bank, Xs[0]
    return torch.as_tensor(kp).to(dev), torch.as_tensor(pts).to(dev), K


def lists(P, dev, seed):
    pairs, scores, counts, _ = synth.two_view_lists([KPTS] * P, KPTS, KPTS, inlier_frac=0.7, seed=seed)
    t = lambda x: torch.as_tensor(x).to(dev)                     # noqa: E731
    return t(pairs), t(scores), t(counts)


def pnp_times(kp, pts, K, P, dev, seed):
    pairs, scores, counts = lists(P, dev, seed)
    s = torch.arange(P, dtype=torch.int32, device=dev) % SCENES
    pidx = torch.stack([s, 3 * s + 1], 1)
    res = {"lists": P, "rows_in": P * KPTS}
    for refine in (0, 10):
        out, tm = timed(lambda: geometry.solve_pnp_device(pts, kp, pairs, scores, counts, K, pair_index=pidx,
                                                          threshold=THRESH, iters=ITERS, refine_iters=refine))
        tm["rows_kept"] = int(out[4].to(torch.int64).sum())
        tm["with_model"] = int((out[0].abs().sum((1, 2)) > 0).sum())
        sc = tm["kernel_ms"].get("pnp_score")
        tm["score_evals_per_s"] = float(f"{P * ITERS * KPTS / (sc * 1e-3):.3g}") if sc else None
        res[f"refine{refine}"] = tm
    return res


def main():
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "warmup": WARMUP, "reps": REPS, "iters": ITERS, "threshold_px": THRESH,
           "rows_per_list": KPTS}
    kp, pts, K = scenes(dev)
    res["c2"] = pnp_times(kp, pts, K, 599, dev, seed=7)

    pairs, scores, counts = lists(2 * SCENES, dev, seed=9)           # lists 0..598: (0, 1); 599..: (1, 2)
    s = torch.arange(SCENES, dtype=torch.int32, device=dev)
    pidx_f = torch.stack([3 * s, 3 * s + 1], 1)
    pidx_t = torch.stack([s, 3 * s + 2], 1)
    a, b = slice(0, SCENES), slice(SCENES, 2 * SCENES)

    def chain():
        F, vp, vs, vc = geometry.verify_fundamental_device(kp, kp, pairs[a], scores[a], counts[a], pair_index=pidx_f,
                                                           threshold=THRESH, iters=ITERS)
        R, t, _, _, _, _, _, mask, X = geometry.recover_pose_device(
            kp, kp, geometry.essential_from_fundamental(F, K), vp, vs, vc, K, pair_index=pidx_f, want_mask=True,
            want_points=True)
        maps = geometry.point_map(vp, vc, X, mask, KPTS, R, t)
        rows, sc, n = geometry.rows_with_points(pairs[b], scores[b], counts[b], maps)
        return geometry.solve_pnp_device(maps, kp, rows, sc, n, K, pair_index=pidx_t, threshold=THRESH,
                                         iters=ITERS) + (n,)
    out, res["c2_chain"] = timed(chain)
    res["c2_chain"]["pnp_rows_in"] = int(out[-1].to(torch.int64).sum())        # rows with a point
    res["c2_chain"]["pnp_rows_kept"] = int(out[4].to(torch.int64).sum())
    del pairs, scores, counts, out
    torch.cuda.empty_cache()
    res["c4"] = pnp_times(kp, pts, K, 32640, dev, seed=8)

    out = os.environ.get("OUT")
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
