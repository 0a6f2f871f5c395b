"""Triangulation under a known pose (csrc/triangulate.cu) and the tracking step with map growth timed:

  c2  599 lists, one per consecutive pair of a 600-frame run
  c4  32 640 lists, as many as all pairs of 256 keyframes
  Both over 599 general-motion scenes (synth.two_view_bank, 2048 keypoints, 0.3 px noise; c4's list p reads
  scene p mod 599 through pair_index): list p pairs the keypoints of cameras 0 and 1, 2048 rows, 30 % outlier
  rows (synth.two_view_lists), under the scene's true relative pose.

sslam_triangulate runs WARMUP + REPS times per workload at refine_iters 0 and 10, timed with CUDA events around
each call; then one geometry.track_and_map step (PnP at 1024 samples against the exact points of camera 0,
carry, triangulation, map fill) is timed at P = 1 (the latency of one sequence) and at P = 599.  Reports ms per
call (median, min, max), the per-kernel ms of one profiled call, the rows kept, and the GPU's name, power limit
and max SM clock read in the same run.  Prints one JSON line; with OUT=<path> in the environment the result is
also written there (indented)."""
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
    """Keypoints (2*SCENES, KPTS, 2): sets 2p, 2p+1 are cameras 0, 1 of scene p; the exact points of camera 0
    (SCENES, KPTS, 3) fp32; the true poses R (SCENES, 9), t (SCENES, 3)."""
    kp = np.empty((2 * SCENES, KPTS, 2), np.float32)
    pts = np.empty((SCENES, KPTS, 3), np.float32)
    R, t = np.empty((SCENES, 9)), np.empty((SCENES, 3))
    K = None
    for p in range(SCENES):
        bank, _, Rs, ts, K, Xs = synth.two_view_bank(2, KPTS, seed=1000 + p, noise=0.3, poses=True, points=True)
        kp[2 * p:2 * p + 2], pts[p], R[p], t[p] = bank, Xs[0], Rs[0].reshape(9), ts[0]
    T = lambda x: torch.as_tensor(x).to(dev)                     # noqa: E731
    return T(kp), T(pts), T(R), T(t), K


def lists(P, dev, seed):
    pairs, scores, counts, _ = synth.two_view_lists([KPTS] * P, KPTS, KPTS, inlier_frac=0.7, seed=seed)
    t = lambda x: torch.as_tensor(x).to(dev)                     # noqa: E731
    return t(pairs), t(scores), t(counts)


def tri_times(kp, R, t, K, P, dev, seed):
    pairs, scores, counts = lists(P, dev, seed)
    s = torch.arange(P, dtype=torch.int32, device=dev) % SCENES
    pidx = torch.stack([2 * s, 2 * s + 1], 1)
    Rp, tp = R[s.long()], t[s.long()]
    res = {"lists": P, "rows_in": P * KPTS}
    for refine in (0, 10):
        out, tm = timed(lambda: geometry.triangulate_device(kp, kp, pairs, scores, counts, Rp, tp, K, pair_index=pidx,
                                                            threshold=THRESH, refine_iters=refine))
        tm["rows_kept"] = int(out[3].to(torch.int64).sum())
        tri = tm["kernel_ms"].get("triangulate")
        tm["rows_per_s"] = float(f"{P * KPTS / (tri * 1e-3):.3g}") if tri else None
        res[f"refine{refine}"] = tm
    return res


def step_times(kp, pts, K, P, dev, seed):
    pairs, scores, counts = lists(P, dev, seed)
    s = torch.arange(P, dtype=torch.int32, device=dev) % SCENES
    pidx = torch.stack([2 * s, 2 * s + 1], 1)
    maps = pts[s.long()].contiguous()
    out, tm = timed(lambda: geometry.track_and_map(maps, kp, kp, pairs, scores, counts, K, pidx, threshold=THRESH,
                                                   iters=ITERS))
    tm["lists"] = P
    tm["pnp_rows_kept"] = int(out[4].to(torch.int64).sum())
    tm["next_map_points"] = int(torch.isfinite(out[5]).all(-1).sum())
    return tm


def main():
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "warmup": WARMUP, "reps": REPS, "threshold_px": THRESH, "rows_per_list": KPTS,
           "pnp_iters": ITERS}
    kp, pts, R, t, K = scenes(dev)
    res["c2"] = tri_times(kp, R, t, K, 599, dev, seed=7)
    res["step_p1"] = step_times(kp, pts, K, 1, dev, seed=9)
    res["step_p599"] = step_times(kp, pts, K, 599, dev, seed=9)
    torch.cuda.empty_cache()
    res["c4"] = tri_times(kp, R, t, K, 32640, dev, seed=8)

    out = os.environ.get("OUT")
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
