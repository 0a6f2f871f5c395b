"""Relative pose (csrc/pose.cu) timed on general-motion match lists:

  c2  599 lists, one per consecutive pair of a 600-frame run
  c4  32 640 lists, as many as all pairs of 256 keyframes
  Both over 599 general-motion two-view scenes (synth.two_view_bank, 2048 keypoints, 0.3 px noise; c4's
  list p reads scene p mod 599 through pair_index) with 2048-row lists, 30 % outliers (synth.two_view_lists).

The lists are verified once by the F RANSAC (iters = 1024 samples, 3 px); E = K^T F K.  Then
sslam_recover_pose runs WARMUP + REPS times per workload at refine_iters 0 and 10, timed with CUDA events
around each call, and F RANSAC + E + pose (refine_iters 10) is timed as one chain on c2.  Reports ms per
batch (median, min, max), the rows entering the pose kernel and the rows it keeps, and the GPU's name and
power limit read in the same run.  Prints one JSON line; with OUT=<path> in the environment the result is
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
    b1, b2 = np.empty((SCENES, KPTS, 2), np.float32), np.empty((SCENES, KPTS, 2), np.float32)
    K = None
    for p in range(SCENES):
        bank, _, _, _, K = synth.two_view_bank(2, KPTS, seed=1000 + p, noise=0.3, poses=True)
        b1[p], b2[p] = bank[0], bank[1]
    return torch.as_tensor(b1).to(dev), torch.as_tensor(b2).to(dev), K


def workload(b1, b2, K, P, dev, seed):
    pairs, scores, counts, _ = synth.two_view_lists([KPTS] * P, KPTS, KPTS, inlier_frac=0.7, seed=seed)
    idx = np.arange(P, dtype=np.int32) % SCENES
    pidx = torch.as_tensor(np.stack([idx, idx], 1)).to(dev)
    t = lambda x: torch.as_tensor(x).to(dev)                     # noqa: E731
    return pidx, t(pairs), t(scores), t(counts)


def pose_times(b1, b2, K, pidx, pairs, scores, counts):
    F, vp, vs, vc = geometry.verify_fundamental_device(b1, b2, pairs, scores, counts, pair_index=pidx,
                                                       threshold=THRESH, iters=ITERS)
    E = geometry.essential_from_fundamental(F, K)
    res = {"pairs": int(pairs.shape[0]), "rows_in": int(vc.to(torch.int64).sum())}
    for refine in (0, 10):
        out, tm = timed(lambda: geometry.recover_pose_device(b1, b2, E, vp, vs, vc, K, pair_index=pidx,
                                                             refine_iters=refine))
        tm["rows_kept"] = int(out[4].to(torch.int64).sum())
        tm["with_pose"] = int((out[1].abs().sum(1) > 0).sum())
        res[f"refine{refine}"] = tm
    return res


def main():
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "warmup": WARMUP, "reps": REPS, "ransac_iters": ITERS, "threshold_px": THRESH,
           "rows_per_list": KPTS}
    b1, b2, K = scenes(dev)
    c2 = workload(b1, b2, K, 599, dev, seed=7)
    res["c2"] = pose_times(b1, b2, K, *c2)
    pidx, pairs, scores, counts = c2

    def chain():
        F, vp, vs, vc = geometry.verify_fundamental_device(b1, b2, pairs, scores, counts, pair_index=pidx,
                                                           threshold=THRESH, iters=ITERS)
        return geometry.recover_pose_device(b1, b2, geometry.essential_from_fundamental(F, K), vp, vs, vc, K,
                                            pair_index=pidx, refine_iters=10)
    _, res["c2_ransac_f_plus_pose"] = timed(chain)
    del c2, pidx, pairs, scores, counts
    torch.cuda.empty_cache()
    res["c4"] = pose_times(b1, b2, K, *workload(b1, b2, K, 32640, dev, seed=8))

    out = os.environ.get("OUT")
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
