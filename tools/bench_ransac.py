"""RANSAC homography verification (csrc/ransac.cu) timed on the match lists of two workloads:

  c2  the 599 consecutive-pair lists of a c2 run (600 synthetic frames 640x480, K = 2048, M1 ratio 0.8)
  c4  all 32 640 pairs of 256 keyframes (frames 0..255 of synthetic sequence 0, K = 2048, M2)

The lists are produced once by the pipeline; then sslam_ransac_homography (iters = 1024, threshold
3 px) runs WARMUP + REPS times per workload and is timed with CUDA events around each call; a separate
profiled call splits the time per kernel.  Reports ms per batch, transfer-error evaluations per second
(sum over pairs of n * iters), the ratio to the c2 step (10.57 ms, DESIGN.md section 5), and the GPU's
name and power limit read in the same run.  Prints one JSON line; with OUT=<path> in the environment the
result is also written there (indented)."""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "semantic-slam-master_b200")]
import torch  # noqa: E402
from models.descriptor_refiner import DescriptorRefiner  # noqa: E402
from sslam_b200 import dist, geometry, matchers, ops, synth  # noqa: E402
from sslam_b200.pipeline import FrontEnd  # noqa: E402

ITERS, THRESH = 1024, 3.0
WARMUP, REPS = int(os.environ.get("WARMUP", 3)), int(os.environ.get("REPS", 20))
C2_STEP_MS = 10.57


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def time_verify(kp1, kp2, pairs, scores, counts, pair_index=None, num_pairs=None):
    P, L = pairs.shape[:2]
    ws = torch.empty(ops._lib.load().sslam_ransac_workspace_bytes(P, L, ITERS), dtype=torch.uint8,
                     device=pairs.device)

    def call():
        return geometry.verify_homography_device(kp1, kp2, pairs, scores, counts, pair_index=pair_index,
                                                 num_pairs=num_pairs, threshold=THRESH, iters=ITERS, workspace=ws)
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
    n = counts.to(torch.int64).clamp(max=L)
    evals = int(n.sum()) * ITERS
    med = statistics.median(ms)
    kept = int(out[3].to(torch.int64).sum())
    return dict(pairs=P, list_stride=L, matches=int(n.sum()), mean_matches=round(float(n.float().mean()), 1),
                kept=kept, iters=ITERS, ms_median=round(med, 4), ms_min=round(min(ms), 4), ms_max=round(max(ms), 4),
                evals=evals, evals_per_s=float("%.4g" % (evals / (med * 1e-3))),
                ratio_to_c2_step=round(med / C2_STEP_MS, 4), kernel_ms=kinds)


def main():
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    refiner = DescriptorRefiner(384, 384, 256, 4).to(dev).eval()
    fe = FrontEnd(refiner, num_keypoints=2048, grid="pixel")
    res = {"gpu": gpu_info(), "warmup": WARMUP, "reps": REPS, "threshold_px": THRESH}

    sal, feat = synth.make_sequence(600, seq_id=0, device=dev)
    feats, pairs, pscores, counts = fe.run_sequence(sal, feat, matchers.M1, ratio_thresh=0.8)
    kp = feats["keypoints_pixel"]
    res["c2"] = time_verify(kp, kp[1:], pairs, pscores, counts, num_pairs=599)
    del sal, feat, feats, pairs, pscores, counts, kp

    sal, feat = synth.make_sequence(256, seq_id=0, device=dev)
    idx = dist.all_pairs_index(256).to(dev)
    feats, pairs, pscores, counts = fe.run_pairs(sal, feat, idx, matchers.M2)
    kp = feats["keypoints_pixel"]
    res["c4"] = time_verify(kp, kp, pairs, pscores, counts, pair_index=idx)

    out = os.environ.get("OUT")
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
