"""RANSAC verification (csrc/ransac.cu) timed for both models — homography and fundamental matrix — on the
match lists of three workloads:

  c2  the 599 consecutive-pair lists of a c2 run (600 synthetic frames 640x480, K = 2048, M1 ratio 0.8)
  c4  all 32 640 pairs of 256 keyframes (frames 0..255 of synthetic sequence 0, K = 2048, M2)
  gm  599 general-motion two-view lists (synth.two_view_bank, one scene per pair, 2048 rows, 0.3 px
      noise, 30 % outliers): the synthetic sequences translate a flat canvas, so most 7-point samples of
      c2 / c4 are degenerate (rank 6) and never scored; here every slot with a real root is

The lists are produced once; then sslam_ransac_homography / sslam_ransac_fundamental (iters = 1024
samples, threshold 3 px) run WARMUP + REPS times per workload and model and are timed with CUDA events
around each call; a separate profiled call splits the time per kernel.  Reports ms per batch, error
evaluations per second (sum over pairs of n * scored hypothesis slots: iters for H, the non-degenerate
slots of 3 * iters for F), the ratio to the c2 step (10.57 ms, DESIGN.md section 5), and the GPU's name
and power limit read in the same run.  Prints one JSON line; with OUT=<path> in the environment the
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
import numpy as np  # noqa: E402
from sslam_b200 import dist, geometry, matchers, ops, synth  # noqa: E402
from sslam_b200.pipeline import FrontEnd  # noqa: E402

ITERS, THRESH = 1024, 3.0
WARMUP, REPS = int(os.environ.get("WARMUP", 3)), int(os.environ.get("REPS", 20))
C2_STEP_MS = 10.57


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def time_verify(kp1, kp2, pairs, scores, counts, pair_index=None, num_pairs=None, model="homography"):
    P, L = pairs.shape[:2]
    ws = torch.empty(ops.ransac_workspace_bytes(P, L, ITERS, model=model), dtype=torch.uint8, device=pairs.device)
    verify = geometry.verify_fundamental_device if model == "fundamental" else geometry.verify_homography_device

    def call():
        return verify(kp1, kp2, pairs, scores, counts, pair_index=pair_index, num_pairs=num_pairs,
                      threshold=THRESH, iters=ITERS, workspace=ws)
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
    hc = ops.ransac_workspace_views(ws, P, L, ITERS, model=model)[0]
    scored = (hc >= 0).to(torch.int64).sum(1)                 # slots the scoring kernel evaluates
    evals = int((n * scored).sum())
    med = statistics.median(ms)
    kept = int(out[3].to(torch.int64).sum())
    return dict(pairs=P, list_stride=L, matches=int(n.sum()), mean_matches=round(float(n.float().mean()), 1),
                kept=kept, iters=ITERS, scored_slots=int(scored.sum()), ms_median=round(med, 4),
                ms_min=round(min(ms), 4), ms_max=round(max(ms), 4), evals=evals,
                evals_per_s=float("%.4g" % (evals / (med * 1e-3))), ratio_to_c2_step=round(med / C2_STEP_MS, 4),
                kernel_ms=kinds, workspace_bytes=ws.numel())


def both(*args, **kw):
    out = {}
    for model in ("homography", "fundamental"):
        out[model] = time_verify(*args, model=model, **kw)
        torch.cuda.empty_cache()
    return out


def general_motion_lists(P=599, K=2048, dev=None):
    """P independent two-view scenes (one per pair): banks (P,K,2) x 2 and lists of K rows, 30 % outliers."""
    b1, b2 = np.empty((P, K, 2), np.float32), np.empty((P, K, 2), np.float32)
    for p in range(P):
        bank, _ = synth.two_view_bank(2, K, seed=1000 + p, noise=0.3)
        b1[p], b2[p] = bank[0], bank[1]
    pairs, scores, counts, _ = synth.two_view_lists([K] * P, K, K, inlier_frac=0.7, seed=7)
    t = lambda x: torch.as_tensor(x).to(dev)                     # noqa: E731
    return t(b1), t(b2), t(pairs), t(scores), t(counts)


def main():
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    refiner = DescriptorRefiner(384, 384, 256, 4).to(dev).eval()
    fe = FrontEnd(refiner, num_keypoints=2048, grid="pixel")
    res = {"gpu": gpu_info(), "warmup": WARMUP, "reps": REPS, "threshold_px": THRESH}

    sal, feat = synth.make_sequence(600, seq_id=0, device=dev)
    feats, pairs, pscores, counts = fe.run_sequence(sal, feat, matchers.M1, ratio_thresh=0.8)
    kp = feats["keypoints_pixel"]
    res["c2"] = both(kp, kp[1:], pairs, pscores, counts, num_pairs=599)
    del sal, feat, feats, pairs, pscores, counts, kp

    sal, feat = synth.make_sequence(256, seq_id=0, device=dev)
    idx = dist.all_pairs_index(256).to(dev)
    feats, pairs, pscores, counts = fe.run_pairs(sal, feat, idx, matchers.M2)
    kp = feats["keypoints_pixel"]
    res["c4"] = both(kp, kp, pairs, pscores, counts, pair_index=idx)
    del sal, feat, feats, pairs, pscores, counts, kp, idx

    res["gm"] = both(*general_motion_lists(dev=dev), num_pairs=599)

    out = os.environ.get("OUT")
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
