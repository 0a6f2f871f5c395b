"""Sliding-window bundle adjustment (csrc/bundle_adjust.cu) and one full sliding-window step timed:

  ba_p1, ba_p599   1 and 599 windows of W = 5 frames of 2048 keypoints (synth.two_view_bank, 0.3 px noise; window
                   p reads scene p mod 64 through frame_index), 2000 tracks each observed in all five frames, N =
                   W * 2048, the last three poses and the points perturbed, at refine_iters 0 and 10
  step_p1, step_p599   track_and_map(want_links) into the fifth frame (PnP at 1024 samples against frame 4's map,
                   2048-row lists with 30 % outlier rows), window_tracks, the adjustment (10 trials) and window_map

Every workload runs WARMUP + REPS times, timed with CUDA events around each call, then once with the library's
per-kernel profiling (kind ``bundle_adjust``).  Reports ms per call (median, min, max), the per-kernel ms, the
accepted trials and the rms before / after, and the GPU's name, power limit and max SM clock read in the same
run.  Prints one JSON line; with OUT=<path> in the environment the result is also written there (indented)."""
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

W, KPTS, TRACKS, SCENES = 5, 2048, 2000, 64
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


def scenes():
    """Bank (SCENES*W, KPTS, 2), the points of every frame in its camera (SCENES, W, KPTS, 3), absolute poses of
    the frames in frame 0's coordinates (SCENES, W, 3, 3), (SCENES, W, 3), K."""
    kp = np.empty((SCENES * W, KPTS, 2), np.float32)
    X = np.empty((SCENES, W, KPTS, 3))
    R, t = np.empty((SCENES, W, 3, 3)), np.empty((SCENES, W, 3))
    K = None
    for s in range(SCENES):
        bank, _, Rs, ts, K, Xs = synth.two_view_bank(W, KPTS, seed=2000 + s, noise=0.3, poses=True, points=True)
        kp[W * s:W * s + W], X[s] = bank, Xs
        R[s, 0], t[s, 0] = np.eye(3), 0.0
        for w in range(1, W):
            R[s, w] = Rs[w - 1] @ R[s, w - 1]
            t[s, w] = Rs[w - 1] @ t[s, w - 1] + ts[w - 1]
    return kp, X, R, t, K


def ba_inputs(P, X, R, t, dev, seed):
    rng = np.random.default_rng(seed)
    s = np.arange(P) % SCENES
    fi = (W * s[:, None] + np.arange(W)[None]).astype(np.int32)
    obs = np.full((P, W * KPTS, W), -1, np.int32)
    obs[:, :TRACKS] = np.arange(TRACKS)[None, :, None]
    pts = np.full((P, W * KPTS, 3), np.nan, np.float32)
    pts[:, :TRACKS] = X[s, 0, :TRACKS] + rng.normal(0, 0.01, (P, TRACKS, 3))
    Rp, tp = R[s].copy(), t[s].copy()
    for p in range(P):
        for w in range(2, W):
            Rp[p, w] = synth._rotation(rng.normal(0, 1e-3, 3)) @ Rp[p, w]
            tp[p, w] += rng.normal(0, 1e-2, 3)
    T = lambda x: torch.as_tensor(x).to(dev)                     # noqa: E731
    return T(fi), T(obs), T(pts), torch.full((P,), TRACKS, dtype=torch.int32, device=dev), T(Rp), T(tp)


def ba_times(P, kpd, X, R, t, K, dev):
    fi, obs, pts, cnt, Rp, tp = ba_inputs(P, X, R, t, dev, seed=P)
    res = {"windows": P, "W": W, "tracks": TRACKS, "N": W * KPTS}
    for refine in (0, 10):
        out, tm = timed(lambda: geometry.bundle_adjust_device(kpd, fi, obs, pts, cnt, Rp, tp, K, refine_iters=refine))
        tm["accepted_mean"] = float(out[4].to(torch.float64).mean())
        tm["rms_before_after_mean"] = [round(float(v), 4) for v in out[3].mean(0)]
        res[f"refine{refine}"] = tm
    return res


def step_times(P, kpd, X, R, t, K, dev):
    """Frames 0-3 carry exact maps and identity links; the step tracks frame 4 from frame 3."""
    s = np.arange(P) % SCENES
    fi = torch.as_tensor((W * s[:, None] + np.arange(W)[None]).astype(np.int32)).to(dev)
    maps = [torch.as_tensor(X[s, w].astype(np.float32)).to(dev) for w in range(W - 1)]
    ident = torch.arange(KPTS, dtype=torch.int32, device=dev).expand(P, KPTS).contiguous()
    links = [(ident, torch.zeros(P, KPTS, dtype=torch.bool, device=dev))] * (W - 2)
    Rw, tw = torch.as_tensor(R[s, :W - 1]).to(dev), torch.as_tensor(t[s, :W - 1]).to(dev)
    pairs, scores, counts, _ = synth.two_view_lists([KPTS] * P, KPTS, KPTS, inlier_frac=0.7, seed=11)
    pr, sc, cn = (torch.as_tensor(x).to(dev) for x in (pairs, scores, counts))
    pidx = fi[:, W - 2:W].contiguous()

    def step():
        Rr, tr_, _, _, _, nxt, lk, bn = geometry.track_and_map(maps[-1], kpd, kpd, pr, sc, cn, K, pidx, want_links=True)
        Rn = Rr @ Rw[:, -1]
        tn = (Rr @ tw[:, -1, :, None])[..., 0] + tr_
        Ra, ta = torch.cat([Rw, Rn[:, None]], 1), torch.cat([tw, tn[:, None]], 1)
        obs, pts, cnt, trk = geometry.window_tracks(torch.stack(maps + [nxt], 1),
                                                    torch.stack([x[0] for x in links] + [lk], 1),
                                                    torch.stack([x[1] for x in links] + [bn], 1), Ra, ta)
        Rb, tb, Xb, rms, acc, mask = geometry.bundle_adjust_device(kpd, fi, obs, pts, cnt, Ra, ta, K, want_mask=True)
        return Rb, tb, rms, acc, cnt, geometry.window_map(trk, Xb, Rb, tb, obs=obs, mask=mask)
    out, tm = timed(step)
    tm["windows"] = P
    tm["tracks_mean"] = float(out[4].to(torch.float64).mean())
    tm["accepted_mean"] = float(out[3].to(torch.float64).mean())
    tm["newest_map_points"] = int(torch.isfinite(out[5][:, -1]).all(-1).sum())
    return tm


def main():
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "warmup": WARMUP, "reps": REPS, "window": W, "keypoints": KPTS}
    kp, X, R, t, K = scenes()
    kpd = torch.as_tensor(kp).to(dev)
    res["ba_p1"] = ba_times(1, kpd, X, R, t, K, dev)
    res["ba_p599"] = ba_times(599, kpd, X, R, t, K, dev)
    res["step_p1"] = step_times(1, kpd, X, R, t, K, dev)
    res["step_p599"] = step_times(599, kpd, X, R, t, K, dev)
    out = os.environ.get("OUT")
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
