#!/usr/bin/env python
"""bench.py — frame-pairs/s for extract+match (BASELINE.json metric), on 1..8 B200.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path, workload c2
    python bench.py --workload c3|c4|c5 [...]                       # the other BASELINE.json configs
    python bench.py --scaling strong [...]                          # c2/c5: ONE sequence split over the ranks
    python bench.py --impl reference [...]                          # the reference's CPU path, host cores
    python bench.py --dump-outputs DIR [...]                        # also write the last timed step's outputs

Workloads (BASELINE.json configs[1..4], made concrete in SURVEY.md §8(d)); inputs are the tensors the
path sees after the backbone: saliency maps (T,H,W,1) fp32 and NHWC feature maps (T,H/16,W/16,384) fp32.
  c2  TUM-RGB-D-shaped sequence, 600 frames 640x480, K=2048, D=256, consecutive pairs, M1 (ratio 0.8),
      fp32 mode (f16x3 on tcgen05: fp32 in/out, 3-term fp16 hi/lo split).          [default, the metric]
  c3  64 independent pairs (frames 2p, 2p+1 of sequence p), K=4096, bf16 similarity, M1 0.8 (+ M3 0.9).
  c4  256 keyframes x K=2048, all 32 640 unordered pairs, M2; sharded by keyframe, descriptor banks
      all-gathered over NCCL, pair tiles dealt block-cyclically, lists gathered on rank 0.
  c5  1280x960 frames, K=8192, sequence of 600 frames, consecutive pairs, M1, fp32 mode.
One *step* is one pass over the workload: every frame is extracted once (decode -> sample -> refiner MLP
-> L2 norm) and every pair is matched.  --scaling weak (default): every rank runs its own sequence /
pair set; strong: the one sequence of c2/c5 is split with shard_frames (one halo frame per rank), c3
pairs are striped; c4 is always one keyframe set split over the ranks.

`value`   : pairs/s with inputs resident in HBM, CUDA events, max over ranks (CUDA-graph replay per step).
`e2e`     : the same step from pinned HOST buffers through the public pipeline entry points, H2D and D2H
            copies inside the timed region; `h2d_ceiling_gbs` is a bare pinned-copy probe of the same
            buffers (no kernels) run right before it on every rank at once.
`roofline`: the dominant kernel of the step: algorithmic flops or bytes / summed CUDA-event durations.
`parity`  : the oracle's match lists for the same inputs (all pairs of c2 at N=1, a bounded sample
            elsewhere) compared with the GPU's.
`cpu_baseline` / --impl reference: the reference's own functions (from baseline/_ref, kind "reference")
            or, when that tree is absent, the oracle port (kind "port"), in a process pool on all host cores.
`gpu_eager_baseline`: the same pipeline in stock PyTorch ops on the same B200 (bounded sample).
"""

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "semantic-slam-master_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

_REAL_STDOUT = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


METRIC = "frame-pairs/sec extract+match @640x480, 2048 kpts"
UNIT = "frame-pairs/s"
C, HID, D = 384, 384, 256

# name -> (H, W, K, frames, similarity mode, matcher, description)
WORKLOADS = {
    "c2": dict(H=480, W=640, K=2048, frames=600, mode="f16x3", kind="sequence",
               text="c2: TUM RGB-D-shaped synthetic sequence, {frames} frames 640x480, consecutive-pair matching "
                    "(M1 ratio 0.8), {K} kpts x 256-D, refiner MLP 384-384-384-256, fp32 mode"),
    "c3": dict(H=480, W=640, K=4096, frames=128, mode="bf16", kind="pairs",
               text="c3: {pairs} independent synthetic frame pairs 640x480, {K} kpts x 256-D, bf16 similarity, "
                    "ratio test 0.8 (M1)"),
    "c4": dict(H=480, W=640, K=2048, frames=256, mode="f16x3", kind="allpairs",
               text="c4: loop-closure style all-pairs matching, {frames} keyframes x {K} kpts x 256-D ({pairs} pairs, "
                    "M2), keyframes sharded, NCCL all-gather of descriptor banks + gather of match lists"),
    "c5": dict(H=960, W=1280, K=8192, frames=600, mode="f16x3", kind="sequence",
               text="c5: high-res 1280x960 synthetic sequence, {frames} frames, consecutive-pair matching (M1 ratio 0.8), "
                    "{K} kpts x 256-D, fp32 mode"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--frames", type=int, default=0, help="override the workload's frame / keyframe count")
    ap.add_argument("--kpts", type=int, default=0, help="override the workload's keypoints per frame")
    ap.add_argument("--mode", default="auto", choices=["auto", "f32", "tf32x3", "f16x3", "bf16"])
    ap.add_argument("--chunk", type=int, default=0, help="frames per extraction launch group (0 = workload default)")
    ap.add_argument("--e2e-chunk", type=int, default=50, help="frames per host->device staging buffer (e2e arm)")
    ap.add_argument("--cpu-sample-frames", type=int, default=0, help="frames per CPU-arm step (0 = sized to a time budget)")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="time budget of the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs); with "
                         "several ranks: rank 0's frames and the match lists of all ranks gathered on rank 0")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    w = WORKLOADS[a.workload]
    a.H, a.W, a.kind = w["H"], w["W"], w["kind"]
    a.frames = a.frames or w["frames"]
    a.kpts = a.kpts or w["K"]
    a.mode_name = w["mode"] if a.mode == "auto" else a.mode
    if a.mode == "auto" and os.environ.get("SSLAM_BENCH_MODE"):
        a.mode_name = os.environ["SSLAM_BENCH_MODE"]
    if not a.chunk:
        a.chunk = 300 if a.workload != "c5" else 75          # ~10 GB of intermediates per launch group
    return a


def total_pairs(a):
    if a.kind == "sequence":
        return a.frames - 1
    if a.kind == "pairs":
        return a.frames // 2
    return a.frames * (a.frames - 1) // 2


def workload_config(a):
    """The `config` object — identical for the b200 and the reference arm (same workload, same keys)."""
    pairs = total_pairs(a)
    return {"workload": WORKLOADS[a.workload]["text"].format(frames=a.frames, K=a.kpts, pairs=pairs),
            "name": a.workload, "frames": a.frames, "kpts": a.kpts, "pairs": pairs,
            "height": a.H, "width": a.W, "descriptor_dim": D, "scaling": a.scaling, "n_gpus": a.gpus}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, \
        "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, rows):
    """dram bytes per launch of `kernel` from the newest committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by profiles/summarize_ncu.py), scaled to this run's rows per
    launch; None when no capture of this kernel is on file."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            rec = json.load(f).get(kernel)
        return rec["dram_bytes_per_row"] * rows if rec else None
    except Exception:
        return None


# --------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons every 10 ms while the timed region runs (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz, self.ok = None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                                            # pragma: no cover
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:                                             # pragma: no cover
                pass
            time.sleep(0.01)

    def summary(self):
        if not self.ok or not self.samples:
            return smi_clocks(self.index)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def smi_clocks(index):
    """Fallback when NVML sampling failed: one nvidia-smi query right after the timed region."""
    import subprocess
    try:
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=20).stdout.strip().split(",")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for n, v in zip(names, out[2:]) if v.strip().lower() == "active"]
        return {"sm_mhz": int(out[0]), "sm_max_mhz": int(out[1]), "reasons": reasons,
                "note": "NVML sampling unavailable; single nvidia-smi sample after the timed region"}
    except Exception as e:                                                # pragma: no cover
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": f"no clock source: {e!r}"}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# --------------------------------------------------------------------------------------- inputs
def frame_plan(a, rank, world):
    """Which frames this rank extracts and which pairs it matches.
    Returns dict(seq, frames=[(seq_id, frame t)], pair_index (local frame indices) or None = consecutive,
    npairs_local, npairs_global)."""
    from sslam_b200 import dist as sdist
    T = a.frames
    if a.kind == "sequence":
        if a.scaling == "strong" and world > 1:
            s, e, n = sdist.shard_frames(T, world, rank)
            return dict(frames=[(0, t) for t in range(s, e)], pair_index=None, npairs_local=n, npairs_global=T - 1,
                        pad_pairs=-(-(T - 1) // world))
        return dict(frames=[(rank, t) for t in range(T)], pair_index=None, npairs_local=T - 1,
                    npairs_global=(T - 1) * world, pad_pairs=T - 1)
    if a.kind == "pairs":
        P = T // 2
        mine = list(range(rank, P, world)) if (a.scaling == "strong" and world > 1) else list(range(P))
        seq_off = 0 if (a.scaling == "strong" or world == 1) else rank * P
        frames, idx = [], []
        for k, p in enumerate(mine):                       # frames (2p, 2p+1) of sequence p (SURVEY §8(d))
            frames += [(seq_off + p, 2 * p), (seq_off + p, 2 * p + 1)]
            idx.append((2 * k, 2 * k + 1))
        glob = P if (a.scaling == "strong" or world == 1) else P * world
        return dict(frames=frames, pair_index=idx, npairs_local=len(mine), npairs_global=glob,
                    pad_pairs=-(-P // world) if a.scaling == "strong" else P)
    # all pairs: keyframes = frames 0, 8, 16, ... of sequence 0, contiguous blocks per rank
    per = T // world
    return dict(frames=[(0, 8 * k) for k in range(rank * per, (rank + 1) * per)], pair_index="allpairs",
                npairs_local=None, npairs_global=T * (T - 1) // 2, pad_pairs=None)


def make_inputs(a, plan, pinned=True):
    """Seeded synthetic frames on the HOST (torch CPU generators: identical to what the oracle / the
    reference arm generates), in pinned buffers that also serve the e2e arm."""
    import torch
    from sslam_b200 import synth
    n = len(plan["frames"])
    sal = torch.empty((n, a.H, a.W, 1), dtype=torch.float32, pin_memory=pinned)
    feat = torch.empty((n, a.H // 16, a.W // 16, C), dtype=torch.float32, pin_memory=pinned)
    canvases = {}
    for i, (seq, t) in enumerate(plan["frames"]):
        cv = canvases.get(seq)
        if cv is None:
            if len(canvases) > 2:
                canvases.clear()
            cv = canvases[seq] = synth.WorldCanvas(seq, a.H, a.W, C, "cpu")
        lg, ft = cv.frame(t)
        sal[i, :, :, 0].copy_(torch.sigmoid(lg))
        feat[i].copy_(ft)
    return sal, feat


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, per_frame, per_pair, descriptors):
    """--dump-outputs: the outputs of the last timed step as <path>/<name>.npy, all float32 (the integer
    outputs are exact there: |value| < 2**24).  Inputs and weights are seeded, so two builds run with the
    same arguments can be compared file for file.

    per_frame / per_pair: name -> tensor whose first axis runs over the frames / the pairs;
    descriptors: (frames, K, D).  The files stay under DUMP_BYTES in all.  The per-pair arrays, then the
    per-frame arrays, are kept whole when they fit an equal share of what is left; otherwise every array
    of that group keeps the same fixed, seeded sample of its rows, whose indices go to pair_rows.npy /
    frame_rows.npy (float64).  The descriptors fill the rest: a seeded sample of the (frame, keypoint)
    rows of the kept frames, written as descriptors.npy (n, D) with descriptor_rows.npy holding
    frame * K + keypoint."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES - 256 * (2 * (len(per_frame) + len(per_pair)) + 4)     # room for the .npy headers

    def sample(n, keep):
        return np.sort(np.random.Generator(np.random.PCG64(0)).choice(n, keep, replace=False))

    def save(name, arr):
        np.save(os.path.join(path, name + ".npy"), arr)
        return arr.nbytes

    def put(group, arrays, share):
        rows = next(iter(arrays.values())).shape[0]
        row_bytes = sum(4 * t.numel() // max(rows, 1) for t in arrays.values())
        idx, used = np.arange(rows), 0
        if rows * row_bytes > share:
            idx = sample(rows, min(rows, share // (row_bytes + 8)))
            used += save(group + "_rows", idx.astype(np.float64))
        sel = torch.from_numpy(idx)
        for name, t in arrays.items():
            used += save(name, t.index_select(0, sel.to(t.device)).float().cpu().numpy())
        return idx, used

    _, used = put("pair", per_pair, left // 3)
    left -= used
    frames, used = put("frame", per_frame, left // 2)
    left -= used
    F, K, D = descriptors.shape
    cand = (frames[:, None] * K + np.arange(K)[None, :]).ravel()
    rows = cand[sample(cand.size, min(cand.size, left // (4 * D + 8)))]
    save("descriptor_rows", rows.astype(np.float64))
    flat = descriptors.reshape(F * K, D)
    save("descriptors", flat.index_select(0, torch.from_numpy(rows).to(flat.device)).float().cpu().numpy())


def refiner_module(dev=None):
    import torch
    from models.descriptor_refiner import DescriptorRefiner
    torch.manual_seed(0)
    m = DescriptorRefiner(C, HID, D, 4)
    return m.to(dev) if dev is not None else m


# --------------------------------------------------------------------------------------- CPU arm
def cpu_arm_kind():
    from oracle import ref_pipeline
    return "reference" if ref_pipeline.available() else "port"


def cpu_pipeline(a, frames, workers):
    """The CPU arm on the first `frames` frames of the c2-style sequence 0 (or pairs of c3 / keyframes):
    returns (pairs/s, seconds, [(count, crc32)] per consecutive pair, kind)."""
    import numpy as np
    import torch
    from oracle import pipeline as opipe, ref_pipeline
    import oracle
    plan = dict(frames=[(0, t) for t in range(frames)])
    sal, feat = make_inputs(a, plan, pinned=False)
    refiner = refiner_module()
    if ref_pipeline.available():
        sd = {k: v.detach().numpy() for k, v in refiner.state_dict().items()}
        rec, sec = ref_pipeline.run_sequence(sal.numpy()[..., 0], feat.numpy(), sd, (C, HID, D, 4), a.kpts, workers)
        kind = "reference"
    else:
        weights = oracle.RefinerWeights.from_state_dict(refiner.state_dict())
        rec, sec = opipe.run_sequence(sal.numpy()[..., 0], feat.numpy(), weights, a.kpts, 1, workers)
        kind = "port"
    del np, torch
    return (frames - 1) / sec, sec, rec, kind


def cpu_sample_text(kind, frames, workers, sec=None):
    what = ("the reference's own select_keypoints / pixel_to_patch / extract_at_keypoints / DescriptorRefiner / "
            "find_matches (baseline/_ref)" if kind == "reference" else "oracle port (NumPy)")
    t = f"{frames} frames / {frames - 1} consecutive pairs of sequence 0 of the workload per step, {what}, " \
        f"{workers}-process pool over frames then pairs"
    return t + (f", {sec:.1f} s" if sec is not None else "")


def run_reference(a):
    """--impl reference: the reference's CPU implementation of the path on every host core."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pipeline as opipe
    cores = opipe.host_cores()
    frames = a.cpu_sample_frames
    if frames <= 0:
        # size the per-step sample so that the whole run (warm-ups + steps) fits the time budget
        probe = 33 if a.kpts <= 4096 and a.H <= 480 else 9
        _, sec, _, _ = cpu_pipeline(a, probe, cores)
        per_frame = sec / probe
        frames = int(a.cpu_budget_s / max(1, a.warmup + a.steps) / per_frame)
        frames = max(17, min(frames, a.frames + 1))
    vals, kind = [], None
    for i in range(a.warmup + a.steps):
        v, sec, _, kind = cpu_pipeline(a, frames, cores)
        if i >= a.warmup:
            vals.append((v, sec))
    value = sum(v for v, _ in vals) / len(vals)
    ms = 1e3 * sum(s for _, s in vals) / len(vals)
    sample = cpu_sample_text(kind, frames, cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": a.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------------------- stock-torch GPU baseline
def gpu_eager_baseline(a, sal, feat, refiner, frames=16):
    """The same pipeline in stock PyTorch ops on the same GPU (quantile / max_pool2d / topk /
    grid_sample / linear + layer_norm (cuBLAS fp32) / normalize / mm / argmax), main decode branch,
    consecutive pairs of the first `frames` frames; CUDA events.  Returns pairs/s."""
    import torch
    import torch.nn.functional as F
    K = a.kpts
    T = min(frames, sal.shape[0])
    if T < 2:
        return None

    def extract(s, f):
        s2 = s[:, :, 0]
        thr = max(torch.quantile(s2.flatten(), 0.5).item(), 0.1)
        pooled = F.max_pool2d(s2[None, None], 5, 1, 2)[0, 0]
        nms = s2 * (s2 == pooled).float()
        cand = torch.where(nms > thr, nms, torch.zeros_like(nms)).flatten()
        sc, idx = torch.topk(cand, K)
        xy = torch.stack([(idx % a.W).float(), (idx // a.W).float()], -1)
        pc = (xy - 8.0) / 16.0
        h, w = f.shape[0], f.shape[1]
        g = torch.stack([2 * pc[:, 0] / (w - 1) - 1, 2 * pc[:, 1] / (h - 1) - 1], -1)[None, None]
        samp = F.grid_sample(f.permute(2, 0, 1)[None], g, mode="bilinear", align_corners=True)[0, :, 0].t()
        return F.normalize(refiner.forward_unnormalized(samp[None]), p=2, dim=-1), sc

    def match(d1, d2):
        S = d1 @ d2.t()
        best, nn12 = S.max(1)
        nn21 = S.argmax(0)
        second = S.scatter(1, nn12[:, None], -1.0).max(1).values
        ok = (nn21[nn12] == torch.arange(S.shape[0], device=S.device)) & (best > second * 0.8)
        return torch.nonzero(ok).squeeze(1), nn12

    with torch.no_grad():
        for rep in range(2):                                   # first pass = warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            prev = None
            for t in range(T):
                d, _ = extract(sal[t], feat[t])
                if prev is not None:
                    match(prev, d)
                prev = d
            e1.record()
            torch.cuda.synchronize()
    return (T - 1) / (e0.elapsed_time(e1) * 1e-3)


# --------------------------------------------------------------------------------------- GPU arm
def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sslam_b200 import dist as sdist
    from sslam_b200 import matchers, ops
    from sslam_b200.pipeline import FrontEnd

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    mode = {"f32": ops.SIM_F32, "tf32x3": ops.SIM_TF32X3, "bf16": ops.SIM_BF16, "f16x3": ops.SIM_F16X3}[a.mode_name]
    variant = matchers.M2 if a.kind == "allpairs" else matchers.M1
    mkw = {} if a.kind == "allpairs" else {"ratio_thresh": 0.8}

    refiner = refiner_module(dev)
    fe = FrontEnd(refiner, num_keypoints=a.kpts, grid="pixel", sim_mode=mode)
    plan = frame_plan(a, rank, world)
    sal_h, feat_h = make_inputs(a, plan)
    sal, feat = sal_h.to(dev), feat_h.to(dev)
    Tl = sal.shape[0]
    in_bytes = sal.numel() * 4 + feat.numel() * 4
    K = a.kpts

    # ---- the device-resident step
    coll_ms = {"all_gather": [], "gather_lists": []}
    if a.kind == "sequence":
        run = lambda timers=None: fe.run_sequence(sal, feat, variant, chunk=a.chunk, timers=timers, **mkw)  # noqa: E731
        pidx_local = None
    elif a.kind == "pairs":
        pidx_local = torch.tensor(plan["pair_index"], dtype=torch.int32, device=dev).reshape(-1, 2)
        run = lambda timers=None: fe.run_pairs(sal, feat, pidx_local, variant, chunk=a.chunk, timers=timers, **mkw)  # noqa: E731
    else:
        all_idx = sdist.all_pairs_index(a.frames)
        mine = sdist.deal_pairs_block_cyclic(all_idx, world, rank, block=16)
        pidx_local = all_idx[mine].to(dev)
        pad = -(-all_idx.shape[0] // world) + 16 * 16 * 2        # dealt tiles differ by up to two tiles

        def run(timers=None):
            f = fe.extract(sal, feat, timers=timers)
            hi, lo, sc = f["descriptors_hi"], f["descriptors_lo"], f["scores"]
            if world > 1:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                ev[0].record()
                hi, lo, sc = sdist.all_gather_bank(hi), sdist.all_gather_bank(lo), sdist.all_gather_bank(sc)
                ev[1].record()
                coll_ms["all_gather"].append(ev)
            fe._mark(timers, "begin")
            pairs, pscores, counts, _ = matchers.match((hi, lo), (hi, lo), variant, pair_index=pidx_local,
                                                       mode=mode, scores1=sc, scores2=sc, **mkw)
            fe._mark(timers, "match")
            return f, pairs, pscores, counts

    replay = None
    use_graph = not a.no_graph and not (a.kind == "allpairs" and world > 1)      # NCCL stays outside graphs
    if use_graph:
        replay, (g_feats, g_pairs, g_pscores, g_counts) = fe.capture(run)

    npl = plan["npairs_local"] if plan["npairs_local"] is not None else int(pidx_local.shape[0])
    pad_pairs = plan["pad_pairs"] if plan["pad_pairs"] is not None else pad
    padded = None
    if world > 1 and pad_pairs != npl:
        padded = (torch.full((pad_pairs, K, 2), -1, dtype=torch.int32, device=dev),
                  torch.zeros((pad_pairs, K), device=dev), torch.zeros((pad_pairs,), dtype=torch.int32, device=dev))

    last_feats = [None]                                      # the bank the latest step wrote

    def step(timers=None, eager=False):
        if replay is not None and not eager:
            replay()
            last_feats[0], pairs, pscores, counts = g_feats, g_pairs, g_pscores, g_counts
        else:
            last_feats[0], pairs, pscores, counts = run(timers)
        gathered = None
        if world > 1:
            if padded is not None:                           # ranks own different numbers of pairs
                for dst, src in zip(padded, (pairs, pscores, counts)):
                    dst[:npl].copy_(src)
                pairs, pscores, counts = padded
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            gathered = sdist.gather_match_lists(pairs, pscores, counts, dst=0)
            ev[1].record()
            coll_ms["gather_lists"].append(ev)
        return pairs, pscores, counts, gathered

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        step()
    fence()
    coll_ms = {k: [] for k in coll_ms}
    sampler = ClockSampler(physical_gpu_index(local))
    sampler.start()
    c0 = ops.launch_count()
    step(eager=True)
    fence()
    launches_per_step = ops.launch_count() - c0              # graph replays bypass the library's counter
    coll_ms = {k: [] for k in coll_ms}
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()          # `ncu --profile-from-start off` sees only the timed steps
    t_beg.record()
    for _ in range(a.steps):
        out = step()
    t_end.record()
    fence()
    torch.cuda.profiler.stop()
    sampler.stop_flag = True
    ms_total = t_beg.elapsed_time(t_end)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / a.steps
    pairs_per_step = plan["npairs_global"]
    value = pairs_per_step / (ms_step * 1e-3)
    coll = {k: (sum(e0.elapsed_time(e1) for e0, e1 in v) / max(len(v), 1) if v else None) for k, v in coll_ms.items()}
    final_pairs, final_scores, final_counts = (t.clone() for t in out[:3])
    if a.dump_outputs and rank == 0:
        # rank 0's frames; with several ranks, the match lists of all ranks as gathered on rank 0
        f = last_feats[0]
        lists = out[3] if world > 1 else (final_pairs, final_scores, final_counts)
        dump_outputs(a.dump_outputs, {"keypoints": f["keypoints_pixel"], "scores": f["scores"]},
                     dict(zip(("pairs", "pair_scores", "counts"), lists)), f["descriptors"])

    # ---- instrumented pass: CUDA events around every kernel launch of the library (per-kernel rooflines)
    ops.profile_enable(True)
    for _ in range(a.steps):
        step(eager=True)
    fence()
    kernel_ms = ops.profile_read()
    ops.profile_enable(False)

    # ---- per-stage device time from event marks (eager launches)
    stage_ms, timer_lists = {}, []
    for _ in range(a.steps):
        tl = []
        step(tl, eager=True)
        timer_lists.append(tl)
    fence()
    for tl in timer_lists:
        for (n0, e0), (n1, e1) in zip(tl[:-1], tl[1:]):
            if n1 != "begin":
                stage_ms[n1] = stage_ms.get(n1, 0.0) + e0.elapsed_time(e1)
    stage_ms = {k: v / a.steps for k, v in stage_ms.items()}

    # ---- e2e: pinned host buffers -> match lists on the host, through the public entry points
    e2e = None
    if not a.no_e2e:
        # bare pinned-copy probe: the same chunks, no kernels, all ranks at once = the H2D ceiling
        stage = [torch.empty((a.e2e_chunk,) + tuple(sal_h.shape[1:]), device=dev),
                 torch.empty((a.e2e_chunk,) + tuple(feat_h.shape[1:]), device=dev)]

        def probe():
            for s in range(0, Tl, a.e2e_chunk):
                e = min(Tl, s + a.e2e_chunk)
                stage[0][:e - s].copy_(sal_h[s:e], non_blocking=True)
                stage[1][:e - s].copy_(feat_h[s:e], non_blocking=True)
        probe()
        fence()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(3):
            probe()
        p1.record()
        fence()
        probe_ms = p0.elapsed_time(p1) / 3
        if world > 1:
            t = torch.tensor([probe_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            probe_ms = float(t.item())
        del stage

        if a.kind == "sequence":
            host_fn = lambda oh: fe.run_sequence_host(sal_h, feat_h, variant, chunk=a.e2e_chunk, out_host=oh, **mkw)  # noqa: E731
        elif a.kind == "pairs":
            host_fn = lambda oh: fe.run_pairs_host(sal_h, feat_h, pidx_local, variant, chunk=a.e2e_chunk, out_host=oh, **mkw)  # noqa: E731
        else:
            def host_fn(oh):                                  # H2D of the keyframes, device step, D2H of the lists
                sal.copy_(sal_h, non_blocking=True)
                feat.copy_(feat_h, non_blocking=True)
                pr, ps, cn, _ = step(eager=True)
                if oh is None:
                    oh = tuple(torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (pr, ps, cn))
                for d_, s_ in zip(oh, (pr, ps, cn)):
                    d_.copy_(s_, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                return oh
        out_h = None
        for _ in range(max(1, min(2, a.warmup))):
            out_h = host_fn(out_h)
        fence()
        w0 = time.perf_counter()
        e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e_beg.record()
        for _ in range(a.steps):
            out_h = host_fn(out_h)
            if world > 1 and a.kind != "allpairs":
                # the lists of every rank are on its own host; the NCCL gather of the device arm is not part
                # of the host-to-host path
                pass
        e_end.record()
        fence()
        wall_ms = (time.perf_counter() - w0) * 1e3
        e_ms = max(e_beg.elapsed_time(e_end), wall_ms)       # host-blocking D2H: wall clock bounds it
        if world > 1:
            t = torch.tensor([e_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_ms = float(t.item())
        d2h = sum(t.numel() * t.element_size() for t in out_h)
        e_step = e_ms / a.steps
        e2e = {"value": pairs_per_step / (e_step * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(in_bytes), "d2h_bytes_per_step": int(d2h), "ms_per_step": e_step,
               "h2d_ceiling_gbs": in_bytes / (probe_ms * 1e-3) / 1e9,
               "h2d_probe_ms": probe_ms, "frac_of_h2d_ceiling": probe_ms / e_step,
               "note": "per rank; h2d_ceiling_gbs = bare pinned copies of the same staging chunks, no kernels, "
                       "every rank at once; frac_of_h2d_ceiling = probe time / e2e step time"}

    # ---- parity against the CPU arm on identical inputs
    parity, cpu = None, None
    if rank == 0:
        gp = final_pairs.cpu().numpy()
        gc = final_counts.cpu().numpy()
        from oracle import pipeline as opipe
        gkp = last_feats[0]["keypoints_pixel"].cpu().numpy()      # (no collective may run on rank 0 alone)

        def gpu_record(p):                                    # consecutive pair p = frames (p, p + 1)
            return opipe.pair_record(gp[p, :int(gc[p])], gkp[p], gkp[p + 1])
        cores = opipe.host_cores()
        if a.kind == "sequence" and not a.no_cpu_baseline and (world == 1 or a.scaling == "strong"):
            # rank 0 holds the first frames of sequence 0 in both scaling modes
            frames = a.cpu_sample_frames or (min(a.frames, Tl) if a.workload == "c2" else 9)
            frames = min(frames, Tl)
            v, sec, rec, kind = cpu_pipeline(a, frames, cores)
            same_n = sum(1 for p, r in enumerate(rec) if gpu_record(p)[0] == r[0])
            same_l = sum(1 for p, r in enumerate(rec) if gpu_record(p) == tuple(r))
            parity = {"pairs": len(rec), "identical_counts": same_n, "identical_lists": same_l,
                      "max_count_delta": max(abs(gpu_record(p)[0] - r[0]) for p, r in enumerate(rec)),
                      "against": kind, "note": "match lists compared by count and by CRC32 of the sorted (x1,y1,x2,y2) keypoint rows (independent "
                                               "of torch.topk's unspecified order of equal scores); lists may differ only by similarity "
                                               "near ties (tests/: margins < 2*(eps+2e-6))"}
            if world == 1:
                cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                       "sample": cpu_sample_text(kind, frames, cores, sec)}
        elif not a.no_cpu_baseline and world == 1:
            # pairs / all-pairs: the oracle on a bounded sample of the same frames
            import oracle
            nfr = 4 if a.kind == "pairs" else 5
            w = oracle.RefinerWeights.from_state_dict(refiner.state_dict())
            t0 = time.perf_counter()
            okp, osc, _ = oracle.select_keypoints(sal_h[:nfr].numpy(), K)
            od = oracle.refiner_forward(w, oracle.extract_at_keypoints(feat_h[:nfr].numpy(), oracle.pixel_to_patch(okp)))
            if a.kind == "pairs":
                plist = [(2 * p, 2 * p + 1, p) for p in range(nfr // 2)]
            else:
                lut = {tuple(r): i for i, r in enumerate(pidx_local.cpu().tolist())}
                plist = [(i, j, lut[(i, j)]) for i in range(nfr) for j in range(i + 1, nfr)]
            agree, refn = 0, 0
            for (i, j, p) in plist:
                if a.kind == "pairs":
                    ref = {(x, y) for x, y, _ in oracle.match_m1(od[i], od[j], 0.8)}
                else:
                    ref = {tuple(r) for r in oracle.match_m2(od[i], od[j], osc[i], osc[j])[0].tolist()}
                got = {tuple(r) for r in gp[p, :int(gc[p])].tolist()}
                agree += len(ref & got)
                refn += len(ref | got)
            sec = time.perf_counter() - t0
            parity = {"pairs": len(plist), "index_agreement": agree / max(refn, 1), "against": "port",
                      "note": "oracle end to end on its own descriptors for the first frames; "
                              + ("bf16 similarity: agreement is a percentage by design" if a.mode_name == "bf16" else
                                 "fp32 mode")}
            cpu = {"value": len(plist) / sec, "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": f"{nfr} frames / {len(plist)} pairs of the same workload, oracle port (NumPy), single process, {sec:.1f} s"}

    eager = None
    if rank == 0 and not a.no_eager_baseline:
        try:
            v = gpu_eager_baseline(a, sal, feat, refiner)
            eager = {"value": v, "unit": UNIT, "kind": "torch_eager_restatement",
                     "sample": "first 16 frames / 15 consecutive pairs, stock PyTorch ops on the same B200 "
                               "(quantile, max_pool2d, topk, grid_sample, cuBLAS fp32 linear + layer_norm, mm, argmax), "
                               "per-frame launches as the reference issues them"}
        except Exception as e:                               # pragma: no cover
            eager = {"value": None, "error": repr(e)[:200]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = measured_peaks()
    peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    hbm = float(peaks["hbm_gbs"])
    rows = Tl * K
    blocks = 2
    mm_flops = 2.0 * K * K * D * npl
    work = {   # algorithmic work per step on this rank (SURVEY.md §8(d), DESIGN.md §4)
        "gemm_f16x3": ("tensor", 2.0 * rows * (C * HID + blocks * 2 * HID * HID + HID * D)),
        "match_tc": ("tensor", mm_flops), "match_f32": ("tensor", mm_flops),
        "decode_scan": ("hbm", (4.0 * a.H * a.W + 12 * K) * Tl),
        "gather": ("hbm", (4.0 * (a.H // 16) * (a.W // 16) * C + 8 * K + 4 * K * C) * Tl),
        # fp32 in, fp32 out, plus the operand copy the matcher reads (fp16 hi/lo pair: 4 B, bf16: 2 B) — written
        # here instead of by a split pass in front of the matcher
        "l2norm": ("hbm", (8.0 + {"f16x3": 4.0, "bf16": 2.0}.get(a.mode_name, 0.0)) * K * D * Tl),
    }
    kernels = {}
    for kind, (ms_tot, n) in kernel_ms.items():
        e = {"ms_per_step": ms_tot / a.steps, "launches_per_step": n / a.steps}
        if kind in work and e["ms_per_step"] > 0:
            bound, w = work[kind]
            if bound == "tensor":
                e["algorithmic_TFLOP/s"] = w / (e["ms_per_step"] * 1e-3) / 1e12
                e["frac_of_bf16_peak"] = e["algorithmic_TFLOP/s"] / peak
            else:
                e["algorithmic_GB/s"] = w / (e["ms_per_step"] * 1e-3) / 1e9
                e["frac_of_hbm_peak"] = e["algorithmic_GB/s"] / hbm
        kernels[kind] = e
    dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
    dk = kernels[dom]
    split_note = ("fp32 accuracy costs three 16-bit MMAs per product (fp16 hi/lo split), so the ceiling of "
                  "this fraction is 1/3 = 0.333 (1/6 for the tf32x3 variant)")
    if work.get(dom, ("", 0))[0] == "tensor":
        ach = dk["algorithmic_TFLOP/s"]
        traffic = ncu_traffic(dom, rows / max(dk["launches_per_step"], 1e-9)) if dom == "gemm_f16x3" else None
        roofline = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                    "frac": ach / peak, "traffic": traffic,
                    "peak_source": peak_src + ", bf16 dense sustained",
                    "launch_ms": dk["ms_per_step"] / dk["launches_per_step"],
                    "launches_per_step": dk["launches_per_step"],
                    "algorithmic_flops_per_step": work[dom][1],
                    "note": ("achieved = algorithmic flops of all launches of this kernel in a step / their "
                             "summed CUDA-event durations (instrumented pass of the same steps); traffic = dram bytes per "
                             "launch from profiles/ncu_traffic.json (null when no capture of this kernel is on file); "
                             + (split_note if (a.mode_name != "bf16" or dom == "gemm_f16x3") else ""))}
    else:
        ach = dk.get("algorithmic_GB/s", float("nan"))
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": hbm, "unit": "GB/s",
                    "frac": ach / hbm, "traffic": None, "peak_source": peak_src,
                    "launch_ms": dk["ms_per_step"] / dk["launches_per_step"]}
    stages = {k: {"ms_per_step": v} for k, v in stage_ms.items()}

    cfg = workload_config(a)
    line = {"metric": METRIC if a.workload == "c2" else f"frame-pairs/sec extract+match, workload {a.workload}",
            "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": a.scaling,
            "vs_baseline": None,
            "dtype": {"f32": "f32", "tf32x3": "tf32x3 (fp32 in/out)", "f16x3": "f16x3 (fp32 in/out)", "bf16": "bf16"}[a.mode_name],
            "data": "synthetic", "config": cfg,
            "run": {"frames_per_rank": Tl, "pairs_per_step": pairs_per_step, "pairs_this_rank": npl,
                    "similarity_mode": a.mode_name, "chunk": a.chunk, "e2e_chunk": a.e2e_chunk,
                    "launch": "CUDA graph replay (one graph per step)" if replay is not None else "eager",
                    "l2_policy": f"inputs larger than L2 ({in_bytes / 1e6:.0f} MB per step per GPU)",
                    "parallelism": (f"{world} ranks, {a.scaling} scaling, one packed NCCL gather of match records"
                                    + (", NCCL all-gather of descriptor banks" if a.kind == "allpairs" else ""))
                    if world > 1 else "single GPU",
                    "collective_ms_per_step": coll},
            "roofline": roofline, "kernels": kernels, "stages": stages, "parity": parity, "cpu_baseline": cpu,
            "gpu_eager_baseline": eager, "e2e": e2e,
            "gpu_launches": int(launches_per_step * a.steps), "clocks": sampler.summary()}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner) are
    # sent to stderr, and the line is written to the saved descriptor at the end.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
