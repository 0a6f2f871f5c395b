"""HBM-resident frame store and the sequence / tracking drivers on top of it (SURVEY.md §8(f) N3).

The reference's drivers re-extract frames and move every result to the host:
``process_spacing`` extracts BOTH frames of every pair (visualize_matches_sequence.py:306-307, for
spacings 1, 5, 10, 15, 20 at :369) and ``TrackingTester.track_frame_sequence`` ends every frame in
``.cpu().numpy()`` before a NumPy matmul (test/test_tracking.py:151-177).  Here every frame is
extracted exactly once into a ring buffer of slots in HBM — keypoints, scores, fp32 descriptors and
the fp16 (hi, lo) operand pair of the tcgen05 matcher — and all matching runs from the resident
slots through ``pair_index`` (slot ids), so nothing leaves the device until the caller asks.

``FrameStore``          ring buffer of ``capacity`` slots; ``push`` extracts a batch of frames into it.
``match_spacings``      frame t against frame t - s for several spacings s at once (one matcher call).
``verify_pairs``        RANSAC homography or fundamental matrix over lists those calls returned, from the
                        resident keypoints.
``TrackingCounters``    the counters of track_frame_sequence (:166-199) accumulated on the device.
"""

import torch

from . import geometry, matchers, ops
from .ops import SIM_BF16, SIM_F16X3


class FrameStore:
    def __init__(self, frontend, capacity):
        """frontend: a pipeline.FrontEnd (decode / sample / refine configuration); capacity: slots."""
        self.fe, self.capacity = frontend, int(capacity)
        self.bank = None
        self.next_frame = 0                        # id of the next frame to be pushed
        self._span = None

    # ---- storage
    def _ensure(self, device):
        if self.bank is None:
            self.bank = self.fe._alloc_bank(self.capacity, device)
            self.frame_of_slot = torch.full((self.capacity,), -1, dtype=torch.int64, device=device)

    def slot_of(self, frame):
        return frame % self.capacity

    def oldest(self):
        return max(0, self.next_frame - self.capacity)

    def holds(self, frame):
        return self.oldest() <= frame < self.next_frame

    @torch.no_grad()
    def push(self, saliency, features):
        """Extract B consecutive frames (B <= capacity) into the ring.  Returns their frame ids
        (range).  A batch that wraps around the end of the ring is written as two slices."""
        B = saliency.shape[0]
        if B > self.capacity:
            raise ValueError("batch larger than the frame store")
        self._ensure(saliency.device)
        first = self.next_frame
        done = 0
        while done < B:
            s = self.slot_of(first + done)
            n = min(B - done, self.capacity - s)
            self.fe.extract(saliency[done:done + n], features[done:done + n],
                            out=self.fe._bank_slice(self.bank, s, s + n))
            self.frame_of_slot[s:s + n] = torch.arange(first + done, first + done + n,
                                                       device=self.frame_of_slot.device)
            done += n
        self.next_frame = first + B
        return range(first, first + B)

    def frame(self, frame):
        """Views of one resident frame: keypoints_pixel (K,2), scores (K,), descriptors (K,D)."""
        if not self.holds(frame):
            raise KeyError(f"frame {frame} is no longer resident (oldest: {self.oldest()})")
        s = self.slot_of(frame)
        kp = self.bank["keypoints"][s]
        if self.fe.grid != "pixel":
            kp = kp * self.fe.patch + self.fe.patch / 2
        return {"keypoints_pixel": kp, "scores": self.bank["scores"][s], "descriptors": self.bank["descriptors"][s]}

    # ---- matching from resident slots
    def pair_index(self, frame_pairs):
        """[(a, b), ...] frame ids -> (P,2) int32 slot ids on the device; all must be resident."""
        for a, b in frame_pairs:
            if not (self.holds(a) and self.holds(b)):
                raise KeyError(f"pair ({a},{b}) touches a frame that is not resident")
        idx = torch.tensor([[self.slot_of(a), self.slot_of(b)] for a, b in frame_pairs], dtype=torch.int32)
        return idx.reshape(-1, 2).to(self.bank["scores"].device)

    @torch.no_grad()
    def match_pairs(self, frame_pairs, variant=matchers.M2, **kw):
        """Match listed (a, b) frame pairs from the ring.  Returns padded (pairs, scores, counts)."""
        idx = self.pair_index(frame_pairs)
        bank = self.fe.bank(self.bank)
        sc = self.bank["scores"]
        return matchers.match(bank, bank, variant, pair_index=idx, mode=self.fe.sim_mode, scores1=sc, scores2=sc,
                              **kw)[:3]

    def spacing_pairs(self, frames, spacings=(1, 5, 10, 15, 20)):
        """(t - s, t) for every new frame t and spacing s whose earlier frame is resident."""
        return [(t - s, t) for s in spacings for t in frames if t - s >= self.oldest()]

    @torch.no_grad()
    def match_spacings(self, frames, spacings=(1, 5, 10, 15, 20), variant=matchers.M2, **kw):
        """All spacings of visualize_matches_sequence.py:369 in ONE matcher launch sequence: frame t
        (for t in ``frames``, typically the range push() returned) against cached frame t - s.
        Returns (frame_pairs, pairs, scores, counts); the lists are ordered spacing-major."""
        fp = self.spacing_pairs(frames, spacings)
        if not fp:
            dev = self.bank["scores"].device
            K = self.fe.K
            return fp, torch.empty(0, K, 2, dtype=torch.int32, device=dev), torch.empty(0, K, device=dev), \
                torch.empty(0, dtype=torch.int32, device=dev)
        return (fp,) + tuple(self.match_pairs(fp, variant, **kw))

    @torch.no_grad()
    def verify_pairs(self, frame_pairs, pairs, scores, counts, model="homography", **ransac):
        """Geometric verification of the lists match_pairs / match_spacings returned for ``frame_pairs``,
        on the resident keypoints (pixel units), against a homography (default) or, with
        ``model="fundamental"``, the epipolar constraint.  ``ransac``: threshold, iters, seed, want_mask.
        Returns geometry.verify_homography_device's (H (P,3,3), pairs, scores, counts[, mask]), or
        verify_fundamental_device's with F in place of H."""
        verify = {"homography": geometry.verify_homography_device,
                  "fundamental": geometry.verify_fundamental_device}.get(model)
        if verify is None:
            raise ValueError(f"verify_pairs: model must be 'homography' or 'fundamental', not {model!r}")
        kp = self.bank["keypoints"]
        if self.fe.grid != "pixel":
            kp = kp * self.fe.patch + self.fe.patch / 2
        return verify(kp, kp, pairs, scores, counts, pair_index=self.pair_index(frame_pairs), **ransac)


class TrackingCounters:
    """Device-side accumulators of TrackingTester.track_frame_sequence (test/test_tracking.py:139-199):
    per comparison the M5 count ``(max_j S[i,j] > match_threshold).sum()`` (:159-161), success when it
    reaches ``min_matches`` (:168-173).  ``update`` takes the counts tensor the matcher produced and
    never synchronises; ``results`` reads everything back once."""

    def __init__(self, num_keypoints, min_matches=50, device=None):
        self.K, self.min_matches = int(num_keypoints), int(min_matches)
        self.device = device
        self.count_chunks = []
        self.tracked = None

    def update(self, counts):
        counts = counts.reshape(-1)
        ok = (counts >= self.min_matches).sum()
        self.tracked = ok if self.tracked is None else self.tracked + ok
        self.count_chunks.append(counts)

    def results(self, sequence="", frame_spacing=1):
        import numpy as np
        if not self.count_chunks:
            return {"sequence": sequence, "frame_spacing": frame_spacing, "total_frames": 0,
                    "tracked_frames": 0, "lost_frames": 0, "tracking_success_rate": 0.0,
                    "match_counts": [], "match_ratios": []}
        mc = torch.cat(self.count_chunks).cpu().numpy().astype(np.int64)
        tracked = int(self.tracked)
        total = int(mc.size)
        ratios = mc / self.K
        return {"sequence": sequence, "frame_spacing": frame_spacing, "total_frames": total,
                "tracked_frames": tracked, "lost_frames": total - tracked,
                "tracking_success_rate": tracked / total if total > 0 else 0.0,
                "mean_matches": np.mean(mc), "std_matches": np.std(mc), "min_matches": np.min(mc),
                "max_matches": np.max(mc), "mean_match_ratio": np.mean(ratios),
                "match_counts": list(mc), "match_ratios": list(ratios)}


@torch.no_grad()
def track_sequence(frontend, saliency, features, frame_spacing=1, max_frames=100, min_matches=50,
                   match_threshold=0.8, chunk=64, capacity=None):
    """``track_frame_sequence`` (test/test_tracking.py:87-199) from device tensors: compare frame
    i - frame_spacing with frame i for i = frame_spacing, 2*frame_spacing, ... (< max_frames *
    frame_spacing), counting rows whose best similarity exceeds ``match_threshold`` (M5, no mutual
    check).  Only the frames that take part are extracted, each once, through a ring buffer; counts
    and the success counters stay on the device until the final read-back."""
    T = saliency.shape[0]
    ids = list(range(0, min(max_frames * frame_spacing, T), frame_spacing))      # frames compared (:140-148)
    store = FrameStore(frontend, capacity or min(len(ids), chunk + 1))
    counters = TrackingCounters(frontend.K, min_matches)
    sel = torch.tensor(ids, device=saliency.device)
    pushed = 0
    while pushed < len(ids):
        n = min(store.capacity - 1 if pushed else store.capacity, len(ids) - pushed)
        part = sel[pushed:pushed + n]
        fr = store.push(saliency.index_select(0, part), features.index_select(0, part))
        pairs = [(t - 1, t) for t in fr if t >= 1]                               # store ids are 0, 1, 2, ...
        if pairs:
            _, _, counts = store.match_pairs(pairs, matchers.M5, match_threshold=match_threshold)
            counters.update(counts)
        pushed += n
    return counters.results(frame_spacing=frame_spacing)
