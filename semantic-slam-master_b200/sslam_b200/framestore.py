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
``relative_poses``      RANSAC fundamental matrix, then the relative pose and the points of a calibrated
                        camera, from the resident keypoints.
``track_poses``         the pose of each list's second frame against 3-D points attached to its first
                        frame's keypoints (geometry.point_map), by RANSAC P3P on the resident keypoints.
``triangulate_pairs``   the 3-D points of the rows of lists under known relative poses, on the resident
                        keypoints.
``track_and_map``       one step of sequence tracking with map growth: track_poses, then the points carried
                        onto each list's second frame and new points triangulated for its other keypoints.
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

    @torch.no_grad()
    def relative_poses(self, frame_pairs, pairs, scores, counts, camera, distance_thresh=50.0, refine_iters=10,
                       want_mask=False, want_points=False, **ransac):
        """Two-view initialisation for the lists match_pairs / match_spacings returned: verify_pairs with
        model="fundamental" (``ransac``: threshold, iters, seed), E = K^T F K, then the relative pose of
        every pair on the resident keypoints.  camera: (fx, fy, cx, cy) or a 3x3 matrix of the frames.
        Returns (R (P,3,3), t (P,3) unit, F (P,3,3), pose pairs, pose scores, pose counts[, mask (P,L)][,
        points (P,L,3)]); the pose lists hold the rows of the F inlier lists that lie in front of both
        cameras.  A pair without an F or without a pose has R, t all zeros and an empty list."""
        F, vp, vs, vc = self.verify_pairs(frame_pairs, pairs, scores, counts, model="fundamental", **ransac)
        kp = self.bank["keypoints"]
        if self.fe.grid != "pixel":
            kp = kp * self.fe.patch + self.fe.patch / 2
        out = geometry.recover_pose_device(kp, kp, geometry.essential_from_fundamental(F, camera), vp, vs, vc,
                                           camera, pair_index=self.pair_index(frame_pairs),
                                           distance_thresh=distance_thresh, refine_iters=refine_iters,
                                           want_mask=want_mask, want_points=want_points)
        return (out[0], out[1], F) + tuple(out[2:5]) + tuple(out[7:])

    @torch.no_grad()
    def track_poses(self, frame_pairs, pairs, scores, counts, point_maps, camera, threshold=3.0, iters=1024, seed=0,
                    refine_iters=10):
        """Camera tracking for the lists match_pairs / match_spacings returned for ``frame_pairs`` (a, b):
        point_maps (P, Ka, 3) holds, for list p, the 3-D point of each keypoint of frame a (NaN where there is
        none; geometry.point_map builds it).  Each list is first restricted, in order, to the rows whose point
        is finite (geometry.rows_with_points: no sample is spent on a row without a point), then the pose of
        frame b against those
        points is estimated by RANSAC P3P on the resident keypoints of b.  camera: (fx, fy, cx, cy) or a 3x3
        matrix of the frames.  Returns (R (P,3,3), t (P,3) in the points' units, pairs, scores, counts): the
        inlier rows, a subset of the input lists in input order.  A list without a model has R, t all zeros
        and an empty list."""
        kp = self.bank["keypoints"]
        if self.fe.grid != "pixel":
            kp = kp * self.fe.patch + self.fe.patch / 2
        maps = point_maps.to(torch.float32).contiguous()
        rows, sc, n = geometry.rows_with_points(pairs, scores, counts, maps)
        P = rows.shape[0]
        dev = rows.device
        idx = self.pair_index(frame_pairs)
        idx = torch.stack([torch.arange(P, dtype=torch.int32, device=dev), idx[:, 1]], 1)
        out = geometry.solve_pnp_device(maps, kp, rows, sc, n, camera,
                                        pair_index=idx, threshold=threshold, iters=iters, seed=seed,
                                        refine_iters=refine_iters)
        return out[:5]


    def _pixel_keypoints(self):
        kp = self.bank["keypoints"]
        return kp * self.fe.patch + self.fe.patch / 2 if self.fe.grid != "pixel" else kp

    @torch.no_grad()
    def triangulate_pairs(self, frame_pairs, pairs, scores, counts, R, t, camera, threshold=3.0, min_parallax_deg=1.0,
                          distance_thresh=50.0, refine_iters=10, want_mask=False):
        """The 3-D points of the rows of the lists match_pairs / match_spacings returned for ``frame_pairs``
        (a, b), under the relative pose (R, t) of each pair (x_b ~ R x_a + t), on the resident keypoints:
        geometry.triangulate_device's (points (P,L,3) in frame a's camera frame, kept pairs, scores,
        counts[, mask])."""
        kp = self._pixel_keypoints()
        return geometry.triangulate_device(kp, kp, pairs, scores, counts, R, t, camera,
                                           pair_index=self.pair_index(frame_pairs), threshold=threshold,
                                           min_parallax_deg=min_parallax_deg, distance_thresh=distance_thresh,
                                           refine_iters=refine_iters, want_mask=want_mask)

    @torch.no_grad()
    def track_and_map(self, frame_pairs, pairs, scores, counts, point_maps, camera, **kw):
        """One step of sequence tracking with map growth for the lists match_pairs / match_spacings returned
        for ``frame_pairs`` (a, b): point_maps (P, Ka, 3) as for track_poses.  The pose of frame b by RANSAC
        P3P against the points of frame a, then the next point maps (P, Kb, 3) of frame b: the PnP inliers'
        points carried over, and points triangulated under that pose for the keypoints that have none
        (geometry.track_and_map, whose keyword arguments ``kw`` takes).  Returns (R (P,3,3), t (P,3), pairs,
        scores, counts, next point maps); a list without a model has R, t all zeros, an empty list and an
        all-NaN map."""
        kp = self._pixel_keypoints()
        return geometry.track_and_map(point_maps, kp, kp, pairs, scores, counts, camera, self.pair_index(frame_pairs),
                                      **kw)

    @torch.no_grad()
    def bundle_adjust(self, windows, obs, points, counts, R, t, camera, **kw):
        """Sliding-window bundle adjustment on the resident keypoints: ``windows`` holds P lists of W resident
        frame ids; obs (P,N,W), points (P,N,3), counts (P,) as geometry.window_tracks returns them, R (P,W,3,3),
        t (P,W,3) the frames' absolute poses.  -> geometry.bundle_adjust_device's (R, t, points, rms,
        accepted[, mask]), whose keyword arguments ``kw`` takes."""
        for frames in windows:
            for f in frames:
                if not self.holds(f):
                    raise KeyError(f"window frame {f} is not resident")
        kp = self._pixel_keypoints()
        fi = torch.tensor([[self.slot_of(f) for f in frames] for frames in windows], dtype=torch.int32)
        return geometry.bundle_adjust_device(kp, fi.to(kp.device), obs, points, counts, R, t, camera, **kw)


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
