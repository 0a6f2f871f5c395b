"""CPU: the oracle port of the whole path end to end against the per-pair records (match count and
CRC32 of the keypoint rows of the match list) stored in tests/golden/pipeline.npz.  The port wrote
those records: its stages are pinned to the reference by test_oracle_golden.py, and every match
decision of this case clears its threshold by more than 5e-4 (asserted below), so last-bit differences
between implementations cannot change them.  Where the reference's own functions are installed
(baseline/_ref, placed there by __graft_entry__.build()), they run on the same inputs and must give
the same records."""

import json

import numpy as np
import torch

import oracle
from oracle import pipeline as opipe, recipes, ref_pipeline
from parity import load_golden
from sslam_b200 import synth


def test_oracle_pipeline_equals_reference_pipeline():
    from models.descriptor_refiner import DescriptorRefiner
    z, meta = load_golden("pipeline")
    T, K, dims = meta["frames"], meta["K"], tuple(meta["refiner"])
    torch.manual_seed(meta["torch_seed"])
    refiner = DescriptorRefiner(*dims)
    sal, feat = synth.make_sequence(T, seq_id=meta["seq_id"], height=meta["height"], width=meta["width"])
    sd = {k: v.detach().numpy() for k, v in refiner.state_dict().items()}
    # the stored records belong to these exact inputs and weights
    assert recipes.sha256(sal.numpy()) == meta["sha256"]["saliency"]
    assert recipes.sha256(feat.numpy()) == meta["sha256"]["features"]
    assert recipes.sha256(np.concatenate([sd[k].ravel() for k in sorted(sd)])) == meta["sha256"]["weights"]
    stored = [tuple(int(v) for v in r) for r in z["records"]]
    assert len(stored) == T - 1 and all(r[0] > 0 for r in stored), json.dumps(meta)
    w = oracle.RefinerWeights.from_state_dict(refiner.state_dict())
    port_rec, _ = opipe.run_sequence(sal.numpy()[..., 0], feat.numpy(), w, K, 1, 1)
    assert [tuple(r) for r in port_rec] == stored
    # mutual nearest neighbours (row and column argmax) and the ratio test of M1 (0.8) are far from ties
    ex = [opipe.extract_frame(sal.numpy()[t, ..., 0], feat.numpy()[t], w, K) for t in range(T)]
    for e1, e2 in zip(ex[:-1], ex[1:]):
        S = e1[2].astype(np.float64) @ e2[2].astype(np.float64).T
        row, col = -np.sort(-S, axis=1)[:, :2], -np.sort(-S.T, axis=1)[:, :2]
        assert (row[:, 0] - row[:, 1]).min() > 5e-4 and (col[:, 0] - col[:, 1]).min() > 5e-4
        assert np.abs(row[:, 0] - 0.8 * row[:, 1]).min() > 5e-4
    if ref_pipeline.available():
        ref_rec, _ = ref_pipeline.run_sequence(sal.numpy()[..., 0], feat.numpy(), sd, dims, K, 2)
        assert [tuple(r) for r in ref_rec] == stored
