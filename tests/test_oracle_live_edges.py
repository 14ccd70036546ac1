"""
Edge cases of the path, oracle vs the unmodified reference (CPU only).  The reference's own tests hold no vectors for the path
(SURVEY.md 8c), so the edge cases its data can produce were pinned by running it (tests/golden/make_golden_edges.py writes
tests/golden/edge_<case>.npz): one segment per video, the ActivityNet maximum of 27 segments, sequences of a single frame / word,
a batch of one video, and equal lengths everywhere.  Loss, and for EVERY parameter gradient its inf-norm, 2-norm and a seeded
sample of its elements.
"""
import os

import numpy as np
import pytest
import torch as th

from coot_videotext_b200 import synthetic as syn
from oracle import coot_oracle as O
from tests.util import GOLDEN_DIR, grad_sample_index, rel_inf

DATA_SEED, PARAM_SEED, CC_SEED = 4242, 31, 77
EDGE_GRAD_SAMPLES = 64  # per gradient tensor: keeps each golden file small; the inf- and 2-norms cover every element


def _shrink_to_single_steps(b, every=3):
    """Sets every `every`-th clip / sentence (and the first video / paragraph) to ONE valid position."""
    for feat, mask, lens in (("clip_feat", "clip_feat_mask", "clip_feat_len"), ("sent_feat", "sent_feat_mask", "sent_feat_len"),
                             ("vid_feat", "vid_feat_mask", "vid_feat_len"), ("par_feat", "par_feat_mask", "par_feat_len")):
        rows = range(1, b[lens].numel(), every) if feat in ("clip_feat", "sent_feat") else [b[lens].numel() - 1]
        for r in rows:
            b[lens][r] = 1
            b[feat][r, 1:] = 0
            b[mask][r, 1:] = True
    return b


CASES = {
    "one_segment_per_video": (syn.WorkloadCfg("e1", 5, 1, 12, 7, 64, 96, ragged=True), None),
    "27_segments": (syn.WorkloadCfg("e2", 2, 27, 6, 5, 64, 96, ragged=True, ragged_clip_num=True, max_vid_frames=20, max_par_words=30), None),
    "single_step_sequences": (syn.WorkloadCfg("e3", 4, 3, 10, 6, 64, 96, ragged=True), _shrink_to_single_steps),
    "one_video": (syn.WorkloadCfg("e4", 1, 3, 9, 5, 64, 96, ragged=True), None),
    "equal_lengths": (syn.WorkloadCfg("e5", 3, 2, 8, 4, 64, 96, ragged=False), None),
}


def edge_case_inputs(case):
    """(workload, host batch, parameters) of one edge case."""
    wl, mutate = CASES[case]
    b = syn.make_batch(wl, DATA_SEED)
    if mutate is not None:
        b = mutate(b)
    return wl, b, syn.make_params(wl.d_vid, wl.d_txt, PARAM_SEED)


def checksums(b, params):
    """float64 sums of every batch field and of every net's parameters: detect a drift of the seeded generators."""
    return (np.array([float(b[k].double().sum()) for k in sorted(b)]),
            np.array([float(sum(p.double().sum() for p in params[n].values())) for n in syn.NET_NAMES]))


def golden_path(case):
    return os.path.join(GOLDEN_DIR, f"edge_{case}.npz")


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_equals_live_reference_on_edge_case(case):
    g = np.load(golden_path(case))
    wl, b, params = edge_case_inputs(case)
    batch_sum, param_sum = checksums(b, params)
    assert np.allclose(batch_sum, g["batch_checksum"], rtol=1e-9) and np.allclose(param_sum, g["param_checksum"], rtol=1e-9), \
        "seeded input generators drifted from the golden run"
    # the multinomial draws of coot/loss_fn.py:311-313 that the reference made in this step
    ci, si = th.from_numpy(g["cc_clip_idx"]), th.from_numpy(g["cc_sent_idx"])
    loss, v, t, grads, parts = O.train_step(params, b, O.LOSS_CFG_ANET, ci, si, use_sampling=True)
    assert th.isfinite(loss) and rel_inf(loss, g["loss"]) < 2e-5, (float(loss), float(g["loss"]))
    row = {str(n): i for i, n in enumerate(g["grad_names"])}
    expected = [f"{net}.{name}" for net in syn.NET_NAMES for name in syn.trainable_names(params[net])]
    assert sorted(row) == sorted(expected)
    worst = 0.0
    for net in syn.NET_NAMES:
        for name in syn.trainable_names(params[net]):
            key = f"{net}.{name}"
            i = row[key]
            got = grads[net][name].flatten()
            assert th.isfinite(got).all(), (net, name)
            ref_inf, ref_l2 = float(g["grad_inf"][i]), float(g["grad_l2"][i])
            scale = max(ref_inf, 1e-5)
            idx = th.from_numpy(grad_sample_index(key, got.numel(), EDGE_GRAD_SAMPLES))
            err = float((got[idx] - th.from_numpy(g["grad_sample"][i])).abs().max()) / scale
            worst = max(worst, err)
            assert err < 2e-4, (case, key, err)
            assert abs(float(got.abs().max()) - ref_inf) / scale < 2e-4, (case, key)
            assert abs(float(got.norm()) - ref_l2) / max(ref_l2, 2e-4) < 2e-4, (case, key)
    print(case, "loss", float(loss), "worst grad err", worst)
