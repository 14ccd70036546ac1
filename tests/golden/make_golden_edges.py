"""
Generates tests/golden/edge_<case>.npz by running the UNMODIFIED reference (imported through oracle/ref_import.py) on the edge
cases of tests/test_oracle_live_edges.py: one training step in eval mode on the CPU, cycle-consistency indices drawn by the
reference from torch's RNG seeded with CC_SEED.
Run where the reference tree is available:  python tests/golden/make_golden_edges.py

Stored per case: the loss, the cycle-consistency indices the reference drew, checksums of the seeded inputs, and for every
parameter gradient its inf-norm, 2-norm and a seeded sample of EDGE_GRAD_SAMPLES elements.
"""
import os
import sys

import numpy as np
import torch as th

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from coot_videotext_b200 import synthetic as syn  # noqa: E402
from oracle import ref_runner as RR  # noqa: E402
from tests.golden.make_golden import draw_cc_indices  # noqa: E402
from tests.test_oracle_live_edges import CASES, CC_SEED, EDGE_GRAD_SAMPLES, checksums, edge_case_inputs, golden_path  # noqa: E402
from tests.util import grad_sample_index  # noqa: E402


def run_case(case):
    wl, b, params = edge_case_inputs(case)
    rs = RR.ReferenceStep(wl, b, params, device="cpu", fp16=False, train=False)
    th.manual_seed(CC_SEED)
    loss = rs.step()
    out = {"loss": loss.numpy()}
    # eval mode: nothing consumes the RNG before the draws of coot/loss_fn.py:311-313, so they are replayed from the same seed
    maxc = int(b["clip_num"].max())
    pad_mask = th.arange(maxc)[None, :] >= b["clip_num"][:, None]
    ci, si = draw_cc_indices(CC_SEED, pad_mask, pad_mask)
    out["cc_clip_idx"], out["cc_sent_idx"] = ci.numpy(), si.numpy()
    out["batch_checksum"], out["param_checksum"] = checksums(b, params)
    names, inf, l2, sample = [], [], [], []
    for net in syn.NET_NAMES:
        named = dict(rs.mgr.model_dict[net].named_parameters())
        for name in syn.trainable_names(params[net]):
            g = named[name].grad.detach().flatten()
            names.append(f"{net}.{name}")
            inf.append(float(g.abs().max()))
            l2.append(float(g.norm()))
            sample.append(g[th.from_numpy(grad_sample_index(f"{net}.{name}", g.numel(), EDGE_GRAD_SAMPLES))].numpy())
    # one array per statistic (row i = gradient names[i]): a member per gradient would make the file mostly zip headers
    out["grad_names"], out["grad_inf"], out["grad_l2"] = np.array(names), np.array(inf, np.float32), np.array(l2, np.float32)
    out["grad_sample"] = np.stack(sample)
    path = golden_path(case)
    np.savez_compressed(path, **out)
    print(path, "loss", float(loss), "bytes", os.path.getsize(path))


if __name__ == "__main__":
    for c in sorted(CASES):
        run_case(c)
