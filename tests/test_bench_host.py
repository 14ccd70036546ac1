"""Host-side arithmetic of bench.py (no GPU): the `roofline` / `attention` blocks are assembled from the per-family CUDA-event
times of a committed bench line and must reproduce that line; the config-5 workload string parses into a size list."""
import json
import os
import re
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from coot_videotext_b200 import synthetic as syn  # noqa: E402


def test_roofline_blocks_reproduce_committed_line():
    line = json.load(open(os.path.join(ROOT, "profiles", "r2_bench_n1_final.json")))
    wl = syn.WORKLOADS[line["config"]["workload"]]
    host = syn.make_batch(wl, 1234)
    fam = bench.family_work(host, wl, int(host["clip_num"].max()))
    breakdown = {n: {"ms_per_step": v["ms_per_step"], "launches_per_step": v["launches_per_step"]} for n, v in line["breakdown"].items()}
    roofline, attention = bench.roofline_blocks(breakdown, fam, line["ms_per_step"])
    json.dumps([roofline, attention])  # serialisable
    assert roofline["family"] == line["roofline"]["family"] == "gemm_nn"
    assert roofline["algorithmic_flops_per_step"] == pytest.approx(line["roofline"]["algorithmic_flops_per_step"], rel=1e-12)
    assert roofline["achieved"] == pytest.approx(line["roofline"]["achieved"], rel=1e-9)
    assert 0.0 < roofline["frac"] < 1.0 and 0.0 < roofline["step_frac_of_tensor_peak"] < 1.0
    assert roofline["achieved"] * 1e12 * breakdown["gemm_nn"]["ms_per_step"] * 1e-3 == pytest.approx(fam["gemm_nn"]["flops"], rel=1e-9)
    # with the committed ncu family totals the traffic is per launch of the dominant family and the attention block carries the counters
    fams = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_families.json")))
    assert roofline["traffic"] == pytest.approx(fams["gemm_nn"]["dram_bytes_per_step"] / breakdown["gemm_nn"]["launches_per_step"])
    for n in ("attn_fwd", "attn_bwd"):
        assert attention[n]["ncu"]["tensor_pipe_pct_time_weighted"] > 0
        assert 0.0 < attention[n]["frac_of_hbm_peak"] < 1.0 and 0.0 < attention[n]["frac_of_tensor_peak"] < 1.0
        assert attention[n]["ms_per_step"] == pytest.approx(line["breakdown"][n]["ms_per_step"])


def test_dumped_outputs_are_whole_under_the_limit_and_a_fixed_sample_above(tmp_path):
    import numpy as np
    rng = np.random.default_rng(1)
    arrays = {"loss": np.float32([1.5]), "grad_a": rng.standard_normal(3000).astype(np.float32),
              "grad_b": rng.standard_normal((10, 100)).astype(np.float32)}
    bench.write_outputs(str(tmp_path / "whole"), arrays)
    for name, a in arrays.items():
        assert np.array_equal(np.load(tmp_path / "whole" / f"{name}.npy"), a)
    for run in ("one", "two"):
        bench.write_outputs(str(tmp_path / run), arrays, limit=8000)
    total = 0
    for name, a in arrays.items():
        s = np.load(tmp_path / "one" / f"{name}.npy")
        assert s.dtype == np.float32 and np.array_equal(s, np.load(tmp_path / "two" / f"{name}.npy"))
        assert np.isin(s, a).all()
        total += s.nbytes
    assert 0 < total <= 8000


def test_cfg5_workload_string():
    pat = r"cfg5_loss_n([\d,]+)(?:_d(\d+))?$"
    assert pat in open(os.path.join(ROOT, "bench.py")).read()
    m = re.match(pat, "cfg5_loss_n16384,4096_d768")
    assert [int(x) for x in m.group(1).split(",") if x] == [16384, 4096] and int(m.group(2)) == 768
    m = re.match(pat, "cfg5_loss_n1024")
    assert [int(x) for x in m.group(1).split(",") if x] == [1024] and m.group(2) is None
