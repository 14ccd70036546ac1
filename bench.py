#!/usr/bin/env python
"""
Benchmark of the COOT retrieval forward/backward hot path (BASELINE.json metric: clip+sentence pairs/sec).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2_anet_b64]

A "step" is one pass of the hot path over one synthetic batch: zero_grad + encode_visual + encode_text + 7 contrastive terms +
cycle-consistency loss + backward (+ embedding all-gather and gradient all-reduce for N > 1) - the body of the reference's train
loop without the optimizer (coot/trainer_retrieval.py:261-284).  One JSON line is printed by rank 0 (see the driver contract).

  value     whole-job pairs/s with the batch already resident in HBM (CUDA events, max over ranks)
  e2e       the same metric through the public drop-in API with HOST (pinned) inputs: H2D copy of the batch and D2H read of
            the loss inside the timed region
  roofline  the kernel family with the LARGEST CUDA-event share of the step (measured live in a profiled pass): algorithmic
            FLOPs / summed CUDA-event duration vs the measured bf16 peak; `attention` = the same for the attention kernels
            (the metric's second half) with the tensor-pipe % / DRAM bytes of the committed ncu capture (profiles/)
  cpu_baseline / --impl reference : the UNMODIFIED reference modules (oracle/_ref, copied by oracle/make_ref.py) on the host
            cores, full batch, train mode (kind "reference"); the oracle port only if that copy is missing (kind "port")
  --impl torch_cuda : the same unmodified reference modules as eager PyTorch on cuda:0 (fp32 and fp16 autocast) - SURVEY 8d's
            "PyTorch-on-B200" bar
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# Rank 0 must print exactly ONE JSON line on stdout: file descriptor 1 is pointed at stderr for the whole run (NCCL prints its
# version banner on stdout from C code) and restored only for the final line.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)

METRIC = "clip+sentence pairs/sec"
UNIT = "pairs/s"
CPU_SAMPLE_VIDEOS = 16
DUMP_LIMIT_BYTES = 64_000_000


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_cuda"])
    ap.add_argument("--workload", default="cfg2_anet_b64")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--api", default="fused_graph", choices=["fused_graph", "fused", "autograd"],
                    help="fused_graph: three C calls replayed from a CUDA graph (default); fused: same without graph; "
                         "autograd: the drop-in autograd composition of step.HotPath")
    ap.add_argument("--padded-h2d", action="store_true",
                    help="e2e: copy the whole padded feature tensors (cudaMemcpy) instead of staging only their valid rows")
    ap.add_argument("--feat", default="fp16_packed", choices=["fp16_packed", "fp32"],
                    help="e2e host feature storage: fp16_packed = data.PackedFeatureStore (packed valid rows, IEEE fp16, SURVEY 8f-2; "
                         "default); fp32 = the padded fp32 tensors of the reference contract (valid rows staged)")
    ap.add_argument("--no-clocks", action="store_true", help="do not sample clocks (use when running under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (loss, and the gradient of every net's parameters) as DIR/<name>.npy, "
                         f"float32, at most {DUMP_LIMIT_BYTES // 10**6} MB in all; the inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload.startswith("cfg5_loss_n")):
        ap.error("--dump-outputs applies to --impl b200 on the training-step workloads")
    return args


def step_outputs(loss, mgr):
    """Host copies of what one training step hands its caller: the loss, and per net the gradient of its trainable parameters
    flattened in named_parameters() order."""
    import torch as th
    from coot_videotext_b200.model_retrieval import NET_NAMES
    out = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
    for net in NET_NAMES:
        grads = [p.grad.detach().flatten() for p in mgr.model_dict[net].parameters() if p.requires_grad]
        out[f"grad_{net}"] = th.cat(grads).float().cpu().numpy()
    return out


def write_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes DIR/<name>.npy.  Above `limit` bytes in all, every array is replaced by the same fixed, seeded sample of its elements
    (flattened, indices ascending) in proportion to its size, so that runs with the same arguments stay comparable."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            keep = max(1, a.size * limit // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def workload_config(wl, n_gpus, input_bytes=None):
    """The SAME dict for every arm (the driver matches the arms on it); what differs between the arms (dropout RNG, sample) is
    reported in the arm's own keys, not here."""
    mb = f"{input_bytes / 1e6:.0f} MB" if input_bytes else "features"
    return {"workload": wl.name, "global_batch_videos": wl.batch * n_gpus, "videos_per_gpu": wl.batch,
            "clips_per_video": wl.clips_per_video, "max_frames": wl.max_frames, "max_words": wl.max_words, "d_vid": wl.d_vid,
            "d_txt": wl.d_txt, "lengths": "ragged U[max/2, max]" if wl.ragged else "full", "parallelism": f"dp{n_gpus}",
            "l2": f"inputs ({mb}/step) + ~1 GB of saved activations per step exceed L2 (126 MB); no explicit flush",
            "dropout": f"train mode, p={wl.dropout} at the 7 nn.Dropout sites of every net",
            "step": "zero_grad+encode_visual+encode_text+contrastive(7)+cycle_cons+backward, no optimizer"}


def host_core_info():
    n = os.cpu_count() or 1
    phys = None
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
    except Exception:  # noqa: BLE001
        pass
    model = None
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except Exception:  # noqa: BLE001
        pass
    return {"logical": n, "physical": phys, "model": model}


# ----------------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_time(wl, steps, warmup):
    """Times the UNMODIFIED reference modules (oracle/_ref via oracle/ref_runner.py) on the host cores: the FULL workload batch,
    train mode (torch dropout), fp32, forward + losses + autograd backward, no optimizer.  Returns
    (pairs/s, threads, sample description, seconds per step, kind)."""
    import torch as th
    from coot_videotext_b200 import synthetic as syn
    from oracle import ref_import
    ncpu = os.cpu_count() or 1
    b = syn.make_batch(wl, 1234)
    params = syn.make_params(wl.d_vid, wl.d_txt, 7)
    pairs = int(b["clip_num"].sum())
    if not ref_import.reference_available():
        return cpu_port_time(wl, steps, warmup) + ("port",)
    from oracle import ref_runner as RR
    rs = RR.ReferenceStep(wl, b, params, device="cpu", fp16=False, train=True)
    # torch's intra-op pool scales badly past a few dozen threads on these tensors: time one step at a few thread counts and keep
    # the fastest, so that the CPU arm runs at ITS best; `cores` reports the threads actually used
    best = (None, 1)
    for nt in sorted({t for t in (16, 32, 64) if t <= ncpu} or {ncpu}):
        th.set_num_threads(nt)
        rs.step()
        t0 = time.perf_counter()
        rs.step()
        dt = time.perf_counter() - t0
        if best[0] is None or dt < best[0]:
            best = (dt, nt)
    th.set_num_threads(best[1])
    for _ in range(warmup):
        rs.step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        rs.step()
        times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    sample = (f"full {wl.name} batch ({wl.batch} videos, {pairs} pairs), {len(times)} timed steps after {warmup} warm-up, train mode "
              f"(torch dropout p={wl.dropout}), fp32, unmodified coot/ + nntrainer/ modules from {os.path.relpath(ref_import.REFERENCE_ROOT, ROOT) if ref_import.REFERENCE_ROOT.startswith(ROOT) else ref_import.REFERENCE_ROOT}")
    return pairs / sec, best[1], sample, sec, "reference"


def cpu_port_time(wl, steps, warmup, sample_videos=CPU_SAMPLE_VIDEOS):
    """Fallback when oracle/_ref is missing: the oracle restatement (oracle/coot_oracle.py) with torch autograd, eval mode, on the
    first `sample_videos` videos.  Returns (pairs/s, cores, sample description, seconds per step)."""
    import torch as th
    from coot_videotext_b200 import synthetic as syn
    from oracle import coot_oracle as O
    ncpu = os.cpu_count() or 1
    b = syn.make_batch(wl, 1234, batch=sample_videos)
    params = syn.make_params(wl.d_vid, wl.d_txt, 7)
    pairs = int(b["clip_num"].sum())
    ci = th.zeros(sample_videos, dtype=th.long)
    th.set_num_threads(min(32, ncpu))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.train_step_autograd(params, b, O.LOSS_CFG_ANET, ci, ci, use_sampling=True)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return (pairs * len(times) / total, min(32, ncpu),
            f"PORT (oracle/_ref missing): first {sample_videos} videos ({pairs} pairs) of {wl.name}, eval mode, {len(times)} steps", total / len(times))


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each step = the full 64-video batch on the host (about 1 - 3 s); bounded so that the arm ends within a few minutes
    steps, warmup = max(1, min(args.steps, 10)), max(1, min(args.warmup, 2))
    value, cores, sample, sec, kind = cpu_reference_time(wl, steps, warmup)
    from coot_videotext_b200 import synthetic as syn
    host = syn.make_batch(wl, 1234)
    in_bytes = sum(host[k].numel() * 4 for k in ("vid_feat", "clip_feat", "par_feat", "sent_feat"))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(wl, args.gpus, in_bytes),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "host": host_core_info(),
                             "timed_steps": steps},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "one rank-0 process on the host cores times ONE GPU's share of the batch (weak scaling: 64 videos per GPU); "
                    "dropout masks come from torch's RNG here and from the stateless hash on the B200 arm (same p)"}
    emit(line)


def run_torch_cuda(args, wl):
    """SURVEY 8d: the reference's own eager PyTorch path on the B200 (unmodified modules from oracle/_ref, use_cuda: true), fp32 and
    fp16 autocast + GradScaler (the shipped configs' fp16_train: true).  Not part of the driver contract; one JSON line."""
    import torch as th
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from coot_videotext_b200 import synthetic as syn
    from oracle import ref_import
    if not ref_import.reference_available() or not th.cuda.is_available():
        emit({"impl": "torch_cuda", "unavailable": "oracle/_ref (python oracle/make_ref.py) and a CUDA device are required"})
        return
    from oracle import ref_runner as RR
    host = syn.make_batch(wl, 1234)
    params = syn.make_params(wl.d_vid, wl.d_txt, 7)
    res = {}
    for name, fp16 in (("fp32", False), ("fp16_autocast", True)):
        th.backends.cuda.matmul.allow_tf32 = False
        v, sec, _, loss = RR.time_reference(wl, host, params, max(3, args.steps), max(3, args.warmup), device="cuda:0", fp16=fp16)
        res[name] = {"value": v, "unit": UNIT, "ms_per_step": sec * 1e3, "loss": loss}
    in_bytes = sum(host[k].numel() * 4 for k in ("vid_feat", "clip_feat", "par_feat", "sent_feat"))
    emit({"impl": "torch_cuda", "metric": METRIC, "value": res["fp16_autocast"]["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": res["fp16_autocast"]["ms_per_step"], "higher_is_better": True, "dtype": "fp16 autocast (value) / fp32",
          "data": "synthetic", "config": workload_config(wl, 1, in_bytes), "variants": res,
          "note": "unmodified reference modules (oracle/_ref) as eager PyTorch on cuda:0, batch resident on the device, wall clock "
                  "around synchronised steps (host-launch bound); torch " + th.__version__})


# ----------------------------------------------------------------------------------------------------- clocks sampling
def bind_to_gpu_numa_node(index):
    """Pins the calling thread to the CPUs NVML reports as local to GPU `index` while the pinned host batch is allocated, so that
    its first-touch pages sit on the GPU's NUMA node; a pinned buffer on the other socket costs ~15 % of the H2D bandwidth, which
    is what bounds e2e.  Returns (previous affinity, number of local CPUs) or (None, 0) when NVML has no answer - the run then
    keeps the affinity it was started with.  The caller restores the affinity right after the allocation."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus or len(cpus) == len(allowed):
            return None, 0
        os.sched_setaffinity(0, cpus)
        return allowed, len(cpus)
    except Exception:  # noqa: BLE001
        return None, 0


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML (in-process thread, ~20 Hz) during the timed region."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, reasons))
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                break
            time.sleep(0.05)

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {self.err}"]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        nv = self.nv
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            mx = None
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                "hw_power_brake_slowdown": 0x80}
        reasons = set()
        for _, r in self.samples:
            for name, bit in bits.items():
                if r & bit:
                    reasons.add(name)
        sm = [x for x, _ in self.samples]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------- B200 arm
def family_work(batch, wl, max_clips):
    """ALGORITHMIC work per kernel family and step (SURVEY.md section 8d formulas, ACTUAL valid lengths; padding does not count,
    except the global nets' padded positions, which the reference computes too).  FLOPs are 1x per product."""
    D = 384
    b = int(batch["clip_num"].shape[0])
    mods = ((batch["vid_feat_len"], batch["clip_feat_len"], wl.d_vid), (batch["par_feat_len"], batch["sent_feat_len"], wl.d_txt))
    T = [float(a.sum() + c.sum()) for a, c, _ in mods]
    T2 = [float((a.double() ** 2).sum() + (c.double() ** 2).sum()) for a, c, _ in mods]
    loc = 2654208.0  # per token: QKV 884736 + out 294912 + FFN 589824 + GenPool 884736
    R = float(b * max_clips)
    glob = R * (1769472.0 + 589824.0) + b * 1179648.0  # per global net: self layer on R rows; cross layer: K,V on R rows, rest on b rows
    inputfc = sum(2.0 * D * t * d for t, (_, _, d) in zip(T, mods))
    nn_fwd = sum(T) * loc + 2 * glob
    attn_fwd = sum(1536.0 * t2 for t2 in T2)
    qkv_bytes = sum(T) * 3 * D * 4.0  # split-bf16 planes: 4 B per element
    ctx_bytes = sum(T) * D * 4.0
    fam = {
        "gemm_inputfc": {"flops": inputfc, "kernel": "gemm_tc5_nn_kernel<BIAS|GELU|PE|OUT_F32|OUT_SPLIT> (input FC, K = d_in)"},
        "gemm_nn": {"flops": 2.0 * nn_fwd, "kernel": "gemm_tc5_nn_kernel<*> family: forward + data-gradient GEMMs of the 4 nets "
                                                     "(QKV, out-proj, FFN x2, GenPool x3; K = 384 / 768), tcgen05 + TMA, split-bf16 x3"},
        "gemm_tt": {"flops": nn_fwd, "kernel": "gemm_tc5_tt_kernel: weight-gradient GEMMs (reduction over tokens, split-K)"},
        "gemm_tt_inputfc": {"flops": inputfc, "kernel": "gemm_tc5_tt_kernel (input-FC weight gradient)"},
        "attn_fwd": {"flops": attn_fwd, "bytes": qkv_bytes + ctx_bytes, "kernel": "attention kernels of csrc/attention*.cu"},
        "attn_bwd": {"flops": 2.5 * attn_fwd, "bytes": 2 * qkv_bytes + 2 * ctx_bytes, "kernel": "attention kernels of csrc/attention*.cu"},
    }
    fam["step"] = {"flops": inputfc * 2 + nn_fwd * 3 + attn_fwd * 3.5}
    return fam


def roofline_blocks(breakdown, fam, step_ms):
    """`roofline` (the kernel family with the largest CUDA-event share) and `attention` blocks of the JSON line from the per-family
    event times of the profiled pass (`breakdown`), the algorithmic work (`family_work`) and the resident step time.  Pure host
    arithmetic (tests/test_bench_host.py)."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernels timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained"
    ncu = {}
    try:  # per-family DRAM bytes / tensor-pipe % of the committed `ncu --set full` capture of this same step (tests/ncu_summary.py)
        ncu = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_families.json")))
    except Exception:  # noqa: BLE001
        pass
    for n in breakdown:
        w = fam.get(n)
        t = breakdown[n]["ms_per_step"] * 1e-3
        if w and t > 0:
            breakdown[n]["algorithmic_gflop_per_step"] = w["flops"] / 1e9
            breakdown[n]["tflops"] = w["flops"] / t / 1e12
            breakdown[n]["frac_of_tensor_peak"] = w["flops"] / t / 1e12 / peak
    # the family with the largest CUDA-event share of the profiled step
    dom = max((n for n in breakdown if n in fam), key=lambda n: breakdown[n]["ms_per_step"])
    d_ms, d_cnt = breakdown[dom]["ms_per_step"], breakdown[dom]["launches_per_step"]
    achieved = fam[dom]["flops"] / (d_ms * 1e-3) / 1e12 if d_ms > 0 else 0.0
    nd = ncu.get(dom, {})
    roofline = {"bound": "tensor", "kernel": fam[dom]["kernel"], "family": dom,
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": (nd.get("dram_bytes_per_step") / d_cnt) if (nd.get("dram_bytes_per_step") and d_cnt) else None,
                "traffic_note": nd.get("source"),
                "peak_source": peak_src, "algorithmic_flops_per_step": fam[dom]["flops"], "launches_per_step": d_cnt,
                "avg_launch_ms": d_ms / d_cnt if d_cnt else None,
                "share_of_profiled_step": d_ms / max(1e-9, sum(v["ms_per_step"] for v in breakdown.values())),
                "share_note": "share among the event-timed families (all GEMM and attention launches); the row kernels, losses and "
                              "small launches are not event-timed (profiles/r2_kernel_rooflines.md lists every family of the ncu launch list)",
                "note": "achieved = algorithmic FLOPs of the family (1x per product, SURVEY 8d formulas with the actual valid lengths) / "
                        "summed CUDA-event duration of its launches in the profiled pass; per launch = /launches_per_step. The "
                        "split-bf16 kernels issue 3 bf16 MMAs per product, so the tensor pipe does 3x this work"}
    roofline["step_frac_of_tensor_peak"] = (fam["step"]["flops"] / (step_ms * 1e-3)) / 1e12 / peak
    # the attention path (the metric's second half): tensor fraction AND HBM fraction of the unfused form it runs in
    at = {}
    for n in ("attn_fwd", "attn_bwd"):
        t = breakdown[n]["ms_per_step"] * 1e-3
        if t > 0:
            at[n] = {"ms_per_step": t * 1e3, "launches_per_step": breakdown[n]["launches_per_step"],
                     "algorithmic_gflop": fam[n]["flops"] / 1e9, "tflops": fam[n]["flops"] / t / 1e12,
                     "frac_of_tensor_peak": fam[n]["flops"] / t / 1e12 / peak,
                     "algorithmic_hbm_bytes": fam[n]["bytes"], "gbs": fam[n]["bytes"] / t / 1e9,
                     "frac_of_hbm_peak": fam[n]["bytes"] / t / 1e9 / hbm_peak,
                     "ncu": ncu.get(n)}
    attention = {"kernels": fam["attn_fwd"]["kernel"], "hbm_peak_gbs": hbm_peak, "tensor_peak_tflops": peak, **at,
                 "note": "algorithmic HBM bytes = split-bf16 Q,K,V read + context written (fwd); Q,K,V,dO,O read + dQ,dK,dV written "
                         "(bwd); `ncu` = sm__pipe_tensor* % and dram bytes of the committed capture (profiles/r2_ncu_families.json)"}
    return roofline, attention


def run_b200(args, wl):
    import torch as th
    import torch.distributed as dist
    from coot_videotext_b200 import build as B
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not th.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    th.cuda.set_device(local_rank)
    if world > 1:
        # optional SM partition between NCCL and the library's persistent kernels (COOT_SM_RESERVE = N: NCCL capped at N CTAs, the
        # kernels sized to SMs - N); off by default (slower at N = 2, see fused.py)
        if int(os.environ.get("COOT_SM_RESERVE", "0")) > 0:
            os.environ.setdefault("NCCL_MAX_CTAS", os.environ["COOT_SM_RESERVE"])
        dist.init_process_group("nccl", device_id=th.device("cuda", local_rank))
    if rank == 0:
        B.build()
    if world > 1:
        dist.barrier()
    from coot_videotext_b200 import lib as L
    from coot_videotext_b200 import synthetic as syn
    from coot_videotext_b200.model_retrieval import NET_NAMES, RetrievalDataBatch, RetrievalModelManager
    from coot_videotext_b200.step import HotPath
    lib = L.load()
    dev = th.device("cuda", local_rank)
    params = syn.make_params(wl.d_vid, wl.d_txt, 7)
    mgr = RetrievalModelManager(vid_feat_dim=wl.d_vid, text_feat_dim=wl.d_txt, dropout_layer=wl.dropout, dropout_pool=wl.dropout)
    mgr.set_model_state({n: params[n] for n in NET_NAMES})
    mgr.cuda()
    mgr.set_all_models_train()
    from coot_videotext_b200.fused import FusedHotPath
    if args.api == "autograd":
        hot = HotPath(mgr)
    else:
        # static_shards: the synthetic batches have one fixed layout on every rank (no per-step layout exchange)
        hot = FusedHotPath(mgr, use_graph=(args.api == "fused_graph"), static_shards=True, dropout_layer=wl.dropout,
                           dropout_pool=wl.dropout)
    host = syn.make_batch(wl, 1234 + rank)
    pairs_local = int(host["clip_num"].sum())
    max_clips = int(host["clip_num"].max())
    prev_affinity, numa_cpus = bind_to_gpu_numa_node(local_rank)  # first touch of the pinned pages on the GPU's NUMA node
    pinned = {k: v.pin_memory() for k, v in host.items()}
    if prev_affinity is not None:
        os.sched_setaffinity(0, prev_affinity)
    resident = RetrievalDataBatch(**{k: v.to(dev) for k, v in host.items()}, max_clips=max_clips, max_sents=max_clips)
    b = host["clip_num"].shape[0]
    g = th.Generator().manual_seed(99)
    clip_idx = th.stack([th.randint(0, int(c), (1,), generator=g)[0] for c in host["clip_num"]]).to(dev)
    sent_idx = th.stack([th.randint(0, int(c), (1,), generator=g)[0] for c in host["sent_num"]]).to(dev)
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())

    def sync_all():
        th.cuda.synchronize()
        if world > 1:
            dist.barrier()
            th.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = th.tensor([ms], dtype=th.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step_resident():
        return hot.train_step(resident, clip_idx, sent_idx)

    from coot_videotext_b200.data import DeviceBatchRing
    # three slots, copies submitted TWO batches ahead: the copy engine always has the next transfer queued, so the step period is
    # max(compute, H2D) and not H2D + the host's submission latency (with two slots the copy of batch i+1 could only be submitted
    # after step i had been launched, which cost 0.06 - 0.45 ms per step depending on how fast the host thread was)
    packed = args.feat == "fp16_packed" and args.api != "autograd" and not args.padded_h2d
    if packed:
        from coot_videotext_b200.data import PackedBatchRing, PackedFeatureStore
        prev_affinity, _ = bind_to_gpu_numa_node(local_rank)
        pinned = PackedFeatureStore(host)  # converted ONCE (preload time), pinned
        if prev_affinity is not None:
            os.sched_setaffinity(0, prev_affinity)
        ring = PackedBatchRing(pinned, dev, depth=3)
    else:
        ring = DeviceBatchRing(host, dev, depth=3, max_clips=max_clips, max_sents=max_clips, valid_rows_only=not args.padded_h2d)

    def step_e2e(prefetch_next=True):
        # every step: H2D of its whole batch from pinned host memory (copy stream, three slots so that the transfer of step
        # i+1 overlaps the compute of step i), the step itself, and the D2H read of the loss of the PREVIOUS step
        batch = ring.acquire()
        loss_t = hot.train_step(batch, clip_idx, sent_idx)
        ring.release()
        if prefetch_next:
            ring.prefetch(pinned)
        return loss_t

    for _ in range(max(args.warmup, 3)):
        loss = step_resident()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0 and not args.no_clocks:
        sampler.start()
    launches0 = lib.coot_launch_count()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step_resident()
    e1.record()
    sync_all()
    ms = max_over_ranks(e0.elapsed_time(e1))
    # taken before anything below runs another step (launch count, e2e, profiled pass) and overwrites the gradients
    outputs = step_outputs(loss, mgr) if (args.dump_outputs and rank == 0) else None
    launches = lib.coot_launch_count() - launches0
    launches_per_step = launches / args.steps
    if launches == 0:  # CUDA-graph replay: the library's launch sites ran once at capture time; count one un-captured step
        c0 = lib.coot_launch_count()
        hot._step_body(resident, clip_idx, sent_idx)
        th.cuda.synchronize()
        launches_per_step = lib.coot_launch_count() - c0
    clocks = sampler.stop() if (rank == 0 and not args.no_clocks) else None
    value = pairs_local * world * args.steps / (ms * 1e-3)

    # ---- end to end: host (pinned) inputs, H2D + D2H inside the timed region
    ring.prefetch(pinned)
    ring.prefetch(pinned)
    for _ in range(4):
        step_e2e()
    sync_all()
    e0.record()
    prev = None
    for i in range(args.steps):
        cur = step_e2e(prefetch_next=True)
        if prev is not None:
            lv = float(prev.item())  # D2H read of the step result (one step delayed so that it does not stall the pipeline)
        prev = cur.clone()
    lv = float(prev.item())
    e1.record()
    sync_all()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    h2d_padded_bytes, h2d_bytes = h2d_bytes, ring.last_h2d_bytes
    e2e = pairs_local * world * args.steps / (ms_e2e * 1e-3)

    # ---- forward only (validation path)
    fwd = (lambda: hot.forward_only(resident)) if args.api == "autograd" else (lambda: hot.encode(resident))
    for _ in range(2):
        fwd()
    sync_all()
    e0.record()
    for _ in range(args.steps):
        fwd()
    e1.record()
    sync_all()
    ms_fwd = max_over_ranks(e0.elapsed_time(e1))

    # ---- roofline of the dominant kernel family (separate profiled pass: CUDA events around every GEMM / attention launch)
    roofline, breakdown, attention = None, None, None
    prof_steps = 3
    lib.coot_set_single_stream(1)  # every kernel timed alone on one stream (eager, no graph): durations are per-kernel, not overlapped
    lib.coot_profile_enable(1 if rank == 0 else 0)
    prof_step = step_resident if args.api == "autograd" else (lambda: hot._step_body(resident, clip_idx, sent_idx))
    for _ in range(prof_steps):  # every rank runs the steps (they contain collectives); only rank 0 records events
        prof_step()
    th.cuda.synchronize()
    lib.coot_profile_enable(0)
    lib.coot_set_single_stream(0)
    if rank == 0:
        import ctypes
        ntags = 16
        ms_by = (ctypes.c_float * ntags)()
        cnt_by = (ctypes.c_int * ntags)()
        lib.coot_profile_collect(ms_by, cnt_by, ntags)
        names = ["other", "gemm_inputfc", "gemm_nn", "gemm_tt", "gemm_tt_inputfc", "attn_fwd", "attn_bwd"]
        breakdown = {n: {"ms_per_step": ms_by[i] / prof_steps, "launches_per_step": cnt_by[i] / prof_steps} for i, n in enumerate(names)}
        fam = family_work(host, wl, max_clips)
        roofline, attention = roofline_blocks(breakdown, fam, ms / args.steps)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, sample, _, kind = cpu_reference_time(wl, 2, 1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "host": host_core_info()}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate; losses fp32)", "data": "synthetic",
                "config": workload_config(wl, world, h2d_padded_bytes), "clocks": clocks,
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                        "h2d_padded_bytes_per_step": h2d_padded_bytes,
                        "staging": ("packed valid rows stored as IEEE fp16 in pinned host memory (data.PackedFeatureStore, converted once at "
                                    "preload; SURVEY 8f-2), widened to fp32 by the first kernel" if packed else
                                    "padded tensors, cudaMemcpyAsync" if args.padded_h2d else
                                    "valid rows of the padded pinned fp32 feature tensors only (coot_stage_valid_rows)"),
                        "feature_storage": "fp16_packed" if packed else "fp32",
                        "ms_per_step": ms_e2e / args.steps,
                        "host_cpus_bound_to_gpu_numa_node": numa_cpus},
                "gpu_launches": int(launches_per_step * args.steps), "gpu_launches_per_step": launches_per_step, "api": args.api,
                "dp_graph_mode": getattr(hot, "dp_graph_mode", None) if world > 1 else None,
                "forward_only": {"value": pairs_local * world * args.steps / (ms_fwd * 1e-3), "unit": UNIT, "ms_per_step": ms_fwd / args.steps},
                "roofline": roofline, "attention": attention if rank == 0 else None, "cpu_baseline": cpu, "breakdown": breakdown, "loss": float(loss), "pairs_per_step": pairs_local * world}
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        emit(line)
    if world > 1:
        # captured graphs hold NCCL kernels: drop them before leaving, and leave without waiting for communicator destruction
        # (observed to block after single-graph data-parallel capture)
        if hasattr(hot, "release_graphs"):
            hot.release_graphs()
        th.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def run_cfg5(args):
    """BASELINE.json configs[4]: global-batch contrastive sweep.  N gathered (im, s) pairs of dim D, sharded over the ranks
    (nl = N / world rows each).  A step = all-gather of both embedding matrices (NCCL over NVLink) + the tensor-core contrastive
    loss with its gradient for this rank's rows (csrc/losses_tc5.cu) + all-reduce of the loss value.  Reports the step rate, the
    loss kernel alone against the tensor roofline (algorithmic FLOPs: scores 2 x (2 nl N D) + gradient products 2 x (2 nl N D)),
    and the all-gather alone against its bytes."""
    import torch as th
    import torch.distributed as dist
    from coot_videotext_b200 import build as B
    m = __import__("re").match(r"cfg5_loss_n([\d,]+)(?:_d(\d+))?$", args.workload)
    sizes, d = [int(x) for x in m.group(1).split(",") if x], int(m.group(2) or 384)  # "cfg5_loss_n1024,4096": a sweep in one process
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    th.cuda.set_device(local_rank)
    dev = th.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        B.build()
    if world > 1:
        dist.barrier()
    from coot_videotext_b200 import lib as L
    lib = L.load()
    for n in sizes:
        _cfg5_one(args, n, d, world, rank, local_rank, dev, lib, L)
    if world > 1:
        th.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def _cfg5_one(args, n, d, world, rank, local_rank, dev, lib, L):
    """One size of the sweep: one JSON line."""
    import torch as th
    import torch.distributed as dist
    nl = n // world
    g = th.Generator().manual_seed(1234 + rank)
    a = th.nn.functional.normalize(th.randn(nl, d, generator=g)).to(dev)
    b = th.nn.functional.normalize(0.6 * a.cpu() + 0.8 * th.nn.functional.normalize(th.randn(nl, d, generator=g))).to(dev)
    send = th.cat([a, b], dim=1).contiguous()                      # ONE all-gather of [im | s] rows
    recv = th.empty(world * nl, 2 * d, device=dev)
    im, s = th.empty(n, d, device=dev), th.empty(n, d, device=dev)
    loss = th.zeros((), device=dev)
    d_im, d_s = th.empty(nl, d, device=dev), th.empty(nl, d, device=dev)
    ws = th.empty(int(lib.coot_contrastive_tc_ws_bytes(n, nl, d)), dtype=th.uint8, device=dev)

    def gather():
        if world > 1:
            dist.all_gather_into_tensor(recv, send)
        else:
            recv.copy_(send)
        im.copy_(recv[:, :d])
        s.copy_(recv[:, d:])

    def loss_step():
        loss.zero_()
        L.check(lib.coot_contrastive_sharded_tc(L.ptr(im), L.ptr(s), n, d, rank * nl, nl, 0.2, 1.0, L.ptr(loss), L.ptr(d_im), L.ptr(d_s),
                                                L.ptr(ws), ws.numel(), L.stream_ptr()), "contrastive_sharded_tc")

    def step():
        gather()
        loss_step()
        if world > 1:
            dist.all_reduce(loss)

    def timed(fn, k):
        for _ in range(max(args.warmup, 3)):
            fn()
        th.cuda.synchronize()
        if world > 1:
            dist.barrier()
            th.cuda.synchronize()
        e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        th.cuda.synchronize()
        t = th.tensor([e0.elapsed_time(e1) / k], dtype=th.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local_rank)
    if rank == 0 and not args.no_clocks:
        sampler.start()
    ms = timed(step, args.steps)
    clocks = sampler.stop() if (rank == 0 and not args.no_clocks) else None
    ms_gather = timed(gather, args.steps)
    ms_loss = timed(loss_step, args.steps)
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak = float(peaks.get("bf16_tflops", 1590.0))  # burst figure: the kernel is timed alone
        flops = 4.0 * 2.0 * nl * n * d  # two passes (row block, column block) x (score tile + gradient product), per rank
        gather_bytes = (world - 1) * nl * 2 * d * 4
        line = {"metric": "contrastive pairs/sec (loss + gradient over N gathered pairs)", "value": n / (ms * 1e-3), "unit": "pairs/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16x3 scores (exact fp32 near the margin), bf16x3 gradient product",
                "data": "synthetic", "config": {"workload": f"cfg5_loss_n{n}" + (f"_d{d}" if d != 384 else ""), "N": n, "D": d, "rows_per_gpu": nl, "parallelism": f"dp{world}",
                                                "l2": "operands re-streamed per tile; no explicit flush (N x D fp32+split = %.0f MB)" % (n * d * 10 / 1e6)},
                "clocks": clocks, "gpu_launches": 5 * args.steps,
                "e2e": None,
                "roofline": {"bound": "tensor", "kernel": "k_contr_tc5 (+ diag, diag-fix, split)", "achieved": flops / (ms_loss * 1e-3) / 1e12,
                             "peak": peak, "unit": "TFLOP/s", "frac": flops / (ms_loss * 1e-3) / 1e12 / peak, "traffic": None,
                             "algorithmic_flops_per_rank": flops, "ms_loss_only": ms_loss,
                             "note": "algorithmic FLOPs 1x per product (the tensor pipe does 3x for the scores, 3x for the 3-plane gradient product)"},
                "all_gather": {"ms": ms_gather, "bytes_received_per_rank": gather_bytes,
                               "gbs_per_rank": gather_bytes / (ms_gather * 1e-3) / 1e9 if world > 1 else None,
                               "nvlink_peak_gbs_per_direction": 770.0},
                "loss": float(loss)}
        emit(line)


def main():
    args = parse_args()
    if args.workload.startswith("cfg5_loss_n"):
        return run_cfg5(args)
    from coot_videotext_b200 import synthetic as syn
    wl = syn.WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    elif args.impl == "torch_cuda":
        run_torch_cuda(args, wl)
    else:
        run_b200(args, wl)


if __name__ == "__main__":
    main()
