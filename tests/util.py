"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch as th

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = {"tiny": ("tiny_s1234_p7.npz", 1234, 7, 99), "small": ("small_s4321_p11.npz", 4321, 11, 5),
                # real feature dims of BASELINE.json configs[1] / configs[3] (K = 1024 / 1536 / 3072 input FC, 512-frame sequences)
                "anet_sub": ("anet_sub_s2468_p13.npz", 2468, 13, 17), "yc2_long": ("yc2_long_s1357_p19.npz", 1357, 19, 23)}
GRAD_SAMPLES = 512


def hash_name(name: str) -> int:
    h = 2166136261
    for ch in name.encode():
        h = ((h ^ ch) * 16777619) & 0xFFFFFFFF
    return h


def grad_sample_index(name: str, numel: int, samples: int = GRAD_SAMPLES) -> np.ndarray:
    rng = np.random.default_rng(abs(hash_name(name)) % (2 ** 32))
    return rng.integers(0, numel, size=min(samples, numel))


def rel_inf(a, b) -> float:
    """The tolerance metric of SURVEY.md section 8d: ||a-b||_inf / max(||b||_inf, tiny)."""
    a = th.as_tensor(a).double()
    b = th.as_tensor(b).double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def load_golden(case: str):
    fname, data_seed, param_seed, cc_seed = GOLDEN_CASES[case]
    return np.load(os.path.join(GOLDEN_DIR, fname)), data_seed, param_seed, cc_seed


# ---------------------------------------------------------------- dropout mask mirror of csrc/common.cuh drop_hash()
def drop_hash_np(seed: int, site: int, rows: np.ndarray, cols: np.ndarray) -> np.ndarray:
    """Bit-exact numpy mirror of drop_hash = drop_bits(drop_row_base(seed, site, row), col) (uint32 wrap-around arithmetic)."""
    M = np.uint64(0xFFFFFFFF)
    rows = rows.astype(np.uint64)
    cols = cols.astype(np.uint64)
    h = np.uint64((seed ^ ((site * 0x9E3779B9) & 0xFFFFFFFF)) & 0xFFFFFFFF)
    h = np.broadcast_to(h, np.broadcast(rows, cols).shape).astype(np.uint64)
    h = h ^ ((rows + np.uint64(0x7F4A7C15) + ((h << np.uint64(6)) & M) + (h >> np.uint64(2))) & M)
    h = h ^ (h >> np.uint64(16))
    h = (h * np.uint64(0x85EBCA6B)) & M
    h = h ^ (h >> np.uint64(13))
    h = (h * np.uint64(0xC2B2AE35)) & M
    h = h ^ (h >> np.uint64(16))  # row base
    h = ((h ^ cols) * np.uint64(0x9E3779B1)) & M
    h = h ^ (h >> np.uint64(15))
    h = (h * np.uint64(0x85EBCA6B)) & M
    h = h ^ (h >> np.uint64(13))
    return h.astype(np.uint32)


def make_mask_fn(seed: int):
    """mask_fn(site_id, rows, cols, p) for oracle.DropCtx: the multiplicative masks (0 or 1/(1-p)) of the CUDA path."""
    def fn(site_id, rows, cols, p):
        if p <= 0:
            return th.ones(th.broadcast_shapes(rows.shape, cols.shape))
        thresh = min(int(p * 4294967296.0), 4294967295)
        h = drop_hash_np(seed, site_id, rows.numpy(), cols.numpy())
        return th.from_numpy(np.where(h < np.uint32(thresh), 0.0, 1.0 / (1.0 - np.float32(p))).astype(np.float32))
    return fn
