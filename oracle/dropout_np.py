"""ORACLE (test infrastructure, never shipped or timed as the product): the head trainer's dropout masks restated in
numpy, so a float64 reference step can use exactly the elements the device dropped.

Port of vmb::dropout_scale (csrc/igemm_sm100.cuh) with explicit uint32 arithmetic: a murmur3 fmix32 over the element
index keyed by (seed, layer).  Activation (level l, Linear j) of a step is dropped under layer id 1 + l * 4 + j, its
element (clip b, time step t, feature c) has index (b * T + t) * H + c, and it is kept when u >= p in float32, with
u = (h >> 8) * 2^-24; a kept element is scaled by 1 / (1 - p) computed in float32.
"""
from __future__ import annotations

import numpy as np

MAX_FC = 4                 # kMaxFc of csrc/mla_train.cu: the layer id stride between levels

_M = np.uint64(0xFFFFFFFF)


def _u32(v) -> np.ndarray:
    return (np.asarray(v, dtype=np.uint64) & _M).astype(np.uint32)


def layer_id(level: int, j: int) -> int:
    return 1 + level * MAX_FC + j


def dropout_scale(seed: int, layer: int, idx: np.ndarray, p: float) -> np.ndarray:
    """float32 inverted-dropout scale (1 / (1 - p) or 0) of elements `idx` (uint64 array) of layer `layer`."""
    idx = np.asarray(idx, dtype=np.uint64)
    p32 = np.float32(p)
    if p32 <= 0:
        return np.ones(idx.shape, np.float32)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    with np.errstate(over="ignore"):
        key = (np.uint32(seed & 0xFFFFFFFF) ^ (np.uint32(seed >> 32) * np.uint32(0x9E3779B1)) ^
               (np.uint32(layer) * np.uint32(0x85EBCA77) + np.uint32(0xC2B2AE3D)))
        h = (_u32(idx) ^ key) * np.uint32(0x9E3779B1) + _u32(idx >> np.uint64(32)) * np.uint32(0x27D4EB2F)
        h ^= h >> np.uint32(16)
        h *= np.uint32(0x85EBCA6B)
        h ^= h >> np.uint32(13)
        h *= np.uint32(0xC2B2AE35)
        h ^= h >> np.uint32(16)
    u = (h >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    keep = np.float32(1) / (np.float32(1) - p32)
    return np.where(u >= p32, keep, np.float32(0)).astype(np.float32)


def step_masks(seed: int, model_conf, batch: int, t_steps: int, hidden: int, p: float) -> dict:
    """{(level, j): float32 array (batch, t_steps, hidden)}: the scale every activation of one training step is
    multiplied by.  `seed` is the step's seed: HeadTrainer passes seed + step_count to step n (step_count counts the
    Adam steps taken so far), the module bridge a value drawn from torch's global generator per forward."""
    idx = np.arange(batch * t_steps * hidden, dtype=np.uint64)
    return {(l, j): dropout_scale(seed, layer_id(l, j), idx, p).reshape(batch, t_steps, hidden)
            for l, n_fc in enumerate(model_conf) for j in range(n_fc)}
