"""ORACLE (test infrastructure): deterministic, platform-independent synthetic checkpoints.

The reference ships no weights (.gitignore:3-9 excludes *.pth). Parity runs therefore need a
state_dict that can be regenerated bit-identically on the build container (where the real
reference is imported to make golden outputs) and on the GPU box (where only this repo exists).
`make_state_dict(spec, seed)` fills every tensor of a reference-format state_dict from a numpy
RandomState keyed by crc32(name) ^ seed; `spec` is the (name, shape, dtype) list dumped from the
reference module itself by make_golden.py into tests/golden/<model>_x<scale>.spec.json.
"""
from __future__ import annotations

import json
import os
import zlib

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# per-model gain on conv/linear weights, chosen so the network branch is O(0.1..1) next to the
# interpolation skip (tune with oracle/make_golden.py --stats)
GAIN = {"MyEfficientLFNet": 0.7, "EPIT": 0.6, "DistgSSR": 0.6, "LF_InterNet": 0.55, "MyEfficientLFNetV4_5": 0.7}


# the patch-pipeline goldens of make_golden.py, split by key prefix so that every file stays under 1 MB
PIPELINE_GOLDENS = {"pipeline.npz": ("div_",),                   # LFdivide
                    "pipeline_tail.npz": ("int_", "met_")}       # LFintegrate, cal_metrics


def save_pipeline_golden(pipe: dict) -> None:
    assert all(k.startswith(sum(PIPELINE_GOLDENS.values(), ())) for k in pipe), "a key without a file"
    for fname, prefixes in PIPELINE_GOLDENS.items():
        np.savez_compressed(os.path.join(GOLDEN_DIR, fname), **{k: v for k, v in pipe.items() if k.startswith(prefixes)})


def load_pipeline_golden() -> dict:
    out = {}
    for fname in PIPELINE_GOLDENS:
        with np.load(os.path.join(GOLDEN_DIR, fname)) as g:
            out.update({k: g[k] for k in g.files})
    return out


def spec_path(model: str, scale: int) -> str:
    return os.path.join(GOLDEN_DIR, f"{model}_x{scale}.spec.json")


def load_spec(model: str, scale: int):
    with open(spec_path(model, scale)) as f:
        return [(n, tuple(s), d) for n, s, d in json.load(f)]


def _fill(name: str, shape, dtype: str, seed: int, gain: float) -> torch.Tensor:
    rs = np.random.RandomState((zlib.crc32(name.encode()) ^ (seed * 2654435761)) & 0xFFFFFFFF)
    if dtype == "int64":
        return torch.zeros(shape, dtype=torch.int64)
    leaf = name.rsplit(".", 1)[-1]
    if leaf == "running_var":
        a = rs.uniform(0.5, 1.5, shape)
    elif leaf == "running_mean":
        a = rs.normal(0.0, 0.1, shape)
    elif len(shape) >= 2:
        fan_in = int(np.prod(shape[1:]))
        b = gain * np.sqrt(3.0 / fan_in)
        a = rs.uniform(-b, b, shape)
    elif leaf == "weight":          # BatchNorm / LayerNorm scale
        a = rs.uniform(0.8, 1.2, shape)
    elif leaf == "bias":
        a = rs.normal(0.0, 0.05, shape)
    elif leaf == "scale":           # LightweightAngularAttention.scale (MyEfficientLFNet.py:252)
        a = rs.uniform(0.05, 0.2, shape)
    else:                           # e.g. SAModulator.combine
        a = rs.normal(0.5, 0.3, shape)
    return torch.from_numpy(np.asarray(a, dtype=np.float32).reshape(shape))


def make_state_dict(model: str, scale: int, seed: int = 1234, spec=None) -> dict:
    spec = spec if spec is not None else load_spec(model, scale)
    g = GAIN.get(model, 1.0)
    return {n: _fill(n, s, d, seed, g) for n, s, d in spec}


def synthetic_patches(batch: int, ang: int = 5, patch: int = 32, seed: int = 0) -> torch.Tensor:
    """uniform [0,1) Y-channel SAI mosaics [B,1,A*P,A*P] (SURVEY.md 8d), numpy-seeded."""
    rs = np.random.RandomState(seed)
    return torch.from_numpy(rs.random_sample((batch, 1, ang * patch, ang * patch)).astype(np.float32))
