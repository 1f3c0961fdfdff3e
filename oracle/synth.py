"""TEST INFRASTRUCTURE ONLY -- deterministic synthetic tensors (no torch RNG).

A counter-based integer hash (splitmix64 finaliser, all uint64 numpy arithmetic) so that the same
(name, shape) yields bit-identical values in the authoring container (where the reference generates
the golden outputs) and on the GPU box (where the tests regenerate the inputs and weights).
"""
import zlib

import numpy as np
import torch

_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)
_GOLD = np.uint64(0x9E3779B97F4A7C15)


def _mix(z):
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
        return z ^ (z >> np.uint64(31))


def uniform(name: str, shape, lo=-1.0, hi=1.0) -> torch.Tensor:
    """float32 tensor, uniform in [lo, hi), a pure function of (name, shape)."""
    n = int(np.prod(shape)) if len(shape) else 1
    seed = np.uint64(zlib.crc32(name.encode()) | (1 << 40))
    with np.errstate(over="ignore"):
        ctr = (np.arange(n, dtype=np.uint64) + np.uint64(1)) * _GOLD + seed * _M2
    bits = _mix(ctr) >> np.uint64(40)  # 24 random bits: exactly representable in float32
    u = bits.astype(np.float64) / float(1 << 24)
    out = (lo + (hi - lo) * u).astype(np.float32).reshape(shape)
    return torch.from_numpy(out)


def normalish(name: str, shape, std=1.0) -> torch.Tensor:
    """Sum of 4 uniforms (variance-matched), roughly bell-shaped, bounded: a stand-in for N(0, std)."""
    acc = sum(uniform(f"{name}#{i}", shape, -1.0, 1.0) for i in range(4))
    return acc * (std * (3.0 / 4.0) ** 0.5)


def copied(k: str, v: torch.Tensor) -> bool:
    """The entries fill_state_dict keeps as they are: integer buffers and rotary frequency tables."""
    return not torch.is_floating_point(v) or k.endswith("rope.freqs") or k.endswith("inv_freq")


def fill_state_dict(sd: dict, tag: str, weight_std: float = 0.05) -> dict:
    """Deterministic weights for every floating tensor of a STDiT3-style state_dict (keeps dtypes).

    Norm weights get ~1, biases and modulation tables small non-zero values, matrices std=weight_std,
    so that no path is multiplied by zero (the reference zero-inits temporal proj/fc2,
    open_sora_transformer_3d.py:508-511, which would hide those kernels from a parity test).
    """
    out = {}
    for k, v in sd.items():
        if copied(k, v):
            out[k] = v.clone()
            continue
        if k.endswith("q_norm.weight") or k.endswith("k_norm.weight"):
            w = 1.0 + 0.2 * uniform(tag + k, tuple(v.shape))
        elif k.endswith(".bias"):
            w = 0.1 * uniform(tag + k, tuple(v.shape))
        elif k.endswith("scale_shift_table"):
            w = normalish(tag + k, tuple(v.shape), std=0.3)
        elif k.endswith("y_embedding"):
            w = normalish(tag + k, tuple(v.shape), std=0.1)
        else:
            w = normalish(tag + k, tuple(v.shape), std=weight_std)
        out[k] = w.to(v.dtype)
    return out
