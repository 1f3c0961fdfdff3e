"""TEST INFRASTRUCTURE ONLY -- Dynamic Sequence Parallelism reshard, restated as single-process index math.

The reference's comm layer cannot run on CPU (gloo has no list all_to_all; the gather asserts CUDA:
core/distributed/comm.py:107,181), so the DSP oracle is the invariant the reference relies on:
every per-rank tensor is a slice of the zero-padded full tensor (SURVEY.md Appendix E).  Pinned in
tests/test_oracle_vs_reference.py against the outputs of the reference's own functions run on simulated ranks
(threads + a fake ``dist``, oracle/gen_golden_pins.py).
"""
from typing import List

import torch


def pad_amount(n: int, sp: int) -> int:
    """set_pad: core/distributed/comm.py:271-275."""
    return (sp - n % sp) % sp


def split_sequence(x: torch.Tensor, sp: int, dim: int, pad_val: float = 0.0) -> List[torch.Tensor]:
    """_split_sequence_func for every rank: comm.py:148-167 (pad at the end, equal chunks)."""
    p = pad_amount(x.shape[dim], sp)
    if p:
        shp = list(x.shape)
        shp[dim] = p
        x = torch.cat([x, torch.full(shp, pad_val, dtype=x.dtype)], dim=dim)
    return [c.contiguous() for c in torch.chunk(x, sp, dim=dim)]


def gather_sequence(parts: List[torch.Tensor], dim: int, pad: int) -> torch.Tensor:
    """_gather_sequence_func: comm.py:170-190."""
    out = torch.cat(parts, dim=dim)
    return out.narrow(dim, 0, out.shape[dim] - pad) if pad else out


def all_to_all_with_pad(parts: List[torch.Tensor], scatter_dim: int, gather_dim: int, scatter_pad: int, gather_pad: int):
    """all_to_all_with_pad + _all_to_all_func on all ranks at once: comm.py:282-304,104-108.

    parts[r] is rank r's local tensor; returns the list of per-rank outputs."""
    sp = len(parts)
    padded = []
    for x in parts:
        if scatter_pad:
            shp = list(x.shape)
            shp[scatter_dim] = scatter_pad
            x = torch.cat([x, torch.zeros(shp, dtype=x.dtype)], dim=scatter_dim)
        padded.append(torch.tensor_split(x, sp, scatter_dim))
    outs = []
    for r in range(sp):
        o = torch.cat([padded[src][r] for src in range(sp)], dim=gather_dim).contiguous()
        if gather_pad:
            o = o.narrow(gather_dim, 0, o.shape[gather_dim] - gather_pad)
        outs.append(o)
    return outs


def dynamic_switch(parts: List[torch.Tensor], T: int, S: int, to_spatial_shard: bool):
    """STDiT3Block.dynamic_switch for video (T > 1): open_sora_transformer_3d.py:288-315.

    parts[r]: [B, t*s, C] in the current layout; T, S are the *global* frame/patch counts."""
    sp = len(parts)
    tp, spd = pad_amount(T, sp), pad_amount(S, sp)
    if to_spatial_shard:  # [B, Tp/sp, S, C] -> [B, T, Sp/sp, C]
        t_loc = (T + tp) // sp
        xs = [p.reshape(p.shape[0], t_loc, S, p.shape[-1]) for p in parts]
        outs = all_to_all_with_pad(xs, 2, 1, spd, tp)
    else:  # [B, T, Sp/sp, C] -> [B, Tp/sp, S, C]
        s_loc = (S + spd) // sp
        xs = [p.reshape(p.shape[0], T, s_loc, p.shape[-1]) for p in parts]
        outs = all_to_all_with_pad(xs, 1, 2, tp, spd)
    new_t, new_s = outs[0].shape[1], outs[0].shape[2]
    return [o.reshape(o.shape[0], new_t * new_s, o.shape[-1]) for o in outs], new_s, new_t
