"""TEST INFRASTRUCTURE ONLY -- compact records of the reference's outputs and the checks against them.

tests/golden/reference_pins.pt.gz (written by oracle/gen_golden_pins.py from the unmodified reference) holds, per output:
  exact  -- shape, dtype and SHA-256 of the bytes: equal records <=> bit-identical tensors;
  close  -- a fixed strided sample of the values (all of them when there are few) and the sums of the values and of their
            magnitudes over each of PARTS contiguous parts of the flattened tensor.  allclose(got, want, rtol, atol) implies
            allclose on the sample and, per part of m values, |sum(got) - sum(want)| <= m * atol + rtol * sum(|want|) (the
            same for sum(|got|)), so both are checked: every value is in a part, a deviation confined to a few values moves
            its part's sums;
  rel    -- the headline model's criterion: ours-vs-fp32 within 1.3 x the reference's own bf16-vs-fp32 error, on the
            sample, and the norm of the output against the fp32 norm within that error over the whole tensor;
and per reference module whose state dict seeds synth.fill_state_dict a template: names with shapes and dtypes, plus the
tensors that fill_state_dict copies as they are (filled(template) rebuilds a state dict it fills identically).
"""
import gzip
import hashlib
import io

import torch

STRIDE = 7919  # prime: (i * STRIDE) % n are n distinct indices for every n it does not divide


def save(records, path):
    """torch.save, gzip-compressed (the many small records are mostly per-tensor container overhead)."""
    buf = io.BytesIO()
    torch.save(records, buf)
    with open(path, "wb") as f:
        f.write(gzip.compress(buf.getvalue(), compresslevel=9, mtime=0))


def load(path):
    with open(path, "rb") as f:
        return torch.load(io.BytesIO(gzip.decompress(f.read())))


def _idx(n, k):
    return torch.arange(min(n, k), dtype=torch.int64) * STRIDE % n


def template(sd):
    from . import synth

    return {k: v.detach().clone() if synth.copied(k, v) else (tuple(v.shape), str(v.dtype).split(".")[-1]) for k, v in sd.items()}


def filled(tmpl, tag):
    """synth.fill_state_dict on the state dict a template was taken from."""
    from . import synth

    sd = {k: v if torch.is_tensor(v) else torch.empty(v[0], dtype=getattr(torch, v[1]), device="meta") for k, v in tmpl.items()}
    return synth.fill_state_dict(sd, tag)


def exact(t):
    b = t.detach().cpu().contiguous().reshape(-1).view(torch.uint8).numpy().tobytes()
    return {"shape": tuple(t.shape), "dtype": str(t.dtype), "sha256": hashlib.sha256(b).hexdigest()}


def assert_exact(got, rec, what=""):
    g = exact(got)
    assert (g["shape"], g["dtype"]) == (rec["shape"], rec["dtype"]), (what, g, rec)
    assert g["sha256"] == rec["sha256"], f"{what}: not bit-identical to the reference's output"


PARTS = 64


def _part_sums(f):
    parts = f.double().tensor_split(min(PARTS, f.numel()))
    return (torch.tensor([p.sum().item() for p in parts], dtype=torch.float64),
            torch.tensor([p.abs().sum().item() for p in parts], dtype=torch.float64),
            torch.tensor([p.numel() for p in parts], dtype=torch.float64))


def close(t, k=256):
    f = t.detach().cpu().reshape(-1)
    s, a, _ = _part_sums(f)
    return {"shape": tuple(t.shape), "sample": f[_idx(f.numel(), k)].clone(), "part_sum": s, "part_abs_sum": a,
            "max_abs": f.double().abs().max().item()}


def assert_close(got, rec, rtol, atol, what=""):
    assert tuple(got.shape) == rec["shape"], (what, tuple(got.shape), rec["shape"])
    g = got.detach().cpu().reshape(-1)
    want = rec["sample"]
    s = g[_idx(g.numel(), want.numel())].to(want.dtype)
    assert torch.allclose(s, want, rtol=rtol, atol=atol), (what, (s - want).abs().max().item())
    gs, ga, m = _part_sums(g)
    assert gs.numel() == rec["part_sum"].numel(), (what, gs.numel(), rec["part_sum"].numel())
    bound = m * atol + (rtol + 1e-12) * rec["part_abs_sum"]
    for name, d in (("sum", gs - rec["part_sum"]), ("sum of magnitudes", ga - rec["part_abs_sum"])):
        i = int((d.abs() - bound).argmax())
        assert bool((d.abs() <= bound).all()), (what, f"{name} of part {i} of {d.numel()}", d[i].item(), bound[i].item())


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


def rel(w16, w32, k=512):
    i = _idx(w32.numel(), k)
    return {"shape": tuple(w32.shape), "w16": w16.reshape(-1)[i].clone(), "w32": w32.reshape(-1)[i].clone(),
            "rel16": _rel(w16, w32), "norm32": w32.double().norm().item()}


def assert_rel(got, rec, what="", factor=1.3, slack=1e-4):
    assert tuple(got.shape) == rec["shape"], (what, tuple(got.shape), rec["shape"])
    s = got.detach().cpu().reshape(-1)[_idx(got.numel(), rec["w32"].numel())]
    e_ours, e_ref = _rel(s, rec["w32"]), _rel(rec["w16"], rec["w32"])
    assert e_ours <= factor * e_ref + slack, (what, e_ours, e_ref)
    n = got.detach().cpu().double().norm().item()
    assert abs(n / rec["norm32"] - 1.0) <= factor * rec["rel16"] + slack, (what, n, rec["norm32"], rec["rel16"])
