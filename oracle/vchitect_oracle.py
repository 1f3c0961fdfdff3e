"""TEST INFRASTRUCTURE ONLY -- CPU/torch restatement of the Vchitect-2.0 transformer (VchitectXLTransformerModel).

Follows models/transformers/vchitect_transformer_3d.py (JointTransformerBlock.forward :116-178, model forward :478-601)
and models/modules/attentions.py (VchitectAttnProcessor :641-949: apply_rotary_emb :688-701, spatial_attn :663-705,
temporal_attention :707-768, cross_attention :770-803, __call__ :805-927), sp_size == 1, PAB via the callback gates.

Pinning (tests/test_oracle_vs_reference.py, against stored outputs of the reference): ``attention`` (the whole processor on a
VchitectAttention's parameters) bit for bit against the reference's own VchitectAttention + VchitectAttnProcessor, incl. the PAB gates
(test_vchitect_attention_vs_reference, test_vchitect_attention_pab_vs_reference); ``transformer_forward`` against the
reference's VchitectXLTransformerModel executed unmodified (test_vchitect_oracle_vs_reference_model: fp32 within summation
order, bf16 bit for bit).  diffusers==0.30.0 is not installed here: for that run oracle/ref_loader.load_vchitect supplies the
five leaf classes the reference file imports from it, restated from their published semantics -- AdaLayerNormZero,
AdaLayerNormContinuous, GELU (tanh), PatchEmbed (cropped 2-D sin-cos table), CombinedTimestepTextProjEmbeddings
(Timesteps(256, flip) + TimestepEmbedding + PixArtAlphaTextProjection(silu)).  Those five leaves are restated here a second
time; everything between them is the reference's own code.
"""
import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


def _lin(sd, p, x):
    return F.linear(x, sd[p + ".weight"], sd[p + ".bias"])


def _ln(x: Tensor, eps: float = 1e-6) -> Tensor:
    return F.layer_norm(x, (x.shape[-1],), None, None, eps)


def freqs_cis(dim: int, end: int, theta: float = 1e6, rope_scaling_factor: float = 1.0) -> Tensor:
    """VchitectXLTransformerModel.precompute_freqs_cis (:331-338), complex64 [end, dim/2]."""
    freqs = 1.0 / (theta ** (torch.arange(0, dim, 2)[: (dim // 2)].float() / dim))
    t = torch.arange(end, dtype=torch.float) / rope_scaling_factor
    freqs = torch.outer(t, freqs).float()
    return torch.polar(torch.ones_like(freqs), freqs)


def apply_rotary_emb(xq: Tensor, xk: Tensor, fc: Tensor):
    """attentions.py:688-701; xq/xk [B', T, H, D], fc [T, D/2] complex."""
    xq_ = torch.view_as_complex(xq.float().reshape(*xq.shape[:-1], -1, 2))
    xk_ = torch.view_as_complex(xk.float().reshape(*xk.shape[:-1], -1, 2))
    f = fc.view(1, xq_.shape[1], 1, xq_.shape[-1])
    return torch.view_as_real(xq_ * f).flatten(3).type_as(xq), torch.view_as_real(xk_ * f).flatten(3).type_as(xk)


def _sdpa(q, k, v):
    return F.scaled_dot_product_attention(q, k, v, dropout_p=0.0, is_causal=False)


def attention(sd: Dict[str, Tensor], p: str, hidden: Tensor, enc: Tensor, fc: Tensor, heads: int, frames: int,
              context_pre_only: bool, gate=None, cache: Optional[dict] = None):
    """VchitectAttnProcessor.__call__ for batchsize 1: hidden [F, S, C], enc [F, L, C]; returns (video, text).
    gate(kind) -> bool (reuse the cached tensor), cache: dict the reference keeps on the attention module."""
    Fr, S, C = hidden.shape
    D = C // heads
    eq, ek, ev = _lin(sd, p + "add_q_proj", enc), _lin(sd, p + "add_k_proj", enc), _lin(sd, p + "add_v_proj", enc)
    cache = {} if cache is None else cache

    # temporal (:707-768)
    if gate is not None and gate("temporal"):
        hid_t, enc_t = cache["temporal"]
    else:
        q = torch.cat([_lin(sd, p + "to_q_temp", hidden), eq], 1).view(Fr, -1, heads, D)
        k = torch.cat([_lin(sd, p + "to_k_temp", hidden), ek], 1).view(Fr, -1, heads, D)
        v = torch.cat([_lin(sd, p + "to_v_temp", hidden), ev], 1).view(Fr, -1, heads, D)
        q, k, v = (t.transpose(0, 1) for t in (q, k, v))  # "(B T) S H C -> (B S) T H C", B = 1
        q, k = apply_rotary_emb(q, k, fc[:Fr])
        o = _sdpa(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2))  # [N, H, F, D]
        o = o.transpose(1, 2).reshape(-1, Fr, C).to(v.dtype).transpose(0, 1)  # "(B S) T C -> (B T) S C"
        hid_t, enc_t = _lin(sd, p + "to_out_temporal", o[:, :S]), o[:, S:]
        if gate is not None:
            cache["temporal"] = (hid_t, enc_t)

    # cross (:770-803): frame 0's text keys / values for every query
    if gate is not None and gate("cross"):
        cross = cache["cross"]
    else:
        qc = torch.cat([_lin(sd, p + "to_q_cross", hidden), eq], 1).view(Fr, -1, heads, D)
        N = qc.shape[1]
        qy = qc.permute(1, 0, 2, 3).reshape(1, N * Fr, heads, D)  # "(B T) S H C -> B (S T) H C"
        ky, vy = ek[0].view(1, -1, heads, D), ev[0].view(1, -1, heads, D)
        o = _sdpa(qy.transpose(1, 2), ky.transpose(1, 2), vy.transpose(1, 2))
        o = o.transpose(1, 2).reshape(1, N, Fr, C).to(qc.dtype)[0].transpose(0, 1)  # "B (S T) C -> (B T) S C"
        cross = _lin(sd, p + "to_out_context", o)
        if gate is not None:
            cache["cross"] = cross

    # spatial (:663-705)
    if gate is not None and gate("spatial"):
        sp = cache["spatial"]
    else:
        q = torch.cat([_lin(sd, p + "to_q", hidden), eq], 1).view(Fr, -1, heads, D)
        k = torch.cat([_lin(sd, p + "to_k", hidden), ek], 1).view(Fr, -1, heads, D)
        v = torch.cat([_lin(sd, p + "to_v", hidden), ev], 1).view(Fr, -1, heads, D)
        sp = _sdpa(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2)).transpose(1, 2).reshape(Fr, -1, C).to(q.dtype)
        if gate is not None:
            cache["spatial"] = sp

    mix = sp * 1.1 + cross  # :897
    hv, he = mix[:, :S], mix[:, S:]
    hv = _lin(sd, p + "to_out.0", hv)
    if Fr == 1:
        hid_t = hid_t * 0
    hv = hv + hid_t
    if not context_pre_only:
        he = _lin(sd, p + "to_add_out", he)
    et = _lin(sd, p + "to_add_out_temporal", enc_t)
    if Fr == 1:
        et = et * 0
    return hv, he + et


def feed_forward(sd, p, x):
    h = F.gelu(_lin(sd, p + "net.0.proj", x), approximate="tanh")
    return _lin(sd, p + "net.2", h)


def ada_zero(sd, p, x, temb):
    """diffusers AdaLayerNormZero.forward(x, emb=temb)."""
    emb = _lin(sd, p + "linear", F.silu(temb))
    sh, sc, g, sh2, sc2, g2 = emb.chunk(6, dim=1)
    return _ln(x) * (1 + sc[:, None]) + sh[:, None], g, sh2, sc2, g2


def ada_continuous(sd, p, x, cond):
    """diffusers AdaLayerNormContinuous.forward: scale first, then shift."""
    emb = _lin(sd, p + "linear", F.silu(cond).to(x.dtype))
    sc, sh = torch.chunk(emb, 2, dim=1)
    return _ln(x) * (1 + sc)[:, None, :] + sh[:, None, :]


def block(sd, p, hidden, enc, temb, fc, heads, frames, context_pre_only, gate=None, cache=None):
    """JointTransformerBlock.forward (:116-178); temb [F, C]."""
    nh, g_msa, sh_mlp, sc_mlp, g_mlp = ada_zero(sd, p + "norm1.", hidden, temb)
    if context_pre_only:
        ne = ada_continuous(sd, p + "norm1_context.", enc, temb)
    else:
        ne, c_g_msa, c_sh_mlp, c_sc_mlp, c_g_mlp = ada_zero(sd, p + "norm1_context.", enc, temb)
    a, ca = attention(sd, p + "attn.", nh, ne, fc, heads, frames, context_pre_only, gate, cache)
    hidden = hidden + g_msa.unsqueeze(1) * a
    nh = _ln(hidden) * (1 + sc_mlp[:, None]) + sh_mlp[:, None]
    hidden = hidden + g_mlp.unsqueeze(1) * feed_forward(sd, p + "ff.", nh)
    if context_pre_only:
        return None, hidden
    enc = enc + c_g_msa.unsqueeze(1) * ca
    ne = _ln(enc) * (1 + c_sc_mlp[:, None]) + c_sh_mlp[:, None]
    enc = enc + c_g_mlp.unsqueeze(1) * feed_forward(sd, p + "ff_context.", ne)
    return enc, hidden


# ---- diffusers embedders, restated (PARITY UNPINNED) ----------------------------------------------------------------------
def _sincos_1d(embed_dim, pos):
    omega = 1.0 / 10000 ** (torch.arange(embed_dim // 2, dtype=torch.float64) / (embed_dim / 2.0))
    out = pos.reshape(-1).double()[:, None] * omega[None]
    return torch.cat([out.sin(), out.cos()], dim=1)


def pos_embed_2d(embed_dim, grid_size, base_size):
    g = torch.arange(grid_size, dtype=torch.float32) / (grid_size / base_size)
    gw, gh = torch.meshgrid(g, g, indexing="xy")
    return torch.cat([_sincos_1d(embed_dim // 2, gw), _sincos_1d(embed_dim // 2, gh)], dim=1).float()


def time_text_embed(sd, p, timestep, pooled):
    half = 128
    e = timestep[:, None].float() * torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32) / half)[None]
    tp = torch.cat([e.cos(), e.sin()], dim=-1).to(pooled.dtype)
    t = _lin(sd, p + "timestep_embedder.linear_2", F.silu(_lin(sd, p + "timestep_embedder.linear_1", tp)))
    y = _lin(sd, p + "text_embedder.linear_2", F.silu(_lin(sd, p + "text_embedder.linear_1", pooled)))
    return t + y


def transformer_forward(sd, cfg: dict, latents: Tensor, enc: Tensor, pooled: Tensor, timestep: Tensor, gate=None,
                        caches: Optional[list] = None) -> Tensor:
    """VchitectXLTransformerModel.forward (:478-601), batch 1.  latents [1, F, Cin, H, W] -> [F, Cout, H, W].
    cfg: heads, head_dim, layers, patch, sample_size, pos_embed_max_size, out_channels."""
    heads, D, p = cfg["heads"], cfg["head_dim"], cfg["patch"]
    C = heads * D
    B, Fr, Cin, Hh, Ww = latents.shape
    dt = sd["proj_out.weight"].dtype
    x = F.conv2d(latents.to(dt).reshape(Fr, Cin, Hh, Ww), sd["pos_embed.proj.weight"], sd["pos_embed.proj.bias"], stride=p)
    x = x.flatten(2).transpose(1, 2)
    m, h, w = cfg["pos_embed_max_size"], Hh // p, Ww // p
    top, left = (m - h) // 2, (m - w) // 2
    pe = sd["pos_embed.pos_embed"].reshape(1, m, m, -1)[:, top : top + h, left : left + w].reshape(1, h * w, -1)
    hidden = (x + pe).to(x.dtype)
    fc = freqs_cis(D, max(Fr, 2), theta=1e6, rope_scaling_factor=cfg.get("rope_scaling_factor", 1.0))
    temb = time_text_embed(sd, "time_text_embed.", timestep, pooled.to(dt))
    e = _lin(sd, "context_embedder", enc.to(dt))
    cur = temb.repeat(Fr, 1)
    for i in range(cfg["layers"]):
        g = (lambda kind, i=i: gate(i, kind)) if gate is not None else None
        e, hidden = block(sd, f"transformer_blocks.{i}.", hidden, e, cur, fc, heads, Fr, i == cfg["layers"] - 1, g,
                          None if caches is None else caches[i])
    hidden = ada_continuous(sd, "norm_out.", hidden, temb)
    hidden = _lin(sd, "proj_out", hidden)
    Co = cfg["out_channels"]
    hidden = hidden.reshape(hidden.shape[0], h, w, p, p, Co)
    hidden = torch.einsum("nhwpqc->nchpwq", hidden)
    return hidden.reshape(hidden.shape[0], Co, h * p, w * p)
