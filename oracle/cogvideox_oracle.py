"""TEST INFRASTRUCTURE ONLY -- CPU/torch restatement of the CogVideoX transformer block (block level).

PINNED against the outputs of the reference's own CogVideoXTransformer3DModel, executed unmodified (tests/test_oracle_vs_reference.py::
test_cogvideox_oracle_vs_reference_model: fp32 within summation order, bf16 and fp16 bit for bit; also
test_cogvideox_layernorm_zero and the DDIM scheduler test).  ``diffusers==0.30.0`` (requirements.txt:25) is not installed
here; oracle/ref_loader.load_cogvideox supplies the leaf classes the reference file imports from it:
  * ``Attention(query_dim, heads, dim_head, qk_norm="layer_norm", eps=1e-6, bias, out_bias)`` = the reference's own vendored
    copy (VchitectAttention, models/modules/attentions.py:321-638: to_q/to_k/to_v Linears, ``norm_q``/``norm_k`` =
    nn.LayerNorm(dim_head, eps=1e-6), to_out[0]), driven by the in-tree CogVideoXAttnProcessor2_0 (:88-175);
  * ``FeedForward(dim, activation_fn="gelu-approximate", final_dropout=True, bias=True)`` = the vendored copy in
    open_sora_plan_v110_transformer_3d.py:1312-1367 (Linear -> tanh-GELU -> Linear);
  * ``Timesteps`` / ``TimestepEmbedding`` / GELU restated there (a few lines each);
  * ``get_3d_sincos_pos_embed`` = ``sincos_3d`` below: the one piece of this model that stays PARITY UNPINNED (restated from
    the library's published semantics; no copy of it exists in the reference tree).
2B configuration: no rotary embedding (use_rotary_positional_embeddings False), sp = 1.

``transformer_forward`` restates CogVideoXTransformer3DModel.forward (:479-589) around the block: CogVideoXPatchEmbed
(models/modules/embeddings.py:14-51), AdaLayerNorm (normalization.py:60-114), unpatchify (:578-581).
"""
import math
from typing import Dict

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


def layer_norm_zero(sd: Dict[str, Tensor], p: str, hidden: Tensor, enc: Tensor, temb: Tensor, eps: float = 1e-5):
    """CogVideoXLayerNormZero.forward: models/modules/normalization.py:51-57."""
    C = hidden.shape[-1]
    shift, scale, gate, e_shift, e_scale, e_gate = F.linear(F.silu(temb), sd[p + "linear.weight"], sd[p + "linear.bias"]).chunk(6, dim=1)
    w, b = sd[p + "norm.weight"], sd[p + "norm.bias"]
    hs = F.layer_norm(hidden, (C,), w, b, eps) * (1 + scale)[:, None, :] + shift[:, None, :]
    es = F.layer_norm(enc, (C,), w, b, eps) * (1 + e_scale)[:, None, :] + e_shift[:, None, :]
    return hs, es, gate[:, None, :], e_gate[:, None, :]


def apply_rotary_emb(x: Tensor, cos: Tensor, sin: Tensor) -> Tensor:
    """models/modules/embeddings.py:367-412 (use_real, unbind dim -1): interleaved pairs, fp32 math, cast back."""
    xr, xi = x.reshape(*x.shape[:-1], -1, 2).unbind(-1)
    rot = torch.stack([-xi, xr], dim=-1).flatten(3)
    return (x.float() * cos[None, None] + rot.float() * sin[None, None]).to(x.dtype)


def rotary_3d(embed_dim: int, crops_coords, grid_size, temporal_size: int, theta: float = 10000.0):
    """get_3d_rotary_pos_embed (models/modules/embeddings.py:283-364): (cos, sin) [T*H*W, embed_dim]; a quarter of the
    channels for the frame, three eighths each for the (cropped, resized) row and column coordinate."""
    (s0, s1), (e0, e1) = crops_coords
    lin = lambda a, b, n: torch.from_numpy(__import__("numpy").linspace(a, b, n, endpoint=False, dtype="float32")).float()  # noqa: E731
    gh, gw, gt = lin(s0, e0, grid_size[0]), lin(s1, e1, grid_size[1]), lin(0, temporal_size, temporal_size)
    dt_, dh = embed_dim // 4, embed_dim // 8 * 3

    def fr(g, d):
        f = 1.0 / (theta ** (torch.arange(0, d, 2).float() / d))
        return torch.einsum("n,f->nf", g, f).repeat_interleave(2, dim=-1)

    ft, fh, fw = fr(gt, dt_), fr(gh, dh), fr(gw, dh)
    T, H, W = temporal_size, grid_size[0], grid_size[1]
    freqs = torch.cat([ft[:, None, None, :].expand(T, H, W, -1), fh[None, :, None, :].expand(T, H, W, -1),
                       fw[None, None, :, :].expand(T, H, W, -1)], dim=-1).reshape(T * H * W, -1)
    return freqs.cos(), freqs.sin()


def resize_crop_region_for_grid(src, tgt_width, tgt_height):
    """pipelines/cogvideox/pipeline_cogvideox.py:758-773."""
    h, w = src
    if h / w > tgt_height / tgt_width:
        rh, rw = tgt_height, int(round(tgt_height / h * w))
    else:
        rw, rh = tgt_width, int(round(tgt_width / w * h))
    top, left = int(round((tgt_height - rh) / 2.0)), int(round((tgt_width - rw) / 2.0))
    return (top, left), (top + rh, left + rw)


def joint_attention(sd, p: str, hidden: Tensor, enc: Tensor, heads: int, rotary=None):
    """CogVideoXAttnProcessor2_0.__call__ with sp_size == 1, no mask: cogvideox_transformer_3d.py:88-175; rotary = (cos, sin)
    of the video tokens (:146-155, CogVideoX-5b) or None."""
    text_len = enc.size(1)
    x = torch.cat([enc, hidden], dim=1)
    B, N, C = x.shape
    D = C // heads
    q = F.linear(x, sd[p + "to_q.weight"], sd.get(p + "to_q.bias"))
    k = F.linear(x, sd[p + "to_k.weight"], sd.get(p + "to_k.bias"))
    v = F.linear(x, sd[p + "to_v.weight"], sd.get(p + "to_v.bias"))
    q = q.view(B, -1, heads, D).transpose(1, 2)
    k = k.view(B, -1, heads, D).transpose(1, 2)
    v = v.view(B, -1, heads, D).transpose(1, 2)
    q = F.layer_norm(q, (D,), sd[p + "norm_q.weight"], sd[p + "norm_q.bias"], 1e-6)
    k = F.layer_norm(k, (D,), sd[p + "norm_k.weight"], sd[p + "norm_k.bias"], 1e-6)
    if rotary is not None:
        n = rotary[0].shape[0]
        q[:, :, text_len : text_len + n] = apply_rotary_emb(q[:, :, text_len : text_len + n], *rotary)
        k[:, :, text_len : text_len + n] = apply_rotary_emb(k[:, :, text_len : text_len + n], *rotary)
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False)
    o = o.transpose(1, 2).reshape(B, -1, C)
    o = F.linear(o, sd[p + "to_out.0.weight"], sd[p + "to_out.0.bias"])
    e, h = o.split([text_len, o.size(1) - text_len], dim=1)
    return h, e


def feed_forward(sd, p: str, x: Tensor) -> Tensor:
    h = F.gelu(F.linear(x, sd[p + "net.0.proj.weight"], sd[p + "net.0.proj.bias"]), approximate="tanh")
    return F.linear(h, sd[p + "net.2.weight"], sd[p + "net.2.bias"])


class BlockPAB:
    def __init__(self):
        self.attn_count = 0
        self.last_attn = None


def block(sd, p: str, hidden: Tensor, enc: Tensor, temb: Tensor, heads: int, pab=None, pab_state=None, timestep_int=None,
          rotary=None):
    """CogVideoXBlock.forward: cogvideox_transformer_3d.py:268-312 (PAB: spatial gate only, :284-295)."""
    text_len = enc.size(1)
    nh, ne, gate, e_gate = layer_norm_zero(sd, p + "norm1.", hidden, enc, temb)
    reuse = False
    if pab is not None and pab.enabled():
        reuse, pab_state.attn_count = pab.gate("spatial", timestep_int, pab_state.attn_count)
    if reuse:
        ah, ae = pab_state.last_attn
    else:
        ah, ae = joint_attention(sd, p + "attn1.", nh, ne, heads, rotary)
        if pab is not None and pab.enabled():
            pab_state.last_attn = (ah, ae)
    hidden = hidden + gate * ah
    enc = enc + e_gate * ae
    nh, ne, gate_ff, e_gate_ff = layer_norm_zero(sd, p + "norm2.", hidden, enc, temb)
    ff = feed_forward(sd, p + "ff.", torch.cat([ne, nh], dim=1))
    hidden = hidden + gate_ff * ff[:, text_len:]
    enc = enc + e_gate_ff * ff[:, :text_len]
    return hidden, enc


def _sincos_1d(embed_dim: int, pos: Tensor) -> Tensor:
    omega = 1.0 / 10000 ** (torch.arange(embed_dim // 2, dtype=torch.float64) / (embed_dim / 2.0))
    out = pos.reshape(-1).double()[:, None] * omega[None]
    return torch.cat([out.sin(), out.cos()], dim=1)


def sincos_3d(embed_dim, spatial_size, temporal_size, spatial_scale=1.0, temporal_scale=1.0) -> Tensor:
    """diffusers get_3d_sincos_pos_embed(embed_dim, (W, H), T, ...): [T, H*W, D] (temporal quarter first)."""
    W, H = spatial_size
    d_sp, d_t = 3 * embed_dim // 4, embed_dim // 4
    gh = torch.arange(H, dtype=torch.float32) / spatial_scale
    gw = torch.arange(W, dtype=torch.float32) / spatial_scale
    grid_w, grid_h = torch.meshgrid(gw, gh, indexing="xy")
    sp = torch.cat([_sincos_1d(d_sp // 2, grid_w), _sincos_1d(d_sp // 2, grid_h)], dim=1)
    tm = _sincos_1d(d_t, torch.arange(temporal_size, dtype=torch.float32) / temporal_scale)
    return torch.cat([tm[:, None, :].expand(-1, H * W, -1), sp[None].expand(temporal_size, -1, -1)], dim=-1).float()


def timestep_sinusoid(timesteps: Tensor, dim: int, flip_sin_to_cos=True, freq_shift=0) -> Tensor:
    """diffusers get_timestep_embedding (fp32)."""
    half = dim // 2
    exponent = -math.log(10000.0) * torch.arange(half, dtype=torch.float32) / (half - freq_shift)
    emb = timesteps[:, None].float() * exponent.exp()[None]
    emb = torch.cat([emb.sin(), emb.cos()], dim=-1)
    return torch.cat([emb[:, half:], emb[:, :half]], dim=-1) if flip_sin_to_cos else emb


def transformer_forward(sd, cfg: dict, hidden: Tensor, enc: Tensor, timestep: Tensor, pab=None, pab_states=None, rotary=None):
    """CogVideoXTransformer3DModel.forward (:479-589), 2B configuration; cfg: heads, head_dim, layers, patch,
    max_text, sample_width/height/frames, spatial_scale, temporal_scale, out_channels, eps."""
    dt = sd["proj_out.weight"].dtype
    heads, D, p = cfg["heads"], cfg["head_dim"], cfg["patch"]
    C = heads * D
    B, Fr, Cin, H, W = hidden.shape
    t_emb = timestep_sinusoid(timestep, C).to(dt)
    emb = F.linear(F.silu(F.linear(t_emb, sd["time_embedding.linear_1.weight"], sd["time_embedding.linear_1.bias"])),
                   sd["time_embedding.linear_2.weight"], sd["time_embedding.linear_2.bias"])
    txt = F.linear(enc.to(dt), sd["patch_embed.text_proj.weight"], sd["patch_embed.text_proj.bias"])
    img = F.conv2d(hidden.to(dt).reshape(-1, Cin, H, W), sd["patch_embed.proj.weight"], sd["patch_embed.proj.bias"], stride=p)
    img = img.view(B, Fr, C, -1).transpose(2, 3).flatten(1, 2)
    x = torch.cat([txt, img], dim=1)
    Nt = txt.shape[1]
    frames = (cfg["sample_frames"] - 1) // 4 + 1
    pos = torch.zeros(1, cfg["max_text"] + (cfg["sample_height"] // p) * (cfg["sample_width"] // p) * frames, C)
    pos[:, cfg["max_text"]:] = sincos_3d(C, (cfg["sample_width"] // p, cfg["sample_height"] // p), frames,
                                         cfg.get("spatial_scale", 1.875), cfg.get("temporal_scale", 1.0)).flatten(0, 1)
    if rotary is None:  # use_rotary_positional_embeddings (CogVideoX-5b) adds no table (:519-524)
        x = x + pos[:, : x.shape[1]].to(dt)
    e, h = x[:, :Nt], x[:, Nt:]
    ts_int = int(timestep[0]) if pab is not None else None
    for i in range(cfg["layers"]):
        h, e = block(sd, f"transformer_blocks.{i}.", h, e, emb, heads, pab, pab_states[i] if pab_states else None, ts_int, rotary)
    eps = cfg.get("eps", 1e-5)
    h = F.layer_norm(h, (C,), sd["norm_final.weight"], sd["norm_final.bias"], eps)
    shift, scale = F.linear(F.silu(emb), sd["norm_out.linear.weight"], sd["norm_out.linear.bias"]).chunk(2, dim=1)
    h = F.layer_norm(h, (C,), sd["norm_out.norm.weight"], sd["norm_out.norm.bias"], eps) * (1 + scale)[:, None, :] + shift[:, None, :]
    h = F.linear(h, sd["proj_out.weight"], sd["proj_out.bias"])
    Co = cfg.get("out_channels", Cin)
    return h.reshape(B, Fr, H // p, W // p, Co, p, p).permute(0, 1, 4, 2, 5, 3, 6).flatten(5, 6).flatten(3, 4)
