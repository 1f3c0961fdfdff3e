"""TEST INFRASTRUCTURE ONLY -- CPU/torch restatement of the Latte transformer blocks (block level).

PINNED against the outputs of the reference's own LatteT2V, executed unmodified (tests/test_oracle_vs_reference.py::
test_latte_oracle_vs_reference_model: fp32 within summation order, bf16 bit for bit).  ``diffusers==0.30.0`` (requirements.txt:25)
is not installed here, so the reference file's diffusers LEAF classes are supplied by oracle/ref_loader.load_latte from the
reference's own vendored copies in open_sora_plan_v110_transformer_3d.py (Attention + AttnProcessor2_0, PatchEmbed,
CombinedTimestepSizeEmbeddings, CaptionProjection, get_1d_sincos_pos_embed_from_grid) plus three restated ones (GELU,
Timesteps, TimestepEmbedding: published semantics, a few lines each).  This file restates the in-tree block code
(models/transformers/latte_transformer_3d.py:357-517 spatial ``BasicTransformerBlock``, :680-824 temporal
``BasicTransformerBlock_``, local ``FeedForward`` :92-148, block loop :1312-1425) and those leaves:
  * ``Attention(query_dim, heads, dim_head, bias=True, cross_attention_dim)`` with the default processor:
    to_q / to_k / to_v Linears, heads split, F.scaled_dot_product_attention (no mask: the Latte pipeline never passes
    one, pipeline_latte.py:854-862), to_out[0] Linear, dropout 0, rescale_output_factor 1;
  * ``GELU(dim, inner, approximate="tanh")`` = Linear then tanh-GELU.
Configuration: norm_type "ada_norm_single", norm_elementwise_affine False, eps 1e-6, activation "gelu-approximate".

``transformer_forward`` restates LatteT2V.forward around the block loop (:1144-1466): the in-tree glue (rearranges, output
head :1436-1443, unpatchify :1446-1456, temp_pos_embed :1468-1470) as written, the diffusers pieces (``PatchEmbed`` with
its 2-D sincos table, ``AdaLayerNormSingle`` -> ``PixArtAlphaCombinedTimestepSizeEmbeddings`` -> ``Timesteps`` /
``TimestepEmbedding``, ``PixArtAlphaTextProjection``) from their published semantics; the whole forward is pinned as above.
"""
import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


def _ln(x: Tensor, eps: float = 1e-6) -> Tensor:
    return F.layer_norm(x, (x.shape[-1],), None, None, eps)


def attention(sd: Dict[str, Tensor], p: str, x: Tensor, enc: Optional[Tensor], heads: int) -> Tensor:
    """diffusers Attention.forward -> AttnProcessor2_0.__call__ (self-attention when enc is None)."""
    B, N, C = x.shape
    D = C // heads
    src = x if enc is None else enc
    q = F.linear(x, sd[p + "to_q.weight"], sd.get(p + "to_q.bias"))
    k = F.linear(src, sd[p + "to_k.weight"], sd.get(p + "to_k.bias"))
    v = F.linear(src, sd[p + "to_v.weight"], sd.get(p + "to_v.bias"))
    q = q.view(B, -1, heads, D).transpose(1, 2)
    k = k.view(B, -1, heads, D).transpose(1, 2)
    v = v.view(B, -1, heads, D).transpose(1, 2)
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False)
    o = o.transpose(1, 2).reshape(B, -1, C).to(q.dtype)
    return F.linear(o, sd[p + "to_out.0.weight"], sd[p + "to_out.0.bias"])


def feed_forward(sd: Dict[str, Tensor], p: str, x: Tensor) -> Tensor:
    """FeedForward(activation_fn='gelu-approximate'): latte_transformer_3d.py:92-148."""
    h = F.gelu(F.linear(x, sd[p + "net.0.proj.weight"], sd[p + "net.0.proj.bias"]), approximate="tanh")
    return F.linear(h, sd[p + "net.2.weight"], sd[p + "net.2.bias"])


def spatial_block(sd, p: str, x: Tensor, enc: Tensor, timestep6: Tensor, heads: int) -> Tensor:
    """BasicTransformerBlock.forward, ada_norm_single, PAB off: latte_transformer_3d.py:357-517.
    x [(b f), S, C]; enc [(b f), L, C]; timestep6 [(b f), 6C]."""
    bs = x.shape[0]
    sh_a, sc_a, g_a, sh_m, sc_m, g_m = (sd[p + "scale_shift_table"][None] + timestep6.reshape(bs, 6, -1)).chunk(6, dim=1)
    n = _ln(x) * (1 + sc_a) + sh_a
    x = g_a * attention(sd, p + "attn1.", n, None, heads) + x
    x = attention(sd, p + "attn2.", x, enc, heads) + x  # ada_norm_single: no norm before cross attention (:447-450)
    n = _ln(x) * (1 + sc_m) + sh_m  # norm2
    return g_m * feed_forward(sd, p + "ff.", n) + x


def temporal_block(sd, p: str, x: Tensor, timestep6: Tensor, heads: int) -> Tensor:
    """BasicTransformerBlock_.forward, ada_norm_single, sp=1, PAB off: latte_transformer_3d.py:680-824.
    x [(b s), F, C]; timestep6 [(b s), 6C]."""
    bs = x.shape[0]
    sh_a, sc_a, g_a, sh_m, sc_m, g_m = (sd[p + "scale_shift_table"][None] + timestep6.reshape(bs, 6, -1)).chunk(6, dim=1)
    n = _ln(x) * (1 + sc_a) + sh_a
    x = g_a * attention(sd, p + "attn1.", n, None, heads) + x
    n = _ln(x) * (1 + sc_m) + sh_m  # norm3 (:778)
    return g_m * feed_forward(sd, p + "ff.", n) + x


def block_stack(sd, x: Tensor, enc: Tensor, timestep6: Tensor, heads: int, depth: int, temp_pos_embed: Optional[Tensor]):
    """The LatteT2V block loop at inference (sp=1, use_image_num=0): latte_transformer_3d.py:1290-1425.
    x [B, F, S, C] -> [B, F, S, C]; enc [B, L, C]; timestep6 [B, 6C]; temp_pos_embed [1, F, C] or None."""
    B, Fr, S, C = x.shape
    enc_sp = enc[:, None].expand(B, Fr, *enc.shape[1:]).reshape(B * Fr, *enc.shape[1:]).contiguous()
    t_sp = timestep6[:, None].expand(B, Fr, -1).reshape(B * Fr, -1).contiguous()
    t_tm = timestep6[:, None].expand(B, S, -1).reshape(B * S, -1).contiguous()
    h = x.reshape(B * Fr, S, C)
    for i in range(depth):
        h = spatial_block(sd, f"transformer_blocks.{i}.", h, enc_sp, t_sp, heads)
        h = h.reshape(B, Fr, S, C).permute(0, 2, 1, 3).reshape(B * S, Fr, C).contiguous()  # (b f) t d -> (b t) f d
        if i == 0 and Fr > 1 and temp_pos_embed is not None:
            h = h + temp_pos_embed
        h = temporal_block(sd, f"temporal_transformer_blocks.{i}.", h, t_tm, heads)
        h = h.reshape(B, S, Fr, C).permute(0, 2, 1, 3).reshape(B * Fr, S, C).contiguous()
    return h.reshape(B, Fr, S, C)


def _sincos_1d(embed_dim: int, pos: Tensor) -> Tensor:
    omega = 1.0 / 10000 ** (torch.arange(embed_dim // 2, dtype=torch.float64) / (embed_dim / 2.0))
    out = pos.reshape(-1).double()[:, None] * omega[None]
    return torch.cat([out.sin(), out.cos()], dim=1)


def sincos_2d(embed_dim: int, grid_size: int, base_size: int, interpolation_scale: float = 1.0) -> Tensor:
    """diffusers get_2d_sincos_pos_embed as PatchEmbed calls it (w-first meshgrid): [grid*grid, D] float32."""
    g = torch.arange(grid_size, dtype=torch.float32) / (grid_size / base_size) / interpolation_scale
    gw, gh = torch.meshgrid(g, g, indexing="xy")
    return torch.cat([_sincos_1d(embed_dim // 2, gw), _sincos_1d(embed_dim // 2, gh)], dim=1).float()


def transformer_forward(sd, cfg: dict, latents: Tensor, timestep: Tensor, text: Tensor) -> Tensor:
    """LatteT2V.forward, inference, sp = 1, ada_norm_single, no micro-conditions (sample_size != 128).
    cfg: heads, head_dim, layers, patch, sample_size, out_channels, video_length."""
    dt = sd["proj_out.weight"].dtype
    heads, D, p = cfg["heads"], cfg["head_dim"], cfg["patch"]
    C = heads * D
    B, Cin, Fr, H, W = latents.shape
    h, w = H // p, W // p
    x = latents.to(dt).permute(0, 2, 1, 3, 4).reshape(B * Fr, Cin, H, W)
    x = F.conv2d(x, sd["pos_embed.proj.weight"], sd["pos_embed.proj.bias"], stride=p).flatten(2).transpose(1, 2)
    grid = cfg["sample_size"] // p
    x = (x + sincos_2d(C, h, base_size=grid, interpolation_scale=max(cfg["sample_size"] // 64, 1))[None].to(dt)).reshape(B, Fr, h * w, C)
    half = 128
    e = timestep[:, None].float() * (-math.log(10000.0) * torch.arange(half, dtype=torch.float32) / half).exp()[None]
    t_emb = torch.cat([e.cos(), e.sin()], dim=-1).to(dt)  # Timesteps(256, flip_sin_to_cos=True, freq_shift=0)
    pre = "adaln_single.emb.timestep_embedder."
    emb = F.linear(F.silu(F.linear(t_emb, sd[pre + "linear_1.weight"], sd[pre + "linear_1.bias"])), sd[pre + "linear_2.weight"],
                   sd[pre + "linear_2.bias"])
    t6 = F.linear(F.silu(emb), sd["adaln_single.linear.weight"], sd["adaln_single.linear.bias"])
    enc = F.linear(F.gelu(F.linear(text.to(dt), sd["caption_projection.linear_1.weight"], sd["caption_projection.linear_1.bias"]),
                          approximate="tanh"), sd["caption_projection.linear_2.weight"], sd["caption_projection.linear_2.bias"])
    tpe = _sincos_1d(C, torch.arange(cfg["video_length"]).float()).float()[None][:, :Fr].to(dt)
    x = block_stack(sd, x, enc, t6, heads, cfg["layers"], tpe if Fr > 1 else None)
    shift, scale = (sd["scale_shift_table"][None] + emb[:, None]).chunk(2, dim=1)  # per sample, broadcast over frames
    y = _ln(x.reshape(B, Fr * h * w, C)) * (1 + scale) + shift
    y = F.linear(y, sd["proj_out.weight"], sd["proj_out.bias"])
    Co = cfg["out_channels"]
    y = torch.einsum("nhwpqc->nchpwq", y.reshape(B * Fr, h, w, p, p, Co)).reshape(B * Fr, Co, h * p, w * p)
    return y.reshape(B, Fr, Co, h * p, w * p).permute(0, 2, 1, 3, 4).contiguous()
