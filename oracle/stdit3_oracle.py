"""TEST INFRASTRUCTURE ONLY -- CPU/torch restatement of the OpenSora STDiT3 denoising hot path.

This file is the *oracle* the CUDA path is checked against.  It is never imported by the product
package (``videosys_b200``); only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may use it.

Every function is a functional restatement (state_dict in, tensors out; no nn.Module, no global
singletons) of the reference code it cites, keeping the reference's *op order and rounding points*:
each eager op rounds to the storage dtype exactly where the reference's eager op does, so on CPU in
the same dtype the two are bit-identical (pinned by the committed golden vectors in tests/golden/, which
tests/test_oracle_vs_reference.py and tests/test_oracle_golden.py check).

Third-party pieces that are not in the reference tree and are restated from their published
semantics (SURVEY.md section 8c): timm ``Mlp`` (fc2(act(fc1(x)))), ``rotary_embedding_torch``
``RotaryEmbedding.rotate_queries_or_keys`` (interleaved pairs, theta 1e4, fp32 math, cast back).
Citations are relative to /root/reference/videosys/.
"""
import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# ----------------------------------------------------------------------------------------------
# leaf ops
# ----------------------------------------------------------------------------------------------
def t2i_modulate(x: Tensor, shift: Tensor, scale: Tensor) -> Tensor:
    """models/transformers/open_sora_transformer_3d.py:47-48."""
    return x * (1 + scale) + shift


def layer_norm_noaffine(x: Tensor, eps: float = 1e-6) -> Tensor:
    """nn.LayerNorm(C, eps=1e-6, elementwise_affine=False): open_sora_transformer_3d.py:117,129."""
    return F.layer_norm(x, (x.shape[-1],), None, None, eps)


def frame_select(x_mask: Tensor, a: Tensor, b: Tensor, T: int, S: int) -> Tensor:
    """t_mask_select: open_sora_transformer_3d.py:152-160.  x_mask [B,T] bool, a/b [B,T*S,C]."""
    B, _, C = a.shape
    out = torch.where(x_mask[:, :, None, None], a.reshape(B, T, S, C), b.reshape(B, T, S, C))
    return out.reshape(B, T * S, C)


def llama_rms_norm(x: Tensor, weight: Tensor, eps: float = 1e-6) -> Tensor:
    """LlamaRMSNorm.forward: models/modules/normalization.py:28-33 (fp32 stats, cast back, then * w)."""
    dt = x.dtype
    h = x.to(torch.float32)
    var = h.pow(2).mean(-1, keepdim=True)
    h = h * torch.rsqrt(var + eps)
    return weight * h.to(dt)


def rope_freqs(head_dim: int, theta: float = 10000.0) -> Tensor:
    """rotary_embedding_torch.RotaryEmbedding(dim=head_dim).freqs ('lang'); open_sora_transformer_3d.py:388-390."""
    return 1.0 / (theta ** (torch.arange(0, head_dim, 2)[: head_dim // 2].float() / head_dim))


def rotate_queries_or_keys(t: Tensor, freqs: Tensor) -> Tensor:
    """RotaryEmbedding.rotate_queries_or_keys(t, seq_dim=-2): positions 0..n-1, interleaved pairs,
    fp32 math then cast back (call site models/modules/attentions.py:76-78)."""
    n = t.shape[-2]
    pos = torch.arange(n, device=t.device, dtype=torch.float32)
    ang = torch.einsum("i,j->ij", pos, freqs.float().to(t.device)).repeat_interleave(2, dim=-1)
    x1, x2 = t.reshape(*t.shape[:-1], -1, 2).unbind(-1)
    rot = torch.stack((-x2, x1), -1).flatten(-2)
    return (t * ang.cos() + rot * ang.sin()).type(t.dtype)


def native_attention(q: Tensor, k: Tensor, v: Tensor, scale: float) -> Tensor:
    """OpenSoraAttention.native_attention: attentions.py:111-120 (op order matters in bf16)."""
    dt = q.dtype
    q = q * scale
    attn = q @ k.transpose(-2, -1)
    attn = attn.to(torch.float32).softmax(dim=-1).to(dt)
    return attn @ v


def gelu_tanh(x: Tensor) -> Tensor:
    """approx_gelu = nn.GELU(approximate='tanh'): models/modules/activations.py:3."""
    return F.gelu(x, approximate="tanh")


def mlp(sd: Dict[str, Tensor], p: str, x: Tensor) -> Tensor:
    """timm Mlp semantics (third party; call sites open_sora_transformer_3d.py:130-132,267)."""
    h = F.linear(x, sd[p + "fc1.weight"], sd[p + "fc1.bias"])
    h = gelu_tanh(h)
    return F.linear(h, sd[p + "fc2.weight"], sd[p + "fc2.bias"])


# ----------------------------------------------------------------------------------------------
# attention modules
# ----------------------------------------------------------------------------------------------
def self_attention(sd, p: str, x: Tensor, num_heads: int, freqs: Optional[Tensor]) -> Tensor:
    """OpenSoraAttention.forward, enable_flash_attn=False: attentions.py:55-109.

    x [B', N, C]; freqs is None for spatial blocks, the rope table for temporal blocks
    (open_sora_transformer_3d.py:438).  N < 30 takes native_attention (attentions.py:58,95-97),
    N == 1 returns v (attentions.py:65-66), otherwise SDPA (attentions.py:100).
    """
    Bq, N, C = x.shape
    D = C // num_heads
    qkv = F.linear(x, sd[p + "qkv.weight"], sd[p + "qkv.bias"])
    qkv = qkv.view(Bq, N, 3, num_heads, D).permute(2, 0, 3, 1, 4)
    q, k, v = qkv.unbind(0)
    if N == 1:
        o = v
    else:
        q = llama_rms_norm(q, sd[p + "q_norm.weight"])
        k = llama_rms_norm(k, sd[p + "k_norm.weight"])
        if freqs is not None:
            q = rotate_queries_or_keys(q, freqs)
            k = rotate_queries_or_keys(k, freqs)
        if N < 30:
            o = native_attention(q, k, v, D**-0.5)
        else:
            o = F.scaled_dot_product_attention(q, k, v)
    o = o.transpose(1, 2).reshape(Bq, N, C)
    return F.linear(o, sd[p + "proj.weight"], sd[p + "proj.bias"])


def cross_attention(sd, p: str, x: Tensor, cond: Tensor, y_lens: List[int], num_heads: int) -> Tensor:
    """OpenSoraMultiHeadCrossAttention.forward + torch_impl: attentions.py:152-185,259-270.

    cond is the packed text [1, sum(L), C]; the reference views k/v as [B, sum(L)/B, H, D]
    (attentions.py:260-262, requires equal lengths) and marks the first y_lens[i] keys attendable
    (bool mask, True = attend: attentions.py:264-266).
    """
    B, N, C = x.shape
    D = C // num_heads
    q = F.linear(x, sd[p + "q_linear.weight"], sd[p + "q_linear.bias"]).view(1, -1, num_heads, D)
    kv = F.linear(cond, sd[p + "kv_linear.weight"], sd[p + "kv_linear.bias"]).view(1, -1, 2, num_heads, D)
    k, v = kv.unbind(2)
    q = q.view(B, -1, num_heads, D).transpose(1, 2)
    k = k.view(B, -1, num_heads, D).transpose(1, 2)
    v = v.view(B, -1, num_heads, D).transpose(1, 2)
    attn_mask = torch.zeros(B, 1, N, k.shape[2], dtype=torch.bool, device=q.device)
    for i, m in enumerate(y_lens):
        attn_mask[i, :, :, :m] = True
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=attn_mask)
    o = o.transpose(1, 2).contiguous().view(B, N, C)
    return F.linear(o, sd[p + "proj.weight"], sd[p + "proj.bias"])


def cross_attention_varlen(sd, p: str, x: Tensor, cond: Tensor, y_lens: List[int], num_heads: int) -> Tensor:
    """OpenSoraMultiHeadCrossAttention.forward with enable_flash_attn=True: attentions.py:152-185 -> flash_attn_impl
    :240-257.  flash_attn_varlen_func (third party, flash-attn) is called with cu_seqlens_q = [0, N, 2N, ..] and
    cu_seqlens_k = cumsum(y_lens): sample i's queries attend exactly the y_lens[i] packed keys of sample i --
    restated as one softmax(q k^T / sqrt(d)) v per sample (the library's published semantics)."""
    B, N, C = x.shape
    D = C // num_heads
    q = F.linear(x, sd[p + "q_linear.weight"], sd[p + "q_linear.bias"]).view(B, N, num_heads, D)
    kv = F.linear(cond, sd[p + "kv_linear.weight"], sd[p + "kv_linear.bias"]).view(-1, 2, num_heads, D)
    outs, start = [], 0
    for i, m in enumerate(y_lens):
        k, v = kv[start:start + m, 0], kv[start:start + m, 1]  # [m, H, D]
        start += m
        o = F.scaled_dot_product_attention(q[i].transpose(0, 1)[None], k.transpose(0, 1)[None], v.transpose(0, 1)[None])
        outs.append(o[0].transpose(0, 1).reshape(N, C))
    o = torch.stack(outs, 0)
    return F.linear(o, sd[p + "proj.weight"], sd[p + "proj.bias"])


# ----------------------------------------------------------------------------------------------
# PAB per-block state (the reference keeps these as attributes on the block: :141-147)
# ----------------------------------------------------------------------------------------------
class BlockPABState:
    def __init__(self):
        self.attn_count = 0
        self.cross_count = 0
        self.last_attn = None
        self.last_cross = None


# ----------------------------------------------------------------------------------------------
# STDiT3Block.forward
# ----------------------------------------------------------------------------------------------
def stdit3_block(
    sd,
    p: str,
    x: Tensor,
    y: Tensor,
    t: Tensor,
    y_lens: List[int],
    x_mask: Optional[Tensor],
    t0: Optional[Tensor],
    T: int,
    S: int,
    num_heads: int,
    temporal: bool,
    freqs: Optional[Tensor] = None,
    pab=None,
    pab_state: Optional[BlockPABState] = None,
    timestep_int: Optional[int] = None,
    spatial_attn_fn=None,
    cross_varlen: bool = False,
) -> Tensor:
    """STDiT3Block.forward: open_sora_transformer_3d.py:162-286 (mlp_broadcast unreachable for OpenSora,
    SURVEY fact 7).  ``pab`` is an oracle.pab_oracle.PABGate or None; ``spatial_attn_fn`` lets the DSP
    oracle wrap the spatial attention with the reshard (lines :208-216)."""
    B, N, C = x.shape
    tab = sd[p + "scale_shift_table"]
    sh_a, sc_a, g_a, sh_m, sc_m, g_m = (tab[None] + t.reshape(B, 6, -1)).chunk(6, dim=1)
    if x_mask is not None:
        sh_a0, sc_a0, g_a0, sh_m0, sc_m0, g_m0 = (tab[None] + t0.reshape(B, 6, -1)).chunk(6, dim=1)

    pab_on = pab is not None and pab.enabled()
    reuse_attn = False
    if pab_on:
        kind = "temporal" if temporal else "spatial"
        reuse_attn, pab_state.attn_count = pab.gate(kind, timestep_int, pab_state.attn_count)

    if pab_on and reuse_attn:
        x_m_s = pab_state.last_attn
    else:
        n1 = layer_norm_noaffine(x)
        x_m = t2i_modulate(n1, sh_a, sc_a)
        if x_mask is not None:
            x_m = frame_select(x_mask, x_m, t2i_modulate(n1, sh_a0, sc_a0), T, S)
        if temporal:
            x_m = x_m.reshape(B, T, S, C).permute(0, 2, 1, 3).reshape(B * S, T, C)
            x_m = self_attention(sd, p + "attn.", x_m, num_heads, freqs)
            x_m = x_m.reshape(B, S, T, C).permute(0, 2, 1, 3).reshape(B, T * S, C)
        elif spatial_attn_fn is not None:
            x_m = spatial_attn_fn(x_m)
        else:
            x_m = x_m.reshape(B * T, S, C)
            x_m = self_attention(sd, p + "attn.", x_m, num_heads, None)
            x_m = x_m.reshape(B, T * S, C)
        x_m_s = g_a * x_m
        if x_mask is not None:
            x_m_s = frame_select(x_mask, x_m_s, g_a0 * x_m, T, S)
        if pab_on:
            pab_state.last_attn = x_m_s
    x = x + x_m_s

    reuse_cross = False
    if pab_on:
        reuse_cross, pab_state.cross_count = pab.gate("cross", timestep_int, pab_state.cross_count)
    if pab_on and reuse_cross:
        x = x + pab_state.last_cross
    else:
        x_cross = (cross_attention_varlen if cross_varlen else cross_attention)(sd, p + "cross_attn.", x, y, y_lens, num_heads)
        if pab_on:
            pab_state.last_cross = x_cross
        x = x + x_cross

    n2 = layer_norm_noaffine(x)
    x_m = t2i_modulate(n2, sh_m, sc_m)
    if x_mask is not None:
        x_m = frame_select(x_mask, x_m, t2i_modulate(n2, sh_m0, sc_m0), T, S)
    x_m = mlp(sd, p + "mlp.", x_m)
    x_m_s = g_m * x_m
    if x_mask is not None:
        x_m_s = frame_select(x_mask, x_m_s, g_m0 * x_m, T, S)
    return x + x_m_s


# ----------------------------------------------------------------------------------------------
# STDiT3.forward glue (embedders, final layer, unpatchify)
# ----------------------------------------------------------------------------------------------
def sinusoid_embedding(t: Tensor, dim: int = 256, max_period: float = 10000.0) -> Tensor:
    """TimestepEmbedder.timestep_embedding: models/modules/embeddings.py:119-138."""
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(0, half, dtype=torch.float32) / half).to(t.device)
    args = t[:, None].float() * freqs[None]
    return torch.cat([torch.cos(args), torch.sin(args)], dim=-1)


def _embed_mlp(sd, p: str, freq: Tensor) -> Tensor:
    h = F.linear(freq, sd[p + "mlp.0.weight"], sd[p + "mlp.0.bias"])
    return F.linear(F.silu(h), sd[p + "mlp.2.weight"], sd[p + "mlp.2.bias"])


def timestep_embed(sd, p: str, t: Tensor, dtype) -> Tensor:
    """TimestepEmbedder.forward: embeddings.py:140-145."""
    return _embed_mlp(sd, p, sinusoid_embedding(t).to(dtype))


def size_embed(sd, p: str, s: Tensor, bs: int) -> Tensor:
    """SizeEmbedder.forward: embeddings.py:164-176 (s is fps.unsqueeze(1): [B,1])."""
    if s.ndim == 1:
        s = s[:, None]
    if s.shape[0] != bs:
        s = s.repeat(bs // s.shape[0], 1)
    b, dims = s.shape
    dtype = sd[p + "mlp.0.weight"].dtype
    out = _embed_mlp(sd, p, sinusoid_embedding(s.reshape(-1)).to(dtype))
    return out.reshape(b, dims * out.shape[-1])


def pos_embed_2d(dim: int, h: int, w: int, scale: float, base_size: int, dtype, device="cpu") -> Tensor:
    """OpenSoraPositionEmbedding2D._get_cached_emb: embeddings.py:247-270 (w goes first in the meshgrid).

    ``inv_freq`` is a (non-persistent) module buffer (embeddings.py:236-237), so ``model.to(bf16)``
    rounds it to the model dtype before the fp32 einsum -- kept, it changes the table in bf16."""
    half = dim // 2
    inv_freq = (1.0 / (10000 ** (torch.arange(0, half, 2).float() / half))).to(dtype).to(device)
    gh = torch.arange(h, device=device) / scale
    gw = torch.arange(w, device=device) / scale
    gh = gh * (base_size / h)
    gw = gw * (base_size / w)
    gh, gw = torch.meshgrid(gw, gh, indexing="ij")
    gh = gh.t().reshape(-1)
    gw = gw.t().reshape(-1)

    def sincos(v):
        o = torch.einsum("i,d->id", v, inv_freq)
        return torch.cat((torch.sin(o), torch.cos(o)), dim=-1)

    return torch.concat([sincos(gh), sincos(gw)], dim=-1).unsqueeze(0).to(dtype)


def patch_embed(sd, p: str, x: Tensor, patch=(1, 2, 2)) -> Tensor:
    """OpenSoraPatchEmbed3D.forward: embeddings.py:84-104 (right/bottom zero pad, Conv3d stride=patch)."""
    _, _, D, H, W = x.shape
    if W % patch[2]:
        x = F.pad(x, (0, patch[2] - W % patch[2]))
    if H % patch[1]:
        x = F.pad(x, (0, 0, 0, patch[1] - H % patch[1]))
    if D % patch[0]:
        x = F.pad(x, (0, 0, 0, 0, 0, patch[0] - D % patch[0]))
    x = F.conv3d(x, sd[p + "proj.weight"], sd[p + "proj.bias"], stride=patch)
    return x.flatten(2).transpose(1, 2)


def encode_text(sd, y: Tensor, mask: Optional[Tensor], hidden: int):
    """STDiT3.encode_text (eval: no token drop): open_sora_transformer_3d.py:526-537."""
    y = mlp(sd, "y_embedder.y_proj.", y)
    if mask is not None:
        if mask.shape[0] != y.shape[0]:
            mask = mask.repeat(y.shape[0] // mask.shape[0], 1)
        mask = mask.squeeze(1).squeeze(1)
        y = y.squeeze(1).masked_select(mask.unsqueeze(-1) != 0).view(1, -1, hidden)
        y_lens = mask.sum(dim=1).tolist()
    else:
        y_lens = [y.shape[2]] * y.shape[0]
        y = y.squeeze(1).view(1, -1, hidden)
    return y, y_lens


def final_layer(sd, x: Tensor, t: Tensor, x_mask, t0, T: int, S: int) -> Tensor:
    """T2IFinalLayer.forward: open_sora_transformer_3d.py:75-87.

    Reference quirk kept on purpose: line :81 rebinds ``x`` to the t-modulated tensor, so the t0
    branch at :84 normalises the *already modulated* activations, not the block output."""
    tab = sd["final_layer.scale_shift_table"]
    shift, scale = (tab[None] + t[:, None]).chunk(2, dim=1)
    out = t2i_modulate(layer_norm_noaffine(x), shift, scale)
    if x_mask is not None:
        shift0, scale0 = (tab[None] + t0[:, None]).chunk(2, dim=1)
        out0 = t2i_modulate(layer_norm_noaffine(out), shift0, scale0)
        out = frame_select(x_mask, out, out0, T, S)
    return F.linear(out, sd["final_layer.linear.weight"], sd["final_layer.linear.bias"])


def unpatchify(x: Tensor, Nt, Nh, Nw, Rt, Rh, Rw, patch=(1, 2, 2), out_ch=8) -> Tensor:
    """STDiT3.unpatchify: open_sora_transformer_3d.py:634-658."""
    B = x.shape[0]
    Tp, Hp, Wp = patch
    x = x.reshape(B, Nt, Nh, Nw, Tp, Hp, Wp, out_ch)
    x = x.permute(0, 7, 1, 4, 2, 5, 3, 6).reshape(B, out_ch, Nt * Tp, Nh * Hp, Nw * Wp)
    return x[:, :, :Rt, :Rh, :Rw]


def stdit3_forward(
    sd: Dict[str, Tensor],
    cfg: dict,
    x: Tensor,
    timestep: Tensor,
    y: Tensor,
    mask: Optional[Tensor] = None,
    x_mask: Optional[Tensor] = None,
    fps: Optional[Tensor] = None,
    height: Optional[Tensor] = None,
    width: Optional[Tensor] = None,
    pab=None,
    pab_states=None,
    valid_depth: Optional[int] = None,
    return_tokens: bool = False,
    cross_varlen: bool = False,
) -> Tensor:
    """STDiT3.forward on one rank (sp=cp=1): open_sora_transformer_3d.py:539-632.

    cfg: dict(hidden_size, num_heads, depth, patch_size, input_sq_size, in_channels, out_channels).
    pab_states: {"spatial": [BlockPABState]*depth, "temporal": [...]} when pab is given.
    """
    C, H_ = cfg["hidden_size"], cfg["num_heads"]
    patch = tuple(cfg.get("patch_size", (1, 2, 2)))
    depth = cfg["depth"] if valid_depth is None else valid_depth
    dtype = sd["x_embedder.proj.weight"].dtype
    _, _, Tx, Hx, Wx = x.shape
    T = -(-Tx // patch[0])
    Hn = -(-Hx // patch[1])
    Wn = -(-Wx // patch[2])
    B = x.shape[0]
    x = x.to(dtype)
    timestep = timestep.to(dtype)
    y = y.to(dtype)

    S = Hn * Wn
    base_size = round(S**0.5)
    resolution_sq = (height[0].item() * width[0].item()) ** 0.5
    scale = resolution_sq / cfg.get("input_sq_size", 512)
    pos = pos_embed_2d(C, Hn, Wn, scale, base_size, dtype, x.device)

    t = timestep_embed(sd, "t_embedder.", timestep, dtype)
    fps_e = size_embed(sd, "fps_embedder.", fps.unsqueeze(1), B)
    t = t + fps_e
    t_mlp = F.linear(F.silu(t), sd["t_block.1.weight"], sd["t_block.1.bias"])
    t0 = t0_mlp = None
    if x_mask is not None:
        t0 = timestep_embed(sd, "t_embedder.", torch.zeros_like(timestep), dtype) + fps_e
        t0_mlp = F.linear(F.silu(t0), sd["t_block.1.weight"], sd["t_block.1.bias"])

    y_tok, y_lens = encode_text(sd, y, mask, C)

    h = patch_embed(sd, "x_embedder.", x, patch)
    h = h.reshape(B, T, S, C) + pos
    h = h.reshape(B, T * S, C)

    freqs = sd["rope.freqs"] if "rope.freqs" in sd else rope_freqs(C // H_)
    ts_int = int(timestep[0]) if pab is not None else None
    for d in range(depth):
        for kind, temporal in (("spatial", False), ("temporal", True)):
            h = stdit3_block(
                sd,
                f"{kind}_blocks.{d}.",
                h,
                y_tok,
                t_mlp,
                y_lens,
                x_mask,
                t0_mlp,
                T,
                S,
                H_,
                temporal,
                freqs if temporal else None,
                pab,
                pab_states[kind][d] if pab_states is not None else None,
                ts_int,
                cross_varlen=cross_varlen,
            )
    if return_tokens:
        return h
    out = final_layer(sd, h, t, x_mask, t0, T, S)
    out = unpatchify(out, T, Hn, Wn, Tx, Hx, Wx, patch, cfg.get("out_channels", 8))
    return out.to(torch.float32)


# ----------------------------------------------------------------------------------------------
# scheduler pieces used by the metric harness
# ----------------------------------------------------------------------------------------------
def timestep_transform(t: Tensor, height: Tensor, width: Tensor, num_frames: Tensor, num_timesteps: int = 1000) -> Tensor:
    """schedulers/scheduling_rflow_open_sora.py:47-70 (base_resolution 512*512, base_num_frames 1, scale 1)."""
    t = t / num_timesteps
    resolution = height * width
    ratio_space = (resolution / (512 * 512)).sqrt()
    if num_frames[0] == 1:
        nf = torch.ones_like(num_frames)
    else:
        nf = num_frames // 17 * 5
    ratio_time = (nf / 1).sqrt()
    ratio = ratio_space * ratio_time * 1.0
    new_t = ratio * t / (1 + (ratio - 1) * t)
    return new_t * num_timesteps


def rflow_timesteps(num_sampling_steps: int, height: float, width: float, num_frames: int, dtype=torch.bfloat16):
    """RFLOW.sample timestep list + the ints PAB sees: scheduling_rflow_open_sora.py:208-223.
    Inputs are dtype tensors as built by prepare_multi_resolution_info (pipelines/open_sora/data_process.py:798-805)."""
    h = torch.tensor([height], dtype=dtype)
    w = torch.tensor([width], dtype=dtype)
    nf = torch.tensor([num_frames], dtype=dtype)
    ts = [(1.0 - i / num_sampling_steps) * 1000 for i in range(num_sampling_steps)]
    ts = [torch.tensor([v] * 1) for v in ts]
    ts = [timestep_transform(v, h, w, nf, 1000) for v in ts]
    ints = [int(v.to(dtype).item()) for v in ts]
    return ts, ints
