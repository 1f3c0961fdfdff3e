"""TEST INFRASTRUCTURE ONLY -- the cases of tests/test_oracle_vs_reference.py, shared with oracle/gen_golden_pins.py (which runs
the UNMODIFIED reference on them) so that both sides use one definition of every configuration, schedule and input."""
import random

import torch

from . import pab_oracle, synth

DT = {torch.float32: "float32", torch.bfloat16: "bfloat16", torch.float16: "float16"}

PAB_TS = [900, 700, 650, 600, 550, 500, 450, 50]

def lnz_inputs(dtype):
    return (synth.normalish("lnz.h", (2, 9, 128)).to(dtype), synth.normalish("lnz.e", (2, 4, 128)).to(dtype),
            synth.normalish("lnz.t", (2, 64)).to(dtype))

COGX_DDIM = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                 set_alpha_to_one=True, steps_offset=0, prediction_type="v_prediction", timestep_spacing="trailing",
                 rescale_betas_zero_snr=True, snr_shift_scale=3.0)

OSP_SMALL = dict(num_attention_heads=2, attention_head_dim=72, in_channels=4, out_channels=8, num_layers=2,
                 cross_attention_dim=144, attention_bias=True, sample_size=(8, 8), patch_size=2, activation_fn="gelu-approximate",
                 norm_type="ada_norm_single", norm_elementwise_affine=False, norm_eps=1e-6, caption_channels=32, video_length=5,
                 attention_mode="math", use_rope=True)

OSP_MIRROR_CASES = [(True, (8, 8), None), (False, (8, 8), None), (True, (12, 8), 2)]

OSP_PAB_MLP = {700: {"block": [0, 1], "skip_count": 2}, 550: {"block": [1], "skip_count": 1}}

OSP_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 850], spatial_range=2, temporal_broadcast=True,
                  temporal_threshold=[100, 850], temporal_range=3, cross_broadcast=True, cross_threshold=[100, 850], cross_range=4,
                  mlp_broadcast=True, mlp_spatial_broadcast_config=OSP_PAB_MLP, mlp_temporal_broadcast_config=OSP_PAB_MLP)

def osp_key(use_rope, HW, scale1d):
    return f"osp.{int(use_rope)}.{HW[0]}x{HW[1]}.{scale1d}"

def osp_inputs(B, Fr, HW, L=7, tag="osp."):
    x = synth.normalish(tag + "x", (B, 4, Fr, *HW))
    enc = synth.normalish(tag + "enc", (B, 1, L, 32))
    m = torch.ones(B, 1, L)
    m[B - 1, 0, L - 2:] = 0  # tokenizer padding on the last sample
    return x, enc, m

LATTE_SMALL = dict(num_attention_heads=2, attention_head_dim=72, in_channels=4, out_channels=8, num_layers=2,
                   cross_attention_dim=144, attention_bias=True, sample_size=8, patch_size=2, activation_fn="gelu-approximate",
                   norm_type="ada_norm_single", norm_elementwise_affine=False, norm_eps=1e-6, caption_channels=32, video_length=6)

LATTE_SMALL_O = dict(heads=2, head_dim=72, layers=2, patch=2, sample_size=8, out_channels=8, video_length=6)

LATTE_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 800], spatial_range=2, temporal_broadcast=True,
                    temporal_threshold=[100, 800], temporal_range=3, cross_broadcast=True, cross_threshold=[100, 800],
                    cross_range=6, mlp_broadcast=True, mlp_spatial_broadcast_config=OSP_PAB_MLP,
                    mlp_temporal_broadcast_config=OSP_PAB_MLP)

def latte_call(ref, x, t, enc, all_ts=(900, 500)):
    """The reference's LatteT2V call."""
    return ref(x, timestep=t, all_timesteps=torch.tensor(list(all_ts)), encoder_hidden_states=enc,
               added_cond_kwargs={"resolution": None, "aspect_ratio": None}, enable_temporal_attentions=True,
               return_dict=False)[0]

COGX_SMALL = dict(num_attention_heads=4, attention_head_dim=64, in_channels=4, out_channels=4, time_embed_dim=64, text_embed_dim=48,
                  num_layers=2, sample_width=16, sample_height=12, sample_frames=9, max_text_seq_length=16)

COGX_SMALL_O = dict(heads=4, head_dim=64, layers=2, patch=2, max_text=16, sample_width=16, sample_height=12, sample_frames=9,
                    out_channels=4)

COGX_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 850], spatial_range=2)

COGX_ROT_GRIDS = [(30, 45), (6, 8), (20, 20), (9, 40)]

def cogx_norms(sd, tag, dtype):
    for k in sd:
        if k.endswith("norm.weight") or k.endswith("norm_final.weight") or k.endswith("norm_q.weight") or k.endswith("norm_k.weight"):
            sd[k] = 1.0 + 0.2 * synth.uniform(tag + k, tuple(sd[k].shape))
    return {k: v.to(dtype) for k, v in sd.items()}

VCH_SMALL = dict(sample_size=8, patch_size=2, in_channels=4, num_layers=3, attention_head_dim=64, num_attention_heads=2,
                 joint_attention_dim=48, caption_projection_dim=128, pooled_projection_dim=40, out_channels=4, pos_embed_max_size=12)

VCH_SMALL_O = dict(heads=2, head_dim=64, layers=3, patch=2, sample_size=8, pos_embed_max_size=12, out_channels=4)

VCH_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 800], spatial_range=2, temporal_broadcast=True,
                  temporal_threshold=[100, 800], temporal_range=3, cross_broadcast=True, cross_threshold=[100, 800], cross_range=4)

def vch_sp_inputs(Fr):
    return synth.normalish("vchsp.lat", (1, Fr, 4, 12, 16)), synth.normalish("vchsp.enc", (1, 9, 48)), synth.normalish("vchsp.pool", (1, 40))

OSP12_SMALL = dict(num_attention_heads=2, attention_head_dim=96, in_channels=4, out_channels=8, num_layers=2, cross_attention_dim=192,
                   attention_bias=True, sample_size=(8, 8), sample_size_t=5, patch_size=2, patch_size_t=1,
                   activation_fn="gelu-approximate", norm_type="ada_norm_single", norm_elementwise_affine=False, norm_eps=1e-6,
                   caption_channels=32, interpolation_scale_h=1.0, interpolation_scale_w=2.0, interpolation_scale_t=1.5,
                   attention_mode="math", downsampler=None, use_rope=True)

OSP12_MIRROR_CASES = [(True, (8, 8)), (False, (8, 8)), (True, (12, 8))]

OSP12_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 850], spatial_range=2, cross_broadcast=True,
                    cross_threshold=[100, 850], cross_range=3)

def osp12_key(use_rope, HW):
    return f"osp12.{int(use_rope)}.{HW[0]}x{HW[1]}"

STDIT3_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 930], spatial_range=2, temporal_broadcast=True,
                     temporal_threshold=[100, 930], temporal_range=3, cross_broadcast=True, cross_threshold=[100, 930], cross_range=4)

STDIT3_PAB_TS = [900.0, 800.0, 700.0, 600.0, 500.0, 50.0]

def stdit3_run(model, inp, dt):
    f = lambda v: v.to(dt) if torch.is_tensor(v) and v.is_floating_point() else v  # noqa: E731
    with torch.no_grad():
        return model(f(inp["x"]), f(inp["timestep"]), f(inp["y"]), mask=inp["mask"], x_mask=inp["x_mask"], fps=f(inp["fps"]),
                     height=f(inp["height"]), width=f(inp["width"]))

def cogx_rotary(T=3, gh=6, gw=8, D=64):
    from oracle import cogvideox_oracle as CO

    return CO.rotary_3d(D, CO.resize_crop_region_for_grid((gh, gw), 45, 30), (gh, gw), T)


# STDiT3 with the reference's OpenSora PAB defaults (pab_oracle.opensora_default on the oracle side)
OPENSORA_PAB_STEPS = [1000, 900, 860, 800, 700, 600, 500, 300]
OPENSORA_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[450, 930], spatial_range=2, temporal_broadcast=True,
                       temporal_threshold=[450, 930], temporal_range=4, cross_broadcast=True, cross_threshold=[450, 930],
                       cross_range=6)
DSP_CASES = [(2, 5, 9), (4, 5, 9), (8, 20, 24), (4, 4, 8), (2, 15, 405)]  # (sp, T, S)
VCH_ATTN_C, VCH_ATTN_H = 64, 4
VCH_ATTN_CASES = [(5, 12, 7, False), (5, 12, 7, True), (1, 12, 7, False)]  # (frames, tokens, text tokens, context_pre_only)
VCH_ATTN_PAB_SHAPE = (4, 10, 6)
VCH_ATTN_PAB_KW = dict(spatial_broadcast=True, spatial_threshold=[100, 800], spatial_range=2, temporal_broadcast=True,
                       temporal_threshold=[100, 800], temporal_range=3, cross_broadcast=True, cross_threshold=[100, 800],
                       cross_range=4)


def pab_gate(kw, steps):
    """pab_oracle.PABGate for a reference PABConfig's attention-broadcast keywords."""
    return pab_oracle.PABGate(steps=steps, **{k: (kw[f"{k}_broadcast"], tuple(kw[f"{k}_threshold"]), kw[f"{k}_range"])
                                              for k in pab_oracle.PABGate.KINDS if kw.get(f"{k}_broadcast")})


def pab_gate_cases(n=20, seed=0):
    """Random PAB configurations: per case the gate spec, the step count and, per kind, the timesteps of 3 x steps calls
    (None = a call without a timestep)."""
    rnd = random.Random(seed)
    out = []
    for _ in range(n):
        spec = {}
        for k in pab_oracle.PABGate.KINDS:
            on = rnd.random() < 0.7
            lo = rnd.randrange(0, 600)
            hi = lo + rnd.randrange(1, 500)
            spec[k] = (on, (lo, hi), rnd.randrange(1, 7))
        steps = rnd.randrange(1, 40)
        ts = {k: [rnd.choice([None, rnd.randrange(0, 1100)]) for _ in range(3 * steps)] for k in pab_oracle.PABGate.KINDS}
        out.append((spec, steps, ts))
    return out


def pab_config_kw(spec):
    """The reference PABConfig keywords of a pab_gate_cases spec."""
    kw = {}
    for k, (on, (lo, hi), rg) in spec.items():
        kw.update({f"{k}_broadcast": on, f"{k}_threshold": [lo, hi], f"{k}_range": rg})
    return kw
