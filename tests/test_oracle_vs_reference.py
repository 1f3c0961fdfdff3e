"""Pins the oracle and the product's host logic to outputs of the UNMODIFIED reference.

tests/golden/reference_pins.pt.gz holds, for every check below, what the reference computed on the same synthetic weights and
inputs (oracle/gen_golden_pins.py executes it, with the configurations and input helpers of this module), in the compact
records of oracle/pins.py: bit-exact comparisons as SHA-256 digests, tolerance comparisons as a fixed sample plus whole-
tensor sums.  The weights are regenerated here from the reference's state-dict templates stored alongside."""
import os

import pytest
import torch

from oracle import cases, dsp_oracle, pab_oracle, pin_cases as PC, pins, stdit3_oracle as O, synth



@pytest.fixture(scope="module")
def pin(golden_dir):
    return pins.load(os.path.join(golden_dir, "reference_pins.pt.gz"))


def _fill(pin, key, tag):
    return pins.filled(pin["tmpl." + key], tag)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_forward_bit_exact(pin, dtype):
    c = cases.small_model_cfg(depth=2)
    sd = _fill(pin, f"stdit3.{PC.DT[dtype]}", "vsref.")
    inp = cases.forward_inputs(dtype)
    with torch.no_grad():
        out = O.stdit3_forward(sd, cases.oracle_cfg(c), **inp)
    pins.assert_exact(out, pin[f"stdit3.forward.{PC.DT[dtype]}"])


def test_forward_with_pab_bit_exact_over_steps(pin):
    """PAB on (attn + cross broadcast; mlp_broadcast=False, the only mode the reference can run for
    OpenSora, SURVEY fact 7): reuse-by-reference semantics and counters over 8 consecutive steps."""
    dtype = torch.bfloat16
    c = cases.small_model_cfg(depth=2)
    sd = _fill(pin, "stdit3.bfloat16", "vsref.")
    steps = PC.OPENSORA_PAB_STEPS
    gate = pab_oracle.opensora_default(len(steps))
    states = {k: [O.BlockPABState() for _ in range(2)] for k in ("spatial", "temporal")}
    inp = cases.forward_inputs(dtype)
    with torch.no_grad():
        for i, t in enumerate(steps):
            inp["x"] = synth.normalish(f"pab.x{i}", tuple(inp["x"].shape))
            inp["timestep"] = torch.tensor([float(t)] * 2)
            o = O.stdit3_forward(sd, cases.oracle_cfg(c), pab=gate, pab_states=states, **inp)
            pins.assert_exact(o, pin[f"stdit3.pab.{i}"], f"step {i} t={t}")


def test_pab_gate_matches_reference_manager(pin):
    got = []
    for spec, steps, ts in PC.pab_gate_cases():
        g = pab_oracle.PABGate(steps=steps, **spec)
        for k in ("spatial", "temporal", "cross"):
            c2 = 0
            for t in ts[k]:
                f2, c2 = g.gate(k, t, c2)
                got.append((int(f2), c2))
    pins.assert_exact(torch.tensor(got, dtype=torch.int64), pin["pab_gate"], "(broadcast, counter) after every call")


@pytest.mark.parametrize("sp,T,S", PC.DSP_CASES)
def test_dsp_reshard_matches_reference_comm(pin, sp, T, S):
    B, C = 2, 16
    full = synth.normalish(f"dsp{sp}{T}{S}", (B, T, S, C))
    tp, spd = dsp_oracle.pad_amount(T, sp), dsp_oracle.pad_amount(S, sp)
    res = dsp_oracle.split_sequence(full, sp, dim=2)
    parts = [p.reshape(B, -1, C) for p in res]
    sw, new_s, new_t = dsp_oracle.dynamic_switch(parts, T, S, to_spatial_shard=False)
    back, s2, t2 = dsp_oracle.dynamic_switch(sw, T, S, to_spatial_shard=True)
    padded_t = torch.cat([full, torch.zeros(B, tp, S, C)], 1)
    recs = pin[f"dsp.{sp}.{T}.{S}"]
    assert len(recs) == sp
    for r in range(sp):
        rx, ra, rb = recs[r]
        pins.assert_exact(res[r], rx, f"rank {r} split")
        a = padded_t[:, r * new_t:(r + 1) * new_t]  # Appendix E: a slice of the T-padded tensor
        pins.assert_exact(a, ra, f"rank {r} to temporal shard")
        assert ra["shape"][1:3] == (new_t, new_s) and torch.equal(a.reshape(B, -1, C), sw[r])
        pins.assert_exact(back[r].reshape(res[r].shape), rb, f"rank {r} back to spatial shard")
        assert rb == rx
    assert torch.equal(dsp_oracle.gather_sequence(res, 2, spd), full)




@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_cogvideox_layernorm_zero(pin, dtype):
    """The in-tree half of the CogVideoX block: CogVideoXLayerNormZero (models/modules/normalization.py:36-57)."""
    from oracle import cogvideox_oracle as CO

    sd = {"n." + k: v for k, v in _fill(pin, f"lnz.{PC.DT[dtype]}", "lnz.").items()}
    sd["n.norm.weight"] = (1 + 0.2 * synth.uniform("lnz.w", (128,))).to(dtype)
    with torch.no_grad():
        got = CO.layer_norm_zero(sd, "n.", *PC.lnz_inputs(dtype))
    want = pin[f"lnz.{PC.DT[dtype]}"]
    assert len(got) == len(want)
    for a, rec in zip(got, want):
        pins.assert_exact(a, rec)




def test_cogvideox_ddim_scheduler_vs_reference(pin):
    """videosys_b200's CogVideoXDDIMScheduler against the reference's own class: trailing timesteps, the SNR-shifted /
    zero-terminal-SNR alphas, and 50 v-prediction steps on random tensors."""
    from videosys_b200.schedulers.scheduling_ddim_cogvideox import CogVideoXDDIMScheduler as Ours

    rec = pin["cogx_ddim"]
    ours = Ours(**PC.COGX_DDIM)
    pins.assert_exact(ours.alphas_cumprod, rec["alphas_cumprod"])
    for n in (50, 30, 7):
        ours.set_timesteps(n)
        assert ours.timesteps.tolist() == rec["timesteps"][n]
    ours.set_timesteps(50)
    g = torch.Generator().manual_seed(0)
    xo = torch.randn(1, 3, 4, 6, 6, generator=g)
    assert len(rec["steps"]) == len(ours.timesteps)
    for t, want in zip(rec["timesteps"][50], rec["steps"]):
        v = torch.randn(xo.shape, generator=g)
        xo = ours.step(v, int(t), xo)[0]
        pins.assert_close(xo.float(), want, rtol=1e-5, atol=1e-6, what=int(t))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Fr,S,L,pre_only", PC.VCH_ATTN_CASES)
def test_vchitect_attention_vs_reference(pin, Fr, S, L, pre_only, dtype):
    """oracle/vchitect_oracle.attention against the reference's own VchitectAttention + VchitectAttnProcessor
    (models/modules/attentions.py:321-949): temporal (RoPE), cross (frame-0 text keys) and spatial joint attention, the
    1.1 mix, the output projections of both streams; bit for bit."""
    from oracle import vchitect_oracle as VO

    C, H = PC.VCH_ATTN_C, PC.VCH_ATTN_H
    sd = {"a." + k: v for k, v in _fill(pin, f"vch_attn.{int(pre_only)}.{PC.DT[dtype]}", "vchattn.").items()}
    nh = synth.normalish("vch.h", (Fr, S, C)).to(dtype)
    ne = synth.normalish("vch.e", (Fr, L, C)).to(dtype)
    fc = VO.freqs_cis(C // H, 64, theta=1e6)
    with torch.no_grad():
        ov, oe = VO.attention(sd, "a.", nh, ne, fc, H, Fr, pre_only)
    rv, re = pin[f"vch_attn.{Fr}.{S}.{L}.{int(pre_only)}.{PC.DT[dtype]}"]
    pins.assert_exact(ov, rv, "video stream")
    pins.assert_exact(oe, re, "text stream")


def test_vchitect_attention_pab_vs_reference(pin):
    """The three PAB gates of the processor (:838-895: temporal, cross, spatial, in this order) over 8 steps."""
    from oracle import vchitect_oracle as VO

    (C, H), (Fr, S, L) = (PC.VCH_ATTN_C, PC.VCH_ATTN_H), PC.VCH_ATTN_PAB_SHAPE
    sd = {"a." + k: v for k, v in _fill(pin, "vch_attn.0.float32", "vchattn.").items()}
    fc = VO.freqs_cis(C // H, 64, theta=1e6)
    counts = {"spatial": 0, "temporal": 0, "cross": 0}
    cache = {}
    G = PC.pab_gate(PC.VCH_ATTN_PAB_KW, len(PC.PAB_TS))
    for step, t in enumerate(PC.PAB_TS):
        nh = synth.normalish(f"vchp.h{step}", (Fr, S, C))
        ne = synth.normalish(f"vchp.e{step}", (Fr, L, C))

        def gate(kind, t=t):
            hit, counts[kind] = G.gate(kind, t, counts[kind])
            return hit

        with torch.no_grad():
            ov, oe = VO.attention(sd, "a.", nh, ne, fc, H, Fr, False, gate, cache)
        rv, re = pin[f"vch_attn_pab.{step}"]
        pins.assert_exact(ov, rv, step)
        pins.assert_exact(oe, re, step)


# ---- Open-Sora-Plan v1.1.0: the product's host logic against the UNMODIFIED reference model --------------------------------




def _osp_net(pin, cfg, key, tag):
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V

    net = LatteT2V(**cfg)
    net.load_state_dict(_fill(pin, key, tag))  # strict: same parameter / buffer names as the reference
    return net.eval()




@pytest.mark.parametrize("use_rope,HW,scale1d", PC.OSP_MIRROR_CASES)
def test_osp_v110_mirror_vs_reference_model(pin, monkeypatch, use_rope, HW, scale1d):
    """videosys_b200's Open-Sora-Plan v1.1.0 front end, its kernel entries replaced by torch stand-ins
    (tests/kernels_emul.py), against the reference's own LatteT2V: RoPE tables (2-D / 1-D, linear scaling), position tables,
    text padding mask, block order, output head."""
    from tests import kernels_emul

    kernels_emul.emulate(monkeypatch)
    key = PC.osp_key(use_rope, HW, scale1d)
    net = _osp_net(pin, dict(PC.OSP_SMALL, use_rope=use_rope, interpolation_scale_1d=scale1d), key, "osp.")
    B, Fr = 2, 5
    x, enc, m = PC.osp_inputs(B, Fr, HW)
    got = net(x, timestep=torch.tensor([500, 500]), all_timesteps=[900, 500], encoder_hidden_states=enc,
              attention_mask=torch.ones(B, Fr, *HW), encoder_attention_mask=m, return_dict=False)[0]
    pins.assert_close(got, pin[key], rtol=1e-4, atol=1e-5)


def test_osp_v110_pab_vs_reference_model(pin, monkeypatch):
    """Eight steps with PAB (attention broadcast on all three gates + the MLP skip windows) on both sides."""
    from tests import kernels_emul
    from videosys_b200.core.pab import pab_mgr as ours

    kernels_emul.emulate(monkeypatch)
    net = _osp_net(pin, PC.OSP_SMALL, "ospp", "ospp.")
    ours.set_pab_manager(ours.PABConfig(**PC.OSP_PAB_KW))
    ours.update_steps(len(PC.PAB_TS))
    net.reset_pab_state()
    try:
        B, Fr, HW = 2, 5, (8, 8)
        for step, t in enumerate(PC.PAB_TS):
            x, enc, m = PC.osp_inputs(B, Fr, HW, tag=f"ospp{step}.")
            got = net(x, timestep=torch.tensor([t, t]), all_timesteps=PC.PAB_TS, encoder_hidden_states=enc, encoder_attention_mask=m,
                      return_dict=False)[0]
            pins.assert_close(got, pin[f"ospp.{step}"], rtol=1e-4, atol=1e-5, what=step)
    finally:
        ours.set_pab_manager(None)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_osp_v110_rope_tables_vs_reference_classes(pin, dtype):
    """The cos / signed-sin tables of vsb_qk_rope_halves against LinearScalingRoPE2D / LinearScalingRoPE1D run on q itself:
    q*cos + partner*sin_signed, evaluated op by op in the dtype, equals the reference's output bit for bit."""
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import rope_tables

    D, Hh, h, w, Fr = 72, 3, 5, 7, 9
    want2, want1 = pin[f"osp_rope.{PC.DT[dtype]}"]
    q2 = synth.normalish("rope.q2", (2, Hh, h * w, D)).to(dtype)
    yx = torch.cartesian_prod(torch.arange(h), torch.arange(w))
    c, s, half = rope_tables(D, [yx[:, 0], yx[:, 1]], 2, dtype, "cpu")
    assert half == 18

    def apply(q, c, s, half):
        partner = q.reshape(*q.shape[:-1], D // (2 * half), 2, half).flip(-2).reshape(q.shape)
        return q * c.to(dtype) + partner * s.to(dtype)

    pins.assert_exact(apply(q2, c, s, half), want2, "2-D")
    q1 = synth.normalish("rope.q1", (4, Hh, Fr, D)).to(dtype)
    c, s, half = rope_tables(D, [torch.arange(Fr)], 2, dtype, "cpu")
    assert half == 36
    pins.assert_exact(apply(q1, c, s, half), want1, "1-D")


# ---- Latte: oracle and product host logic against the UNMODIFIED reference model ---------------------------------------------


def _latte_sd(pin, dtype=torch.float32):
    return {k: v.to(dtype) for k, v in _fill(pin, f"latte.{PC.DT[dtype]}", "lattep.").items()}




@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_latte_oracle_vs_reference_model(pin, dtype):
    """oracle/latte_oracle.transformer_forward against the reference's own LatteT2V (models/transformers/
    latte_transformer_3d.py): the whole forward -- PatchEmbed + 2-D sin-cos table, AdaLayerNormSingle, caption projection,
    both block kinds, temp_pos_embed, output head, un-patchify.  fp32: equal up to summation order; bf16: bit for bit."""
    from oracle import latte_oracle as LO

    sd = _latte_sd(pin, dtype)
    x = synth.normalish("lattep.x", (2, 4, 6, 8, 8)).to(dtype)
    enc = synth.normalish("lattep.enc", (2, 7, 32)).to(dtype)
    with torch.no_grad():
        got = LO.transformer_forward(sd, PC.LATTE_SMALL_O, x, torch.tensor([500, 500]), enc)
    if dtype == torch.float32:
        pins.assert_close(got, pin["latte.float32"], rtol=1e-4, atol=1e-5)
    else:
        pins.assert_exact(got, pin["latte.bfloat16"], "latte oracle bf16")


def test_latte_mirror_vs_reference_model(pin, monkeypatch):
    """videosys_b200's LatteT2V (kernel entries = torch stand-ins) against the reference model, fp32, incl. 8 PAB steps with the
    MLP skip on both sides."""
    from tests import kernels_emul
    from videosys_b200.core.pab import pab_mgr as ours
    from videosys_b200.models.transformers.latte_transformer_3d import LatteT2V

    kernels_emul.emulate(monkeypatch)
    net = LatteT2V(**PC.LATTE_SMALL)
    net.load_state_dict(_latte_sd(pin))
    net.eval()
    x = synth.normalish("lattep.x", (2, 4, 6, 8, 8))
    enc = synth.normalish("lattep.enc", (2, 7, 32))
    got = net(x, timestep=torch.tensor([500, 500]), all_timesteps=[900, 500], encoder_hidden_states=enc, return_dict=False)[0]
    pins.assert_close(got, pin["latte.float32"], rtol=1e-4, atol=1e-5)
    ours.set_pab_manager(ours.PABConfig(**PC.LATTE_PAB_KW))
    ours.update_steps(len(PC.PAB_TS))
    net.reset_pab_state()
    try:
        for step, tv in enumerate(PC.PAB_TS):
            x = synth.normalish(f"lattep.x{step}", (2, 4, 6, 8, 8))
            got = net(x, timestep=torch.tensor([tv, tv]), all_timesteps=PC.PAB_TS, encoder_hidden_states=enc, return_dict=False)[0]
            pins.assert_close(got, pin[f"latte.pab.{step}"], rtol=1e-4, atol=1e-5, what=step)
    finally:
        ours.set_pab_manager(None)


# ---- CogVideoX: oracle and product host logic against the UNMODIFIED reference model ------------------------------------------


def cogx_weights(pin, key, tag, dtype):
    """synth weights for the reference's CogVideoX state dict (fp32 template), LayerNorm weights around 1 (fill_state_dict
    treats them as matrices), cast to dtype."""
    return PC.cogx_norms(_fill(pin, key, tag), tag, dtype)




@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_cogvideox_oracle_vs_reference_model(pin, dtype):
    """oracle/cogvideox_oracle.transformer_forward against the reference's own CogVideoXTransformer3DModel: patch / text
    embedding, position table, LayerNormZero blocks with the joint-attention processor, norm_final + AdaLayerNorm head,
    un-patchify."""
    from oracle import cogvideox_oracle as CO

    sd = cogx_weights(pin, f"cogxp.{PC.DT[dtype]}", "cogxp.", dtype)
    lat = synth.normalish("cogxp.lat", (2, 3, 4, 12, 16)).to(dtype)
    txt = synth.normalish("cogxp.txt", (2, 16, 48)).to(dtype)
    with torch.no_grad():
        got = CO.transformer_forward(sd, PC.COGX_SMALL_O, lat, txt, torch.tensor([499, 499]))
    if dtype == torch.float32:
        pins.assert_close(got, pin["cogx.float32"], rtol=1e-4, atol=1e-5)
    else:
        pins.assert_exact(got, pin[f"cogx.{PC.DT[dtype]}"], f"cogvideox oracle {dtype}")


def test_cogvideox_mirror_vs_reference_model(pin, monkeypatch):
    """videosys_b200's CogVideoXTransformer3DModel (kernel entries = torch stand-ins) against the reference model, fp32, plain
    and over 8 PAB steps."""
    from tests import kernels_emul
    from videosys_b200.core.pab import pab_mgr as ours
    from videosys_b200.models.transformers.cogvideox_transformer_3d import CogVideoXTransformer3DModel

    kernels_emul.emulate(monkeypatch)
    sd = cogx_weights(pin, "cogxp.float32", "cogxp.", torch.float32)
    net = CogVideoXTransformer3DModel(**PC.COGX_SMALL)
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert not missing and all(".attn1.to_" in k and ("_temp" in k or "_cross" in k or "_context" in k or "temporal" in k)
                               for k in unexpected), (missing, unexpected)  # the vendored Attention's Vchitect-only members
    net.eval()
    lat = synth.normalish("cogxp.lat", (2, 3, 4, 12, 16))
    txt = synth.normalish("cogxp.txt", (2, 16, 48))
    got = net(lat, txt, torch.tensor([499, 499]), return_dict=False)[0]
    pins.assert_close(got, pin["cogx.float32"], rtol=1e-4, atol=1e-5)
    ours.set_pab_manager(ours.PABConfig(**PC.COGX_PAB_KW))
    ours.update_steps(len(PC.PAB_TS))
    net.reset_pab_state()
    try:
        for step, tv in enumerate(PC.PAB_TS):
            lat = synth.normalish(f"cogxp.lat{step}", (2, 3, 4, 12, 16))
            got = net(lat, txt, torch.tensor([tv, tv]), return_dict=False)[0]
            pins.assert_close(got, pin[f"cogx.pab.{step}"], rtol=1e-4, atol=1e-5, what=step)
    finally:
        ours.set_pab_manager(None)


# ---- Vchitect: oracle and product host logic against the UNMODIFIED reference transformer ---------------------------------------


def _vch_sd(pin, dtype=torch.float32):
    """The reference's weights: synth fill of its state dict, its own sin-cos position table kept (not a weight; the product
    module builds the same table, checked bit for bit against the reference's)."""
    from videosys_b200.models.transformers.vchitect_transformer_3d import VchitectXLTransformerModel

    table = VchitectXLTransformerModel(**PC.VCH_SMALL).state_dict()["pos_embed.pos_embed"].float()
    pins.assert_exact(table.to(dtype), pin[f"vchm.pos_embed.{PC.DT[dtype]}"], "position table")
    sd = _fill(pin, f"vchm.{PC.DT[dtype]}", "vchm.")
    sd["pos_embed.pos_embed"] = table
    return {k: v.to(dtype) for k, v in sd.items()}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Fr", [5, 1])
def test_vchitect_oracle_vs_reference_model(pin, Fr, dtype):
    """oracle/vchitect_oracle.transformer_forward against the reference's VchitectXLTransformerModel (vchitect_transformer_3d.py
    on the reference's VchitectAttention): per-frame text broadcast in the first block, context_pre_only last block, the three
    attentions, norm_out, un-patchify."""
    from oracle import vchitect_oracle as VO

    sd = _vch_sd(pin, dtype)
    lat = synth.normalish("vchm.lat", (1, Fr, 4, 12, 16)).to(dtype)
    enc = synth.normalish("vchm.enc", (1, 9, 48)).to(dtype)
    pooled = synth.normalish("vchm.pool", (1, 40)).to(dtype)
    with torch.no_grad():
        got = VO.transformer_forward(sd, PC.VCH_SMALL_O, lat, enc, pooled, torch.tensor([500.0]))
    if dtype == torch.float32:
        pins.assert_close(got, pin[f"vch.{Fr}.float32"], rtol=1e-4, atol=1e-5)
    else:
        pins.assert_exact(got, pin[f"vch.{Fr}.bfloat16"], "vchitect oracle bf16")


def test_vchitect_mirror_vs_reference_model(pin, monkeypatch):
    """videosys_b200's VchitectXLTransformerModel (kernel entries = torch stand-ins) against the reference model: strict
    state-dict compatibility, fp32 forward, and 8 steps with the three PAB gates on both sides."""
    from tests import kernels_emul
    from videosys_b200.core.pab import pab_mgr as ours
    from videosys_b200.models.transformers.vchitect_transformer_3d import VchitectXLTransformerModel

    kernels_emul.emulate(monkeypatch)
    net = VchitectXLTransformerModel(**PC.VCH_SMALL)
    net.load_state_dict(_vch_sd(pin))  # strict
    net.eval()
    enc = synth.normalish("vchm.enc", (1, 9, 48))
    pooled = synth.normalish("vchm.pool", (1, 40))
    for pab in (False, True):
        steps = PC.PAB_TS if pab else [500]
        if pab:
            ours.set_pab_manager(ours.PABConfig(**PC.VCH_PAB_KW))
            ours.update_steps(len(steps))
            net.reset_pab_state()
        try:
            for step, tv in enumerate(steps):
                lat = synth.normalish(f"vchm.lat{step}", (1, 4, 4, 12, 16))
                got = net(lat, enc, pooled, torch.tensor([float(tv)]), return_dict=False)[0]
                pins.assert_close(got, pin[f"vch.mirror.{int(pab)}.{step}"], rtol=1e-4, atol=1e-5, what=(pab, step))
        finally:
            ours.set_pab_manager(None)




def _vch_sp_worker(rank, world, port, Fr, sd, q):
    import traceback

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    try:
        import torch.distributed as dist

        from tests import kernels_emul
        from videosys_b200.core.distributed.parallel_mgr import initialize
        from videosys_b200.models.transformers.vchitect_transformer_3d import VchitectXLTransformerModel

        kernels_emul.emulate_global()
        initialize(rank, world)

        def a2a(out_list, in_list, group=None):  # gloo has no all_to_all: the same exchange through all_to_all_single
            send = torch.stack([t.contiguous() for t in in_list])
            recv = torch.empty_like(send)
            dist.all_to_all_single(recv, send, group=group)
            for o, r in zip(out_list, recv.unbind(0)):
                o.copy_(r)

        dist.all_to_all = a2a
        net = VchitectXLTransformerModel(**PC.VCH_SMALL)
        net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        net.eval()
        net.enable_parallel(1, world, False)
        lat, enc, pooled = PC.vch_sp_inputs(Fr)
        got = net(lat, enc, pooled, torch.tensor([500.0]), return_dict=False)[0]
        q.put((rank, got.detach().numpy(), None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:  # pragma: no cover
        q.put((rank, None, traceback.format_exc()))


@pytest.mark.parametrize("Fr", [4, 5, 2])  # 5 frames: a zero frame pads the last rank; 2: one frame per rank (temporal branch * 0)
def test_vchitect_sequence_parallel_vs_reference_gloo_world2(pin, monkeypatch, Fr):
    """Two gloo ranks running videosys_b200's transformer (kernel entries = torch stand-ins) under frame-sharded sequence
    parallelism against what the UNMODIFIED reference transformer computed on every rank under the same sharding, incl. the
    reference's quirks under sp (cross attention against the text keys of the rank's own first frame, cur_frame == 1 judged
    on the local frame count)."""
    import multiprocessing as mp

    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")  # CPU ranks on gloo: with a GPU visible, initialize() picks NCCL
    world, port = 2, 30700 + (os.getpid() % 250) + Fr
    sd = {k: v.numpy() for k, v in _vch_sd(pin).items()}  # by value: no shared-memory handles that die with the worker
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_vch_sp_worker, args=(r, world, port, Fr, sd, q)) for r in range(world)]
    [p.start() for p in procs]
    recs = pin[f"vch.sp.{Fr}"]
    for _ in range(world):
        r, got, tb = q.get(timeout=300)
        assert tb is None, tb
        pins.assert_close(torch.from_numpy(got), recs[r], rtol=0.0, atol=1e-4 * max(recs[r]["max_abs"], 1.0), what=r)
    [p.join(timeout=60) for p in procs]


# ---- Open-Sora-Plan v1.2.0: the product's host logic against the UNMODIFIED reference model --------------------------------




def _osp12_net(pin, cfg, key, tag):
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V

    net = OpenSoraT2V(**cfg)
    net.load_state_dict(_fill(pin, key, tag))  # strict
    return net.eval()


@pytest.mark.parametrize("use_rope,HW", PC.OSP12_MIRROR_CASES)
def test_osp_v120_mirror_vs_reference_model(pin, monkeypatch, use_rope, HW):
    """videosys_b200's OpenSoraT2V (kernel entries = torch stand-ins) against the reference's own OpenSoraT2V: RoPE3D tables
    with per-axis interpolation scales, absolute position tables when RoPE is off, text padding mask, block order, output
    head / un-patchify."""
    from tests import kernels_emul

    kernels_emul.emulate(monkeypatch)
    key = PC.osp12_key(use_rope, HW)
    net = _osp12_net(pin, dict(PC.OSP12_SMALL, use_rope=use_rope), key, "osp12.")
    x, enc, m = PC.osp_inputs(2, 5, HW, tag="osp12.")
    got = net(x, timestep=torch.tensor([500, 500]), encoder_hidden_states=enc, encoder_attention_mask=m, return_dict=False)[0]
    pins.assert_close(got, pin[key], rtol=1e-4, atol=1e-5)


def test_osp_v120_pab_vs_reference_model(pin, monkeypatch):
    from tests import kernels_emul
    from videosys_b200.core.pab import pab_mgr as ours

    kernels_emul.emulate(monkeypatch)
    net = _osp12_net(pin, PC.OSP12_SMALL, "osp12p", "osp12p.")
    ours.set_pab_manager(ours.PABConfig(**PC.OSP12_PAB_KW))
    ours.update_steps(len(PC.PAB_TS))
    net.reset_pab_state()
    try:
        for step, t in enumerate(PC.PAB_TS):
            x, enc, m = PC.osp_inputs(2, 5, (8, 8), tag=f"osp12p{step}.")
            got = net(x, timestep=torch.tensor([t, t]), encoder_hidden_states=enc, encoder_attention_mask=m, return_dict=False)[0]
            pins.assert_close(got, pin[f"osp12p.{step}"], rtol=1e-4, atol=1e-5, what=step)
    finally:
        ours.set_pab_manager(None)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_osp_v120_rope3d_tables_vs_reference_class(pin, dtype):
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import rope3d_tables

    D, Hh, T, h, w = 96, 3, 4, 3, 5
    q = synth.normalish("rope3.q", (2, Hh, T * h * w, D)).to(dtype)
    c, s, half = rope3d_tables(D, T, h, w, (1.5, 1.0, 2.0), dtype, "cpu")
    assert half == 16
    partner = q.reshape(*q.shape[:-1], D // (2 * half), 2, half).flip(-2).reshape(q.shape)
    pins.assert_exact(q * c.to(dtype) + partner * s.to(dtype), pin[f"osp12_rope3d.{PC.DT[dtype]}"])






def test_stdit3_mirror_vs_reference_model(pin, monkeypatch):
    """The headline model's front end (videosys_b200 STDiT3, kernel entries = torch stand-ins, bf16 as it insists) against
    the reference STDiT3: within the reference's own bf16-vs-fp32 error, with PAB off and over 6 PAB steps (hoisted text
    projections, modulation tables, per-frame mask select, final layer on the shard, un-patchify)."""
    from tests import kernels_emul
    from videosys_b200.core.pab import pab_mgr as ours
    from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config

    kernels_emul.emulate(monkeypatch)
    c = cases.small_model_cfg(depth=2)
    net = STDiT3(STDiT3Config(**c)).to(torch.bfloat16)
    net.load_state_dict(_fill(pin, "stde.bfloat16", "stde."))
    net.eval()
    inp = cases.forward_inputs(torch.bfloat16)
    pins.assert_rel(PC.stdit3_run(net, inp, torch.bfloat16), pin["stde.0"], "PAB off")
    ours.set_pab_manager(ours.PABConfig(**PC.STDIT3_PAB_KW))
    ours.update_steps(len(PC.STDIT3_PAB_TS))
    net.reset_pab_state()
    try:
        for i, t in enumerate(PC.STDIT3_PAB_TS):
            inp["timestep"] = torch.tensor([t, t], dtype=torch.bfloat16)
            pins.assert_rel(PC.stdit3_run(net, inp, torch.bfloat16), pin[f"stde.{i + 1}"], i)
    finally:
        ours.set_pab_manager(None)


# ---- CogVideoX-5b: rotary position embeddings ------------------------------------------------------------------------------------


def test_cogvideox_rotary_helpers_vs_reference(pin):
    """oracle rotary_3d / resize_crop_region_for_grid / apply_rotary_emb and the pipeline mirror's
    _prepare_rotary_positional_embeddings against the reference's own functions (models/modules/embeddings.py:283-412,
    pipelines/cogvideox/pipeline_cogvideox.py:758-773 -- the pipeline module itself needs diffusers: its crop helper is
    compared through its published formula on the oracle side)."""
    from oracle import cogvideox_oracle as CO
    from videosys_b200.pipelines.cogvideox.pipeline_cogvideox import CogVideoXPipeline

    for (gh, gw) in PC.COGX_ROT_GRIDS:
        rc, rs = pin[f"cogx_rot.grid.{gh}x{gw}"]
        oc, os_ = CO.rotary_3d(64, CO.resize_crop_region_for_grid((gh, gw), 45, 30), (gh, gw), 5)
        pins.assert_exact(oc, rc, (gh, gw))
        pins.assert_exact(os_, rs, (gh, gw))
        pipe = CogVideoXPipeline.__new__(CogVideoXPipeline)
        pipe.transformer = type("T", (), {"config": type("C", (), {"patch_size": 2, "attention_head_dim": 64})()})()
        pc, ps = pipe._prepare_rotary_positional_embeddings(gh * 16, gw * 16, 5, "cpu")
        pins.assert_exact(pc, rc, ("pipeline", gh, gw))
        pins.assert_exact(ps, rs, ("pipeline", gh, gw))
    for dtype in (torch.float32, torch.bfloat16):
        x = synth.normalish("rot.x", (2, 3, 3 * 6 * 8, 64)).to(dtype)
        c, s = PC.cogx_rotary()
        pins.assert_exact(CO.apply_rotary_emb(x, c, s), pin[f"cogx_rot.apply.{PC.DT[dtype]}"], dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_cogvideox_rotary_oracle_and_mirror_vs_reference_model(pin, monkeypatch, dtype):
    """use_rotary_positional_embeddings=True (CogVideoX-5b): oracle forward (bf16 bit for bit) and, in fp32, the product front end
    on the kernel stand-ins (identity rope rows for the text tokens, RoPE-only pre-pass) against the reference model."""
    from oracle import cogvideox_oracle as CO
    from tests import kernels_emul
    from videosys_b200.models.transformers.cogvideox_transformer_3d import CogVideoXTransformer3DModel

    cfg = dict(PC.COGX_SMALL, use_rotary_positional_embeddings=True)
    sd = cogx_weights(pin, f"cogxr.{PC.DT[dtype]}", "cogxr.", dtype)
    lat = synth.normalish("cogxr.lat", (2, 3, 4, 12, 16)).to(dtype)
    txt = synth.normalish("cogxr.txt", (2, 16, 48)).to(dtype)
    ts = torch.tensor([499, 499])
    rot = PC.cogx_rotary()
    with torch.no_grad():
        got = CO.transformer_forward(sd, PC.COGX_SMALL_O, lat, txt, ts, rotary=rot)
    if dtype == torch.float32:
        pins.assert_close(got, pin["cogx_rot.float32"], rtol=1e-4, atol=1e-5)
        kernels_emul.emulate(monkeypatch)
        net = CogVideoXTransformer3DModel(**cfg)
        missing, unexpected = net.load_state_dict(sd, strict=False)
        assert not missing
        out = net.eval()(lat, txt, ts, image_rotary_emb=rot, return_dict=False)[0]
        pins.assert_close(out, pin["cogx_rot.float32"], rtol=1e-4, atol=1e-5)
    else:
        pins.assert_exact(got, pin["cogx_rot.bfloat16"], "cogvideox rotary oracle bf16")
