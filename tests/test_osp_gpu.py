"""Open-Sora-Plan v1.1.0 on the kernels against outputs of the UNMODIFIED reference model (tests/golden/osp_v110.pt, written
by oracle/gen_golden_osp.py in the authoring container; inputs and weights are regenerated here from oracle/osp_cases.py):
the half-rotation RoPE kernel against the reference's eager formula, the transformer forward (with / without RoPE, at the
released model's width), eight PAB steps incl. the MLP skip, the pipeline surface."""
import os

import pytest
import torch

from oracle import osp_cases as OC, pins, synth

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


@pytest.fixture(scope="module")
def gold(golden_dir):
    return torch.load(os.path.join(golden_dir, "osp_v110.pt"))


def _net(name, dt):
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V

    net = LatteT2V(**OC.CASES[name][0])
    net.load_state_dict(OC.weights(net.state_dict(), name, dt))
    return net.to(dt).to("cuda:0").eval()


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("H,D,half,rows,pos_div,pos_mod", [(16, 72, 18, 700, 1, 35),    # 2-D: (y, x) halves of the head, 5 x 7 grid
                                                            (16, 72, 36, 900, 60, 15),   # 1-D over frames, 60 patches per frame
                                                            (24, 96, 16, 333, 1, 111),   # 3-D (v1.2.0's head_dim 96 = 3 x 32)
                                                            (3, 64, 32, 77, 7, 11)])
def test_qk_rope_halves_kernel(H, D, half, rows, pos_div, pos_mod, dt):
    """vsb_qk_rope_halves against the reference's formula tokens*cos + rotate_half(tokens)*sin (RoPE1D.apply_rope1d,
    open_sora_plan_v110_transformer_3d.py:224-228) evaluated in the 16-bit dtype per rotation block: bit for bit; v untouched."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from videosys_b200 import kernels as K

    qkv = synth.normalish(f"ropek.{H}.{D}.{rows}", (rows, 3, H, D)).to(dt)
    ang = synth.uniform(f"ropek.ang.{pos_mod}.{D}", (pos_mod, D // (2 * half), half), -3.0, 3.0).to(dt)  # 16-bit angles
    ang = torch.cat([ang, ang], dim=-1)  # cat(freqs, freqs) per block
    cos, sin = ang.cos(), ang.sin()  # in the dtype, as the reference computes them
    sign = torch.cat([-torch.ones(half), torch.ones(half)])
    c32 = cos.float().reshape(pos_mod, D).contiguous()
    s32 = (sin.float() * sign).reshape(pos_mod, D).contiguous()
    got = K.qk_rope_halves_(qkv.clone().cuda(), c32.cuda(), s32.cuda(), H, D, half, pos_div, pos_mod).cpu()
    pos = (torch.arange(rows) // pos_div) % pos_mod
    want = qkv.clone()
    for i in (0, 1):
        t = qkv[:, i].reshape(rows, H, D // (2 * half), 2 * half)
        rot = torch.cat((-t[..., half:], t[..., :half]), dim=-1)  # rotate_half
        cc = cos.reshape(pos_mod, 1, D // (2 * half), 2 * half)[pos]
        ss = sin.reshape(pos_mod, 1, D // (2 * half), 2 * half)[pos]
        want[:, i] = ((t * cc) + (rot * ss)).reshape(rows, H, D)
    assert torch.equal(got[:, 2], qkv[:, 2]), "v must stay untouched"
    eq = (got == want).float().mean().item()
    print(f"[parity] qk_rope_halves {dt} H={H} D={D} half={half}: bit-equal {eq*100:.3f} %")
    assert torch.equal(got, want)


@pytest.mark.parametrize("dt,dn", [(torch.bfloat16, "bf16"), (torch.float16, "fp16")])
@pytest.mark.parametrize("name", list(OC.CASES))
def test_osp_v110_forward_vs_reference_golden(gold, name, dt, dn):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    net = _net(name, dt)
    x, enc, m, tt = OC.inputs(name, dt)
    out = net(x.cuda(), timestep=tt.cuda(), all_timesteps=[900, 500], encoder_hidden_states=enc.cuda(),
              attention_mask=torch.ones(x.shape[0], x.shape[2], x.shape[3], x.shape[4]), encoder_attention_mask=m,
              return_dict=False)[0].cpu()
    if f"{name}.{dn}.rel" in gold:  # stored as a sample and the norms (oracle/pins.rel): the full outputs exceed 1 MB
        pins.assert_rel(out, gold[f"{name}.{dn}.rel"], f"osp v110 {name} {dn}")
        return
    r32, r16 = gold[f"{name}.fp32"], gold[f"{name}.{dn}"]
    e_ours, e_ref = _rel(out, r32), _rel(r16, r32)
    print(f"[parity] osp v110 {name} {dn}: ours-vs-reference fp32 {e_ours:.3e}, reference {dn}-vs-fp32 {e_ref:.3e}, "
          f"bit-equal to the reference's {dn} output {(out == r16).float().mean().item()*100:.1f} %")
    assert out.shape == r32.shape
    assert e_ours <= 1.3 * e_ref + 1e-4


def test_osp_v110_pab_steps_vs_reference_golden(gold):
    """Eight steps with attention broadcast on all gates and the MLP skip windows; per step within the reference's own
    bf16 error, fewer kernels on the steps that reuse, every stored MLP output consumed."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from videosys_b200 import kernels
    from videosys_b200.core.pab import pab_mgr

    dt = torch.bfloat16
    net = _net("small_rope", dt)
    pab_mgr.set_pab_manager(pab_mgr.PABConfig(**OC.PAB_KW))
    pab_mgr.update_steps(len(OC.PAB_TIMESTEPS))
    net.reset_pab_state()
    try:
        launches = []
        for step, t in enumerate(OC.PAB_TIMESTEPS):
            x, enc, m, _ = OC.inputs("small_rope", dt, step)
            n0 = kernels.launch_count()
            out = net(x.cuda(), timestep=torch.tensor([t, t]).cuda(), all_timesteps=OC.PAB_TIMESTEPS,
                      encoder_hidden_states=enc.cuda(), encoder_attention_mask=m, return_dict=False, ts_int=t)[0].cpu()
            launches.append(kernels.launch_count() - n0)
            r32, r16 = gold[f"pab.{step}.fp32"], gold[f"pab.{step}.bf16"]
            e_ours, e_ref = _rel(out, r32), _rel(r16, r32)
            print(f"[parity] osp v110 PAB step {step} t={t}: ours-vs-reference fp32 {e_ours:.3e}, reference bf16-vs-fp32 {e_ref:.3e}, "
                  f"kernels {launches[-1]}")
            assert e_ours <= 1.3 * e_ref + 1e-4, step
        assert min(launches) < launches[0], launches
        assert not pab_mgr.PAB_MANAGER.get_spatial_mlp_outputs() and not pab_mgr.PAB_MANAGER.get_temporal_mlp_outputs()
    finally:
        pab_mgr.set_pab_manager(None)


def test_osp_pipeline_generate():
    """Public surface: OpenSoraPlanConfig(version='v110') -> VideoSysEngine.generate (tiny transformer, 6 PNDM steps = 15
    transformer evaluations), PAB off and on."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from videosys_b200 import OpenSoraPlanConfig, OpenSoraPlanV110PABConfig, VideoSysEngine, kernels
    from videosys_b200.core.pab import pab_mgr

    tc = dict(OC.CASES["small_rope"][0])
    kw = dict(num_inference_steps=6, guidance_scale=7.5, seed=0, height=64, width=64, max_sequence_length=24)
    eng = VideoSysEngine(OpenSoraPlanConfig(version="v110", transformer_type="65x512x512", transformer_config=tc))
    assert eng.driver_worker._dtype == torch.float16  # reference pipeline_open_sora_plan.py:262
    n0 = kernels.launch_count()
    out = eng.generate("Sunset over the sea.", **kw).video
    n_plain = kernels.launch_count() - n0
    assert out.shape == (1, 4, 5, 8, 8) and torch.isfinite(out).all()
    assert torch.equal(eng.generate("Sunset over the sea.", **kw).video, out), "same seed, same prompt -> same latents"
    eng.shutdown()
    pab = OpenSoraPlanV110PABConfig(spatial_threshold=(0, 1001), temporal_threshold=(0, 1001), cross_threshold=(0, 1001),
                                    mlp_spatial_broadcast_config={}, mlp_temporal_broadcast_config={})
    eng = VideoSysEngine(OpenSoraPlanConfig(version="v110", transformer_type="65x512x512", transformer_config=tc,
                                            enable_pab=True, pab_config=pab))
    try:
        n0 = kernels.launch_count()
        out2 = eng.generate("Sunset over the sea.", **kw).video
        n_pab = kernels.launch_count() - n0
        assert torch.isfinite(out2).all() and out2.shape == out.shape
        print(f"[pipeline] open-sora-plan v110 kernels launched: plain {n_plain}, PAB {n_pab}")
        assert n_pab < n_plain
    finally:
        pab_mgr.set_pab_manager(None)
        eng.shutdown()


# ---- Open-Sora-Plan v1.2.0 (OpenSoraT2V, head_dim 96) ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gold12(golden_dir):
    return torch.load(os.path.join(golden_dir, "osp_v120.pt"))


def _net12(name, dt):
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V

    net = OpenSoraT2V(**OC.CASES12[name][0])
    net.load_state_dict(OC.weights(net.state_dict(), "v120." + name, dt))
    return net.to(dt).to("cuda:0").eval()


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("nb,nq,nk,H,D,lens", [(2, 200, 200, 3, 96, None),        # self attention, ragged tiles (200 = 3 x 64 + 8)
                                               (3, 130, 77, 2, 96, [77, 13, 64]),  # cross attention with per-sample key counts
                                               (1, 64, 512, 4, 96, None),
                                               (2, 70, 100, 2, 128, [100, 1]),
                                               (2, 33, 65, 5, 32, None)])
def test_attn_mma_kernel(nb, nq, nk, H, D, lens, dt):
    """vsb_attn_flash for head dims without a tcgen05 layout (csrc/attn_mma.cu) against fp32 attention on the same 16-bit
    inputs: packed qkv (self) or separate q / kv buffers (cross), strided views, per-batch key counts."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from videosys_b200 import kernels as K

    C = H * D
    scale = D**-0.5
    if nq == nk and lens is None:  # packed qkv [nb, n, 3, C]
        qkv = synth.normalish(f"mma.qkv.{nb}.{nq}.{D}", (nb, nq, 3, C)).to(dt)
        g = qkv.cuda()
        q3 = g.view(nb * nq, 3, C)
        out = K.attn_flash(q3[:, 0], q3[:, 1], q3[:, 2], nb, nq, nk, H, D, 3 * C, nq * 3 * C, 3 * C, nk * 3 * C, scale).cpu()
        q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    else:
        q = synth.normalish(f"mma.q.{nb}.{nq}.{D}", (nb, nq, C)).to(dt)
        kv = synth.normalish(f"mma.kv.{nb}.{nk}.{D}", (nb, nk, 2, C)).to(dt)
        gq, gkv = q.cuda(), kv.cuda().view(nb * nk, 2, C)
        out = K.attn_flash(gq, gkv[:, 0], gkv[:, 1], nb, nq, nk, H, D, C, nq * C, 2 * C, nk * 2 * C, scale, kv_lens=lens).cpu()
        k, v = kv[:, :, 0], kv[:, :, 1]
    qh, kh, vh = (t.float().view(nb, -1, H, D).transpose(1, 2) for t in (q, k, v))
    mask = None
    if lens is not None:
        mask = torch.arange(nk).view(1, 1, 1, nk) < torch.tensor(lens).view(nb, 1, 1, 1)
    want = torch.nn.functional.scaled_dot_product_attention(qh, kh, vh, attn_mask=mask, scale=scale).transpose(1, 2).reshape(nb, nq, C)
    err = (out.float() - want).abs().max().item()
    rel = _rel(out, want)
    print(f"[parity] attn_mma {dt} nb={nb} nq={nq} nk={nk} H={H} D={D}: rel L2 {rel:.3e}, max abs {err:.3e}")
    assert rel < (6e-3 if dt == torch.bfloat16 else 1e-3)


@pytest.mark.parametrize("dt,dn", [(torch.bfloat16, "bf16"), (torch.float16, "fp16")])
@pytest.mark.parametrize("name", list(OC.CASES12))
def test_osp_v120_forward_vs_reference_golden(gold12, name, dt, dn):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    net = _net12(name, dt)
    x, enc, m, tt = OC.inputs12(name, dt)
    out = net(x.cuda(), timestep=tt.cuda(), encoder_hidden_states=enc.cuda(), encoder_attention_mask=m, return_dict=False)[0].cpu()
    r32, r16 = gold12[f"{name}.fp32"], gold12[f"{name}.{dn}"]
    e_ours, e_ref = _rel(out, r32), _rel(r16, r32)
    print(f"[parity] osp v120 {name} {dn}: ours-vs-reference fp32 {e_ours:.3e}, reference {dn}-vs-fp32 {e_ref:.3e}")
    assert out.shape == r32.shape
    assert e_ours <= 1.3 * e_ref + 1e-4


def test_osp_v120_pab_steps_vs_reference_golden(gold12):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from videosys_b200 import kernels
    from videosys_b200.core.pab import pab_mgr

    dt = torch.bfloat16
    net = _net12("small_rope", dt)
    pab_mgr.set_pab_manager(pab_mgr.PABConfig(**OC.PAB12_KW))
    pab_mgr.update_steps(len(OC.PAB_TIMESTEPS))
    net.reset_pab_state()
    try:
        launches = []
        for step, t in enumerate(OC.PAB_TIMESTEPS):
            x, enc, m, _ = OC.inputs12("small_rope", dt, step)
            n0 = kernels.launch_count()
            out = net(x.cuda(), timestep=torch.tensor([t, t]).cuda(), encoder_hidden_states=enc.cuda(), encoder_attention_mask=m,
                      return_dict=False, ts_int=t)[0].cpu()
            launches.append(kernels.launch_count() - n0)
            r32, r16 = gold12[f"pab.{step}.fp32"], gold12[f"pab.{step}.bf16"]
            e_ours, e_ref = _rel(out, r32), _rel(r16, r32)
            print(f"[parity] osp v120 PAB step {step} t={t}: ours-vs-reference fp32 {e_ours:.3e}, reference bf16-vs-fp32 {e_ref:.3e}, "
                  f"kernels {launches[-1]}")
            assert e_ours <= 1.3 * e_ref + 1e-4, step
        assert min(launches) < launches[0], launches
    finally:
        pab_mgr.set_pab_manager(None)


def test_osp_v120_pipeline_generate():
    """OpenSoraPlanConfig(version='v120') -> VideoSysEngine.generate on a tiny OpenSoraT2V: 6 ancestral Euler steps, PAB off / on."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from videosys_b200 import OpenSoraPlanConfig, OpenSoraPlanV120PABConfig, VideoSysEngine, kernels
    from videosys_b200.core.pab import pab_mgr

    tc = dict(OC.CASES12["small_rope"][0])
    kw = dict(num_inference_steps=6, guidance_scale=7.5, seed=0, max_sequence_length=24)
    eng = VideoSysEngine(OpenSoraPlanConfig(version="v120", transformer_type="29x480p", transformer_config=tc))
    n0 = kernels.launch_count()
    out = eng.generate("Sunset over the sea.", **kw).video
    n_plain = kernels.launch_count() - n0
    assert out.shape == (1, 4, 5, 8, 8) and torch.isfinite(out).all()
    assert torch.equal(eng.generate("Sunset over the sea.", **kw).video, out), "same seed, same prompt -> same latents"
    eng.shutdown()
    pab = OpenSoraPlanV120PABConfig(spatial_threshold=(0, 1001), cross_threshold=(0, 1001))
    eng = VideoSysEngine(OpenSoraPlanConfig(version="v120", transformer_type="29x480p", transformer_config=tc, enable_pab=True,
                                            pab_config=pab))
    try:
        n0 = kernels.launch_count()
        out2 = eng.generate("Sunset over the sea.", **kw).video
        n_pab = kernels.launch_count() - n0
        assert torch.isfinite(out2).all() and out2.shape == out.shape
        print(f"[pipeline] open-sora-plan v120 kernels launched: plain {n_plain}, PAB {n_pab}")
        assert n_pab < n_plain
    finally:
        pab_mgr.set_pab_manager(None)
        eng.shutdown()
