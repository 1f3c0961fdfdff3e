"""Host logic of the model mirrors that widen the path (SURVEY.md section 8 (f)4) on the CPU: every kernel entry is replaced
by its torch stand-in (tests/kernels_emul.py, test infrastructure), so what is checked here is what the front end does
around the kernels -- layouts and strides handed to the attention entries, weight fusion, PAB bookkeeping, un-patchify --
against the oracle in fp32 (tight tolerance: same arithmetic, different op order).  The GPU parity of the same models is
in tests/test_vchitect_gpu.py / tests/test_osp_gpu.py."""
import pytest
import torch

from oracle import pab_oracle, synth
from tests import kernels_emul

VCH = dict(sample_size=8, patch_size=2, in_channels=4, num_layers=3, attention_head_dim=64, num_attention_heads=2,
           joint_attention_dim=48, caption_projection_dim=128, pooled_projection_dim=40, out_channels=4, pos_embed_max_size=12)
VCH_O = dict(heads=2, head_dim=64, layers=3, patch=2, sample_size=8, pos_embed_max_size=12, out_channels=4)


def _vchitect(tag="vch."):
    from videosys_b200.models.transformers.vchitect_transformer_3d import VchitectXLTransformerModel

    net = VchitectXLTransformerModel(**VCH)
    sd = synth.fill_state_dict(net.state_dict(), tag)
    sd["pos_embed.pos_embed"] = net.state_dict()["pos_embed.pos_embed"]  # the sin-cos table is not a weight
    net.load_state_dict(sd)
    return net.eval(), sd


@pytest.mark.parametrize("Fr", [5, 1, 34, 66])  # 66 frames: RoPE pre-pass + flash attention on strided views
def test_vchitect_forward_host_logic(monkeypatch, Fr):
    from oracle import vchitect_oracle as VO

    kernels_emul.emulate(monkeypatch)
    net, sd = _vchitect()
    lat = synth.normalish("vch.lat", (1, Fr, 4, 12, 16))
    enc = synth.normalish("vch.enc", (1, 9, 48))
    pooled = synth.normalish("vch.pool", (1, 40))
    ts = torch.tensor([500])
    out = net(lat, enc, pooled, ts, return_dict=False)[0]
    with torch.no_grad():
        ref = VO.transformer_forward(sd, VCH_O, lat, enc, pooled, ts)
    assert out.shape == ref.shape == (Fr, 4, 12, 16)
    assert torch.allclose(out, ref, rtol=1e-4, atol=1e-5), (out - ref).abs().max()


def test_vchitect_pab_host_logic(monkeypatch):
    """Eight steps with the three gates on: the mirror's counters / caches follow the reference's (pinned per attention
    in test_oracle_vs_reference.py::test_vchitect_attention_pab_vs_reference)."""
    from oracle import vchitect_oracle as VO
    from videosys_b200.core.pab import pab_mgr

    kernels_emul.emulate(monkeypatch)
    net, sd = _vchitect()
    cfg = pab_mgr.PABConfig(spatial_broadcast=True, spatial_threshold=[100, 800], spatial_range=2, temporal_broadcast=True,
                            temporal_threshold=[100, 800], temporal_range=3, cross_broadcast=True, cross_threshold=[100, 800],
                            cross_range=4)
    pab_mgr.set_pab_manager(cfg)
    pab_mgr.update_steps(8)
    net.reset_pab_state()
    try:
        G = pab_oracle.PABGate((True, (100, 800), 2), (True, (100, 800), 3), (True, (100, 800), 4), 8)
        L = VCH["num_layers"]
        counts = [{"spatial": 0, "temporal": 0, "cross": 0} for _ in range(L)]
        caches = [{} for _ in range(L)]
        enc = synth.normalish("vchp.enc", (1, 9, 48))
        pooled = synth.normalish("vchp.pool", (1, 40))
        hits = 0
        for step, t in enumerate([900, 700, 650, 600, 550, 500, 450, 50]):
            lat = synth.normalish(f"vchp.lat{step}", (1, 4, 4, 12, 16))

            def gate(i, kind, t=t):
                nonlocal hits
                hit, counts[i][kind] = G.gate(kind, t, counts[i][kind])
                hits += hit
                return hit

            ts = torch.tensor([t])
            out = net(lat, enc, pooled, ts, return_dict=False)[0]
            with torch.no_grad():
                ref = VO.transformer_forward(sd, VCH_O, lat, enc, pooled, ts, gate, caches)
            assert torch.allclose(out, ref, rtol=1e-4, atol=1e-5), (step, (out - ref).abs().max())
        assert hits > 0
    finally:
        pab_mgr.set_pab_manager(None)


@pytest.mark.parametrize("name", ["small_rope", "small_norope"])
def test_osp_v110_host_logic_vs_reference_golden(monkeypatch, golden_dir, name):
    """The Open-Sora-Plan v1.1.0 front end on the torch stand-ins, fp32, against the fp32 output of the UNMODIFIED reference
    model stored in tests/golden/osp_v110.pt (runs wherever the fixture is: no reference tree needed)."""
    import os

    from oracle import osp_cases as OC
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V

    kernels_emul.emulate(monkeypatch)
    gold = torch.load(os.path.join(golden_dir, "osp_v110.pt"))
    net = LatteT2V(**OC.CASES[name][0])
    net.load_state_dict(OC.weights(net.state_dict(), name, torch.float32))
    x, enc, m, tt = OC.inputs(name, torch.float32)
    out = net.eval()(x, timestep=tt, all_timesteps=[900, 500], encoder_hidden_states=enc, encoder_attention_mask=m,
                     return_dict=False)[0]
    assert torch.allclose(out, gold[f"{name}.fp32"], rtol=1e-4, atol=1e-5), (out - gold[f"{name}.fp32"]).abs().max()


def test_osp_v110_pab_host_logic_vs_reference_golden(monkeypatch, golden_dir):
    import os

    from oracle import osp_cases as OC
    from videosys_b200.core.pab import pab_mgr
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V

    kernels_emul.emulate(monkeypatch)
    gold = torch.load(os.path.join(golden_dir, "osp_v110.pt"))
    net = LatteT2V(**OC.CASES["small_rope"][0])
    net.load_state_dict(OC.weights(net.state_dict(), "small_rope", torch.float32))
    net.eval()
    pab_mgr.set_pab_manager(pab_mgr.PABConfig(**OC.PAB_KW))
    pab_mgr.update_steps(len(OC.PAB_TIMESTEPS))
    net.reset_pab_state()
    try:
        for step, t in enumerate(OC.PAB_TIMESTEPS):
            x, enc, m, _ = OC.inputs("small_rope", torch.float32, step)
            out = net(x, timestep=torch.tensor([t, t]), all_timesteps=OC.PAB_TIMESTEPS, encoder_hidden_states=enc,
                      encoder_attention_mask=m, return_dict=False)[0]
            want = gold[f"pab.{step}.fp32"]
            assert torch.allclose(out, want, rtol=1e-4, atol=1e-5), (step, (out - want).abs().max())
    finally:
        pab_mgr.set_pab_manager(None)


def _bare_pipeline(cls, config, transformer, scheduler, dtype=torch.float32):
    """A pipeline object without its CUDA-only constructor: generate()'s host logic (CFG batching, scheduler stepping,
    timestep bookkeeping) runs on the CPU stand-ins."""
    pipe = cls.__new__(cls)
    pipe._config, pipe._device, pipe._dtype = config, torch.device("cpu"), dtype
    pipe.transformer, pipe.scheduler = transformer, scheduler
    return pipe


def test_vchitect_pipeline_generate_host_logic(monkeypatch):
    from videosys_b200 import VchitectConfig, VchitectXLPipeline
    from videosys_b200.schedulers.scheduling_flow_match_euler import FlowMatchEulerDiscreteScheduler

    kernels_emul.emulate(monkeypatch)
    net, _ = _vchitect("vchg.")
    pipe = _bare_pipeline(VchitectXLPipeline, VchitectConfig(transformer_config=VCH), net, FlowMatchEulerDiscreteScheduler(shift=3.0))
    kw = dict(num_inference_steps=4, guidance_scale=7.5, seed=0, frames=3, height=96, width=128)
    out = pipe.generate("Sunset over the sea.", **kw).video
    assert out.shape == (1, 3, 4, 12, 16) and torch.isfinite(out).all()
    assert torch.equal(pipe.generate("Sunset over the sea.", **kw).video, out)
    assert not torch.equal(pipe.generate("A different prompt.", **kw).video, out)


def test_osp_pipeline_generate_host_logic(monkeypatch):
    from oracle import osp_cases as OC
    from videosys_b200 import OpenSoraPlanConfig, OpenSoraPlanPipeline
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V
    from videosys_b200.schedulers.scheduling_pndm import PNDMScheduler

    kernels_emul.emulate(monkeypatch)
    tc = OC.CASES["small_rope"][0]
    net = LatteT2V(**tc)
    net.load_state_dict(OC.weights(net.state_dict(), "small_rope", torch.float32))
    cfg = OpenSoraPlanConfig(version="v110", transformer_type="65x512x512", transformer_config=tc)
    pipe = _bare_pipeline(OpenSoraPlanPipeline, cfg, net.eval(), PNDMScheduler())
    kw = dict(num_inference_steps=5, guidance_scale=7.5, seed=0, height=64, width=64, max_sequence_length=24)
    out = pipe.generate("Sunset over the sea.", **kw).video
    assert out.shape == (1, 4, 5, 8, 8) and torch.isfinite(out).all()
    assert pipe.scheduler.counter == len(pipe.scheduler.timesteps) == 12 + 2  # 4 Runge-Kutta steps x 3 evaluations + 2 multi-step
    assert torch.equal(pipe.generate("Sunset over the sea.", **kw).video, out)
    assert OpenSoraPlanPipeline.latent_frames(65) == 17 and OpenSoraPlanPipeline.latent_frames(221) == 56


# ---- sequence / CFG parallelism of the model front ends over gloo, world_size 2 (kernel entries = torch stand-ins) -------------
def _sp_worker(rank, world, port, which, enable_cp, q):
    import os
    import traceback

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    try:
        import torch.distributed as dist

        from oracle import osp_cases as OC
        from videosys_b200.core.distributed.parallel_mgr import initialize

        kernels_emul.emulate_global()
        initialize(rank, world)
        if which == "osp_v110":
            from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V

            net = LatteT2V(**OC.CASES["small_rope"][0])
            net.load_state_dict(OC.weights(net.state_dict(), "small_rope", torch.float32))
            x, enc, m, tt = OC.inputs("small_rope", torch.float32)
            call = lambda: net(x, timestep=tt, all_timesteps=[900, 500], encoder_hidden_states=enc, encoder_attention_mask=m,  # noqa: E731
                               return_dict=False)[0]
        elif which == "stdit3":  # OpenSora: S-sharded resident layout, spatial blocks switch to a frame shard (NCCL transport here)
            from oracle import cases
            from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config

            os.environ["VSB_DSP_P2P"] = "0"  # the peer-memory windows need CUDA IPC; all_to_all_single carries the switch
            net = STDiT3(STDiT3Config(**cases.small_model_cfg(depth=2))).to(torch.bfloat16)
            net.load_state_dict(synth.fill_state_dict(net.state_dict(), "spstd."))
            inp = cases.forward_inputs(torch.bfloat16)
            call = lambda: net(inp["x"], inp["timestep"], inp["y"], mask=inp["mask"], x_mask=inp["x_mask"], fps=inp["fps"],  # noqa: E731
                               height=inp["height"], width=inp["width"]).float()
        elif which == "osp_v120":
            from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V

            net = OpenSoraT2V(**OC.CASES12["small_rope"][0])
            net.load_state_dict(OC.weights(net.state_dict(), "v120.small_rope", torch.float32))
            x, enc, m, tt = OC.inputs12("small_rope", torch.float32)
            call = lambda: net(x, timestep=tt, encoder_hidden_states=enc, encoder_attention_mask=m, return_dict=False)[0]  # noqa: E731
        elif which == "latte":
            from videosys_b200.models.transformers.latte_transformer_3d import LatteT2V

            net = LatteT2V(num_attention_heads=2, attention_head_dim=72, in_channels=4, out_channels=8, num_layers=2, sample_size=8,
                           caption_channels=32, video_length=5, cross_attention_dim=144)
            net.load_state_dict(synth.fill_state_dict(net.state_dict(), "spl."))
            x = synth.normalish("spl.x", (2, 4, 5, 8, 8))
            enc = synth.normalish("spl.enc", (2, 7, 32))
            tt = torch.tensor([500, 500])
            call = lambda: net(x, timestep=tt, all_timesteps=[900, 500], encoder_hidden_states=enc, return_dict=False)[0]  # noqa: E731
        else:
            from oracle import cogvideox_oracle as CO
            from videosys_b200.models.transformers.cogvideox_transformer_3d import CogVideoXTransformer3DModel

            rope = which == "cogvideox_rope"  # CogVideoX-5b: rotary tables follow the head-scatter exchange (pad rows = identity)
            net = CogVideoXTransformer3DModel(num_attention_heads=4, attention_head_dim=64, in_channels=4, out_channels=4,
                                              time_embed_dim=64, text_embed_dim=48, num_layers=2, sample_width=16, sample_height=12,
                                              sample_frames=9, max_text_seq_length=16, use_rotary_positional_embeddings=rope)
            net.load_state_dict(synth.fill_state_dict(net.state_dict(), "spc."))
            lat = synth.normalish("spc.lat", (2, 3, 4, 12, 14))  # 6 x 7 = 42 patches per frame: 126 video rows, odd chunking
            txt = synth.normalish("spc.txt", (2, 16, 48))
            tt = torch.tensor([499, 499])
            rot = CO.rotary_3d(64, CO.resize_crop_region_for_grid((6, 7), 45, 30), (6, 7), 3) if rope else None
            call = lambda: net(lat, txt, tt, image_rotary_emb=rot, return_dict=False)[0]  # noqa: E731
        net.eval()
        want = call()  # unsharded (parallel_manager None)
        net.enable_parallel(1, world, enable_cp)
        got = call()
        q.put((rank, float((got - want).abs().max()), float(want.abs().max()), tuple(got.shape) == tuple(want.shape), None))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:  # pragma: no cover
        q.put((rank, None, None, None, traceback.format_exc()))


@pytest.mark.parametrize("which,enable_cp", [("osp_v110", False), ("osp_v110", True), ("latte", False), ("cogvideox", False),
                                             ("cogvideox", True), ("osp_v120", False), ("stdit3", False),
                                             ("cogvideox_rope", False)])
def test_model_parallelism_gloo_world2(monkeypatch, which, enable_cp):
    """Two ranks: frame-sharded DSP (Latte / Open-Sora-Plan v1.1.0: temporal blocks switch to a patch shard, with the RoPE
    tables following the switch), head-scatter sequence parallelism (CogVideoX) or CFG parallelism reproduce the single-rank
    forward on every rank (fp32; the exchanges move data, the per-sequence arithmetic is unchanged)."""
    import multiprocessing as mp
    import os

    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")  # CPU ranks on gloo: with a GPU visible, initialize() picks NCCL
    world, port = 2, 30100 + (os.getpid() % 300) + 7 * ["osp_v110", "latte", "cogvideox", "osp_v120", "stdit3", "cogvideox_rope"].index(which) + int(enable_cp)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sp_worker, args=(r, world, port, which, enable_cp, q)) for r in range(world)]
    [p.start() for p in procs]
    for _ in range(world):
        r, err_abs, scale, same_shape, tb = q.get(timeout=300)
        assert tb is None, tb
        assert same_shape and err_abs <= 1e-4 * max(scale, 1.0), (which, r, err_abs, scale)
    [p.join(timeout=60) for p in procs]


@pytest.mark.parametrize("name", ["small_rope", "small_abspos"])
def test_osp_v120_host_logic_vs_reference_golden(monkeypatch, golden_dir, name):
    """OpenSoraT2V's front end on the torch stand-ins, fp32, against the fp32 output of the UNMODIFIED reference model stored
    in tests/golden/osp_v120.pt."""
    import os

    from oracle import osp_cases as OC
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V

    kernels_emul.emulate(monkeypatch)
    gold = torch.load(os.path.join(golden_dir, "osp_v120.pt"))
    net = OpenSoraT2V(**OC.CASES12[name][0])
    net.load_state_dict(OC.weights(net.state_dict(), "v120." + name, torch.float32))
    x, enc, m, tt = OC.inputs12(name, torch.float32)
    out = net.eval()(x, timestep=tt, encoder_hidden_states=enc, encoder_attention_mask=m, return_dict=False)[0]
    assert torch.allclose(out, gold[f"{name}.fp32"], rtol=1e-4, atol=1e-5), (out - gold[f"{name}.fp32"]).abs().max()


def test_osp_v120_pipeline_generate_host_logic(monkeypatch):
    from oracle import osp_cases as OC
    from videosys_b200 import OpenSoraPlanConfig, OpenSoraPlanPipeline
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V
    from videosys_b200.schedulers.scheduling_euler_ancestral import EulerAncestralDiscreteScheduler

    kernels_emul.emulate(monkeypatch)
    tc = OC.CASES12["small_rope"][0]
    net = OpenSoraT2V(**tc)
    net.load_state_dict(OC.weights(net.state_dict(), "v120.small_rope", torch.float32))
    cfg = OpenSoraPlanConfig(version="v120", transformer_type="29x480p", transformer_config=tc)
    pipe = _bare_pipeline(OpenSoraPlanPipeline, cfg, net.eval(), EulerAncestralDiscreteScheduler())
    kw = dict(num_inference_steps=5, guidance_scale=7.5, seed=0, max_sequence_length=24)
    out = pipe.generate("Sunset over the sea.", **kw).video
    assert out.shape == (1, 4, 5, 8, 8) and torch.isfinite(out).all()
    assert torch.equal(pipe.generate("Sunset over the sea.", **kw).video, out)  # the ancestral noise follows the seed
    assert OpenSoraPlanPipeline.latent_frames(29) == 8 and OpenSoraPlanPipeline.latent_frames(93) == 24


def test_widened_models_from_pretrained_local_snapshot(tmp_path):
    """Vchitect / Open-Sora-Plan v1.1.0 / v1.2.0 load hub-style LOCAL snapshots (config.json with list-valued sample sizes and
    the library's bookkeeping keys + safetensors) strictly under the reference's parameter names (the layouts
    pipeline_vchitect.py:222-225 and pipeline_open_sora_plan.py:294-300 read: ``<root>/transformer`` and ``<root>/<type>``)."""
    import json

    from safetensors.torch import save_file

    from oracle import osp_cases as OC
    from videosys_b200.models.transformers.open_sora_plan_v110_transformer_3d import LatteT2V
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V
    from videosys_b200.models.transformers.vchitect_transformer_3d import VchitectXLTransformerModel

    def lists(cfg):
        return {k: (list(v) if isinstance(v, tuple) else v) for k, v in cfg.items()}

    for cls, cfg, sub in ((VchitectXLTransformerModel, VCH, "transformer"),
                          (LatteT2V, OC.CASES["small_rope"][0], "65x512x512"),
                          (OpenSoraT2V, OC.CASES12["small_rope"][0], "29x480p")):
        src = cls(**cfg)
        d = tmp_path / cls.__name__ / sub
        d.mkdir(parents=True)
        (d / "config.json").write_text(json.dumps(dict(lists(cfg), _class_name=cls.__name__, _diffusers_version="0.30.0")))
        save_file({k: v.contiguous() for k, v in src.state_dict().items()}, str(d / "diffusion_pytorch_model.safetensors"))
        got = cls.from_pretrained(str(tmp_path / cls.__name__), subfolder=sub)
        assert set(got.state_dict()) == set(src.state_dict())
        assert all(torch.equal(got.state_dict()[k], v) for k, v in src.state_dict().items()), cls.__name__
