"""CPU-side tests of the product's host logic: C-ABI surface, PAB mirror, DSP comm over gloo (world_size 2),
state_dict compatibility.  No kernel launches (there is no GPU here)."""
import json
import os
import re
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import cases, dsp_oracle, pab_oracle, stdit3_oracle as O, synth
from tests.helpers import stdit3_state_dict_template

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from videosys_b200 import _lib

    hdr = open(os.path.join(ROOT, "include", "vsb200.h")).read()
    declared = set(re.findall(r"\b(vsb_[a-z0-9_]+)\s*\(", hdr))
    lib = _lib.load()
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/vsb200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_lib.SIGNATURES) == declared
    assert lib.vsb_version() >= 100


def test_no_cpu_fallback_without_device():
    from videosys_b200 import _lib, kernels

    lib = _lib.load()
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert lib.vsb_init(0) == -4  # VSB_ERR_NO_DEVICE
    assert b"no CPU fallback" in lib.vsb_last_error()
    with pytest.raises(_lib.VsbError):
        kernels.residual_add(torch.zeros(8, dtype=torch.bfloat16), torch.zeros(8, dtype=torch.bfloat16))
    from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config

    net = STDiT3(STDiT3Config(**cases.small_model_cfg())).to(torch.bfloat16)
    inp = cases.forward_inputs(torch.bfloat16)
    with pytest.raises(RuntimeError, match="no CPU path"):
        net(**inp)


def test_product_does_not_import_the_oracle():
    """The product package must never route through oracle/ (tier rule 3)."""
    bad = []
    for dp, _, files in os.walk(os.path.join(ROOT, "videosys_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "from oracle" in src:
                    bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_state_dict_is_reference_compatible():
    """Key set and shapes of the B200 module == the reference STDiT3 (SURVEY.md Appendix D)."""
    from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config

    cfg = cases.small_model_cfg(depth=2)
    ours = STDiT3(STDiT3Config(**cfg)).state_dict()
    tmpl = stdit3_state_dict_template(cfg)
    assert set(ours) == set(tmpl)
    for k in tmpl:
        assert tuple(ours[k].shape) == tuple(tmpl[k].shape), k
    net = STDiT3(STDiT3Config(**cfg))
    for blk in net.temporal_blocks:  # reference zero-inits these (open_sora_transformer_3d.py:508-511)
        assert blk.attn.proj.weight.abs().sum() == 0 and blk.mlp.fc2.weight.abs().sum() == 0


def test_pab_mirror_matches_oracle_and_known_answers(golden_dir):
    from videosys_b200.core.pab import pab_mgr as P

    kat = json.load(open(os.path.join(golden_dir, "pab_schedules.json")))
    try:
        for name, steps in (("240p_51f_30", 30), ("720p_68f_50", 50)):
            P.set_pab_manager(P.PABConfig(spatial_broadcast=True, spatial_threshold=[450, 930], spatial_range=2,
                                          temporal_broadcast=True, temporal_threshold=[450, 930], temporal_range=4,
                                          cross_broadcast=True, cross_threshold=[450, 930], cross_range=6))
            P.update_steps(steps)
            assert P.enable_pab()
            for kind, fn in (("spatial", P.if_broadcast_spatial), ("temporal", P.if_broadcast_temporal), ("cross", P.if_broadcast_cross)):
                c, bits = 0, []
                for _ in range(2):
                    for t in kat[name]["timesteps"]:
                        f, c = fn(t, c)
                        bits.append("1" if f else "0")
                assert "".join(bits[:steps]) == kat[name][kind]
                assert "".join(bits[steps:]) == kat[name][kind + "_second_run"]
        # edges: strict bounds, None timestep, kind off, manager off
        P.set_pab_manager(P.PABConfig(spatial_broadcast=True, spatial_threshold=[450, 930], spatial_range=2))
        P.update_steps(4)
        assert P.if_broadcast_spatial(450, 1) == (False, 2) and P.if_broadcast_spatial(930, 1) == (False, 2)
        assert P.if_broadcast_spatial(451, 1) == (True, 2) and P.if_broadcast_spatial(451, 3) == (True, 0)
        assert P.if_broadcast_spatial(None, 1) == (False, 2) and P.if_broadcast_cross(500, 1) == (False, 2)
        P.set_pab_manager(P.PABConfig(mlp_broadcast=True))
        assert not P.enable_pab() and P.if_broadcast_spatial(500, 3) == (False, 3)
    finally:
        P.set_pab_manager(None)


def test_pab_mlp_skip_spec():
    """Latte/OSP MLP broadcast (core/pab/pab_mgr.py:93-174): save at the key step, reuse for skip_count steps, delete at the end."""
    from videosys_b200.core.pab import pab_mgr as P

    ts = [980, 960, 940, 920, 900, 880]
    cfg = P.PABConfig(spatial_broadcast=True, spatial_threshold=[100, 800], spatial_range=2, mlp_broadcast=True,
                      mlp_spatial_broadcast_config={960: {"block": [0, 1], "skip_count": 2}},
                      mlp_temporal_broadcast_config={960: {"block": [0], "skip_count": 1}})
    P.set_pab_manager(cfg)
    P.update_steps(len(ts))
    try:
        assert P.if_broadcast_mlp(980, 0, 0, ts) == (False, 0, False, [960, 940, 920])
        flag, cnt, nxt, rng = P.if_broadcast_mlp(960, 0, 0, ts)
        assert (flag, cnt, nxt, rng) == (False, 1, True, [960, 920])
        P.save_mlp_output(960, 0, "tensor@960")
        flag, cnt, nxt, rng = P.if_broadcast_mlp(940, 1, 0, ts)
        assert (flag, cnt, nxt) == (True, 0, False) and P.get_mlp_output(rng, 940, 0) == "tensor@960"
        flag, cnt, nxt, rng = P.if_broadcast_mlp(920, 0, 0, ts)
        assert flag and P.get_mlp_output(rng, 920, 0) == "tensor@960"
        with pytest.raises(ValueError):
            P.get_mlp_output(rng, 920, 0)  # deleted at the end of the window
        assert P.if_broadcast_mlp(940, 0, 5, ts)[0] is False  # block not listed
    finally:
        P.set_pab_manager(None)


# ---- DSP comm over gloo, world_size 2 ------------------------------------------------------------------------
def _dsp_worker(rank, world, port, T, S, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    try:
        from videosys_b200.core.distributed import comm
        from videosys_b200.core.distributed.parallel_mgr import ParallelManager, initialize

        initialize(rank, world)
        pm = ParallelManager(1, 1, world)
        assert pm.sp_size == world and pm.sp_rank == rank
        B, C = 2, 16
        full = synth.normalish(f"gloo{T}{S}", (B, T, S, C))
        comm.set_pad("temporal", T, pm.sp_group)
        comm.set_pad("spatial", S, pm.sp_group)
        x = comm.split_sequence(full, pm.sp_group, dim=2, pad=comm.get_pad("spatial"))
        a = comm.all_to_all_with_pad(x, pm.sp_group, scatter_dim=1, gather_dim=2, scatter_pad=comm.get_pad("temporal"),
                                     gather_pad=comm.get_pad("spatial"))
        b = comm.all_to_all_with_pad(a, pm.sp_group, scatter_dim=2, gather_dim=1, scatter_pad=comm.get_pad("spatial"),
                                     gather_pad=comm.get_pad("temporal"))
        g = comm.gather_sequence(b, pm.sp_group, dim=2, pad=comm.get_pad("spatial"))
        q.put((rank, x.numpy(), a.numpy(), b.numpy(), g.numpy(), None))  # by value: a tensor's shared-memory file dies with the worker
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:  # pragma: no cover
        import traceback

        q.put((rank, None, None, None, None, traceback.format_exc()))


@pytest.mark.parametrize("T,S", [(5, 9), (4, 8)])
def test_dsp_comm_gloo_world2(monkeypatch, T, S):
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")  # CPU ranks on gloo: with a GPU visible, initialize() picks NCCL
    world, port = 2, 29600 + (os.getpid() % 200) + T
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dsp_worker, args=(r, world, port, T, S, q)) for r in range(world)]
    [p.start() for p in procs]
    res = {}
    for _ in range(world):
        r, x, a, b, g, err = q.get(timeout=120)
        assert err is None, err
        res[r] = tuple(torch.from_numpy(v).clone() for v in (x, a, b, g))
    [p.join(timeout=60) for p in procs]
    B, C = 2, 16
    full = synth.normalish(f"gloo{T}{S}", (B, T, S, C))
    shards = dsp_oracle.split_sequence(full, world, dim=2)
    sw, new_s, new_t = dsp_oracle.dynamic_switch([p.reshape(B, -1, C) for p in shards], T, S, to_spatial_shard=False)
    for r in range(world):
        x, a, b, g = res[r]
        assert torch.equal(x, shards[r])
        assert torch.equal(a.reshape(B, -1, C), sw[r]) and (a.shape[1], a.shape[2]) == (new_t, new_s)
        assert torch.equal(b, x)
        assert torch.equal(g, full)


def _ulysses_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    try:
        from videosys_b200.core.distributed import comm
        from videosys_b200.core.distributed.parallel_mgr import ParallelManager, initialize

        initialize(rank, world)
        pm = ParallelManager(1, 1, world)
        B, Nt, Nv, H, D = 2, 3, 8, 4, 2
        full = synth.normalish("ulysses", (B, Nt + Nv, 3, H, D))
        Nl = Nv // world
        mine = torch.cat([full[:, :Nt], full[:, Nt + rank * Nl : Nt + (rank + 1) * Nl]], 1).contiguous()
        a = comm.ulysses_scatter_heads(mine, Nt, pm.sp_group)  # every row, my heads
        o = a[:, :, 0].reshape(B, Nt + Nv, -1).contiguous()    # stand-in attention output: my heads of q
        back = comm.ulysses_gather_heads(o, Nt, pm.sp_group)    # my rows, every head
        q.put((rank, a.contiguous().numpy(), back.contiguous().numpy(), None))  # by value
        dist.barrier()
        dist.destroy_process_group()
    except Exception:  # pragma: no cover
        import traceback

        q.put((rank, None, None, traceback.format_exc()))


def test_ulysses_head_scatter_gloo_world2(monkeypatch):
    """CogVideoX's head-scatter exchange (reference cogvideox_transformer_3d.py:44-165): after the scatter a rank holds
    every row of its head group, after the way back its own rows (text + its chunk) with every head."""
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")  # CPU ranks on gloo: with a GPU visible, initialize() picks NCCL
    world, port = 2, 29800 + (os.getpid() % 150)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_ulysses_worker, args=(r, world, port, q)) for r in range(world)]
    [p.start() for p in procs]
    res = {}
    for _ in range(world):
        r, a, back, err = q.get(timeout=120)
        assert err is None, err
        res[r] = (torch.from_numpy(a).clone(), torch.from_numpy(back).clone())
    [p.join(timeout=60) for p in procs]
    B, Nt, Nv, H, D = 2, 3, 8, 4, 2
    full = synth.normalish("ulysses", (B, Nt + Nv, 3, H, D))
    Hn, Nl = H // world, Nv // world
    for r in range(world):
        a, back = res[r]
        assert torch.equal(a, full[:, :, :, r * Hn : (r + 1) * Hn])
        rows = torch.cat([full[:, :Nt, 0], full[:, Nt + r * Nl : Nt + (r + 1) * Nl, 0]], 1)  # q of my rows, every head
        assert torch.equal(back, rows.reshape(B, Nt + Nl, H * D))


def test_rflow_timesteps_match_reference_known_answers(golden_dir):
    """The scheduler mirror reproduces the reference's transformed timesteps: int(bf16(t)) == SURVEY Appendix A."""
    from videosys_b200.schedulers.scheduling_rflow_open_sora import RFLOW

    kat = json.load(open(os.path.join(golden_dir, "pab_schedules.json")))
    for name, (hh, ww, nf, steps) in {"240p_51f_30": (240, 426, 51, 30), "720p_68f_50": (720, 1280, 68, 50)}.items():
        bf = torch.bfloat16
        margs = dict(height=torch.tensor([hh], dtype=bf), width=torch.tensor([ww], dtype=bf), num_frames=torch.tensor([nf], dtype=bf))
        ts = RFLOW(num_sampling_steps=steps, use_timestep_transform=True).prepare_timesteps(1, "cpu", margs)
        assert [int(t.to(bf).item()) for t in ts] == kat[name]["timesteps"]
        # and bit-identical to the oracle's restatement (which is pinned against the reference)
        ots, _ = O.rflow_timesteps(steps, hh, ww, nf)
        assert all(torch.equal(a, b) for a, b in zip(ts, ots))


def test_latent_and_image_size_tables():
    from videosys_b200.pipelines.open_sora.pipeline_open_sora import get_image_size, get_latent_size, get_num_frames

    assert get_image_size("720p", "9:16") == (720, 1280) and get_image_size("240p", "9:16") == (240, 426)
    assert get_latent_size(68, 720, 1280) == (20, 90, 160) and get_latent_size(51, 240, 426) == (15, 30, 53)  # SURVEY App. B
    assert get_num_frames("2s") == 51 and get_num_frames(68) == 68
    with pytest.raises(ValueError):
        get_image_size("720p", "3:8")


def test_bench_kernel_fractions():
    """bench.py's per-kernel roofline fractions: pure arithmetic on the measured peaks."""
    import bench

    peaks = dict(tflops=1386.7, tflops_burst=1674.1, hbm=6572.9, src="t")
    shares = {"gemm": {"ms_per_step": 206.4, "launches_per_step": 392.0, "achieved": 1453.0, "unit": "TFLOP/s"},
              "gate_residual": {"ms_per_step": 17.8, "launches_per_step": 112.0, "achieved": 6246.0, "unit": "GB/s"},
              "dsp_switch": {"ms_per_step": 5.5, "launches_per_step": 56.0, "achieved": 367.0, "unit": "GB/s"}}
    out = bench.kernel_fractions(shares, peaks)
    assert abs(out["gemm"]["frac_of_peak"] - 1453.0 / 1386.7) < 1e-9
    assert abs(out["gate_residual"]["frac_of_peak"] - 6246.0 / 6572.9) < 1e-9
    assert abs(out["dsp_switch"]["frac_of_peak"] - 367.0 / 770.0) < 1e-9
    assert shares["gemm"].get("frac_of_peak") is None  # input left untouched


def test_bench_step_flops_match_survey():
    """SURVEY 8(d): 720p/68f step = 3.782e14 dense FLOPs, 7.841e13 of them attention; 240p/51f = 2.706e13 / 1.60e12."""
    import bench

    attn, total = bench.step_flops(bench.WORKLOADS["opensora_720p_68f_50step"])
    assert abs(attn / 7.841e13 - 1) < 2e-3 and abs(total / 3.782e14 - 1) < 2e-3
    attn, total = bench.step_flops(bench.WORKLOADS["opensora_240p_51f_30step"])
    assert abs(attn / 1.60e12 - 1) < 1e-2 and abs(total / 2.706e13 - 1) < 1e-2
    r = bench.attention_roofline(bench.WORKLOADS["opensora_720p_68f_50step"], 0.437, dict(tflops=1386.7))
    assert 0.12 < r["frac_attention_only"] < 0.14 and 0.60 < r["frac_all_dense_flops"] < 0.65


def test_bench_line_contract():
    """The ours-arm JSON line carries every key the bench contract names (built from fake timings, no GPU)."""
    import argparse
    import json

    import bench

    args = argparse.Namespace(steps=4, warmup=3, workload="opensora_720p_68f_50step", pab=False, gpus=1, opt=[], depth=0)
    W = bench.WORKLOADS[args.workload]
    peaks = dict(tflops=1386.7, tflops_burst=1674.1, hbm=6572.9, src="t")
    shares = bench.kernel_fractions({"gemm": {"ms_per_step": 206.4, "launches_per_step": 392.0, "achieved": 1453.0, "unit": "TFLOP/s"}}, peaks)
    roofline = {"bound": "tensor", "achieved": 1453.0, "peak": 1386.7, "unit": "TFLOP/s", "frac": 1453.0 / 1386.7, "traffic": None}
    clocks = {"sm_mhz": 1700, "sm_max_mhz": 1965, "reasons": ["sw_power_cap"]}
    line = bench.make_line(args, W, 1, 4 * 0.437, 4 * 0.435, 4 * 0.44, 3472, roofline, shares, None, clocks, peaks, 28, 4608000, 4608000)
    json.dumps(line)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert key in line, key
    assert abs(line["value"] - 68 / (50 * 0.437)) < 1e-9 and abs(line["ms_per_step"] - 437.0) < 1e-6
    assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert line["config"]["workload"] == args.workload and "model" not in line["config"]


def test_from_pretrained_local_snapshot(tmp_path):
    """SURVEY 8(f)3: the three denoisers load hub-style LOCAL snapshots (config.json + safetensors / .bin) strictly, under
    the reference's parameter names; a path that is not a directory fails loudly (no hub download)."""
    import json

    import torch
    from safetensors.torch import save_file

    from videosys_b200.models.transformers.cogvideox_transformer_3d import CogVideoXTransformer3DModel
    from videosys_b200.models.transformers.latte_transformer_3d import LatteT2V
    from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config

    cfg = dict(hidden_size=144, num_heads=2, depth=1, caption_channels=32, model_max_length=8)
    src = STDiT3(STDiT3Config(**cfg))
    d = tmp_path / "stdit3"
    d.mkdir()
    (d / "config.json").write_text(json.dumps(dict(cfg, _name_or_path="x", architectures=["STDiT3"], model_type="STDiT3")))
    save_file({k: v.contiguous() for k, v in src.state_dict().items()}, str(d / "model.safetensors"))
    got = STDiT3.from_pretrained(str(d), enable_flash_attn=True)
    assert got.config.enable_flash_attn is True and got.depth == 1
    for k, v in src.state_dict().items():
        assert torch.equal(got.state_dict()[k], v), k

    cx = dict(num_attention_heads=2, attention_head_dim=64, in_channels=4, out_channels=4, time_embed_dim=32, text_embed_dim=16,
              num_layers=1, sample_width=8, sample_height=8, sample_frames=5, max_text_seq_length=4)
    srcx = CogVideoXTransformer3DModel(**cx)
    dx = tmp_path / "cogx" / "transformer"
    dx.mkdir(parents=True)
    (dx / "config.json").write_text(json.dumps(dict(cx, _class_name="CogVideoXTransformer3DModel")))
    torch.save(srcx.state_dict(), str(dx / "diffusion_pytorch_model.bin"))
    gotx = CogVideoXTransformer3DModel.from_pretrained(str(tmp_path / "cogx"))
    assert all(torch.equal(gotx.state_dict()[k], v) for k, v in srcx.state_dict().items())

    lt = dict(num_attention_heads=2, attention_head_dim=72, num_layers=1, sample_size=8, caption_channels=16)
    srcl = LatteT2V(**lt, video_length=4)
    dl = tmp_path / "latte" / "transformer"
    dl.mkdir(parents=True)
    (dl / "config.json").write_text(json.dumps(lt))
    sd = {k: v.contiguous() for k, v in srcl.state_dict().items()}
    half = len(sd) // 2
    keys = list(sd)
    save_file({k: sd[k] for k in keys[:half]}, str(dl / "a.safetensors"))
    save_file({k: sd[k] for k in keys[half:]}, str(dl / "b.safetensors"))
    (dl / "diffusion_pytorch_model.safetensors.index.json").write_text(json.dumps(
        {"weight_map": {**{k: "a.safetensors" for k in keys[:half]}, **{k: "b.safetensors" for k in keys[half:]}}}))
    gotl = LatteT2V.from_pretrained(str(tmp_path / "latte"), video_length=4)
    assert all(torch.equal(gotl.state_dict()[k], v) for k, v in srcl.state_dict().items())

    with pytest.raises(FileNotFoundError):
        STDiT3.from_pretrained("hpcai-tech/OpenSora-STDiT-v3")
    bad = dict(src.state_dict())
    bad.pop("t_block.1.bias")
    save_file({k: v.contiguous() for k, v in bad.items()}, str(d / "model.safetensors"))
    with pytest.raises(RuntimeError):
        STDiT3.from_pretrained(str(d))


def test_pab_plan_matches_known_answer_schedules(golden_dir):
    """STDiT3.pab_plan (the per-step skip decisions taken on the host before anything is launched = the key of the step
    graphs) reproduces the reference's skip bitmaps (SURVEY Appendix A, generated by executing the reference) for every
    block over two consecutive 50-step videos, and the number of distinct plans is what core/graph_step.py captures."""
    from videosys_b200.core.pab import pab_mgr as P
    from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config
    from videosys_b200.pipelines.open_sora.pipeline_open_sora import OpenSoraPABConfig

    kat = json.load(open(os.path.join(golden_dir, "pab_schedules.json")))["720p_68f_50"]
    net = STDiT3(STDiT3Config(hidden_size=144, num_heads=2, depth=3, caption_channels=32, model_max_length=8))
    assert net.pab_plan(500) is None  # PAB off
    try:
        P.set_pab_manager(OpenSoraPABConfig())
        P.update_steps(50)
        rows = {"spatial": [], "temporal": [], "cross": []}
        plans = set()
        for rep in range(2):
            for t in kat["timesteps"]:
                plan = net.pab_plan(t)
                plans.add(plan)
                assert len(plan) == 2 * net.depth
                for d in range(net.depth):
                    (sa, sc), (ta, tc) = plan[2 * d], plan[2 * d + 1]
                    assert (sa, sc, ta, tc) == (plan[0][0], plan[0][1], plan[1][0], plan[1][1])  # every block pair alike
                    assert sc == tc  # one cross gate per block, same counter history
                rows["spatial"].append("1" if plan[0][0] else "0")
                rows["temporal"].append("1" if plan[1][0] else "0")
                rows["cross"].append("1" if plan[0][1] else "0")
        for kind in rows:
            assert "".join(rows[kind][:50]) == kat[kind] and "".join(rows[kind][50:]) == kat[kind + "_second_run"], kind
        assert 2 <= len(plans) <= 13, len(plans)  # lcm(2, 4, 6) = 12 skip patterns + "nothing reused"
    finally:
        P.set_pab_manager(None)
