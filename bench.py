#!/usr/bin/env python
"""bench.py -- frames/sec of the OpenSora-v1.2 denoising loop on the vsb200 sm_100a path (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--pab] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one iteration of the RFLOW sampling loop (schedulers/scheduling_rflow_open_sora.py:238-250 in the
reference): CFG batch of 2 through STDiT3.forward (28 spatial + 28 temporal blocks), guidance combine, Euler update,
on synthetic latents and random-init weights of the named architecture.  metric = output frames / (sampling steps x
seconds per step).  N > 1 shards the sequence with DSP (strong scaling: the same video, split over N GPUs).

A step runs as a replayed CUDA graph (videosys_b200/core/graph_step.py; --no-graph launches every kernel from the host).

JSON line: value (inputs resident in HBM), e2e (host buffers, H2D/D2H inside the timed region; timed interleaved with
the resident arm), roofline (the GEMM kernel: CUDA-event pairs around every GEMM launch of an eager pass of the same
steps, on the launching stream -- events cannot be read back from inside a replayed graph), kernels (the same for the
other kernels), cpu_baseline (the oracle port on the host cores, bounded sample, 3 repetitions), gpu_baseline (N = 1:
the reference's eager path = the oracle restatement on torch/cuBLAS/SDPA library kernels on the same GPU), dsp_parity
(N > 1: sharded == unsharded, bit for bit, before anything is timed), clocks, gpu_launches.
--impl reference times the reference's CPU path (oracle port).
--dump-outputs DIR writes the latents the last timed step returned (DIR/latent.npy from the resident arm, DIR/latent_e2e.npy
from the host-buffer arm, float32): weights and inputs are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (height, width, frames, sampling steps, latent T,H,W, text tokens)
    "opensora_720p_68f_50step": dict(h=720, w=1280, frames=68, steps=50, lat=(20, 90, 160), L=300),
    "opensora_240p_51f_30step": dict(h=240, w=426, frames=51, steps=30, lat=(15, 30, 53), L=300),
}
MODEL = dict(hidden_size=1152, num_heads=16, depth=28, caption_channels=4096, model_max_length=300)
# BASELINE.json configs[3]: CogVideoX-2B, 49 frames 480x720, 50 DDIM steps, fp16, 1 GPU (PAB with --pab)
COGVIDEOX = dict(frames=49, steps=50, h=480, w=720, lat=(13, 16, 60, 90), text=(226, 4096), heads=30, head_dim=64, layers=30)
# not a BASELINE.json config (SURVEY section 8 (f)4 widening): Vchitect-2.0-2B, the reference's example call (40 frames 288x480,
# 100 steps, pipeline_vchitect.py:84-93), bf16, 1 GPU
# not a BASELINE.json config either: Open-Sora-Plan v1.2.0 29x480p (480 x 640 video -> 8 x 60 x 80 latent), 100 ancestral Euler steps
OSP_V120 = dict(frames=29, steps=100, lat=(4, 8, 60, 80), sample_size=(60, 80), text=(512, 4096), layers=32)
VCHITECT = dict(frames=40, steps=100, h=288, w=480, lat=(40, 16, 36, 60), text=(333, 4096), pooled=2048, heads=24, head_dim=64,
                layers=24)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d.get("bf16_tflops_sustained", 1386.7), tflops_burst=d.get("bf16_tflops", 1674.1),
                    hbm=d.get("hbm_gbs", 6572.9), src="measured (MEASURED_PEAKS.json, sustained bf16 GEMM)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


def step_flops(W, depth=28, C=1152, B=2):
    """Algorithmic FLOPs of one denoising step (SURVEY 8(d)): returns (attention QK^T + PV only, everything dense)."""
    T, Hl, Wl = W["lat"]
    S = ((Hl + 1) // 2) * ((Wl + 1) // 2)  # 2x2 spatial patches, odd sizes padded
    N, L = B * T * S, W["L"]
    spatial = depth * 4.0 * (B * T) * S * S * C
    temporal = depth * 4.0 * (B * S) * T * T * C
    cross = 2 * depth * 4.0 * N * L * C
    linear = 2 * depth * (2.0 * N * C * 3 * C + 2.0 * N * C * C + 2.0 * N * C * C + 2.0 * (B * L) * C * 2 * C + 2.0 * N * C * C
                          + 16.0 * N * C * C)
    attn = spatial + temporal + cross
    return attn, attn + linear


def attention_roofline(W, sec_per_step, peaks, depth=28):
    """north_star: frames/s 'as achieved fraction of the attention-FLOP roofline' = the time the attention FLOPs alone
    need at the measured tensor peak, over the measured step time (and the same for all dense FLOPs of the step)."""
    attn, total = step_flops(W, depth)
    return {"attention_flops_per_step": attn, "dense_flops_per_step": total, "peak_tflops": peaks["tflops"],
            "frac_attention_only": attn / (peaks["tflops"] * 1e12) / sec_per_step,
            "frac_all_dense_flops": total / (peaks["tflops"] * 1e12) / sec_per_step,
            "note": "fraction of the step time that the listed FLOPs would take at the measured sustained bf16 peak"}


def kernel_fractions(shares, peaks, nvlink_gbs=770.0):
    """Adds `frac_of_peak` to every per-kernel entry: achieved / the measured peak that bounds it (SURVEY 8(d): tensor
    pipe for GEMM and attention, HBM copy bandwidth for the elementwise passes and the short attention, NVLink peer copy
    for the DSP reshard -- 770 GB/s is what a bulk peer copy reached on this pool's boxes)."""
    out = {}
    for k, v in shares.items():
        v = dict(v)
        if v.get("unit") == "TFLOP/s":
            v["frac_of_peak"], v["peak"] = v["achieved"] / peaks["tflops"], f"{peaks['tflops']:.0f} TFLOP/s sustained bf16 GEMM"
        elif k.startswith("dsp_"):
            v["frac_of_peak"], v["peak"] = v["achieved"] / nvlink_gbs, f"{nvlink_gbs:.0f} GB/s peer copy"
        else:
            v["frac_of_peak"], v["peak"] = v["achieved"] / peaks["hbm"], f"{peaks['hbm']:.0f} GB/s HBM copy"
        out[k] = v
    return out


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown"}
            while not self._halt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.1)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port (CPU restatement of the reference's eager path) on the host cores
# ------------------------------------------------------------------------------------------------------------
def cpu_reference(workload):
    """The bounded CPU sample of one denoising step: ONE of the 28 (spatial, temporal) block pairs of the oracle port, bf16
    eager, all host threads, each block on the sequences it really sees --
      spatial block : CFG batch 2 x ONE latent frame x all S patches (spatial attention over S keys; every frame costs
                      the same, so x T),
      temporal block: CFG batch 2 x all T frames x S_t of the S patches (temporal attention over the real T-frame
                      sequences with RoPE, i.e. native_attention for T < 30; every patch costs the same, so x S / S_t),
    with the full text length in both.  Returns (sample(), describe, cores): sample() runs the pair once and returns
    the seconds of a FULL step extrapolated as 28 x (t_spatial x T + t_temporal x S / S_t)."""
    from oracle import stdit3_oracle as O

    torch.set_num_threads(os.cpu_count())
    W = WORKLOADS[workload]
    T, Hl, Wl = W["lat"]
    S = -(-Hl // 2) * -(-Wl // 2)
    C, H = MODEL["hidden_size"], MODEL["num_heads"]
    g = torch.Generator().manual_seed(0)
    bf = torch.bfloat16

    def rnd(*shape, std=0.02):
        return (torch.randn(*shape, generator=g) * std).to(bf)

    sd = {}
    for kind in ("spatial", "temporal"):
        p = f"{kind}_blocks.0."
        sd[p + "scale_shift_table"] = rnd(6, C, std=C**-0.5)
        for name, (o, i) in {"attn.qkv": (3 * C, C), "attn.proj": (C, C), "cross_attn.q_linear": (C, C),
                             "cross_attn.kv_linear": (2 * C, C), "cross_attn.proj": (C, C), "mlp.fc1": (4 * C, C),
                             "mlp.fc2": (C, 4 * C)}.items():
            sd[p + name + ".weight"] = rnd(o, i)
            sd[p + name + ".bias"] = rnd(o)
        sd[p + "attn.q_norm.weight"] = torch.ones(C // H, dtype=bf)
        sd[p + "attn.k_norm.weight"] = torch.ones(C // H, dtype=bf)
    freqs = O.rope_freqs(C // H).to(bf)
    L, B = W["L"], 2
    St = max(1, S // T)  # patches of the temporal sample: as many tokens as the spatial sample has
    y = rnd(1, B * L, C, std=1.0)
    t, t0 = rnd(B, 6 * C, std=0.5), rnd(B, 6 * C, std=0.5)
    xs, xt = rnd(B, 1 * S, C, std=1.0), rnd(B, T * St, C, std=1.0)

    def sample():
        with torch.no_grad():
            a = time.perf_counter()
            O.stdit3_block(sd, "spatial_blocks.0.", xs, y, t, [L] * B, torch.ones(B, 1, dtype=torch.bool), t0, 1, S, H, False)
            b = time.perf_counter()
            O.stdit3_block(sd, "temporal_blocks.0.", xt, y, t, [L] * B, torch.ones(B, T, dtype=torch.bool), t0, T, St, H, True, freqs)
            c = time.perf_counter()
        return 28.0 * ((b - a) * T + (c - b) * S / St)

    desc = (f"{workload}: 1 of 28 (spatial, temporal) block pairs of the oracle port (CPU restatement of the reference's eager "
            f"path), bf16, all host threads; spatial block on CFG batch 2 x 1 of {T} latent frames x {S} patches, temporal "
            f"block on CFG batch 2 x {T} frames x {St} of {S} patches (real {T}-frame sequences), {L} text tokens; "
            f"step = 28 x (t_spatial x {T} + t_temporal x {S}/{St})")
    return sample, desc, os.cpu_count()


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    W = WORKLOADS[args.workload]
    sample, desc, cores = cpu_reference(args.workload)
    per_step = []
    for i in range(args.warmup + args.steps):
        t = sample()
        if i >= args.warmup:
            per_step.append(t)
    sec = statistics.mean(per_step)
    val = W["frames"] / (W["steps"] * sec)
    spread = {"min_s": min(per_step), "max_s": max(per_step), "n": len(per_step)}
    line = {
        "impl": "reference", "metric": "frames/sec", "value": val, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": _config(args, W),
        "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc,
                         "step_seconds_extrapolated": spread,
                         "note": "ms_per_step is EXTRAPOLATED from the bounded sample (the full step would take hours on the "
                                 "host cores); /root/reference itself cannot travel to the GPU box, the port is pinned "
                                 "bit-exact to it by tests/test_oracle_vs_reference.py"},
        "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT = 64 << 20


def dump_outputs(path, arrays):
    """Writes each tensor as <path>/<name>.npy in float32 (at most DUMP_LIMIT bytes in all); rank 0 only."""
    import numpy as np

    if int(os.environ.get("RANK", 0)) != 0:
        return
    size = sum(4 * t.numel() for t in arrays.values())
    if size > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {size} bytes of outputs exceed {DUMP_LIMIT}")
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def _config(args, W):
    return {"workload": args.workload, "resolution": f"{W['h']}x{W['w']}", "frames": W["frames"],
            "sampling_steps": W["steps"], "latent": list(W["lat"]), "cfg_batch": 2, "text_tokens": W["L"],
            "architecture": "STDiT3-XL/2 (hidden 1152, 16 heads x 72, 28+28 blocks)", "pab": bool(args.pab),
            "parallelism": f"dsp{args.gpus}" if args.gpus > 1 else "single",
            "l2": "per-step working set (activations 332 MB/tensor at 720p) exceeds the 126 MB L2; no flush needed"}


def make_line(args, W, world, sec, sec_e2e, sec_profiled, launches, roofline, shares, cpu_base, clocks, peaks, depth,
              h2d_bytes, d2h_bytes, extra=None):
    """The one JSON line of the ours arm (pure: unit-tested on CPU).  sec / sec_e2e / sec_profiled: seconds for
    args.steps steps of the resident arm, the host-buffer arm and the all-kernels-profiled (eager) pass."""
    frames, nsteps = W["frames"], W["steps"]
    per = sec / args.steps
    line = {
        "metric": "frames/sec", "value": frames / (nsteps * per), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": _config(args, W),
        "e2e": {"value": frames / (nsteps * sec_e2e / args.steps), "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": sec_e2e / args.steps * 1e3},
        "gpu_launches": launches, "roofline": roofline,
        "attention_flop_roofline": attention_roofline(W, per * world, peaks, depth),
        "kernels": shares,
        "kernels_note": "per-kernel CUDA-event pairs come from an eager pass of the same steps with events around every "
                        f"launch ({sec_profiled / args.steps * 1e3:.1f} ms/step with that overhead); value / e2e are "
                        "timed without any per-kernel event",
        "cpu_baseline": cpu_base,
        "clocks": clocks,
    }
    if extra:
        line.update(extra)
    if args.opt:
        line["config"]["options"] = args.opt
    if args.depth:
        line["config"]["depth_override"] = args.depth
        line["invalid"] = "reduced depth (debug run): not a bench value"
    return line


def gpu_eager_baseline(W, dev, steps=5):
    """The reference's own 1-GPU PyTorch path: the oracle's op-for-op restatement of STDiT3.forward executed by torch
    library kernels (cuBLAS GEMMs, F.scaled_dot_product_attention, eager elementwise) on this GPU -- the denominator of
    north_star's ">= 6x the reference's own 1-GPU PyTorch path".  Two SDPA settings: torch's default backend choice
    and cuDNN attention forced (SURVEY 2.3).  A reported baseline; none of its kernels is ours."""
    from oracle import stdit3_oracle as O
    from tests.helpers import stdit3_state_dict_template

    bf = torch.bfloat16
    g = torch.Generator(device="cpu").manual_seed(0)
    sd = {}
    for k, v in stdit3_state_dict_template(dict(MODEL), bf).items():
        if k.endswith("rope.freqs"):
            sd[k] = O.rope_freqs(MODEL["hidden_size"] // MODEL["num_heads"]).to(bf).to(dev)
        elif v.ndim >= 2:
            sd[k] = (torch.randn(v.shape, generator=g) * 0.02).to(bf).to(dev)
        else:
            sd[k] = (torch.randn(v.shape, generator=g) * 0.02 + (1.0 if "norm" in k else 0.0)).to(bf).to(dev)
    T, Hl, Wl = W["lat"]
    inp = dict(
        x=torch.randn(2, 4, T, Hl, Wl, generator=g).to(dev, bf), timestep=torch.tensor([900.0, 900.0], device=dev),
        y=torch.randn(2, 1, W["L"], MODEL["caption_channels"], generator=g).to(dev, bf),
        mask=torch.ones(1, W["L"], dtype=torch.long, device=dev), x_mask=torch.ones(2, T, dtype=torch.bool, device=dev),
        fps=torch.tensor([24.0, 24.0], device=dev, dtype=bf), height=torch.tensor([float(W["h"])] * 2, device=dev, dtype=bf),
        width=torch.tensor([float(W["w"])] * 2, device=dev, dtype=bf),
    )
    ocfg = dict(hidden_size=MODEL["hidden_size"], num_heads=MODEL["num_heads"], depth=MODEL["depth"])

    def run(n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            O.stdit3_forward(sd, ocfg, **inp)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    out = {"what": "reference eager path (oracle restatement of STDiT3.forward on torch/cuBLAS/SDPA library kernels), same "
                   "GPU, one forward of the CFG pair per step (no guidance / Euler update)", "steps_timed": steps}
    from torch.nn.attention import SDPBackend, sdpa_kernel

    with torch.no_grad():
        run(1)
        ms = run(steps)
        out["default_sdpa"] = {"ms_per_step": ms, "frames_per_s": W["frames"] / (W["steps"] * ms / 1e3),
                               "backends_enabled": {"flash": torch.backends.cuda.flash_sdp_enabled(),
                                                    "mem_efficient": torch.backends.cuda.mem_efficient_sdp_enabled(),
                                                    "cudnn": torch.backends.cuda.cudnn_sdp_enabled(),
                                                    "math": torch.backends.cuda.math_sdp_enabled()}}
        try:
            with sdpa_kernel([SDPBackend.CUDNN_ATTENTION]):
                run(1)
                ms2 = run(steps)
            out["cudnn_sdpa"] = {"ms_per_step": ms2, "frames_per_s": W["frames"] / (W["steps"] * ms2 / 1e3)}
        except Exception as e:  # cuDNN may reject the masked cross-attention: report, do not fail the bench
            out["cudnn_sdpa"] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    del sd, inp
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    import videosys_b200  # noqa: F401
    from videosys_b200 import kernels
    from videosys_b200.core.distributed.parallel_mgr import initialize
    from videosys_b200.core.graph_step import StepGraph
    from videosys_b200.core.pab import pab_mgr
    from videosys_b200.models.transformers.open_sora_transformer_3d import STDiT3, STDiT3Config
    from videosys_b200.pipelines.open_sora.pipeline_open_sora import OpenSoraPABConfig
    from videosys_b200.schedulers.scheduling_rflow_open_sora import RFLOW

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        initialize(rank=rank, world_size=world)
    W = WORKLOADS[args.workload]
    bf = torch.bfloat16

    for kv in args.opt:
        k, v = kv.split("=")
        kernels.set_option(k, int(v))
    torch.manual_seed(0)
    cfg = dict(MODEL)
    if args.depth:
        cfg["depth"] = args.depth
    net = STDiT3(STDiT3Config(**cfg)).to(bf).to(dev).eval()
    net.enable_parallel(dp_size=1, sp_size=world)
    sched = RFLOW(num_sampling_steps=W["steps"], cfg_scale=7.0, use_timestep_transform=True)

    def pab_on(on):
        pab_mgr.set_pab_manager(OpenSoraPABConfig() if on else None)
        if on:
            pab_mgr.update_steps(W["steps"])
        net.reset_pab_state()

    T, Hl, Wl = W["lat"]
    g = torch.Generator(device="cpu").manual_seed(1)
    z_host = torch.randn(1, 4, T, Hl, Wl, generator=g).pin_memory()
    y = torch.randn(1, 1, W["L"], MODEL["caption_channels"], generator=g).to(dev, bf)
    y_null = net.y_embedder.y_embedding[None, None].to(bf)
    margs = dict(
        y=torch.cat([y, y_null], 0), mask=torch.ones(1, W["L"], dtype=torch.long, device=dev),
        height=torch.tensor([W["h"]], device=dev, dtype=bf), width=torch.tensor([W["w"]], device=dev, dtype=bf),
        num_frames=torch.tensor([W["frames"]], device=dev, dtype=bf), fps=torch.tensor([24], device=dev, dtype=bf),
    )
    # the timestep schedule is host arithmetic (50 tiny transforms): keep it off the GPU launch list
    margs_cpu = {k: v.cpu() for k, v in margs.items() if k in ("height", "width", "num_frames")}
    ts_cpu = sched.prepare_timesteps(1, "cpu", margs_cpu)
    timesteps = [t.to(dev) for t in ts_cpu]
    ts_int = [int(t.to(bf).item()) for t in ts_cpu]  # what the reference's int(timestep[0]) sees (bf16 timestep)
    fwd_args = {k: v for k, v in margs.items() if k != "num_frames"}
    fwd_args["x_mask"] = torch.ones(2, T, dtype=torch.bool, device=dev)  # generate() always passes an all-true mask
    n_ts = len(timesteps)
    # PAB only broadcasts inside (450, 930): a short bench that started at schedule index 0 would time no PAB step
    # (at 720p the timestep transform keeps t above 930 until schedule index ~20: SURVEY Appendix A)
    first = args.first_step if args.first_step >= 0 else (22 if (args.pab and args.steps + args.warmup < n_ts) else 0)
    dts = [((timesteps[i] - timesteps[i + 1] if i < n_ts - 1 else timesteps[i]) / 1000.0) for i in range(n_ts)]

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, i0=0):
        """n calls of fn(i) between events; returns seconds (max over ranks)."""
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i0 + i)
        e1.record()
        sync_all()
        sec = e0.elapsed_time(e1) / 1e3
        if world > 1:
            t = torch.tensor([sec], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = t.item()
        return sec

    # ---- N > 1: parity before anything is timed (VERDICT r1 item 1) ----
    dsp_parity = None
    if world > 1:
        dsp_parity = _dsp_parity(net, sched, z_host.to(dev, bf), timesteps, dts, fwd_args, dev, dist, args)

    pab_on(args.pab)
    stepper = StepGraph(net, 7.0, enabled=not args.no_graph)
    state = {"z": z_host.to(dev, bf)}

    def step_resident(i):
        k = (first + i) % n_ts
        state["z"] = stepper.step(state["z"], timesteps[k], dts[k], fwd_args, ts_int=ts_int[k])

    # ---- e2e arm: host (pinned) latents in, host latents out, every step ----
    out_host = torch.empty(1, 4, T, Hl, Wl, dtype=torch.float32).pin_memory()
    zdev = torch.empty(1, 4, T, Hl, Wl, device=dev, dtype=torch.float32)

    def step_e2e(i):
        k = (first + i) % n_ts
        zdev.copy_(z_host, non_blocking=True)
        znew = stepper.step(zdev.to(bf), timesteps[k], dts[k], fwd_args, ts_int=ts_int[k])
        out_host.copy_(znew.float(), non_blocking=True)

    # warm-up: at least 3 steps; with graphs the first step of a pattern is eager, the second captures
    for i in range(max(args.warmup, 3)):
        step_resident(i)
    step_e2e(0)
    if args.pab:  # warm (capture) every PAB pattern the timed steps will meet, then rewind the counters
        net.reset_pab_state()
        for rep_ in range(2):
            for i in range(args.steps):
                step_resident(i)
            net.reset_pab_state()
    sampler = ClockSampler(local)
    sampler.start()
    # timed region: resident and e2e arms INTERLEAVED in blocks (run-order / clock-ramp noise hits both alike)
    nblk = 2 if args.steps >= 4 and not args.pab else 1
    per_blk = [args.steps // nblk + (1 if b < args.steps % nblk else 0) for b in range(nblk)]
    sec = sec_e2e = 0.0
    l0 = kernels.launch_count()
    r0 = stepper.replayed_launches
    done = 0
    for b in range(nblk):
        net.reset_pab_state() if args.pab else None
        sec += timed(step_resident, per_blk[b], done)
        net.reset_pab_state() if args.pab else None
        sec_e2e += timed(step_e2e, per_blk[b], done)
        done += per_blk[b]
    # our launches inside the two timed regions: host launches + the launches baked into every replayed graph
    launches = ((kernels.launch_count() - l0) + (stepper.replayed_launches - r0)) // 2
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latent": state["z"], "latent_e2e": out_host})

    # ---- per-kernel pass: EAGER steps with CUDA-event pairs around every launch of ours (not part of value) ----
    eager = StepGraph(net, 7.0, enabled=False)
    state["z"] = z_host.to(dev, bf)

    def step_eager(i):
        k = (first + i) % n_ts
        state["z"] = eager.step(state["z"], timesteps[k], dts[k], fwd_args, ts_int=ts_int[k])

    net.reset_pab_state()
    step_eager(0)
    net.reset_pab_state()
    kernels.PROFILE, kernels.PROFILE_KINDS = [], None
    sec_profiled = timed(step_eager, args.steps)
    prof = kernels.PROFILE
    kernels.PROFILE = None

    by_kind = {}
    for kind, a, b, work in prof:
        ms = a.elapsed_time(b)
        d = by_kind.setdefault(kind, [0.0, 0.0, 0])
        d[0] += ms
        d[1] += work
        d[2] += 1
    peaks = _peaks()
    gm = by_kind.get("gemm", [1e-9, 0.0, 1])
    gemm_tflops = gm[1] / (gm[0] * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and args.workload == "opensora_720p_68f_50step":
        traffic = json.load(open(tpath)).get("gemm_720p_n1")
    roofline = {"kernel": "gemm2_bf16_tn_kernel / gemm_bf16_tn_kernel (every Linear layer of the step)",
                "bound": "tensor", "achieved": gemm_tflops,
                "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": gemm_tflops / peaks["tflops"], "traffic": traffic,
                "peak_source": peaks["src"], "launches_timed": gm[2],
                "timed_in": "an eager pass of the same steps, CUDA-event pair around every GEMM launch on the launching "
                            "stream (the value / e2e regions replay CUDA graphs, whose launches carry no events)",
                "share_of_step": gm[0] / (sec_profiled * 1e3)}
    tflop_kinds = ("gemm", "attn_flash")
    shares = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[2] / args.steps,
                  "achieved": (v[1] / (v[0] * 1e-3) / 1e12) if k in tflop_kinds else (v[1] / (v[0] * 1e-3) / 1e9),
                  "unit": "TFLOP/s" if k in tflop_kinds else "GB/s"} for k, v in by_kind.items()}
    shares = kernel_fractions(shares, peaks)

    if rank == 0:
        cpu_base = None
        extra = {"cuda_graph": not args.no_graph, "first_schedule_index": first,
                 "tensor_map_cache": dict(zip(("hits", "host_encodes"), kernels.tmap_cache_stats()))}
        if dsp_parity is not None:
            extra["dsp_parity"] = dsp_parity
        if world == 1 and not args.no_cpu_baseline:
            sample, desc, cores = cpu_reference(args.workload)
            sample()  # warm the thread pool / allocator
            ts = [sample() for _ in range(3)]
            v = W["frames"] / (W["steps"] * statistics.mean(ts))
            cpu_base = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc,
                        "step_seconds_extrapolated": {"mean": statistics.mean(ts), "min": min(ts), "max": max(ts), "n": 3}}
        if world == 1 and not args.no_gpu_baseline and not args.depth:
            state.clear()
            torch.cuda.empty_cache()
            extra["gpu_baseline"] = gpu_eager_baseline(W, dev)
        line = make_line(args, W, world, sec, sec_e2e, sec_profiled, int(launches), roofline, shares, cpu_base, clocks,
                         peaks, cfg["depth"], z_host.numel() * 4, out_host.numel() * 4, extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        # the captured step graphs hold NCCL work (the final gather): release them before the communicator goes away --
        # destroying the process group under live graphs hung the N = 2 run after its line had been printed
        import gc

        del stepper, eager
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)  # every rank has passed the barrier; no communicator / interpreter teardown that could wait on a peer


def _dsp_parity(net, sched, z0, timesteps, dts, fwd_args, dev, dist, args):
    """Sharded == unsharded, bit for bit, on THIS workload's shapes: (1) one forward of the first 2 block pairs;
    (2) 4 full-depth denoising steps through the replayed step graph (28 spatial blocks x 4 steps = 112 uses of each DSP
    window and flag array: the window-reuse argument of DESIGN.md section 5 under load).  The unsharded run is the same
    network with its parallel manager taken away, on every rank; the reshard is a permutation and every kernel is
    row-independent, so ANY difference is a bug."""
    from videosys_b200.core.graph_step import StepGraph

    res = {"transport": ("p2p-fused" if net._fuse_dsp else "p2p-scatter") if os.environ.get("VSB_DSP_P2P", "1") == "1" else "nccl"}
    z_in, tt = torch.cat([z0, z0], 0), torch.cat([timesteps[0], timesteps[0]], 0)
    pm = net.parallel_manager

    def unsharded(fn):
        net.parallel_manager = None
        try:
            return fn()
        finally:
            net.parallel_manager = pm

    a = net(z_in, tt, valid_depth=2, **fwd_args)
    b = unsharded(lambda: net(z_in, tt, valid_depth=2, **fwd_args))
    ok1 = torch.equal(a, b)
    d1 = (a.float() - b.float()).abs().max().item()

    def run4(graph):
        st = StepGraph(net, 7.0, enabled=graph)
        z = z0.clone()
        for i in range(4):
            z = st.step(z, timesteps[i], dts[i], fwd_args)
        return z

    zs = run4(not args.no_graph)
    zu = unsharded(lambda: run4(False))
    ok2 = torch.equal(zs, zu)
    d2 = (zs.float() - zu.float()).abs().max().item()
    flags = torch.tensor([int(ok1), int(ok2)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    res["depth2_forward"] = "bit_equal" if flags[0].item() else f"DIFFERS (max abs {d1:.3e} on rank {dist.get_rank()})"
    res["steps4_depth28_graph_replay" if not args.no_graph else "steps4_depth28"] = (
        "bit_equal" if flags[1].item() else f"DIFFERS (max abs {d2:.3e} on rank {dist.get_rank()})")
    res["ranks"] = dist.get_world_size()
    if args.depth:
        res["note"] = f"depth override {args.depth}"
    return res


def run_cogvideox(args):
    """configs[3]: one DDIM step of CogVideoX-2B = CFG pair through CogVideoXTransformer3DModel (30 blocks, joint text + video
    attention over 226 + 17 550 tokens, fp16 as the reference runs it), guidance, DDIM update.  N > 1: the reference's
    head-scatter sequence parallelism (30 heads: N in {2, 3, 5, 6}), or with --cp its CFG parallelism (N = 2)."""
    import torch.distributed as dist

    import videosys_b200  # noqa: F401
    from videosys_b200 import kernels
    from videosys_b200.core.pab import pab_mgr
    from videosys_b200.models.transformers.cogvideox_transformer_3d import CogVideoXTransformer3DModel
    from videosys_b200.pipelines.cogvideox.pipeline_cogvideox import CogVideoXPABConfig
    from videosys_b200.schedulers.scheduling_ddim_cogvideox import CogVideoXDDIMScheduler

    from videosys_b200.core.distributed.parallel_mgr import initialize

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N > 1")
    W = COGVIDEOX
    dev = torch.device("cuda", local)
    torch.cuda.set_device(local)
    if world > 1:
        initialize(rank=rank, world_size=world)
    dt = torch.float16
    torch.manual_seed(0)
    layers = args.depth or W["layers"]
    net = CogVideoXTransformer3DModel(num_layers=layers)
    for prm in net.parameters():  # random-init weights of the named architecture (small, so 30 blocks stay finite in fp16)
        if prm.ndim >= 2:
            torch.nn.init.normal_(prm, std=0.02)
    net = net.to(dt).to(dev).eval()
    if world > 1:
        net.enable_parallel(1, world, enable_cp=args.cp)
    pm = net.parallel_manager
    par = "single" if world == 1 else (f"cp{pm.cp_size}" if pm.sp_size == 1 else (f"sp{pm.sp_size}" if pm.cp_size == 1 else f"cp{pm.cp_size}xsp{pm.sp_size}"))
    sched = CogVideoXDDIMScheduler()
    sched.set_timesteps(W["steps"], dev)
    ts = [int(v) for v in sched.timesteps.tolist()]
    if args.pab:
        pab_mgr.set_pab_manager(CogVideoXPABConfig())
        pab_mgr.update_steps(W["steps"])
    Fr, Cc, Hl, Wl = W["lat"]
    g = torch.Generator(device="cpu").manual_seed(1)
    z_host = torch.randn(1, Fr, Cc, Hl, Wl, generator=g).pin_memory()
    pe = torch.randn(2, *W["text"], generator=g).to(dev, dt)
    first = args.first_step if args.first_step >= 0 else (8 if (args.pab and args.steps + args.warmup < len(ts)) else 0)
    state = {"z": z_host.to(dev, dt)}

    def one(z, k):
        t = ts[k]
        inp = torch.cat([z, z])
        tt = torch.full((2,), t, device=dev, dtype=torch.int64)
        noise = net(inp, pe, tt, return_dict=False, ts_int=t if args.pab else None)[0].float()
        un, tx = noise.chunk(2)
        return sched.step(un + 6.0 * (tx - un), t, z)[0].to(dt)

    def step_resident(i):
        state["z"] = one(state["z"], (first + i) % len(ts))

    out_host = torch.empty(1, Fr, Cc, Hl, Wl, dtype=torch.float32).pin_memory()
    zdev = torch.empty(1, Fr, Cc, Hl, Wl, device=dev, dtype=torch.float32)

    def step_e2e(i):
        zdev.copy_(z_host, non_blocking=True)
        out_host.copy_(one(zdev.to(dt), (first + i) % len(ts)).float(), non_blocking=True)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        sync_all()
        sec = e0.elapsed_time(e1) / 1e3
        if world > 1:
            t = torch.tensor([sec], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = t.item()
        return sec

    sp_parity = None
    if world > 1:  # sharded == single GPU, bit for bit, on this workload's shapes (2 blocks), before anything is timed
        z0 = state["z"]
        tt0 = torch.full((2,), ts[0], device=dev, dtype=torch.int64)
        keep, blocks = net._stack[0].transformer_blocks, net._stack[0].transformer_blocks
        net._stack[0].transformer_blocks = torch.nn.ModuleList(list(blocks)[:2])
        try:
            a = net(torch.cat([z0, z0]), pe, tt0, return_dict=False)[0]
            net.parallel_manager = None
            b = net(torch.cat([z0, z0]), pe, tt0, return_dict=False)[0]
        finally:
            net.parallel_manager = pm
            net._stack[0].transformer_blocks = keep
        flag = torch.tensor([1 if torch.equal(a, b) else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        sp_parity = {"mode": par, "depth2_forward": "bit_equal" if int(flag.item()) else "MISMATCH", "ranks": world}
        del a, b

    for i in range(max(args.warmup, 3)):
        step_resident(i)
    net.reset_pab_state()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = kernels.launch_count()
    sec = timed(step_resident, args.steps)
    launches = kernels.launch_count() - l0
    net.reset_pab_state()
    sec_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs:  # the e2e arm leaves state["z"] alone; the profiled pass below advances it
        dump_outputs(args.dump_outputs, {"latent": state["z"], "latent_e2e": out_host})
    net.reset_pab_state()
    kernels.PROFILE, kernels.PROFILE_KINDS = [], None
    sec_prof = timed(step_resident, args.steps)
    prof, kernels.PROFILE = kernels.PROFILE, None
    by = {}
    for kind, a, b, work in prof:
        d = by.setdefault(kind, [0.0, 0.0, 0])
        d[0] += a.elapsed_time(b)
        d[1] += work
        d[2] += 1
    peaks = _peaks()
    tf = ("gemm", "attn_flash")
    shares = kernel_fractions({k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[2] / args.steps,
                                   "achieved": v[1] / (v[0] * 1e-3) / (1e12 if k in tf else 1e9),
                                   "unit": "TFLOP/s" if k in tf else "GB/s"} for k, v in by.items()}, peaks)
    at = by.get("attn_flash", [1e-9, 0.0, 1])
    a_tf = at[1] / (at[0] * 1e-3) / 1e12
    per = sec / args.steps
    line = {
        "metric": "frames/sec", "value": W["frames"] / (W["steps"] * per), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "cogvideox_2b_49f_480x720_50step", "resolution": "480x720", "frames": 49, "sampling_steps": 50,
                   "latent": list(W["lat"]), "cfg_batch": 2, "text_tokens": 226, "joint_sequence": 226 + 13 * 30 * 45,
                   "architecture": "CogVideoX-2B transformer (hidden 1920, 30 heads x 64, 30 blocks)", "pab": bool(args.pab),
                   "parallelism": par, "first_schedule_index": first,
                   "l2": "per-step working set (136 MB per activation tensor, 30 blocks) exceeds the 126 MB L2; no flush needed"},
        "e2e": {"value": W["frames"] / (W["steps"] * sec_e2e / args.steps), "unit": "frames/s",
                "h2d_bytes_per_step": z_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4,
                "ms_per_step": sec_e2e / args.steps * 1e3},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "attn_flash (joint text + video attention, 17 776 tokens, head_dim 64): 60 % of the step's FLOPs",
                     "bound": "tensor", "achieved": a_tf, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": a_tf / peaks["tflops"],
                     "traffic": None, "peak_source": peaks["src"], "launches_timed": at[2],
                     "timed_in": "a second pass of the same steps with CUDA-event pairs around every launch",
                     "share_of_step": at[0] / (sec_prof * 1e3)},
        "kernels": shares, "cpu_baseline": None,
        "cpu_baseline_note": "not sampled for this workload: one CogVideoX block on the host needs the full 17 776-token joint "
                             "attention (2.4 TFLOP in 16-bit eager) -- minutes per sample; the headline workload carries the CPU arm",
        "clocks": clocks, "cuda_graph": False,
    }
    if args.depth:
        line["config"]["depth_override"] = args.depth
        line["invalid"] = "reduced depth (debug run): not a bench value"
    if sp_parity is not None:
        line["sp_parity"] = sp_parity
    if rank == 0:
        print(json.dumps(line), flush=True)
    pab_mgr.set_pab_manager(None)
    if world > 1:
        sync_all()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def _simple_bench(args, name, net, one, n_sched, z_host, dt, frames, steps, config, roof_kind, roof_label, dtype_str, first):
    """Timing / profiling / JSON tail shared by the single-GPU workloads of the widened models: ``one(z, k)`` is one denoising
    step on a resident latent (schedule index k); the e2e variant copies the latent in from pinned host memory and the result
    back out inside the timed region."""
    from videosys_b200 import kernels
    from videosys_b200.core.pab import pab_mgr

    dev = torch.device("cuda", 0)
    state = {"z": z_host.to(dev, dt)}

    def step_resident(i):
        state["z"] = one(state["z"], (first + i) % n_sched)

    out_host = torch.empty(z_host.shape, dtype=torch.float32).pin_memory()
    zdev = torch.empty(z_host.shape, device=dev, dtype=torch.float32)

    def step_e2e(i):
        zdev.copy_(z_host, non_blocking=True)
        out_host.copy_(one(zdev.to(dt), (first + i) % n_sched).float(), non_blocking=True)

    def timed(fn, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3

    for i in range(max(args.warmup, 3)):
        step_resident(i)
    net.reset_pab_state()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = kernels.launch_count()
    sec = timed(step_resident, args.steps)
    launches = kernels.launch_count() - l0
    net.reset_pab_state()
    sec_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs:  # the e2e arm leaves state["z"] alone; the profiled pass below advances it
        dump_outputs(args.dump_outputs, {"latent": state["z"], "latent_e2e": out_host})
    net.reset_pab_state()
    kernels.PROFILE, kernels.PROFILE_KINDS = [], None
    sec_prof = timed(step_resident, args.steps)
    prof, kernels.PROFILE = kernels.PROFILE, None
    by = {}
    for kind, a, b, work in prof:
        d = by.setdefault(kind, [0.0, 0.0, 0])
        d[0] += a.elapsed_time(b)
        d[1] += work
        d[2] += 1
    peaks = _peaks()
    tf = ("gemm", "attn_flash")
    shares = kernel_fractions({k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[2] / args.steps,
                                   "achieved": v[1] / (v[0] * 1e-3) / (1e12 if k in tf else 1e9),
                                   "unit": "TFLOP/s" if k in tf else "GB/s"} for k, v in by.items()}, peaks)
    rk = by.get(roof_kind, [1e-9, 0.0, 1])
    r_tf = rk[1] / (rk[0] * 1e-3) / 1e12
    per = sec / args.steps
    line = {
        "metric": "frames/sec", "value": frames / (steps * per), "unit": "frames/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": dtype_str, "data": "synthetic", "config": dict(config, workload=name, pab=bool(args.pab), parallelism="single",
                                                                first_schedule_index=first),
        "e2e": {"value": frames / (steps * sec_e2e / args.steps), "unit": "frames/s", "h2d_bytes_per_step": z_host.numel() * 4,
                "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": sec_e2e / args.steps * 1e3},
        "gpu_launches": int(launches),
        "roofline": {"kernel": roof_label, "bound": "tensor", "achieved": r_tf, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": r_tf / peaks["tflops"], "traffic": None, "peak_source": peaks["src"], "launches_timed": rk[2],
                     "timed_in": "a second pass of the same steps with CUDA-event pairs around every launch",
                     "share_of_step": rk[0] / (sec_prof * 1e3)},
        "kernels": shares, "cpu_baseline": None,
        "cpu_baseline_note": "not sampled for this workload (not a BASELINE.json config); the headline workload carries the CPU arm",
        "clocks": clocks, "cuda_graph": False,
    }
    if args.depth:
        line["config"]["depth_override"] = args.depth
        line["invalid"] = "reduced depth (debug run): not a bench value"
    print(json.dumps(line), flush=True)
    pab_mgr.set_pab_manager(None)


def run_vchitect(args):
    """One denoising step of Vchitect-2.0-2B as the reference runs it (pipeline_vchitect.py:916-954): the unconditional and
    the text forward (batch 1 each) through VchitectXLTransformerModel (24 MMDiT blocks, three joint attentions each),
    cosine-ramped guidance, flow-match Euler update.  1 GPU."""
    import videosys_b200  # noqa: F401
    from videosys_b200.core.pab import pab_mgr
    from videosys_b200.models.transformers.vchitect_transformer_3d import VchitectXLTransformerModel
    from videosys_b200.pipelines.vchitect.pipeline_vchitect import VchitectPABConfig
    from videosys_b200.schedulers.scheduling_flow_match_euler import FlowMatchEulerDiscreteScheduler

    if args.gpus != 1 or int(os.environ.get("WORLD_SIZE", 1)) != 1:
        raise SystemExit("the Vchitect workload is a 1-GPU bench line (the model's frame-sharded parallelism has no bench leg)")
    W = VCHITECT
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dt = torch.bfloat16
    torch.manual_seed(0)
    net = VchitectXLTransformerModel(num_layers=args.depth or W["layers"], num_attention_heads=W["heads"],
                                     attention_head_dim=W["head_dim"], caption_projection_dim=W["heads"] * W["head_dim"])
    for prm in net.parameters():  # random-init weights of the named architecture (incl. the three zero-initialised projections)
        if prm.ndim >= 2:
            torch.nn.init.normal_(prm, std=0.02)
    net = net.to(dt).to(dev).eval()
    sched = FlowMatchEulerDiscreteScheduler(shift=3.0)
    sched.set_timesteps(W["steps"], dev)
    ts = [float(v) for v in sched.timesteps.tolist()]
    if args.pab:
        pab_mgr.set_pab_manager(VchitectPABConfig())
        pab_mgr.update_steps(W["steps"])
    g = torch.Generator(device="cpu").manual_seed(1)
    z_host = torch.randn(1, *W["lat"], generator=g).pin_memory()
    pe = [torch.randn(1, *W["text"], generator=g).to(dev, dt) for _ in range(2)]
    pp = [torch.randn(1, W["pooled"], generator=g).to(dev, dt) for _ in range(2)]

    def one(z, k):
        t = ts[k]
        tt = sched.timesteps[k].expand(1)
        un, tx = (net(z, encoder_hidden_states=e, pooled_projections=p, timestep=tt, return_dict=False,
                      ts_int=int(t) if args.pab else None)[0] for e, p in zip(pe, pp))
        sched._step_index = k
        return sched.step(un + 7.5 * (tx - un), t, z)[0]

    S, L = (W["h"] // 16) * (W["w"] // 16), W["text"][0]
    config = {"resolution": "288x480", "frames": 40, "sampling_steps": 100, "latent": list(W["lat"]), "forwards_per_step": 2,
              "text_tokens": L, "tokens_per_frame": S + L,
              "architecture": "Vchitect-2.0-2B transformer (hidden 1536, 24 heads x 64, 24 MMDiT blocks)",
              "l2": "per-step working set (107 MB per joint activation tensor, 24 blocks) exceeds what stays in the 126 MB L2 "
                    "across a block; no flush needed"}
    _simple_bench(args, "vchitect_2b_40f_288x480_100step", net, one, len(ts), z_host, dt, W["frames"], W["steps"], config, "gemm",
                  "gemm2_bf16_tn_kernel / gemm_bf16_tn_kernel (every Linear of the two forwards)", "bf16",
                  args.first_step if args.first_step >= 0 else (20 if args.pab else 0))


def run_osp_v120(args):
    """One denoising step of Open-Sora-Plan v1.2.0 29x480p (pipeline_open_sora_plan.py:1095-1160): the CFG pair through
    OpenSoraT2V (32 blocks, full 3-D attention over 8 x 30 x 40 = 9600 tokens, 24 heads x 96 -> csrc/attn_mma.cu), guidance,
    ancestral Euler update.  fp16 as the reference, 1 GPU."""
    import videosys_b200  # noqa: F401
    from videosys_b200.core.pab import pab_mgr
    from videosys_b200.models.transformers.open_sora_plan_v120_transformer_3d import OpenSoraT2V
    from videosys_b200.pipelines.open_sora_plan.pipeline_open_sora_plan import OpenSoraPlanV120PABConfig
    from videosys_b200.schedulers.scheduling_euler_ancestral import EulerAncestralDiscreteScheduler

    if args.gpus != 1 or int(os.environ.get("WORLD_SIZE", 1)) != 1:
        raise SystemExit("the Open-Sora-Plan workload is a 1-GPU bench line")
    W = OSP_V120
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dt = torch.float16
    torch.manual_seed(0)
    net = OpenSoraT2V(num_layers=args.depth or W["layers"], sample_size=W["sample_size"], sample_size_t=W["lat"][1],
                      interpolation_scale_h=1.0, interpolation_scale_w=1.0, interpolation_scale_t=1.0)
    for prm in net.parameters():  # random-init weights of the named architecture (small, so 32 blocks stay finite in fp16)
        if prm.ndim >= 2:
            torch.nn.init.normal_(prm, std=0.01)
    net = net.to(dt).to(dev).eval()
    sched = EulerAncestralDiscreteScheduler()
    sched.set_timesteps(W["steps"], dev)
    ts = [float(v) for v in sched.timesteps.tolist()]
    if args.pab:
        pab_mgr.set_pab_manager(OpenSoraPlanV120PABConfig())
        pab_mgr.update_steps(W["steps"])
    g = torch.Generator(device="cpu").manual_seed(1)
    z_host = torch.randn(1, *W["lat"], generator=g).pin_memory()
    pe = (0.1 * torch.randn(2, 1, *W["text"], generator=g)).to(dev, dt)
    mask = torch.ones(2, 1, W["text"][0])
    mask[0, 0, 1:] = 0   # the empty negative prompt
    mask[1, 0, 60:] = 0  # a 60-token caption, the rest is tokenizer padding

    def one(z, k):
        t = ts[k]
        sched._step_index = k
        inp = sched.scale_model_input(torch.cat([z, z]), t).to(dt)
        tt = torch.full((2,), t, device=dev, dtype=torch.float32)
        noise = net(inp, timestep=tt, encoder_hidden_states=pe, encoder_attention_mask=mask, return_dict=False,
                    ts_int=int(t) if args.pab else None)[0]
        un, tx = noise.chunk(2)
        noise = (un + 7.5 * (tx - un)).chunk(2, dim=1)[0]  # learned sigma: keep the mean prediction
        return sched.step(noise, t, z)[0].to(dt)

    config = {"resolution": "480x640", "frames": 29, "sampling_steps": 100, "latent": list(W["lat"]), "cfg_batch": 2,
              "text_tokens": W["text"][0], "tokens": W["lat"][1] * (W["sample_size"][0] // 2) * (W["sample_size"][1] // 2),
              "architecture": "OpenSoraT2V-ROPE-L/122 (hidden 2304, 24 heads x 96, 32 blocks, full 3-D attention)",
              "l2": "per-step working set (88 MB per activation tensor, 32 blocks) exceeds what stays in the 126 MB L2 across a "
                    "block; no flush needed"}
    _simple_bench(args, "osp_v120_29f_480p_100step", net, one, len(ts), z_host, dt, W["frames"], W["steps"], config, "attn_flash",
                  "attn_mma_kernel<96> behind vsb_attn_flash (3-D self attention over 9600 tokens + text cross attention)", "f16",
                  args.first_step if args.first_step >= 0 else (20 if args.pab else 0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="opensora_720p_68f_50step", choices=sorted(WORKLOADS) + ["cogvideox_2b_49f_480x720_50step", "vchitect_2b_40f_288x480_100step",
                                                                                           "osp_v120_29f_480p_100step"])
    ap.add_argument("--pab", action="store_true", help="enable Pyramid Attention Broadcast (config 5)")
    ap.add_argument("--cp", action="store_true", help="CogVideoX workload, N > 1: CFG parallelism instead of a factor 2 of sequence parallelism")
    ap.add_argument("--depth", type=int, default=0, help="debug only: fewer block pairs (marks the line invalid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the eager torch/cuBLAS/SDPA baseline (N = 1)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying CUDA graphs")
    ap.add_argument("--first-step", type=int, default=-1, help="schedule index of the first timed step (default 0; 22 with --pab: inside the broadcast range)")
    ap.add_argument("--opt", action="append", default=[], help="kernel selection knob name=value (vsb_set_option)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the latents of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm times a CPU sample, not the denoising step")
    if args.workload.startswith("cogvideox"):
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm is defined for the OpenSora workloads"}))
        else:
            run_cogvideox(args)
    elif args.workload.startswith("vchitect") or args.workload.startswith("osp_"):
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the CPU reference arm is defined for the OpenSora workloads"}))
        else:
            (run_vchitect if args.workload.startswith("vchitect") else run_osp_v120)(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
