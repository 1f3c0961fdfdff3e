"""Generates tests/golden/reference_pins.pt.gz by EXECUTING THE UNMODIFIED REFERENCE (needs the reference tree, see ref_loader).

    python -m oracle.gen_golden_pins

For every check of tests/test_oracle_vs_reference.py it runs the reference's side exactly as that test sets it up (same
configurations, synth tags, inputs and PAB schedules, from oracle/pin_cases.py) and stores what the test compares
against, in the compact forms of oracle/pins.py, together with the state-dict templates the test fills its weights from.
"""
import importlib
import os
import threading

import torch

from . import cases, pin_cases as PC, pins, ref_loader, synth

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_pins.pt.gz")
DT = PC.DT


def _stdit3(G, P):
    c = cases.small_model_cfg(depth=2)
    for dtype in (torch.float32, torch.bfloat16):
        net = ref_loader.build_stdit3(dtype=dtype, **c)
        G[f"tmpl.stdit3.{DT[dtype]}"] = pins.template(net.state_dict())
        net.load_state_dict(synth.fill_state_dict(net.state_dict(), "vsref."))
        inp = cases.forward_inputs(dtype)
        G[f"stdit3.forward.{DT[dtype]}"] = pins.exact(net(inp["x"], inp["timestep"], inp["y"], mask=inp["mask"],
                                                          x_mask=inp["x_mask"], fps=inp["fps"], height=inp["height"],
                                                          width=inp["width"]))
    steps = PC.OPENSORA_PAB_STEPS
    P.set_pab_manager(P.PABConfig(**PC.OPENSORA_PAB_KW))
    P.update_steps(len(steps))
    inp = cases.forward_inputs(torch.bfloat16)
    try:
        for i, t in enumerate(steps):
            inp["x"] = synth.normalish(f"pab.x{i}", tuple(inp["x"].shape))
            inp["timestep"] = torch.tensor([float(t)] * 2)
            G[f"stdit3.pab.{i}"] = pins.exact(net(inp["x"], inp["timestep"], inp["y"], mask=inp["mask"], x_mask=inp["x_mask"],
                                                  fps=inp["fps"], height=inp["height"], width=inp["width"]))
    finally:
        P.PAB_MANAGER = None


def _pab_gate(G, P):
    got = []
    try:
        for spec, steps, ts in PC.pab_gate_cases():
            P.set_pab_manager(P.PABConfig(**PC.pab_config_kw(spec)))
            P.update_steps(steps)
            for k, fn in (("spatial", P.if_broadcast_spatial), ("temporal", P.if_broadcast_temporal), ("cross", P.if_broadcast_cross)):
                c1 = 0
                for t in ts[k]:
                    f1, c1 = fn(t, c1)
                    got.append((int(f1), c1))
    finally:
        P.PAB_MANAGER = None
    G["pab_gate"] = pins.exact(torch.tensor(got, dtype=torch.int64))


class _FakeDist:
    """Thread-per-rank stand-in for torch.distributed so the reference comm functions run on CPU."""

    def __init__(self, sp):
        self.sp = sp
        self.board = [None] * sp
        self.bar = threading.Barrier(sp)
        self.local = threading.local()
        self.ProcessGroup = object

    def get_world_size(self, group=None):
        return self.sp

    def get_rank(self, group=None):
        return self.local.rank

    def all_to_all(self, output_list, input_list, group=None):
        r = self.local.rank
        self.board[r] = input_list
        self.bar.wait()
        for src in range(self.sp):
            output_list[src].copy_(self.board[src][r])
        self.bar.wait()


def _run_ranks(comm, sp, fn):
    fake = _FakeDist(sp)
    old = comm.dist
    comm.dist = fake
    outs, errs = [None] * sp, []

    def body(r):
        fake.local.rank = r
        try:
            outs[r] = fn(r)
        except Exception as e:
            errs.append(e)
            fake.bar.abort()

    try:
        th = [threading.Thread(target=body, args=(r,)) for r in range(sp)]
        [t.start() for t in th]
        [t.join() for t in th]
    finally:
        comm.dist = old
    assert not errs, errs
    return outs


def _dsp(G, comm):
    from . import dsp_oracle

    for sp, T, S in PC.DSP_CASES:
        full = synth.normalish(f"dsp{sp}{T}{S}", (2, T, S, 16))
        tp, spd = dsp_oracle.pad_amount(T, sp), dsp_oracle.pad_amount(S, sp)

        def fn(r):
            x = comm._split_sequence_func(full, None, 2, spd)
            a = comm.all_to_all_with_pad(x, None, scatter_dim=1, gather_dim=2, scatter_pad=tp, gather_pad=spd)
            b = comm.all_to_all_with_pad(a, None, scatter_dim=2, gather_dim=1, scatter_pad=spd, gather_pad=tp)
            return [pins.exact(v) for v in (x, a, b)]

        G[f"dsp.{sp}.{T}.{S}"] = _run_ranks(comm, sp, fn)


def _cogvideox_small_pieces(G, ref):
    for dtype in (torch.float32, torch.bfloat16):
        mod = ref.normalization.CogVideoXLayerNormZero(64, 128, True, 1e-5, bias=True).to(dtype)
        G[f"tmpl.lnz.{DT[dtype]}"] = pins.template(mod.state_dict())
        sd = synth.fill_state_dict(mod.state_dict(), "lnz.")
        sd["norm.weight"] = (1 + 0.2 * synth.uniform("lnz.w", (128,))).to(dtype)
        mod.load_state_dict(sd)
        h, e, t = PC.lnz_inputs(dtype)
        G[f"lnz.{DT[dtype]}"] = [pins.exact(v) for v in mod(h, e, t)]

    Ref = ref_loader.load_cogvideox_scheduler()
    s = Ref(**PC.COGX_DDIM)
    rec = {"alphas_cumprod": pins.exact(s.alphas_cumprod), "timesteps": {}}
    for n in (50, 30, 7):
        s.set_timesteps(n)
        rec["timesteps"][n] = s.timesteps.tolist()
    s.set_timesteps(50)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 3, 4, 6, 6, generator=g)
    rec["steps"] = []
    for t in s.timesteps:
        x = s.step(torch.randn(x.shape, generator=g), t, x, return_dict=False)[0]
        rec["steps"].append(pins.close(x.float(), k=x.numel()))  # every value: 432 per step
    G["cogx_ddim"] = rec


def _vchitect_attention(G, ref):
    A, P = ref.attentions, ref.pab_mgr
    C, H = PC.VCH_ATTN_C, PC.VCH_ATTN_H

    def build(pre_only, dtype):
        attn = A.VchitectAttention(query_dim=C, cross_attention_dim=None, added_kv_proj_dim=C, dim_head=C // H, heads=H,
                                   out_dim=C, context_pre_only=pre_only, bias=True, processor=A.VchitectAttnProcessor())
        attn = attn.to(dtype).eval()
        attn.parallel_manager = ref_loader.SingleRankPM()
        G[f"tmpl.vch_attn.{int(pre_only)}.{DT[dtype]}"] = pins.template(attn.state_dict())
        attn.load_state_dict(synth.fill_state_dict(attn.state_dict(), "vchattn."))
        return attn

    from . import vchitect_oracle as VO

    fc = VO.freqs_cis(C // H, 64, theta=1e6)
    for dtype in (torch.float32, torch.bfloat16):
        for Fr, S, L, pre_only in PC.VCH_ATTN_CASES:
            attn = build(pre_only, dtype)
            nh = synth.normalish("vch.h", (Fr, S, C)).to(dtype)
            ne = synth.normalish("vch.e", (Fr, L, C)).to(dtype)
            rv, re = attn(hidden_states=nh, encoder_hidden_states=ne, freqs_cis=fc, full_seqlen=Fr, Frame=Fr,
                          timestep=torch.tensor([500]))
            G[f"vch_attn.{Fr}.{S}.{L}.{int(pre_only)}.{DT[dtype]}"] = [pins.exact(rv), pins.exact(re)]
    attn = build(False, torch.float32)
    Fr, S, L = PC.VCH_ATTN_PAB_SHAPE
    P.set_pab_manager(P.PABConfig(**PC.VCH_ATTN_PAB_KW))
    P.update_steps(len(PC.PAB_TS))
    try:
        for step, t in enumerate(PC.PAB_TS):
            nh = synth.normalish(f"vchp.h{step}", (Fr, S, C))
            ne = synth.normalish(f"vchp.e{step}", (Fr, L, C))
            rv, re = attn(hidden_states=nh, encoder_hidden_states=ne, freqs_cis=fc, full_seqlen=Fr, Frame=Fr,
                          timestep=torch.tensor([t]))
            G[f"vch_attn_pab.{step}"] = [pins.exact(rv), pins.exact(re)]
    finally:
        P.PAB_MANAGER = None


def _osp_v110(G, P):
    def pair(cfg, tag, key):
        net = ref_loader.build_osp_v110(**cfg)
        G[f"tmpl.{key}"] = pins.template(net.state_dict())
        net.load_state_dict(synth.fill_state_dict(net.state_dict(), tag))
        return net

    def call(net, x, t, all_ts, enc, m):
        return net(x, timestep=t, all_timesteps=torch.tensor(all_ts), encoder_hidden_states=enc,
                   added_cond_kwargs={"resolution": None, "aspect_ratio": None},
                   attention_mask=torch.ones(x.shape[0], *x.shape[2:]), encoder_attention_mask=m, return_dict=False)[0]

    for use_rope, HW, scale1d in PC.OSP_MIRROR_CASES:
        key = PC.osp_key(use_rope, HW, scale1d)
        net = pair(dict(PC.OSP_SMALL, use_rope=use_rope, interpolation_scale_1d=scale1d), "osp.", key)
        x, enc, m = PC.osp_inputs(2, 5, HW)
        G[key] = pins.close(call(net, x, torch.tensor([500, 500]), [900, 500], enc, m))
    net = pair(PC.OSP_SMALL, "ospp.", "ospp")
    P.set_pab_manager(P.PABConfig(**PC.OSP_PAB_KW))
    P.update_steps(len(PC.PAB_TS))
    try:
        for step, t in enumerate(PC.PAB_TS):
            x, enc, m = PC.osp_inputs(2, 5, (8, 8), tag=f"ospp{step}.")
            G[f"ospp.{step}"] = pins.close(call(net, x, torch.tensor([t, t]), PC.PAB_TS, enc, m))
    finally:
        P.PAB_MANAGER = None
    M = ref_loader.load_osp_v110()
    D, Hh, h, w, Fr = 72, 3, 5, 7, 9
    for dtype in (torch.bfloat16, torch.float16, torch.float32):
        q2 = synth.normalish("rope.q2", (2, Hh, h * w, D)).to(dtype)
        want2 = M.LinearScalingRoPE2D(scaling_factor=2)(q2, M.PositionGetter2D()(2, h, w, "cpu"))
        q1 = synth.normalish("rope.q1", (4, Hh, Fr, D)).to(dtype)
        want1 = M.LinearScalingRoPE1D(scaling_factor=2)(q1, M.PositionGetter1D()(4, Fr, "cpu"))
        G[f"osp_rope.{DT[dtype]}"] = [pins.exact(want2), pins.exact(want1)]


def _latte(G, P):
    ref32 = None
    for dtype in (torch.float32, torch.bfloat16):
        ref = ref_loader.build_latte(dtype=dtype, **PC.LATTE_SMALL)
        sd0 = {k: v.float() for k, v in ref.state_dict().items()}
        G[f"tmpl.latte.{DT[dtype]}"] = pins.template(sd0)
        ref.load_state_dict({k: v.to(dtype) for k, v in synth.fill_state_dict(sd0, "lattep.").items()})
        x = synth.normalish("lattep.x", (2, 4, 6, 8, 8)).to(dtype)
        enc = synth.normalish("lattep.enc", (2, 7, 32)).to(dtype)
        want = PC.latte_call(ref, x, torch.tensor([500, 500]), enc)
        G[f"latte.{DT[dtype]}"] = pins.close(want) if dtype == torch.float32 else pins.exact(want)
        ref32 = ref32 if dtype != torch.float32 else ref
    ref = ref32
    P.set_pab_manager(P.PABConfig(**PC.LATTE_PAB_KW))
    P.update_steps(len(PC.PAB_TS))
    enc = synth.normalish("lattep.enc", (2, 7, 32))
    try:
        for step, tv in enumerate(PC.PAB_TS):
            x = synth.normalish(f"lattep.x{step}", (2, 4, 6, 8, 8))
            G[f"latte.pab.{step}"] = pins.close(PC.latte_call(ref, x, torch.tensor([tv, tv]), enc, PC.PAB_TS))
    finally:
        P.PAB_MANAGER = None


def _cogx_ref(dtype, cfg, tag, G):
    ref = ref_loader.build_cogvideox(dtype=dtype, **cfg)
    sd0 = {k: v.float() for k, v in ref.state_dict().items()}
    G[f"tmpl.{tag}{DT[dtype]}"] = pins.template(sd0)
    ref.load_state_dict(PC.cogx_norms(synth.fill_state_dict(sd0, tag), tag, dtype))
    return ref


def _cogvideox(G, P):
    ref32 = None
    for dtype in (torch.float32, torch.bfloat16, torch.float16):
        ref = _cogx_ref(dtype, PC.COGX_SMALL, "cogxp.", G)
        lat = synth.normalish("cogxp.lat", (2, 3, 4, 12, 16)).to(dtype)
        txt = synth.normalish("cogxp.txt", (2, 16, 48)).to(dtype)
        want = ref(lat, txt, torch.tensor([499, 499]), return_dict=False)[0]
        G[f"cogx.{DT[dtype]}"] = pins.close(want) if dtype == torch.float32 else pins.exact(want)
        ref32 = ref32 if dtype != torch.float32 else ref
    ref = ref32
    txt = synth.normalish("cogxp.txt", (2, 16, 48))
    P.set_pab_manager(P.PABConfig(**PC.COGX_PAB_KW))
    P.update_steps(len(PC.PAB_TS))
    try:
        for step, tv in enumerate(PC.PAB_TS):
            lat = synth.normalish(f"cogxp.lat{step}", (2, 3, 4, 12, 16))
            G[f"cogx.pab.{step}"] = pins.close(ref(lat, txt, torch.tensor([tv, tv]), return_dict=False)[0])
    finally:
        P.PAB_MANAGER = None
    ref_loader.load_cogvideox()
    E = importlib.import_module("videosys.models.modules.embeddings")
    from . import cogvideox_oracle as CO

    for gh, gw in PC.COGX_ROT_GRIDS:
        rc, rs = E.get_3d_rotary_pos_embed(64, CO.resize_crop_region_for_grid((gh, gw), 45, 30), (gh, gw), 5, use_real=True)
        G[f"cogx_rot.grid.{gh}x{gw}"] = [pins.exact(rc), pins.exact(rs)]
    for dtype in (torch.float32, torch.bfloat16):
        x = synth.normalish("rot.x", (2, 3, 3 * 6 * 8, 64)).to(dtype)
        G[f"cogx_rot.apply.{DT[dtype]}"] = pins.exact(E.apply_rotary_emb(x, PC.cogx_rotary()))
    for dtype in (torch.float32, torch.bfloat16):
        ref = _cogx_ref(dtype, dict(PC.COGX_SMALL, use_rotary_positional_embeddings=True), "cogxr.", G)
        lat = synth.normalish("cogxr.lat", (2, 3, 4, 12, 16)).to(dtype)
        txt = synth.normalish("cogxr.txt", (2, 16, 48)).to(dtype)
        want = ref(lat, txt, torch.tensor([499, 499]), image_rotary_emb=PC.cogx_rotary(), return_dict=False)[0]
        G[f"cogx_rot.{DT[dtype]}"] = pins.close(want) if dtype == torch.float32 else pins.exact(want)


def _vch_ref(dtype=torch.float32, G=None):
    ref = ref_loader.build_vchitect(dtype=dtype, **PC.VCH_SMALL)
    sd0 = {k: v.float() for k, v in ref.state_dict().items()}
    if G is not None:
        G[f"tmpl.vchm.{DT[dtype]}"] = pins.template(sd0)
        G[f"vchm.pos_embed.{DT[dtype]}"] = pins.exact(sd0["pos_embed.pos_embed"].to(dtype))
    sd = synth.fill_state_dict(sd0, "vchm.")
    sd["pos_embed.pos_embed"] = sd0["pos_embed.pos_embed"]
    ref.load_state_dict({k: v.to(dtype) for k, v in sd.items()})
    return ref


def _vchitect(G, P):
    for dtype in (torch.float32, torch.bfloat16):
        ref = _vch_ref(dtype, G)
        for Fr in (5, 1):
            lat = synth.normalish("vchm.lat", (1, Fr, 4, 12, 16)).to(dtype)
            enc = synth.normalish("vchm.enc", (1, 9, 48)).to(dtype)
            pooled = synth.normalish("vchm.pool", (1, 40)).to(dtype)
            want = ref(lat, encoder_hidden_states=enc, pooled_projections=pooled, timestep=torch.tensor([500.0]),
                       return_dict=False)[0]
            G[f"vch.{Fr}.{DT[dtype]}"] = pins.close(want) if dtype == torch.float32 else pins.exact(want)
    ref = _vch_ref()
    enc = synth.normalish("vchm.enc", (1, 9, 48))
    pooled = synth.normalish("vchm.pool", (1, 40))
    for pab in (False, True):
        steps = PC.PAB_TS if pab else [500]
        if pab:
            P.set_pab_manager(P.PABConfig(**PC.VCH_PAB_KW))
            P.update_steps(len(steps))
        try:
            for step, tv in enumerate(steps):
                lat = synth.normalish(f"vchm.lat{step}", (1, 4, 4, 12, 16))
                want = ref(lat, encoder_hidden_states=enc, pooled_projections=pooled, timestep=torch.tensor([float(tv)]),
                           return_dict=False)[0]
                G[f"vch.mirror.{int(pab)}.{step}"] = pins.close(want)
        finally:
            P.PAB_MANAGER = None


def _vch_sp_ref_worker(rank, world, port, Fr, q):
    """One gloo rank running the reference transformer under frame-sharded sequence parallelism."""
    import traceback
    import types

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    try:
        import torch.distributed as dist

        from videosys_b200.core.distributed.parallel_mgr import initialize

        initialize(rank, world)

        def a2a(out_list, in_list, group=None):  # gloo has no all_to_all: the same exchange through all_to_all_single
            send = torch.stack([t.contiguous() for t in in_list])
            recv = torch.empty_like(send)
            dist.all_to_all_single(recv, send, group=group)
            for o, r in zip(out_list, recv.unbind(0)):
                o.copy_(r)

        dist.all_to_all = a2a
        RC = ref_loader.load().comm

        def gather_cpu(input_, pg, dim, pad):  # the reference's _gather_sequence_func (comm.py:170-190) minus its CUDA assert
            parts = [torch.empty_like(input_.contiguous()) for _ in range(dist.get_world_size(pg))]
            dist.all_gather(parts, input_.contiguous(), group=pg)
            out = torch.cat(parts, dim=dim)
            return out.narrow(dim, 0, out.size(dim) - pad) if pad > 0 else out

        RC._gather_sequence_func = gather_cpu
        ref = _vch_ref()
        pm = types.SimpleNamespace(sp_size=world, sp_group=dist.group.WORLD, cp_size=1, sp_rank=rank)
        ref.parallel_manager = pm
        for mod in ref.modules():
            if hasattr(mod, "parallel_manager"):
                mod.parallel_manager = pm
        lat, enc, pooled = PC.vch_sp_inputs(Fr)
        with torch.no_grad():
            want = ref(lat, encoder_hidden_states=enc, pooled_projections=pooled, timestep=torch.tensor([500.0]),
                       return_dict=False)[0]
        rec = {k: v.numpy() if torch.is_tensor(v) else v for k, v in pins.close(want).items()}  # by value: no shared-memory
        q.put((rank, rec, None))                                                                  # handles that die with the worker
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        q.put((rank, None, traceback.format_exc()))


def _vchitect_sp(G):
    import multiprocessing as mp

    ctx = mp.get_context("spawn")
    for Fr in (4, 5, 2):
        world, port = 2, 30950 + (os.getpid() % 40) + Fr
        q = ctx.Queue()
        procs = [ctx.Process(target=_vch_sp_ref_worker, args=(r, world, port, Fr, q)) for r in range(world)]
        [p.start() for p in procs]
        recs = [None] * world
        for _ in range(world):
            r, rec, tb = q.get(timeout=300)
            assert tb is None, tb
            recs[r] = {k: torch.from_numpy(v) if hasattr(v, "dtype") else v for k, v in rec.items()}
        [p.join(timeout=60) for p in procs]
        G[f"vch.sp.{Fr}"] = recs


def _osp_v120(G, P):
    def pair(cfg, tag, key):
        net = ref_loader.build_osp_v120(**cfg)
        G[f"tmpl.{key}"] = pins.template(net.state_dict())
        net.load_state_dict(synth.fill_state_dict(net.state_dict(), tag))
        return net

    def call(net, x, t, enc, m):
        return net(x, timestep=t, encoder_hidden_states=enc, attention_mask=torch.ones(x.shape[0], *x.shape[2:]),
                   encoder_attention_mask=m, return_dict=False)[0]

    for use_rope, HW in PC.OSP12_MIRROR_CASES:
        key = PC.osp12_key(use_rope, HW)
        net = pair(dict(PC.OSP12_SMALL, use_rope=use_rope), "osp12.", key)
        x, enc, m = PC.osp_inputs(2, 5, HW, tag="osp12.")
        G[key] = pins.close(call(net, x, torch.tensor([500, 500]), enc, m))
    net = pair(PC.OSP12_SMALL, "osp12p.", "osp12p")
    P.set_pab_manager(P.PABConfig(**PC.OSP12_PAB_KW))
    P.update_steps(len(PC.PAB_TS))
    try:
        for step, t in enumerate(PC.PAB_TS):
            x, enc, m = PC.osp_inputs(2, 5, (8, 8), tag=f"osp12p{step}.")
            G[f"osp12p.{step}"] = pins.close(call(net, x, torch.tensor([t, t]), enc, m))
    finally:
        P.PAB_MANAGER = None
    M = ref_loader.load_osp_v120()
    D, Hh, T, h, w = 96, 3, 4, 3, 5
    for dtype in (torch.bfloat16, torch.float16, torch.float32):
        q = synth.normalish("rope3.q", (2, Hh, T * h * w, D)).to(dtype)
        want = M.RoPE3D(interpolation_scale_thw=(1.5, 1.0, 2.0))(q, M.PositionGetter3D()(2, T, h, w, "cpu"))
        G[f"osp12_rope3d.{DT[dtype]}"] = pins.exact(want)


def _stdit3_mirror(G, P):
    c = cases.small_model_cfg(depth=2)
    ref16 = ref_loader.build_stdit3(dtype=torch.bfloat16, **c)
    G["tmpl.stde.bfloat16"] = pins.template(ref16.state_dict())
    sd = synth.fill_state_dict(ref16.state_dict(), "stde.")
    ref16.load_state_dict(sd)
    ref32 = ref_loader.build_stdit3(dtype=torch.float32, **c)
    ref32.load_state_dict({k: v.float() for k, v in sd.items()})
    inp = cases.forward_inputs(torch.bfloat16)
    G["stde.0"] = pins.rel(PC.stdit3_run(ref16, inp, torch.bfloat16), PC.stdit3_run(ref32, inp, torch.float32))
    res = {}
    for model, dt in ((ref16, torch.bfloat16), (ref32, torch.float32)):
        P.set_pab_manager(P.PABConfig(**PC.STDIT3_PAB_KW))
        P.update_steps(len(PC.STDIT3_PAB_TS))
        try:
            for t in PC.STDIT3_PAB_TS:
                inp["timestep"] = torch.tensor([t, t], dtype=torch.bfloat16)
                res.setdefault(dt, []).append(PC.stdit3_run(model, inp, dt))
        finally:
            P.PAB_MANAGER = None
    for i in range(len(PC.STDIT3_PAB_TS)):
        G[f"stde.{i + 1}"] = pins.rel(res[torch.bfloat16][i], res[torch.float32][i])


@torch.no_grad()
def main():
    G = {}
    ref = ref_loader.load()
    P = ref.pab_mgr
    _stdit3(G, P)
    _pab_gate(G, P)
    _dsp(G, ref.comm)
    _cogvideox_small_pieces(G, ref)
    _vchitect_attention(G, ref)
    _osp_v110(G, P)
    _latte(G, P)
    _cogvideox(G, P)
    _vchitect(G, P)
    _osp_v120(G, P)
    _stdit3_mirror(G, P)
    torch.set_grad_enabled(True)
    _vchitect_sp(G)
    pins.save(G, OUT)
    print(len(G), "records,", os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
