"""N > 1 path.  CPU part: world_size-2 gloo processes check the shard plan and that
"each rank denoises its chunk -> all-gather -> ordered blend" equals the single-process oracle.
GPU part (needs >= 2 GPUs): the sharded MultiDiffusion delegate, NCCL and fused
peer-memory exchange, must be bit-identical to the single-GPU result on every rank."""
import os
import socket
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import blend, synth, tiling

CASE = dict(N=2, C=4, W=128, H=128, tw=96, th=96, ov=48, bs=4)      # T = 4: ranks get 2 tiles each
CASE2 = dict(N=2, C=4, W=512, H=512, tw=96, th=96, ov=48, bs=4)     # BASELINE cfg2, T = 100


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _init(rank, world, port, backend):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group(backend, rank=rank, world_size=world)


def _oracle(c, x):
    plan = tiling.GridPlan(c["W"], c["H"], c["tw"], c["th"], c["ov"], c["bs"], False)
    return plan, blend.multidiffusion_step(x, plan.batched_bboxes, plan.weights, lambda t, bb: synth.fake_denoise(t, bb, c["N"]))


def _gloo_worker(rank, world, port, result_dir):
    from multidiffusion_upscaler_for_automatic1111_b200 import parallel
    _init(rank, world, port, "gloo")
    try:
        for c in (CASE, dict(CASE, W=160, H=64, tw=32, th=24, ov=8)):   # second case: T not divisible by world
            x = synth.latent(17, (c["N"], c["C"], c["H"], c["W"]), torch.float16)
            plan, want = _oracle(c, x)
            T, N = len(plan.bboxes), c["N"]
            sh = parallel.TileShard(T, rank, world)
            assert sh.chunk == -(-T // world) and 0 <= sh.begin <= sh.end <= T
            mine = plan.bboxes[sh.begin:sh.end]
            local = torch.zeros((sh.chunk * N, c["C"], plan.tile_h, plan.tile_w), dtype=x.dtype)
            if mine:
                local[:len(mine) * N] = synth.fake_denoise(blend.scatter_tiles(x, mine), mine, N)
            gathered = parallel.gather_tile_outputs(local)
            acc = torch.zeros_like(x)
            for b in range(sh.num_chunks):
                bbs = plan.bboxes[b * sh.chunk:min((b + 1) * sh.chunk, T)]
                blend.accumulate_md(acc, gathered[b * sh.chunk * N:(b * sh.chunk + len(bbs)) * N], bbs, N)
            got = blend.normalise_md(acc, torch.from_numpy(plan.weights).view(1, 1, c["H"], c["W"]))
            assert torch.equal(got, want), f"rank {rank}: sharded result differs"
        open(os.path.join(result_dir, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


def test_tile_shard_plan():
    from multidiffusion_upscaler_for_automatic1111_b200.parallel import TileShard
    for T, world in [(100, 8), (4, 2), (7, 4), (1, 2), (36, 8), (121, 8)]:
        shards = [TileShard(T, r, world) for r in range(world)]
        assert sum(s.num_local for s in shards) == T
        assert [s.begin for s in shards][1:] == [s.end for s in shards][:-1] or T < world * shards[0].chunk
        covered = [t for s in shards for t in range(s.begin, s.end)]
        assert covered == list(range(T))
        assert all(shards[0].owner(t) == r for r, s in enumerate(shards) for t in range(s.begin, s.end))
        assert shards[0].num_chunks == -(-T // shards[0].chunk)


def test_gloo_world2_sharded_step_equals_single(tmp_path):
    mp.spawn(_gloo_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def _gloo_delegate_worker(rank, world, port, result_dir):
    """The tile-sharded DELEGATES (MultiDiffusion all-gather path, Mixture of Diffusers) on CPU tensors over gloo, with the
    device kernels swapped for the oracle's scatter / blend: every rank must return the single-process result."""
    from multidiffusion_upscaler_for_automatic1111_b200 import MixtureOfDiffusers, MultiDiffusion, engine, host
    from multidiffusion_upscaler_for_automatic1111_b200.tile_methods import abstractdiffusion

    def bbs(g):
        return [tuple(int(v) for v in r) for r in engine.grid_bboxes_xywh(g)]

    def scatter_tiles(g, x, out=None, tile_begin=0, tile_end=None, flags=0):
        return blend.scatter_tiles(x, bbs(g)[tile_begin:tile_end])

    def blend_multidiffusion(g, outs, N, C, tile_bs, weights, acc_dtype, x_buffer=None, flags=0, out=None, rcp_weights=None):
        buf = torch.zeros((N, C, g.H, g.W), dtype=acc_dtype)
        blend.accumulate_md(buf, torch.cat(list(outs), dim=0), bbs(g), N)
        return blend.normalise_md(buf, weights)

    def blend_mixture(g, outs, N, C, tile_bs, tile_weights, rescale, x_buffer, flags=0):
        x_buffer.zero_()
        blend.accumulate_mod(x_buffer, torch.cat(list(outs), dim=0), bbs(g), N, tile_weights, rescale)
        return x_buffer
    engine.scatter_tiles, engine.blend_multidiffusion, engine.blend_mixture = scatter_tiles, blend_multidiffusion, blend_mixture
    abstractdiffusion.AbstractDiffusion._check_input = lambda self, x: x.contiguous()
    host.device = lambda: torch.device("cpu")        # the delegates' buffers on CPU too, also where a GPU is present

    _init(rank, world, port, "gloo")
    try:
        for c in (CASE, dict(CASE, W=160, H=64, tw=32, th=24, ov=8, bs=2)):
            N = c["N"]
            x = synth.latent(19, (N, c["C"], c["H"], c["W"]), torch.float16)
            p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a")
            cond = {"c_crossattn": [torch.zeros(N, 77, 8)], "c_concat": [torch.zeros(N, 5, 1, 1)]}
            state = {"i": 0}

            # MultiDiffusion, all-gather exchange
            def unet(x_tile, sigma, cond=None):
                bb = d.local_batched_bboxes[state["i"]]
                state["i"] += 1
                return synth.fake_denoise(x_tile, bb, N)
            sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=types.SimpleNamespace(forward=unet), image_cfg_scale=None))
            d = MultiDiffusion(p, sampler)
            d.init_grid_bbox(c["tw"], c["th"], c["ov"], c["bs"])
            d.init_done()
            sh = d.init_tile_shard(None, fused=False)
            d.hook()
            out = sampler.model_wrap_cfg.inner_model.forward(x, torch.ones(N), cond=cond)
            _, want = _oracle(c, x)
            assert torch.equal(out, want), f"rank {rank}: sharded MultiDiffusion delegate differs"
            assert state["i"] == len(d.local_batched_bboxes) and sum(len(b) for b in d.local_batched_bboxes) == sh.num_local

            # Mixture of Diffusers
            state["i"] = 0

            def apply_model(x_tile, t, c_):
                bb = m.local_batched_bboxes[state["i"]]
                state["i"] += 1
                return synth.fake_denoise(x_tile, bb, N)
            model = types.SimpleNamespace(apply_model=apply_model, cond_stage_key="txt", model=types.SimpleNamespace(conditioning_key="crossattn"))
            host.use_shared(types.SimpleNamespace(state=types.SimpleNamespace(interrupted=False, sampling_step=0, sampling_steps=1), sd_model=model))
            m = MixtureOfDiffusers(p, types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=types.SimpleNamespace(forward=None), image_cfg_scale=None)))
            m.init_grid_bbox(c["tw"], c["th"], c["ov"], c["bs"])
            m.init_done()
            m.init_tile_shard(None)
            m.hook()
            got = model.apply_model(x, torch.ones(N), cond).clone()
            MixtureOfDiffusers.unhook()
            plan = tiling.GridPlan(c["W"], c["H"], c["tw"], c["th"], c["ov"], c["bs"], True)
            want = blend.mixture_step(x, plan.batched_bboxes, plan.tile_weights, plan.rescale_factor, lambda t, bb: synth.fake_denoise(t, bb, N))
            assert torch.equal(got, want), f"rank {rank}: sharded Mixture of Diffusers delegate differs"
            host.use_shared(None)
        open(os.path.join(result_dir, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


def test_gloo_world2_sharded_delegates_equal_single(tmp_path):
    mp.spawn(_gloo_delegate_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def _gloo_demofusion_worker(rank, world, port, result_dir):
    """Tile-sharded DemoFusion (local windows and global views split over the ranks, grid and random jitter) on CPU
    stand-ins over gloo: every rank must reproduce the single-process oracle."""
    from helpers import DTYPES, install_demofusion_stand_ins
    from oracle import demofusion as odf
    from oracle.make_golden import DEMO_CFG, demo_denoise, position_aware_denoise
    from test_demofusion import _jitter_delegate, _jitter_oracle, _jitter_p, _oracle
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    install_demofusion_stand_ins()
    _init(rank, world, port, "gloo")
    try:
        c = DEMO_CFG
        for jitter, dn, mixture in [(False, "f32", True), (False, "f16", False), (True, "f32", True), (True, "f16", False)]:
            if jitter:
                x, x_step, want, local, sizes = _jitter_oracle(DTYPES[dn], mixture)
                d = _jitter_delegate(mixture)            # same seed on every rank -> same windows
                unet = position_aware_denoise(d)
            else:
                x, want, local, sizes = _oracle(DTYPES[dn], mixture)
                x_step = x
                p = _jitter_p(mixture)
                p.random_jitter = False
                inner = types.SimpleNamespace(forward=None)
                d = DemoFusion(p, types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, forward=None)))
                d.window_size, d.sig = c["window"], c["sig"]
                d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
                unet = lambda xt, sigma, cond=None: demo_denoise(xt)
            calls = []

            def counted(xt, sigma, cond=None, unet=unet):
                calls.append(xt.shape[0] // c["N"])
                return unet(xt, sigma, cond=cond)
            d.sampler_forward = counted
            sh = d.init_tile_shard(None)
            assert sh.num_tiles == len(local) and d._view_shard.num_tiles == sizes[2]
            d.cosine_factor = odf.cosine_factor(c["current_step"], c["t_enc"])
            cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8)], "c_concat": [torch.zeros(c["N"], 5, 1, 1)]}
            got = d.sample_one_step(x_step, torch.ones(c["N"]), cond)
            tol = 3e-6 if dn == "f32" else 2e-3
            err = (got.float() - want.float()).abs().max().item()
            assert got.shape == want.shape and err <= tol * max(1.0, want.float().abs().max().item()), f"rank {rank} jitter={jitter} {dn}: err {err}"
            assert sum(calls) == sh.num_local + d._view_shard.num_local      # this rank denoised only its own windows and views
        open(os.path.join(result_dir, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


def test_gloo_world2_sharded_demofusion_equals_single(tmp_path):
    mp.spawn(_gloo_demofusion_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()



# ------------------------------------------------------------------------------------------- strip shard plan (no GPU)
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8, 12])
@pytest.mark.parametrize("geom", [(512, 512, 96, 96, 48), (128, 200, 32, 24, 8), (96, 97, 96, 96, 48), (1024, 2048, 96, 96, 48)])
def test_strip_shard_plan_covers_and_reproduces_the_single_device_blend(world, geom):
    """parallel.StripShard: every canvas row is owned by exactly one rank; the rows a rank receives as tile halo are
    exactly what its strip needs from foreign tile rows; the latent halo covers its scatter extent; and blending each
    strip from own + halo rows only is bit-identical to the single-device step."""
    import numpy as np
    from multidiffusion_upscaler_for_automatic1111_b200 import engine, parallel
    W, H, tw, th, ov = geom
    N, C = (2, 4) if H * W <= 512 * 512 else (1, 1)
    plan = tiling.GridPlan(W, H, tw, th, ov, 4, False)
    g = engine.make_grid(W, H, tw, th, ov, 4)
    ys, cols = list(g.ys[:g.rows]), g.cols
    x = synth.latent(1, (N, C, H, W), torch.float16)
    full = blend.multidiffusion_step(x, plan.batched_bboxes, plan.weights, lambda t, bb: t * 0.5)
    outs = [x[:, :, y:y + h, xx:xx + w] * 0.5 for (xx, y, w, h) in plan.bboxes]
    wgt = torch.from_numpy(plan.weights).view(1, 1, H, W)
    got = torch.zeros_like(full)
    cover = np.zeros(H, int)
    shards = [parallel.StripShard(ys, cols, th, H, r, world) for r in range(world)]
    for r, sh in enumerate(shards):
        lo, hi = sh.strip()
        assert hi <= lo or (lo % 8 == 0 and (hi % 8 == 0 or hi == H))
        if hi <= lo:
            assert sh.halo_in() == []      # an empty strip (its tiles may still feed other ranks' strips)
            continue
        cover[lo:hi] += 1
        avail = {i: (0, th) for i in sh.bands()}
        for (i, pr, v0, v1) in sh.halo_in():
            assert sh.owner_of_band(i) == pr and (i, r, v0, v1) in shards[pr].halo_out()
            avail[i] = (v0, v1)
        buf = torch.zeros((N, C, H, W), dtype=torch.float16)
        for t, (xx, y, w, h) in enumerate(plan.bboxes):
            i = t // cols
            if i not in avail:
                assert y + h <= lo or y >= hi, "a tile row that touches the strip is neither owned nor received"
                continue
            v0, v1 = avail[i]
            a, b = max(y, lo), min(y + h, hi)
            if b > a:
                assert a >= y + v0 and b <= y + v1, "halo rows do not cover the strip part of the tile"
                buf[:, :, a:b, xx:xx + w] += outs[t][:, :, a - y:b - y]
        o = torch.where(wgt > 1, buf / wgt, buf)
        got[:, :, lo:hi] = o[:, :, lo:hi]
        s0, s1 = sh.scatter_rows()
        have = np.zeros(H, bool)
        have[lo:hi] = True
        for (q, a, b) in sh.x_in():
            assert (r, a, b) in shards[q].x_out()
            have[a:b] = True
        assert have[s0:s1].all(), "latent halo does not cover the scatter extent"
    assert (cover == 1).all()
    assert torch.equal(got, full)


# ------------------------------------------------------------------------------------------- GPU
def _gpu_worker(rank, world, port, result_dir):
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    torch.cuda.set_device(rank)
    _init(rank, world, port, "nccl")
    try:
        for c in (CASE, CASE2):
            x = synth.latent(23, (c["N"], c["C"], c["H"], c["W"]), torch.float16)
            plan, want = _oracle(c, x)
            for fused in (False, True):
                def unet(x_tile, sigma, cond=None):
                    bbs = d.local_batched_bboxes[state["i"]]
                    state["i"] += 1
                    return synth.fake_denoise(x_tile, bbs, c["N"])
                state = {"i": 0}
                inner = types.SimpleNamespace(forward=unet)
                sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None))
                p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a")
                d = MultiDiffusion(p, sampler)
                d.init_grid_bbox(c["tw"], c["th"], c["ov"], c["bs"])
                d.init_done()
                sh = d.init_tile_shard(None, fused=fused, mode="replicate")
                d.hook()
                cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8, device="cuda")], "c_concat": [torch.zeros(c["N"], 5, 1, 1, device="cuda")]}
                for step in range(3):    # several steps: double-buffered exchange + monotonic flags
                    state["i"] = 0
                    out = inner.forward(x.cuda(), torch.ones(c["N"], device="cuda"), cond=cond)
                    torch.cuda.synchronize()
                    assert torch.equal(out.cpu(), want), f"rank {rank} fused={fused} step {step}: differs from single-GPU oracle"
                assert state["i"] == len(d.local_batched_bboxes) and sh.num_local == sh.end - sh.begin
                if d._exchange is not None:
                    dist.barrier()
                    d._exchange.close()
        # row-strip shard (default fused mode): each rank blends its own rows from own + halo tile rows; several steps
        for c in (CASE, CASE2, dict(CASE2, W=256, H=640, N=1)):
            # a different latent every step: a halo left over from the previous step would not go unnoticed
            xs = [synth.latent(31 + k, (c["N"], c["C"], c["H"], c["W"]), torch.float16) for k in range(3)]
            wants = [_oracle(c, xk)[1] for xk in xs]

            def unet(x_tile, sigma, cond=None):
                bbs = d.local_batched_bboxes[state["i"]]
                state["i"] += 1
                return synth.fake_denoise(x_tile, bbs, c["N"])
            state = {"i": 0}
            inner = types.SimpleNamespace(forward=unet)
            sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None))
            p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a")
            d = MultiDiffusion(p, sampler)
            d.init_grid_bbox(c["tw"], c["th"], c["ov"], c["bs"])
            d.init_done()
            d.init_tile_shard(None, fused=True)
            assert d._shard_mode == "strip"
            d.hook()
            cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8, device="cuda")], "c_concat": [torch.zeros(c["N"], 5, 1, 1, device="cuda")]}
            for step in range(3):
                state["i"] = 0
                x, want = xs[step], wants[step]
                out = inner.forward(x.cuda(), torch.ones(c["N"], device="cuda"), cond=cond)
                torch.cuda.synchronize()
                sh = d._strip
                lo, hi = sh.strip()
                assert torch.equal(out[:, :, lo:hi].cpu(), want[:, :, lo:hi]), f"rank {rank} strip rows differ at step {step}"
                for (q, a, b) in sh.x_in():
                    assert torch.equal(out[:, :, a:b].cpu(), want[:, :, a:b]), f"rank {rank}: latent halo from rank {q} differs at step {step}"
                assert state["i"] == len(d.local_batched_bboxes)
                dist.barrier()      # the next step's halo pushes must not overtake this step's checks
            full = d.gather_latent(out)
            assert torch.equal(full.cpu(), want), f"rank {rank}: gathered latent differs"
            dist.barrier()
            d._strip_exchange.close()
        # tiled VAE, tiles sharded over the ranks: fast mode (no collective until the canvas all-reduce) and slow mode
        # (GroupNorm statistics all-reduced every round) must both reproduce the single-process oracle on every rank
        from multidiffusion_upscaler_for_automatic1111_b200 import tilevae
        from oracle import vae as ovae
        from oracle.make_golden import vae_case_inputs
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        for fast in (True, False):
            net, z = vae_case_inputs(True, 40, 52)
            with torch.no_grad():
                want = ovae.vae_hook_call(net, z, 16, True, fast, False)
            net_gpu, _ = vae_case_inputs(True, 40, 52)
            hook = tilevae.VAEHook(net_gpu.cuda(), 16, True, fast_decoder=fast, fast_encoder=fast, color_fix=False)
            hook.init_tile_shard(None)
            with torch.no_grad():
                got = hook(z.cuda())
            err = (got.cpu() - want).abs().max().item()
            assert err <= 3e-4 * max(1.0, want.abs().max().item()), f"rank {rank} sharded VAE fast={fast}: err {err}"
        open(os.path.join(result_dir, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_gpu_sharded_multidiffusion_bit_identical(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_gpu_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def _gpu_mod_worker(rank, world, port, result_dir):
    from multidiffusion_upscaler_for_automatic1111_b200 import MixtureOfDiffusers, host
    torch.cuda.set_device(rank)
    _init(rank, world, port, "nccl")
    try:
        for c in (CASE, CASE2):
            N = c["N"]
            x = synth.latent(29, (N, c["C"], c["H"], c["W"]), torch.float16)
            plan = tiling.GridPlan(c["W"], c["H"], c["tw"], c["th"], c["ov"], c["bs"], True)
            want = blend.mixture_step(x, plan.batched_bboxes, plan.tile_weights, plan.rescale_factor, lambda t, bb: synth.fake_denoise(t, bb, N))
            state = {"i": 0}

            def apply_model(x_tile, t, c_):
                bb = m.local_batched_bboxes[state["i"]]
                state["i"] += 1
                return synth.fake_denoise(x_tile, bb, N)
            model = types.SimpleNamespace(apply_model=apply_model, cond_stage_key="txt", model=types.SimpleNamespace(conditioning_key="crossattn"))
            host.use_shared(types.SimpleNamespace(state=types.SimpleNamespace(interrupted=False, sampling_step=0, sampling_steps=1), sd_model=model))
            p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a")
            m = MixtureOfDiffusers(p, types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=types.SimpleNamespace(forward=None), image_cfg_scale=None)))
            m.init_grid_bbox(c["tw"], c["th"], c["ov"], c["bs"])
            m.init_done()
            m.init_tile_shard(None)
            m.hook()
            cond = {"c_crossattn": [torch.zeros(N, 77, 8, device="cuda")], "c_concat": [torch.zeros(N, 5, 1, 1, device="cuda")]}
            for step in range(2):
                state["i"] = 0
                got = model.apply_model(x.cuda(), torch.ones(N, device="cuda"), cond)
                torch.cuda.synchronize()
                assert torch.equal(got.cpu(), want), f"rank {rank} step {step}: sharded Mixture of Diffusers differs"
            MixtureOfDiffusers.unhook()
            host.use_shared(None)
        open(os.path.join(result_dir, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


# first hardware run pending (written after the round-1 GPU budget was spent)
@pytest.mark.gpu
def test_two_gpu_sharded_mixture_bit_identical(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_gpu_mod_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def _gpu_demofusion_worker(rank, world, port, result_dir):
    from helpers import DTYPES
    from oracle import demofusion as odf
    from oracle.make_golden import DEMO_CFG, demo_denoise, position_aware_denoise
    from test_demofusion import _jitter_delegate, _jitter_oracle, _jitter_p, _oracle
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    torch.cuda.set_device(rank)
    _init(rank, world, port, "nccl")
    try:
        c = DEMO_CFG
        for jitter, dn, mixture in [(False, "f32", True), (False, "f16", False), (True, "f32", True)]:
            if jitter:
                x, x_step, want, local, sizes = _jitter_oracle(DTYPES[dn], mixture)
                d = _jitter_delegate(mixture)
                d.sampler_forward = position_aware_denoise(d)
            else:
                x, want, local, sizes = _oracle(DTYPES[dn], mixture)
                x_step = x
                p = _jitter_p(mixture)
                p.random_jitter = False
                inner = types.SimpleNamespace(forward=None)
                d = DemoFusion(p, types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, forward=None)))
                d.window_size, d.sig = c["window"], c["sig"]
                d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
                d.sampler_forward = lambda xt, sigma, cond=None: demo_denoise(xt)
            d.init_tile_shard(None)
            d.cosine_factor = odf.cosine_factor(c["current_step"], c["t_enc"])
            cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8, device="cuda")], "c_concat": [torch.zeros(c["N"], 5, 1, 1, device="cuda")]}
            got = d.sample_one_step(x_step.cuda(), torch.ones(c["N"], device="cuda"), cond)
            torch.cuda.synchronize()
            tol = 3e-6 if dn == "f32" else 2e-3
            err = (got.cpu().float() - want.float()).abs().max().item()
            assert err <= tol * max(1.0, want.float().abs().max().item()), f"rank {rank} jitter={jitter} {dn}: err {err}"
        open(os.path.join(result_dir, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


# first hardware run pending (written after the round-1 GPU budget was spent)
@pytest.mark.gpu
def test_two_gpu_sharded_demofusion_matches_oracle(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_gpu_demofusion_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
