"""DemoFusion (tile_methods/demofusion.py:219-324, jitter off): oracle vs the reference's fixtures (CPU),
and the sm_100a class path vs oracle (GPU)."""
import os
import types

import numpy as np
import pytest
import torch

from helpers import DTYPES, assert_trace, bits, digest, stub_webui
from oracle import demofusion as odf
from oracle import synth, tiling
from oracle.make_golden import DEMO_CASES, DEMO_CFG, demo_denoise


def _oracle(dtype, mixture):
    c = DEMO_CFG
    x = synth.latent(31, (c["N"], c["C"], c["H"], c["W"]), dtype)
    local, _, _ = tiling.demofusion_views(c["W"], c["H"], c["window"], c["overlap"])
    nb = -(-len(local) // c["tile_bs"]); tbs = -(-len(local) // nb)
    lb = [local[i * tbs:(i + 1) * tbs] for i in range(nb)]
    views = odf.global_views(c["scale"], mixture)
    gnb = -(-len(views) // c["tile_bs_g"]); gtbs = -(-len(views) // gnb)
    gb = [views[i * gtbs:(i + 1) * gtbs] for i in range(gnb)]
    cf = odf.cosine_factor(c["current_step"], c["t_enc"])
    y = odf.sample_one_step(x, lb, gb, c["scale"], mixture, True, c["sig"], cf, c["cs2"], c["cs3"],
                            lambda t, b: demo_denoise(t), lambda t, b: demo_denoise(t))
    return x, y, local, (tbs, gtbs, len(views))


@pytest.mark.parametrize("case", DEMO_CASES, ids=[c[0] for c in DEMO_CASES])
def test_oracle_matches_reference_fixture(golden_dir, case):
    name, dn, mixture = case
    g = np.load(os.path.join(golden_dir, "demofusion_small.npz"))
    _, y, local, sizes = _oracle(DTYPES[dn], mixture)
    assert np.array_equal(np.array(local, np.int32), g[name + "_local"])
    assert list(sizes) == list(g[name + "_tile_bs"])
    assert str(y.dtype) == str(g[name + "_dtype"])
    want = torch.from_numpy(g[name].view(np.float32 if dn == "f32" else np.float16).copy())
    tol = 2e-6 if dn == "f32" else 2e-3     # another CPU's conv kernels: round-off only
    assert (y.float() - want.float()).abs().max().item() <= tol * max(1.0, want.float().abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("case", DEMO_CASES, ids=[c[0] for c in DEMO_CASES])
def test_demofusion_class_matches_oracle(case):
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    name, dn, mixture = case
    c = DEMO_CFG
    x, want, local, sizes = _oracle(DTYPES[dn], mixture)
    p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a", current_scale_num=c["scale"], mixture=mixture,
                              gaussian_filter=True, random_jitter=False, cosine_scale_1=c["cs1"], cosine_scale_2=c["cs2"],
                              cosine_scale_3=c["cs3"], current_step=c["current_step"], steps=20, t_enc=c["t_enc"], sd_model=None)
    calls = []

    def fwd(x_tile, sigma, cond=None):
        calls.append(tuple(x_tile.shape))
        assert sigma.shape[0] == x_tile.shape[0] and cond["c_crossattn"][0].shape[0] == x_tile.shape[0]
        return demo_denoise(x_tile)
    inner = types.SimpleNamespace(forward=fwd)
    sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, forward=None))
    d = DemoFusion(p, sampler)
    d.window_size, d.sig = c["window"], c["sig"]
    d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
    assert [(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb] == local
    assert (d.tile_bs, d.global_tile_bs, d.global_num_tiles) == sizes
    d.sampler_forward = fwd
    d.cosine_factor = odf.cosine_factor(c["current_step"], c["t_enc"])
    cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8, device="cuda")], "c_concat": [torch.zeros(c["N"], 5, 1, 1, device="cuda")]}
    got = d.sample_one_step(x.cuda(), torch.ones(c["N"], device="cuda"), cond)
    assert got.dtype == DTYPES[dn] and got.shape == want.shape
    assert len(calls) == d.num_batches + d.global_num_batches
    tol = 3e-6 if dn == "f32" else 2e-3
    err = (got.cpu().float() - want.float()).abs().max().item()
    assert err <= tol * max(1.0, want.float().abs().max().item()), f"{name}: max err {err}"


@pytest.mark.gpu
def test_demofusion_cfg5_size_matches_oracle():
    """BASELINE cfg5's step (bench.py --config cfg5): latent [2,4,768,768] fp16, 121 windows of 128^2, scale 4, mixture --
    the class on the sm_100a kernels against the oracle run on the host at the same size."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    c = bench.DEMO
    d, fwd, calls = bench._demo_job(torch.device("cuda"), torch.float16, True, False)
    d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
    half = lambda x_tile, sigma=None, cond=None: demo_denoise(x_tile)
    d.sampler_forward = half
    cf = odf.cosine_factor(c["current_step"], c["t_enc"])
    d.cosine_factor = cf
    L = c["lat"]
    x = synth.latent(77, (c["N"], c["C"], L, L), torch.float16)
    local, _, _ = tiling.demofusion_views(L, L, c["window"], c["overlap"])
    assert [(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb] == local and len(local) == 121
    lb = [local[i * d.tile_bs:(i + 1) * d.tile_bs] for i in range(d.num_batches)]
    views = odf.global_views(c["scale"], True)
    gb = [views[i * d.global_tile_bs:(i + 1) * d.global_tile_bs] for i in range(d.global_num_batches)]
    want = odf.sample_one_step(x, lb, gb, c["scale"], True, True, c["sig"], cf, c["cs2"], c["cs3"],
                               lambda t, b: demo_denoise(t), lambda t, b: demo_denoise(t))
    cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8, device="cuda")], "c_concat": [torch.zeros(c["N"], 5, 1, 1, device="cuda")]}
    got = d.sample_one_step(x.cuda(), torch.ones(c["N"], device="cuda"), cond)
    assert got.dtype == torch.float16 and got.shape == want.shape
    err = (got.cpu().float() - want.float()).abs().max().item()
    assert err <= 2e-3 * max(1.0, want.float().abs().max().item()), f"max err {err}"


@pytest.mark.gpu
def test_dilated_gather_and_combine_are_exact():
    """Index work is bit-exact: gather == strided slices; combine == the eager add-back + mix in fp16."""
    import ctypes
    from multidiffusion_upscaler_for_automatic1111_b200._cabi import check, current_stream_ptr, lib
    N, C, H, W, s = 2, 4, 48, 64, 2
    x = synth.latent(5, (N, C, H, W), torch.float16).cuda()
    g_ = synth.latent(6, (N, C, H, W), torch.float16).cuda()
    views = [(0, 0), (1, 0), (0, 1), (1, 1)] * 2
    second = [0] * 4 + [1] * 4
    oh, ow = H // s, W // s
    out = torch.empty((8 * N, C, oh, ow), dtype=torch.float16, device="cuda")
    arr = lambda v: (ctypes.c_int32 * len(v))(*v)
    check(lib.td_dilated_gather(x.data_ptr(), g_.data_ptr(), out.data_ptr(), N, C, H, W, s, oh, ow, arr([v[0] for v in views]),
                                arr([v[1] for v in views]), arr(second), 8, 0, current_stream_ptr()))
    want = torch.cat([(g_ if sec else x)[:, :, by::s, bx::s] for (bx, by), sec in zip(views, second)], dim=0)
    assert torch.equal(out, want)
    x_local = synth.latent(7, (N, C, H, W), torch.float16).cuda()
    res = torch.empty_like(x_local)
    ptrs = (ctypes.c_void_p * 2)(out[:4 * N].data_ptr(), out[4 * N:].data_ptr())
    c2 = 0.3125
    check(lib.td_demofusion_combine(x_local.data_ptr(), ptrs, 2, 4, 8, res.data_ptr(), N, C, H, W, s, oh, ow, H, W, 1, c2, 1 - c2, 0,
                                    current_stream_ptr()))
    xg = torch.zeros_like(x_local)
    for idx, (bx, by) in enumerate(views):
        xg[:, :, by::s, bx::s] += out[idx * N:(idx + 1) * N]
    want = x_local * (1 - c2) + (xg / 2) * c2
    assert torch.equal(res, want)


# ------------------------------------------------------------------------------------------ random jitter
def _jitter_oracle(dtype, mixture):
    """Oracle run of the jitter fixtures: seeded windows, padded latent, position-aware local UNet stand-in."""
    import random
    import torch.nn.functional as F
    from oracle.make_golden import DEMO_JITTER_SEED
    c = DEMO_CFG
    x = synth.latent(31, (c["N"], c["C"], c["H"], c["W"]), dtype)
    local, _, _, jr = tiling.demofusion_views_jitter(c["W"], c["H"], c["window"], c["overlap"], random.Random(DEMO_JITTER_SEED))
    nb = -(-len(local) // c["tile_bs"]); tbs = -(-len(local) // nb)
    lb = [local[i * tbs:(i + 1) * tbs] for i in range(nb)]
    views = odf.global_views(c["scale"], mixture)
    gnb = -(-len(views) // c["tile_bs_g"]); gtbs = -(-len(views) // gnb)
    gb = [views[i * gtbs:(i + 1) * gtbs] for i in range(gnb)]
    cf = odf.cosine_factor(c["current_step"], c["t_enc"])
    xp = F.pad(x, (jr, jr, jr, jr), "constant", value=0)
    y = odf.sample_one_step(xp, lb, gb, c["scale"], mixture, True, c["sig"], cf, c["cs2"], c["cs3"],
                            lambda t, b: synth.fake_denoise(t, b, c["N"]), lambda t, b: demo_denoise(t), jitter_range=jr)
    return x, xp, y, local, (tbs, gtbs, len(views), jr)


def _jitter_p(mixture):
    c = DEMO_CFG
    return types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a", current_scale_num=c["scale"], mixture=mixture,
                                 gaussian_filter=True, random_jitter=True, cosine_scale_1=c["cs1"], cosine_scale_2=c["cs2"],
                                 cosine_scale_3=c["cs3"], current_step=c["current_step"], steps=20, t_enc=c["t_enc"], sd_model=None)


def _jitter_delegate(mixture):
    import random
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    from oracle.make_golden import DEMO_JITTER_SEED
    c = DEMO_CFG
    inner = types.SimpleNamespace(forward=None)
    d = DemoFusion(_jitter_p(mixture), types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, forward=None)))
    d.window_size, d.sig = c["window"], c["sig"]
    random.seed(DEMO_JITTER_SEED)
    d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
    return d


def test_jitter_oracle_and_windows_match_reference_fixture(golden_dir):
    from oracle.make_golden import DEMO_JITTER_CASES
    g = np.load(os.path.join(golden_dir, "demofusion_jitter.npz"))
    for name, dn, mixture in DEMO_JITTER_CASES:
        _, _, y, local, sizes = _jitter_oracle(DTYPES[dn], mixture)
        assert np.array_equal(np.array(local, np.int32), g[name + "_local"])
        assert list(sizes) == list(g[name + "_sizes"])
        want = torch.from_numpy(g[name].view(np.float32 if dn == "f32" else np.float16).copy())
        assert y.shape == want.shape and str(y.dtype) == str(g[name + "_dtype"])
        tol = 2e-6 if dn == "f32" else 2e-3
        assert (y.float() - want.float()).abs().max().item() <= tol * max(1.0, want.float().abs().max().item())
        # the delegate draws the same windows from Python's `random` (host-side bookkeeping, no kernel involved)
        d = _jitter_delegate(mixture)
        assert [(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb] == [tuple(int(v) for v in r) for r in g[name + "_local"]]
        assert [d.tile_bs, d.global_tile_bs, d.global_num_tiles, d.jitter_range] == list(g[name + "_sizes"])


def _forward_one_step(webui, cls):
    """forward_one_step (demofusion.py:185-214) of a `cls` delegate with the tiled step itself replaced by a stub: checks
    the zero padding the stub sees and returns the cropped CFG output."""
    import random
    from oracle.make_golden import DEMO_JITTER_SEED
    c = DEMO_CFG
    g = torch.Generator().manual_seed(1)
    x = torch.randn(c["N"], c["C"], c["H"], c["W"], generator=g)
    px, pn = torch.randn(x.shape, generator=g), torch.randn(x.shape, generator=g)
    p = _jitter_p(True)
    p.x, p.noise, p.disable_extra_networks, p.batch_size = px, pn, True, 1
    seen = {}

    def forward_ori(x_in, sigma, **kw):
        return cfg.inner_model.forward(x_in, sigma, kw.get("cond"))
    inner = types.SimpleNamespace(forward="original")
    cfg = types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, forward=forward_ori, step=0)

    class _S(webui.KDiffusionSampler):
        pass
    sampler = _S()
    sampler.model_wrap_cfg = cfg
    d = cls(p, sampler)
    d.window_size, d.sig = c["window"], c["sig"]
    random.seed(DEMO_JITTER_SEED)
    d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
    d.hook()

    def fake_step(x_in, sigma, cond, seen=seen):
        seen["shape"] = tuple(x_in.shape)
        seen["border"] = float(x_in[:, :, :d.jitter_range].abs().max())
        return x_in * 2 + 1
    d.sample_one_step = fake_step
    out = cfg.forward(x, torch.full((c["N"],), 3.0), cond=None)
    assert cfg.inner_model.forward == "original"                 # restored after the call
    jr = d.jitter_range
    assert jr == 6 and seen["shape"] == (c["N"], c["C"], c["H"] + 2 * jr, c["W"] + 2 * jr) and seen["border"] == 0.0
    assert out.shape == x.shape
    return out


def reference_traces(ref):
    """The reference's side of test_forward_one_step_pads_and_crops_like_the_reference (oracle/make_reference_traces.py)."""
    return {"demofusion_forward_one_step": [digest(_forward_one_step(ref, ref.demofusion.DemoFusion))]}


def test_forward_one_step_pads_and_crops_like_the_reference(monkeypatch):
    """Skip-residual mix, zero-pad by jitter_range, CFG forward with the tiled step patched in, crop back: our delegate on
    CPU under the stub WebUI against the reference's output under the same stub (tests/golden/reference_traces.npz)."""
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    with stub_webui(monkeypatch) as webui:
        out = _forward_one_step(webui, DemoFusion)
    assert_trace([digest(out)], "demofusion_forward_one_step")


# ------------------------------------------------------------------------------------------ delegate host logic on CPU
def _oracle_engine_for_demofusion(monkeypatch):
    from helpers import install_demofusion_stand_ins
    install_demofusion_stand_ins(monkeypatch.setattr)


@pytest.mark.parametrize("jitter", [False, True], ids=["grid", "jitter"])
@pytest.mark.parametrize("dn,mixture", [("f32", True), ("f32", False), ("f16", True)])
def test_delegate_plumbing_on_cpu_stand_ins(monkeypatch, jitter, dn, mixture):
    import random
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    from oracle.make_golden import DEMO_JITTER_SEED, position_aware_denoise
    _oracle_engine_for_demofusion(monkeypatch)
    c = DEMO_CFG
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
    assert [(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb] == local
    d.cosine_factor = odf.cosine_factor(c["current_step"], c["t_enc"])
    cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8)], "c_concat": [torch.zeros(c["N"], 5, 1, 1)]}
    got = d.sample_one_step(x_step, torch.ones(c["N"]), cond)
    assert got.dtype == DTYPES[dn] and got.shape == want.shape
    tol = 3e-6 if dn == "f32" else 2e-3
    err = (got.float() - want.float()).abs().max().item()
    assert err <= tol * max(1.0, want.float().abs().max().item()), f"max err {err}"
