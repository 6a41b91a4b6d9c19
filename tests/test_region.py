"""Region prompt control (custom bboxes, SURVEY.md section 8(f)-1): feather masks, region rectangles, weight canvases
and one full step of MultiDiffusion / Mixture of Diffusers with BACKGROUND and FOREGROUND regions.

The expected values are fixtures generated from the UNMODIFIED reference (tests/golden/region_small.npz,
oracle/make_golden.py::gen_region).  CPU tests pin the oracle restatement and the C-ABI bookkeeping, and run the
delegates' host logic with the device kernels swapped for the oracle's scatter / blend (the kernels themselves are
pinned by tests/test_gpu_diffusion.py).  The `gpu` test runs the same delegates on the real kernels.
"""
import os
import types

import numpy as np
import pytest
import torch

from helpers import region_composite_reference, DTYPES, assert_bit_equal
from oracle import blend, region, synth, tiling
from oracle.make_golden import REGION_CASES, REGION_DTYPES, REGION_GRID

G = REGION_GRID


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "region_small.npz"))


def _want(gold, key):
    dt = getattr(torch, str(gold[key + "_dtype"]).split(".")[-1])
    raw = gold[key]
    t = torch.from_numpy(raw.view(np.int16 if raw.dtype == np.uint16 else np.int32).copy())
    return t.view(dt)


def _p():
    # the prompt fields are only read when a WebUI prompt parser is importable (the reference shim provides a stand-in)
    return types.SimpleNamespace(width=G["W"] * 8, height=G["H"] * 8, sampler_name="Euler a", disable_extra_networks=True,
                                 batch_size=1, steps=20, styles=None, all_prompts=["a photo"], all_negative_prompts=["blurry"])


class _KSampler:
    def __init__(self, fwd=None):
        inner = types.SimpleNamespace(forward=fwd)
        self.model_wrap_cfg = types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, step=0)


def _x(name, dn):
    return synth.latent(synth.case_seed("region_" + name, dn), (G["N"], G["C"], G["H"], G["W"]), DTYPES[dn])


# ------------------------------------------------------------------------------------------------ bookkeeping
def test_feather_mask_cabi_and_oracle_match_reference(gold):
    from multidiffusion_upscaler_for_automatic1111_b200.tile_utils import utils
    for w, h, r in gold["mask_cases"]:
        w, h = int(w), int(h)
        want = gold[f"mask_{w}x{h}_{r}"]
        assert np.array_equal(utils.feather_mask_np(w, h, float(r)).view(np.uint32), want.view(np.uint32))
        assert np.array_equal(region.feather_mask(w, h, float(r)).view(np.uint32), want.view(np.uint32))
    m = utils.feather_mask(10, 8, 0.5)
    assert m.dtype == torch.float32 and tuple(m.shape) == (8, 10)


@pytest.mark.parametrize("case", REGION_CASES, ids=[c[0] for c in REGION_CASES])
def test_region_rects_and_weights_match_reference(gold, case):
    from multidiffusion_upscaler_for_automatic1111_b200 import MixtureOfDiffusers, MultiDiffusion
    name, bg, rows = case
    rects = gold[f"{name}_rects"]
    regs = region.make_regions(rows, G["W"], G["H"])
    assert [(r["x"], r["y"], r["w"], r["h"]) for r in regs] == [tuple(int(v) for v in r) for r in rects]
    for method, cls in (("md", MultiDiffusion), ("mod", MixtureOfDiffusers)):
        d = cls(_p(), _KSampler())
        d.init_grid_bbox(G["tw"], G["th"], G["ov"], G["bs"])
        d.init_custom_bbox({i: row for i, row in enumerate(rows)}, bg, False)
        d.init_done()
        assert [(b.x, b.y, b.w, b.h) for b in d.custom_bboxes] == [tuple(int(v) for v in r) for r in rects]
        assert d.enable_grid_bbox == bg and d.total_bboxes == (d.num_batches if bg else 0) + len(rects)
        want_w = gold[f"{name}_{method}_weights"]
        assert np.array_equal(d.weights[0, 0].cpu().numpy().view(np.uint32), want_w.view(np.uint32)), method
        plan = tiling.GridPlan(G["W"], G["H"], G["tw"], G["th"], G["ov"], G["bs"], method == "mod")
        ow = region.weights_with_regions(plan.weights if bg else None, regs, G["H"], G["W"], method)
        assert np.array_equal(ow.view(np.uint32), want_w.view(np.uint32)), "oracle " + method


def test_disabled_or_degenerate_rows_leave_nothing_to_paint():
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    from multidiffusion_upscaler_for_automatic1111_b200.tile_utils.utils import DEFAULT_BBOX_SETTINGS, build_bbox_settings
    d = MultiDiffusion(_p(), _KSampler())
    d.init_custom_bbox({0: DEFAULT_BBOX_SETTINGS, 1: (True, 1.5, 0.1, 0.2, 0.2, "", "", "Background", 0.2, -1)}, False, False)
    assert not d.enable_custom_bbox and not d.enable_grid_bbox
    with pytest.raises(AssertionError, match="Nothing to paint"):
        d.init_done()
    flat = [True, 0.12345678, 0.2, 0.3, 0.4, "p", "n", "Foreground", 0.23456, 7.0] + list(DEFAULT_BBOX_SETTINGS)
    st = build_bbox_settings(flat)
    assert list(st) == [0] and st[0].x == 0.1235 and st[0].feather_ratio == 0.2346 and st[0].seed == 7


# ------------------------------------------------------------------------------------------------ oracle step
@pytest.mark.parametrize("case", REGION_CASES, ids=[c[0] for c in REGION_CASES])
@pytest.mark.parametrize("method", ["md", "mod"])
@pytest.mark.parametrize("dn", REGION_DTYPES)
def test_oracle_region_step_matches_reference_fixture(gold, case, method, dn):
    name, bg, rows = case
    x = _x(name, dn)
    N = x.shape[0]
    plan = tiling.GridPlan(G["W"], G["H"], G["tw"], G["th"], G["ov"], G["bs"], method == "mod")
    regs = region.make_regions(rows, G["W"], G["H"])
    w = region.weights_with_regions(plan.weights if bg else None, regs, G["H"], G["W"], method)

    def den(t, bb):
        return synth.fake_denoise(t, bb, N)
    if method == "md":
        got = region.multidiffusion_region_step(x, plan.batched_bboxes, w, regs, den, synth.fake_region_denoise, bg)
    else:
        got = region.mixture_region_step(x, plan.batched_bboxes, plan.tile_weights, w, regs, den, synth.fake_region_denoise, bg)
    assert_bit_equal(got, _want(gold, f"{name}_{method}_{dn}"), "oracle region step")


# ------------------------------------------------------------------------------------------------ delegates
def _oracle_engine(monkeypatch):
    """Swap the three device entry points for the oracle so the delegates' host logic runs on CPU tensors (their
    buffers too, also where a GPU is present)."""
    from multidiffusion_upscaler_for_automatic1111_b200 import engine, host
    from multidiffusion_upscaler_for_automatic1111_b200.tile_methods import abstractdiffusion

    def bbs(g):
        return [tuple(int(v) for v in r) for r in engine.grid_bboxes_xywh(g)]

    def scatter_tiles(g, x, out=None, tile_begin=0, tile_end=None, flags=0):
        return blend.scatter_tiles(x, bbs(g)[tile_begin:tile_end])

    def blend_multidiffusion(g, outs, N, C, tile_bs, weights, acc_dtype, x_buffer=None, flags=0, out=None, rcp_weights=None):
        buf = torch.zeros((N, C, g.H, g.W), dtype=acc_dtype)
        blend.accumulate_md(buf, torch.cat(list(outs), dim=0), bbs(g), N)
        if x_buffer is not None:
            x_buffer.copy_(buf)
        return blend.normalise_md(buf, weights)

    def blend_mixture(g, outs, N, C, tile_bs, tile_weights, rescale, x_buffer, flags=0):
        x_buffer.zero_()
        blend.accumulate_mod(x_buffer, torch.cat(list(outs), dim=0), bbs(g), N, tile_weights, rescale)
        return x_buffer

    monkeypatch.setattr(engine, "region_composite", region_composite_reference)
    monkeypatch.setattr(engine, "scatter_tiles", scatter_tiles)
    monkeypatch.setattr(engine, "blend_multidiffusion", blend_multidiffusion)
    monkeypatch.setattr(engine, "blend_mixture", blend_mixture)
    monkeypatch.setattr(abstractdiffusion.AbstractDiffusion, "_check_input", lambda self, x: x.contiguous())
    monkeypatch.setattr(host, "device", lambda: torch.device("cpu"))


def _run_delegate(method, x, bg, rows, device):
    """One step of OUR delegate with custom bboxes; returns (delegate, output)."""
    from multidiffusion_upscaler_for_automatic1111_b200 import MixtureOfDiffusers, MultiDiffusion, host
    N = x.shape[0]
    it = {"i": 0}
    cond = {"c_crossattn": [torch.zeros(N, 2, 4, device=device)], "c_concat": [torch.zeros(N, 5, 1, 1, device=device)]}

    def custom(x_tile, bbox_id, bbox):
        return synth.fake_region_denoise(x_tile, bbox_id)

    if method == "md":
        d = MultiDiffusion(_p(), _KSampler())
        d.init_grid_bbox(G["tw"], G["th"], G["ov"], G["bs"])
        d.init_custom_bbox({i: row for i, row in enumerate(rows)}, bg, False)
        d.init_done()
        out = d.sample_one_step(x.to(device), None, lambda t, bb: synth.fake_denoise(t, bb, N), custom)
        return d, out

    def apply_model(x_tile, t, c):
        bb = d.batched_bboxes[it["i"]]
        it["i"] += 1
        return synth.fake_denoise(x_tile, bb, N)

    model = types.SimpleNamespace(apply_model=apply_model, cond_stage_key="txt", model=types.SimpleNamespace(conditioning_key="crossattn"))
    host.use_shared(types.SimpleNamespace(state=types.SimpleNamespace(interrupted=False, sampling_step=0, sampling_steps=1), sd_model=model))
    try:
        d = MixtureOfDiffusers(_p(), _KSampler())
        d.init_grid_bbox(G["tw"], G["th"], G["ov"], G["bs"])
        d.init_custom_bbox({i: row for i, row in enumerate(rows)}, bg, False)
        d.init_done()
        d.custom_apply_model = lambda x_tile, t, c, bbox_id, bbox: custom(x_tile, bbox_id, bbox)
        d.hook()
        out = model.apply_model(x.to(device), torch.ones(N, device=device), cond)
        d.unhook()
        return d, out.clone()
    finally:
        host.use_shared(None)


@pytest.mark.parametrize("case", REGION_CASES, ids=[c[0] for c in REGION_CASES])
@pytest.mark.parametrize("method", ["md", "mod"])
@pytest.mark.parametrize("dn", REGION_DTYPES)
def test_delegate_region_step_host_logic_on_oracle_engine(gold, monkeypatch, case, method, dn):
    name, bg, rows = case
    _oracle_engine(monkeypatch)
    d, out = _run_delegate(method, _x(name, dn), bg, rows, "cpu")
    assert_bit_equal(out, _want(gold, f"{name}_{method}_{dn}"), f"{method} delegate, oracle engine")


def test_interrupt_during_region_pass_returns_input(monkeypatch):
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion, host
    _oracle_engine(monkeypatch)
    st = types.SimpleNamespace(interrupted=False, sampling_step=0, sampling_steps=1)
    host.use_shared(types.SimpleNamespace(state=st, sd_model=None))
    try:
        d = MultiDiffusion(_p(), _KSampler())
        d.init_grid_bbox(G["tw"], G["th"], G["ov"], G["bs"])
        d.init_custom_bbox({i: row for i, row in enumerate(REGION_CASES[0][2])}, True, False)
        d.init_done()
        x = _x("bg_fg", "f16")

        def custom(x_tile, bbox_id, bbox):
            st.interrupted = True            # the user cancels while the first region is being denoised
            return x_tile
        assert d.sample_one_step(x, None, lambda t, bb: t, custom) is x
    finally:
        host.use_shared(None)
