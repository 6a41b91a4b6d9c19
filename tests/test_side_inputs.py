"""ControlNet / StableSR tile caches (SURVEY.md section 8(f)-2): the per-batch hint tiles our delegate caches and
hands to the extension objects must equal the reference's, for k-diffusion and DDIM samplers, grid and custom bboxes.

CPU: our delegate under the stub WebUI of oracle/ref_shim.py, with the scatter kernel swapped for the oracle's scatter
(the kernel itself is pinned by tests/test_gpu_diffusion.py), against what the UNMODIFIED reference cached under the
same stub (`reference_traces` below, stored in tests/golden/reference_traces.npz).  GPU: the same caches through
td_scatter_tiles on the x8-scaled tile plan, against plain slicing.
"""
import types

import pytest
import torch

from helpers import assert_trace, digest, stub_webui
from oracle import blend, ref_shim

W, H = 64, 48
ROWS = [(True, 0.1, 0.2, 0.5, 0.4, "a cat", "", "Background", 0.2, -1),
        (True, 0.4, 0.3, 0.45, 0.6, "a dog", "ugly", "Foreground", 0.3, 5)]


def _p():
    return types.SimpleNamespace(width=W * 8, height=H * 8, sampler_name="Euler a", disable_extra_networks=True,
                                 batch_size=1, steps=20, styles=None, all_prompts=["a photo"], all_negative_prompts=["blurry"])


def _hints(device="cpu"):
    a = (torch.arange(1 * 3 * H * 8 * W * 8, dtype=torch.float32, device=device).view(1, 3, H * 8, W * 8) % 1021) / 1021.0
    b = (torch.arange(3 * H * 8 * W * 8, dtype=torch.float32, device=device).view(3, H * 8, W * 8) % 509) / 509.0   # 3-d: unsqueezed in place
    return [a, b]


def _controlnet_script(device="cpu"):
    params = [types.SimpleNamespace(hint_cond=t) for t in _hints(device)]
    return types.SimpleNamespace(latest_network=types.SimpleNamespace(control_params=params))


def _oracle_scatter(monkeypatch):
    from multidiffusion_upscaler_for_automatic1111_b200 import engine

    def scatter_tiles(g, x, out=None, tile_begin=0, tile_end=None, flags=0):
        bbs = [tuple(int(v) for v in r) for r in engine.grid_bboxes_xywh(g)]
        return blend.scatter_tiles(x, bbs[tile_begin:tile_end])
    monkeypatch.setattr(engine, "scatter_tiles", scatter_tiles)


def _delegate(cls, sampler, settings, with_regions):
    d = cls(_p(), sampler)
    d.init_grid_bbox(16, 16, 8, 4)
    if with_regions:
        d.init_custom_bbox(settings, True, False)
    return d


def _sampler(webui, kdiff):
    if kdiff:
        return ref_shim.make_kdiff_sampler(lambda x, s, cond=None: x)

    class _S(webui.CompVisSampler):
        pass
    s = _S()
    s.model_wrap_cfg = types.SimpleNamespace(inner_model=types.SimpleNamespace(forward=None), image_cfg_scale=None, step=0)
    return s


def _controlnet_trace(d, cs, tensor_cpu, with_regions):
    """Digests of the hint tiles `d` caches for the ControlNet units of `cs`, then of the hints it hands them at the first
    and last batch (condition / denoise), at a custom region and after the reset."""
    d.init_controlnet(cs, tensor_cpu)
    d.init_done()
    if getattr(d, "pbar", None) is not None:
        d.pbar.disable = True
    hints = lambda: [digest(u.hint_cond) for u in cs.latest_network.control_params]
    out = [digest(t) for per_unit in d.control_tensor_batch for t in per_unit]
    if with_regions:
        out += [digest(t) for per_unit in d.control_tensor_custom for t in per_unit]
    for batch_id in (0, d.num_batches - 1):
        n_tiles = len(d.batched_bboxes[batch_id])
        for is_denoise in (False, True):
            d.switch_controlnet_tensors(batch_id, 2, n_tiles, is_denoise=is_denoise)
            out += hints()
    if with_regions:
        d.set_custom_controlnet_tensors(1, 3)
        out += hints()
    d.reset_controlnet_tensors()
    return out + hints()


def _stablesr_trace(d, latent):
    """Digests of the latent tiles `d` caches for StableSR, then of the latent it hands the model per batch and at a
    custom region; after the reset the model must hold the caller's latent again."""
    model = types.SimpleNamespace(set_image_hooks={}, latent_image=None)
    d.init_stablesr(types.SimpleNamespace(stablesr_model=model))
    d.init_done()
    if getattr(d, "pbar", None) is not None:
        d.pbar.disable = True
    model.set_image_hooks["TiledDiffusion"](latent)
    out = [digest(t) for t in d.stablesr_tensor_batch]
    for b in range(d.num_batches):
        d.switch_stablesr_tensors(b)
        out.append(digest(model.latent_image))
    d.set_custom_stablesr_tensors(1)
    out.append(digest(model.latent_image))
    d.reset_stablesr_tensors()
    assert model.latent_image is latent
    return out


CONTROLNET_CASES = [(kdiff, with_regions, tensor_cpu) for kdiff in (True, False) for with_regions in (False, True) for tensor_cpu in (False, True)]


def _latent():
    return torch.arange(2 * 4 * H * W, dtype=torch.float32).view(2, 4, H, W)


def reference_traces(ref):
    """The reference's side of the tests below (oracle/make_reference_traces.py)."""
    out = {}
    settings = {i: ref.utils.BBoxSettings(*r) for i, r in enumerate(ROWS)}
    for kdiff, with_regions, tensor_cpu in CONTROLNET_CASES:
        d = _delegate(ref.multidiffusion.MultiDiffusion, _sampler(ref, kdiff), settings, with_regions)
        assert d.is_kdiff == kdiff
        out[f"controlnet_{kdiff}_{with_regions}_{tensor_cpu}"] = _controlnet_trace(d, _controlnet_script(), tensor_cpu, with_regions)
    d = _delegate(ref.multidiffusion.MultiDiffusion, ref_shim.make_kdiff_sampler(lambda x, s, cond=None: x), settings, True)
    out["stablesr"] = _stablesr_trace(d, _latent())
    return out


@pytest.mark.parametrize("kdiff", [True, False], ids=["kdiff", "ddim"])
@pytest.mark.parametrize("with_regions", [False, True], ids=["grid", "grid+regions"])
@pytest.mark.parametrize("tensor_cpu", [False, True], ids=["dev", "cpu_cache"])
def test_controlnet_tile_caches_like_the_reference(monkeypatch, kdiff, with_regions, tensor_cpu):
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    with stub_webui(monkeypatch) as webui:
        _oracle_scatter(monkeypatch)
        d = _delegate(MultiDiffusion, _sampler(webui, kdiff), {i: r for i, r in enumerate(ROWS)}, with_regions)
        assert d.is_kdiff == kdiff
        cs = _controlnet_script()
        trace = _controlnet_trace(d, cs, tensor_cpu, with_regions)
    assert len(d.control_tensor_batch) == 2 and all(len(per_unit) == d.num_batches for per_unit in d.control_tensor_batch)
    assert all(u.hint_cond.shape == (1, 3, H * 8, W * 8) for u in cs.latest_network.control_params)
    assert_trace(trace, f"controlnet_{kdiff}_{with_regions}_{tensor_cpu}")


def test_stablesr_tile_caches_like_the_reference(monkeypatch):
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    with stub_webui(monkeypatch):
        _oracle_scatter(monkeypatch)
        d = _delegate(MultiDiffusion, ref_shim.make_kdiff_sampler(lambda x, s, cond=None: x), {i: r for i, r in enumerate(ROWS)}, True)
        trace = _stablesr_trace(d, _latent())
    assert d.enable_stablesr
    assert_trace(trace, "stablesr")


def test_scaled_grid_is_the_tile_plan_times_opt_f():
    from multidiffusion_upscaler_for_automatic1111_b200 import engine
    g = engine.make_grid(W, H, 16, 16, 8, 4)
    s = engine.scaled_grid(g, 8)
    assert (s.H, s.W, s.tile_h, s.tile_w, s.rows, s.cols, s.num_tiles, s.tile_bs) == (H * 8, W * 8, 128, 128, g.rows, g.cols, g.num_tiles, g.tile_bs)
    assert (engine.grid_bboxes_xywh(s) == engine.grid_bboxes_xywh(g) * 8).all()
