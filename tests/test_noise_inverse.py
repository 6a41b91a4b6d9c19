"""Tiled noise inversion (SURVEY.md section 8(f)-3): `init_noise_inverse` replaces the sampler's `sample_img2img`; the
Euler inversion loop runs the tiled denoiser (`get_noise`), the result is mixed with fresh noise under the retouch mask.

Our delegate runs on CPU under the stub WebUI of oracle/ref_shim.py, with the device kernels swapped for the oracle's
scatter / blend (pinned by tests/test_gpu_diffusion.py); its outputs must be identical to those of the UNMODIFIED
reference under the same stub (`reference_traces` below, stored in tests/golden/reference_traces.npz).
"""
import types

import numpy as np
import pytest
import torch

from helpers import assert_trace, digest, reference_trace, stub_webui
from oracle import blend

W, H = 64, 48
ROWS = [(True, 0.1, 0.2, 0.5, 0.4, "a cat", "", "Background", 0.2, -1),
        (True, 0.4, 0.3, 0.45, 0.6, "a dog", "ugly", "Foreground", 0.3, 5)]


class _DNW:
    """CompVisDenoiser look-alike: the three calls find_noise_for_image_sigma_adjustment makes."""

    def get_sigmas(self, n):
        return torch.cat([torch.linspace(14.0, 0.5, n), torch.zeros(1)])

    def get_scalings(self, sigma):
        return -sigma, 1 / (sigma ** 2 + 1) ** 0.5

    def sigma_to_t(self, sigma):
        return sigma * 7 + 1


def _image():
    from PIL import Image
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, size=(H * 8, W * 8, 3)).astype(np.uint8)
    a[: H * 4] = (a[: H * 4] // 64) * 64          # a flat half and a busy half
    return Image.fromarray(a)


def _job(ref, cls, settings, draw_background, with_regions, cache_type):
    """(delegate, sampler, p, cache) ready for sampler.sample_img2img(...)."""
    sd_model = types.SimpleNamespace(sd_model_hash="abc", get_learned_conditioning=lambda prompts: torch.full((len(prompts), 77, 8), 0.25))
    g = torch.Generator().manual_seed(5)
    p = types.SimpleNamespace(width=W * 8, height=H * 8, sampler_name="Euler", disable_extra_networks=True, batch_size=1, steps=6,
                              styles=None, all_prompts=["a photo"], all_negative_prompts=["blurry"], sd_model=sd_model,
                              init_latent=torch.randn(1, 4, H, W, generator=g), image_conditioning=torch.zeros(1, 5, 1, 1),
                              init_images=[_image()], show_tile_progress=False)

    class _Sampler(ref.KDiffusionSampler):
        pass
    sampler = _Sampler()
    sampler.model_wrap = _DNW()
    sampler.model_wrap_cfg = types.SimpleNamespace(inner_model=types.SimpleNamespace(forward=None), image_cfg_scale=None, step=0)
    sampler.get_sigmas = lambda p_, steps: torch.linspace(9.0, 0.0, steps + 1)
    sampler.sample_img2img = lambda p_, x, noise, c, uc, steps=None, image_conditioning=None: ("sampled", x, noise, steps)

    cache = {"v": None, "sets": 0}

    def get_cache():
        return cache["v"]

    def set_cache(x0, xt, prompts):
        cache["sets"] += 1
        cache["v"] = cache_type("abc", x0, xt, 4, 1.5, prompts)

    d = cls(p, sampler)
    d.init_grid_bbox(16, 16, 8, 4)
    if with_regions:
        d.init_custom_bbox(settings, draw_background, False)
    d.init_noise_inverse(4, 1.5, get_cache, set_cache, 1.0, 8)
    d.init_done()
    if getattr(d, "pbar", None) is not None:
        d.pbar.disable = True
    return d, sampler, p, cache


def _oracle_engine(monkeypatch):
    from multidiffusion_upscaler_for_automatic1111_b200 import engine
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

    from helpers import region_composite_reference
    monkeypatch.setattr(engine, "region_composite", region_composite_reference)
    monkeypatch.setattr(engine, "scatter_tiles", scatter_tiles)
    monkeypatch.setattr(engine, "blend_multidiffusion", blend_multidiffusion)
    monkeypatch.setattr(abstractdiffusion.AbstractDiffusion, "_check_input", lambda self, x: x.contiguous())


MODES = ["grid", "grid+regions", "regions_only"]


def _invert(webui, cls, settings, cache_type, mode):
    """Two img2img starts of the same job, the second one served from the cache: digests of the inverted latent and of
    both combined noises, and the step count handed to the sampler."""
    # region prompts at a noise-inversion step go through the (stand-in) prompt parser: [tokens] -> unsqueeze -> apply_model
    webui.shared.sd_model.apply_model = lambda x, t, cond=None: x * 0.5 + t.view(-1, 1, 1, 1) * 1e-3 + cond["c_crossattn"][0].mean() * 0.1
    if hasattr(webui.shared.sd_model, "apply_model_original_md"):
        del webui.shared.sd_model.apply_model_original_md
    webui.shared.state.sampling_step = 0
    with_regions, bg = mode != "grid", mode != "regions_only"
    noise = torch.randn(1, 4, H, W, generator=torch.Generator().manual_seed(9))
    x = torch.zeros(1, 4, H, W)
    d, sampler, p, cache = _job(webui, cls, settings, bg, with_regions, cache_type)
    assert sampler.sample_img2img.__func__ is not None          # replaced by a bound method of the sampler
    first = sampler.sample_img2img(p, x, noise, None, None)
    assert cache["sets"] == 1
    second = sampler.sample_img2img(p, x, noise, None, None)     # cache hit: no second inversion
    assert cache["sets"] == 1
    assert first[0] == second[0] == "sampled"
    assert torch.isfinite(first[2]).all() and not torch.equal(first[2], noise)
    return [digest(cache["v"].xt), digest(first[2]), digest(second[2])], str(first[3])


def reference_traces(ref):
    """The reference's side of the test below (oracle/make_reference_traces.py)."""
    out = {}
    for mode in MODES:
        out[f"noise_inverse_{mode}"], out[f"noise_inverse_{mode}_steps"] = _invert(
            ref, ref.multidiffusion.MultiDiffusion, {i: ref.utils.BBoxSettings(*r) for i, r in enumerate(ROWS)}, ref.utils.NoiseInverseCache, mode)
    return out


@pytest.mark.parametrize("mode", MODES)
def test_noise_inversion_like_the_reference(monkeypatch, mode):
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    from multidiffusion_upscaler_for_automatic1111_b200.tile_utils import utils
    with stub_webui(monkeypatch) as webui:
        _oracle_engine(monkeypatch)
        trace, steps = _invert(webui, MultiDiffusion, {i: r for i, r in enumerate(ROWS)}, utils.NoiseInverseCache, mode)
    assert steps == str(reference_trace(f"noise_inverse_{mode}_steps"))
    assert_trace(trace, f"noise_inverse_{mode}")
