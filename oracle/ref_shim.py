"""TEST INFRASTRUCTURE ONLY -- stub A1111 host so the UNMODIFIED reference imports.

The reference (the original extension, CC BY-NC-SA) is a WebUI extension whose
modules import `modules.*` (A1111), `ldm`, `k_diffusion` and `gradio` at import time
(tile_utils/utils.py:11-14, tile_utils/typing.py:6-29, scripts/tilevae.py:60-70,
tile_utils/attn.py:8-10).  None of those exist here.  `install()` injects empty
`types.ModuleType` stand-ins for exactly the names those import lines need (plus a
deterministic prompt parser); the CPU tests run our delegate under that stub host.
`load()` additionally puts the reference checkout named by $TD_REFERENCE_ROOT on
`sys.path` and returns the reference's own modules, so that the fixture generators
(`oracle/make_*.py`) can call the reference's real code.  No test needs the
reference: they compare with what those generators stored under tests/golden/.
No reference source is copied; this file contains only stubs.
"""
from __future__ import annotations

import contextlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("TD_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "tile_methods", "multidiffusion.py"))


class _State:
    """modules.shared.state look-alike (utils.py:13; polled at multidiffusion.py:152)."""
    interrupted = False
    sampling_step = 0
    sampling_steps = 1
    job_count = 0

    def nextjob(self):
        pass


class _Opts:
    pass


class _CmdOpts:
    md_max_regions = 8


_created = []


def _mod(name: str, **attrs) -> types.ModuleType:
    m = sys.modules.get(name)
    if m is None:
        m = types.ModuleType(name)
        sys.modules[name] = m
        _created.append(name)
        parent, _, child = name.rpartition(".")
        if parent:
            setattr(_mod(parent), child, m)
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


# --- deterministic stand-in for the WebUI's prompt parser (region prompt control tests) ---------------------------
# A "conditioning" is just the tuple of prompt strings; reconstructing it at a sampler step yields a tensor
# [len(prompts), 77 * chunks, 8] whose values depend on the prompt text and the step, chunks = 1 + len(prompt) // 40
# (so that long prompts have a different token count, like the real CLIP chunking).
FAKE_TOKEN_DIM = 8


def _fake_tokens(prompts, step):
    import hashlib

    import torch
    chunks = max(1 + len(p) // 40 for p in prompts)
    rows = []
    for p in prompts:
        h = int.from_bytes(hashlib.sha256(f"{p}|{step}".encode()).digest()[:4], "little")
        base = (h % 997) / 997.0
        rows.append(base + torch.arange(77 * chunks * FAKE_TOKEN_DIM, dtype=torch.float32).view(77 * chunks, FAKE_TOKEN_DIM) / 4096.0)
    return torch.stack(rows)


def fake_multicond(model, prompts, steps):
    return ("multicond", tuple(prompts), steps)


def fake_learned(model, prompts, steps):
    return ("learned", tuple(prompts), steps)


def fake_reconstruct_multicond(cond, step):
    return None, _fake_tokens(cond[1], step)


def fake_reconstruct_cond(cond, step):
    return _fake_tokens(cond[1], step)


_installed = False


def _host() -> types.SimpleNamespace:
    return types.SimpleNamespace(shared=sys.modules["modules.shared"], devices=sys.modules["modules.devices"],
                                 KDiffusionSampler=sys.modules["modules.sd_samplers_kdiffusion"].KDiffusionSampler,
                                 CompVisSampler=sys.modules["modules.sd_samplers_timesteps"].CompVisSampler)


def install(device: str = "cpu") -> types.SimpleNamespace:
    """Inject the stub host (needs no reference) and return its `shared`, `devices` and sampler classes.  Idempotent."""
    global _installed
    import torch

    if _installed:
        sys.modules["modules.devices"].device = torch.device(device)
        return _host()

    class KDiffusionSampler:  # isinstance() target, abstractdiffusion.py:77-79
        pass

    class CompVisSampler:
        pass

    class CompVisDenoiser:
        def forward(self, *a, **k):  # multidiffusion.py:53 asserts attribute exists
            raise NotImplementedError

    class CompVisVDenoiser(CompVisDenoiser):
        pass

    class LatentDiffusion:
        def apply_model(self, *a, **k):  # mixtureofdiffusers.py:62
            raise NotImplementedError

    class _Dummy:
        pass

    def test_for_nans(x, where):
        if torch.isnan(x).any():
            raise RuntimeError(f"NaN in {where}")

    @contextlib.contextmanager
    def autocast(*a, **k):
        yield

    dev = torch.device(device)
    _mod("modules")
    _mod("modules.devices", device=dev, cpu=torch.device("cpu"), autocast=autocast,
         torch_gc=lambda: None, test_for_nans=test_for_nans,
         get_optimal_device=lambda: dev, get_optimal_device_name=lambda: str(dev))
    sd_model = types.SimpleNamespace(cond_stage_key="txt", parameterization="eps",
                                     model=types.SimpleNamespace(conditioning_key="crossattn"))
    _mod("modules.shared", state=_State(), sd_model=sd_model, opts=_Opts(), cmd_opts=_CmdOpts(),
         batch_cond_uncond=True, State=_State)
    _mod("modules.shared_state", State=_State)
    _mod("modules.prompt_parser", MulticondLearnedConditioning=_Dummy, ScheduledPromptConditioning=_Dummy,
         get_multicond_learned_conditioning=fake_multicond, get_learned_conditioning=fake_learned,
         reconstruct_multicond_batch=fake_reconstruct_multicond, reconstruct_cond_batch=fake_reconstruct_cond)
    _mod("modules.extra_networks", ExtraNetworkParams=_Dummy, parse_prompts=lambda prompts: (list(prompts), {}),
         activate=lambda p, data: None, deactivate=lambda p, data: None)
    _mod("modules.sd_samplers_common", setup_img2img_steps=lambda p, steps=None: (steps if steps is not None else p.steps, p.steps - 1),
         store_latent=lambda x: None)
    _mod("modules.processing", opt_f=8, StableDiffusionProcessing=_Dummy,
         StableDiffusionProcessingImg2Img=_Dummy, Processed=_Dummy)
    _mod("modules.sd_samplers_kdiffusion", KDiffusionSampler=KDiffusionSampler, CFGDenoiser=_Dummy,
         CFGDenoiserKDiffusion=_Dummy)
    _mod("modules.sd_samplers_timesteps", CompVisSampler=CompVisSampler, CFGDenoiserTimesteps=_Dummy,
         CompVisTimestepsDenoiser=CompVisDenoiser, CompVisTimestepsVDenoiser=CompVisVDenoiser)
    _mod("modules.scripts", Script=_Dummy, AlwaysVisible=object())
    _mod("modules.ui", gr_show=lambda *a, **k: None)
    _mod("modules.sd_vae_approx", cheap_approximation=lambda x: x[:3])
    _mod("modules.sd_hijack", model_hijack=types.SimpleNamespace(optimization_method=None))
    _mod("modules.sd_hijack_optimizations", get_available_vram=lambda: 0,
         get_xformers_flash_attention_op=lambda *a: None, sub_quad_attention=None)
    _mod("gradio")
    _mod("gradio.components", Component=_Dummy)
    _mod("k_diffusion")
    _mod("k_diffusion.utils", append_dims=lambda x, target_dims: x[(...,) + (None,) * (target_dims - x.ndim)])
    _mod("k_diffusion.external", CompVisDenoiser=CompVisDenoiser, CompVisVDenoiser=CompVisVDenoiser)
    _mod("ldm")
    _mod("ldm.models")
    _mod("ldm.models.diffusion")
    _mod("ldm.models.diffusion.ddpm", LatentDiffusion=LatentDiffusion)
    _mod("ldm.modules")
    _mod("ldm.modules.diffusionmodules")
    _mod("ldm.modules.diffusionmodules.model", AttnBlock=_Dummy, MemoryEfficientAttnBlock=_Dummy)
    _installed = True
    return _host()


def uninstall() -> None:
    """Drop the stand-in modules `install()` created, so that code run afterwards sees no WebUI."""
    global _installed
    for name in reversed(_created):
        sys.modules.pop(name, None)
    _created.clear()
    _installed = False


def load(device: str = "cpu"):
    """Return the stub host of `install()` plus the reference's own (unmodified) modules."""
    if not available():
        raise RuntimeError("reference tree not found: set TD_REFERENCE_ROOT to a checkout of the original extension")
    ns = install(device)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib

    ns.utils = importlib.import_module("tile_utils.utils")
    ns.abstractdiffusion = importlib.import_module("tile_methods.abstractdiffusion")
    ns.multidiffusion = importlib.import_module("tile_methods.multidiffusion")
    ns.mixtureofdiffusers = importlib.import_module("tile_methods.mixtureofdiffusers")
    ns.demofusion = importlib.import_module("tile_methods.demofusion")
    ns.tilevae = importlib.import_module("scripts.tilevae")
    ns.attn = importlib.import_module("tile_utils.attn")
    return ns


def make_p(width: int, height: int, sampler_name: str = "Euler a"):
    """Minimal StableDiffusionProcessing stand-in (abstractdiffusion.py:6-33)."""
    return types.SimpleNamespace(width=width, height=height, sampler_name=sampler_name,
                                 disable_extra_networks=True, batch_size=1, steps=20, styles=None,
                                 all_prompts=["a photo"], all_negative_prompts=["blurry"])


def make_kdiff_sampler(inner_forward):
    """Fake k-diffusion sampler: `.model_wrap_cfg.inner_model.forward` is what
    MultiDiffusion.hook patches (multidiffusion.py:22-23)."""
    ref = install()

    class _Sampler(ref.KDiffusionSampler):
        pass

    s = _Sampler()
    inner = types.SimpleNamespace(forward=inner_forward)
    s.model_wrap_cfg = types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, step=0)
    return s
