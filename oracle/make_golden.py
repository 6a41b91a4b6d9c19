"""TEST INFRASTRUCTURE -- generate tests/golden/*.npz FROM THE UNMODIFIED REFERENCE.

Needs a checkout of the original extension:

    TD_REFERENCE_ROOT=<checkout of the original extension> python -m oracle.make_golden

Every array below is an output of the reference's own code
(tile_utils/utils.py, tile_methods/{multidiffusion,mixtureofdiffusers}.py,
scripts/tilevae.py) executed under the stub host of `oracle/ref_shim.py`, on the
platform-stable synthetic inputs of `oracle/synth.py`.  The fixtures pin the
oracle (tests/test_oracle_golden.py) and, through it and directly, the CUDA path.
"""
from __future__ import annotations

import hashlib
import itertools
import os
import sys

import numpy as np
import torch

from . import ref_shim, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

BBOX_SWEEP = [c for c in itertools.product([13, 64, 100, 128, 160, 512], [16, 64, 77, 128, 512],
                                           [8, 16, 96, 128], [8, 24, 96, 128], [0, 4, 8, 16, 48, 64])]

GRID_CASES = [  # (W, H, tile_w, tile_h, overlap, tile_bs)  latent units
    (64, 64, 16, 16, 4, 4), (72, 72, 24, 16, 6, 3), (128, 128, 96, 96, 4, 4), (128, 128, 96, 96, 48, 4),
    (100, 77, 32, 24, 8, 5), (160, 64, 96, 96, 48, 2), (64, 160, 200, 48, 16, 1), (57, 43, 16, 16, 12, 8),
    (512, 512, 96, 96, 48, 4), (512, 512, 96, 96, 8, 4), (1024, 1024, 96, 96, 4, 8),
]

BLEND_CASES = [  # (name, N, C, W, H, tile_w, tile_h, overlap, tile_bs)
    ("a", 2, 4, 72, 72, 24, 16, 6, 3),
    ("b", 2, 4, 64, 48, 16, 16, 8, 4),
    ("c", 1, 4, 57, 43, 16, 16, 12, 8),     # odd canvas: generic (non-vector) kernels
    ("d", 3, 4, 96, 64, 40, 24, 4, 2),
    ("e", 2, 4, 128, 128, 96, 96, 48, 4),   # the UI default tile at a small canvas
]

HASH_CASES = [  # full-size configs, only a sha256 of the output bytes is stored
    ("cfg2_ov48", 2, 4, 512, 512, 96, 96, 48, 4),
    ("cfg2_ov8", 2, 4, 512, 512, 96, 96, 8, 4),
    ("cfg1", 2, 4, 1024, 1024, 96, 96, 4, 8),
]

DTYPES = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}

VAE_SUBSAMPLE = 3
VAE_CASES = [  # name, is_decoder, fast_mode, color_fix, H, W, tile_size
    ("dec_slow", True, False, False, 40, 52, 16),
    ("dec_fast", True, True, False, 40, 52, 16),
    ("enc_slow", False, False, False, 200, 264, 64),
    ("enc_fast", False, True, False, 200, 264, 64),
    ("enc_fast_colorfix", False, True, True, 200, 264, 64),
    ("dec_tiny_bypass", True, True, False, 20, 30, 16),
]


DEMO_CASES = [("f32_mixture", "f32", True), ("f32_plain", "f32", False), ("f16_mixture", "f16", True), ("f16_plain", "f16", False)]
DEMO_CFG = dict(N=2, C=4, H=48, W=64, scale=2, window=24, overlap=12, tile_bs=4, tile_bs_g=2, sig=0.6, cs1=3.0, cs2=1.0, cs3=1.0,
                current_step=3, t_enc=14)


# region prompt control: rows of the UI (enable, x, y, w, h, prompt, neg_prompt, blend_mode, feather_ratio, seed)
_BG, _FG = "Background", "Foreground"
REGION_GRID = dict(N=2, C=4, W=64, H=48, tw=16, th=16, ov=8, bs=4)
REGION_CASES = [  # name, draw_background, rows
    ("bg_fg", True, [(True, 0.1, 0.2, 0.5, 0.4, "a cat", "", _BG, 0.2, -1),
                     (False, 0.0, 0.0, 0.3, 0.3, "off", "", _BG, 0.2, -1),
                     (True, 0.4, 0.3, 0.45, 0.6, "a dog", "ugly", _FG, 0.3, 5),
                     (True, 1.2, 0.3, 0.2, 0.2, "outside", "", _FG, 0.3, 5),
                     (True, 0.55, 0.05, 0.6, 0.7, "a bird", "", _FG, 0.8, 7)]),
    ("no_background", False, [(True, 0.0, 0.0, 0.7, 0.8, "left", "", _BG, 0.2, -1),
                              (True, 0.3, 0.25, 0.7, 0.75, "right", "", _BG, 0.2, -1),
                              (True, 0.25, 0.3, 0.4, 0.4, "middle", "", _FG, 1.0, 3)]),
    ("fg_only", True, [(True, 0.2, 0.2, 0.33, 0.5, "one", "", _FG, 0.5, 1),
                       (True, 0.3, 0.4, 0.5, 0.5, "two", "", _FG, 0.0, 2)]),
    ("bg_only", True, [(True, 0.05, 0.1, 0.9, 0.3, "strip", "", _BG, 0.2, -1),
                       (True, 0.5, 0.0, 0.5, 1.0, "half", "", _BG, 0.2, -1)]),
]
REGION_DTYPES = ("f16", "f32")


def run_reference_region_step(ref, method: str, x: torch.Tensor, draw_background: bool, rows):
    """One step of the reference WITH custom bboxes; grid UNet = synth.fake_denoise, region UNet = synth.fake_region_denoise."""
    c = REGION_GRID
    N = x.shape[0]
    p = ref_shim.make_p(c["W"] * 8, c["H"] * 8)
    cond = {"c_crossattn": [torch.zeros(N, 2, 4)], "c_concat": [torch.zeros(N, 5, 1, 1)]}
    state = {}

    def unet(x_tile, sigma, cond=None):
        return synth.fake_denoise(x_tile, state["bboxes"], N)

    sampler = ref_shim.make_kdiff_sampler(unet)
    cls = ref.multidiffusion.MultiDiffusion if method == "md" else ref.mixtureofdiffusers.MixtureOfDiffusers
    d = cls(p, sampler)
    d.init_grid_bbox(c["tw"], c["th"], c["ov"], c["bs"])
    settings = {i: ref.utils.BBoxSettings(*row) for i, row in enumerate(rows)}
    d.init_custom_bbox(settings, draw_background, False)
    d.init_done()
    d.pbar.disable = True

    def custom_func(x_tile, bbox_id, bbox):
        return synth.fake_region_denoise(x_tile, bbox_id)

    if method == "md":
        def repeat_func(x_tile, bboxes):
            state["bboxes"] = bboxes
            return unet(x_tile, None)
        out = d.sample_one_step(x, None, repeat_func, custom_func)
    else:
        batches = iter(d.batched_bboxes)

        def apply_model(x_tile, t, c_):
            state["bboxes"] = next(batches)
            return unet(x_tile, None)
        ref.shared.sd_model.apply_model = apply_model
        d.custom_apply_model = lambda x_tile, t, c_, bbox_id, bbox: custom_func(x_tile, bbox_id, bbox)   # instance attribute
        d.hook()
        try:
            out = ref.shared.sd_model.apply_model(x, torch.ones(N), cond)
        finally:
            d.unhook()
    return d, out.clone()


def gen_region(ref):
    """9. region prompt control (custom bboxes): feather masks, rectangles, weights and one full step ------------"""
    c = REGION_GRID
    out = {}
    masks = [(10, 8, 0.5), (29, 29, 0.3), (39, 34, 0.8), (26, 20, 1.0), (33, 24, 0.0), (7, 5, 0.2), (64, 48, 0.2)]
    for (w, h, r) in masks:
        out[f"mask_{w}x{h}_{r}"] = ref.utils.feather_mask(w, h, r).numpy()
    out["mask_cases"] = np.array(masks, np.float64)
    for name, bg, rows in REGION_CASES:
        for method in ("md", "mod"):
            for dn in REGION_DTYPES:
                x = synth.latent(synth.case_seed("region_" + name, dn), (c["N"], c["C"], c["H"], c["W"]), DTYPES[dn])
                d, o = run_reference_region_step(ref, method, x, bg, rows)
                key = f"{name}_{method}_{dn}"
                out[key] = _bits(o)
                out[key + "_dtype"] = np.array(str(o.dtype))
            out[f"{name}_{method}_weights"] = d.weights[0, 0].numpy()
            out[f"{name}_rects"] = np.array([(b.x, b.y, b.w, b.h) for b in d.custom_bboxes], np.int32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "region_small.npz"), **out)


def gen_demofusion_jitter(ref):
    """10. DemoFusion with random jitter (demofusion.py:101-139, :204, :279-310): seeded windows, padded latent ------"""
    import torch.nn.functional as F
    out = {}
    for name, dn, mixture in DEMO_JITTER_CASES:
        d, x, cond = demofusion_reference_case(ref, DTYPES[dn], mixture, jitter_seed=DEMO_JITTER_SEED)
        jr = d.jitter_range
        y = d.sample_one_step(F.pad(x, (jr, jr, jr, jr), "constant", value=0), torch.ones(x.shape[0]), cond)
        out[name] = _bits(y)
        out[name + "_dtype"] = np.array(str(y.dtype))
        out[name + "_local"] = np.array([(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb], np.int32)
        out[name + "_sizes"] = np.array([d.tile_bs, d.global_tile_bs, d.global_num_tiles, jr], np.int32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "demofusion_jitter.npz"), **out)


def demo_denoise(x_tile, *_a, **_k):
    """Deterministic stand-in for the UNet in the DemoFusion fixtures (exact: scale by 0.5)."""
    return (x_tile.float() * 0.5).to(x_tile.dtype)


DEMO_JITTER_SEED = 20240922
DEMO_JITTER_CASES = [("f32_mixture_jitter", "f32", True), ("f16_plain_jitter", "f16", False)]


def position_aware_denoise(delegate):
    """UNet stand-in for the jitter fixtures: local windows are scaled by their (jittered) position, global views by
    0.5.  The delegate hands the window list to `repeat_cond_dict` right before every UNet call; wrapping that
    (an instance attribute, the class is untouched) tells the stand-in which windows it is looking at."""
    state = {}
    orig = delegate.repeat_cond_dict

    def spy(cond_in, bboxes, mode):
        state["bboxes"], state["mode"] = bboxes, mode
        return orig(cond_in, bboxes, mode)
    delegate.repeat_cond_dict = spy

    def unet(xt, sigma, cond=None):
        if state["mode"] == 0:
            return synth.fake_denoise(xt, state["bboxes"], xt.shape[0] // len(state["bboxes"]))
        return demo_denoise(xt)
    return unet


def demofusion_reference_case(ref, dtype, mixture, jitter_seed=None):
    """The reference's DemoFusion delegate set up like tileglobal.py does, without a WebUI."""
    import random
    import types
    from . import demofusion as odf
    c = DEMO_CFG
    sys.modules['modules.sd_samplers_common'].setup_img2img_steps = lambda p, steps=None: (p.steps, p.t_enc)
    x = synth.latent(31, (c["N"], c["C"], c["H"], c["W"]), dtype)
    p = ref_shim.make_p(c["W"] * 8, c["H"] * 8)
    p.current_scale_num, p.mixture, p.gaussian_filter, p.random_jitter = c["scale"], mixture, True, jitter_seed is not None
    p.cosine_scale_1, p.cosine_scale_2, p.cosine_scale_3 = c["cs1"], c["cs2"], c["cs3"]
    p.current_step, p.steps, p.t_enc = c["current_step"], 20, c["t_enc"]
    p.sd_model = types.SimpleNamespace(apply_model=lambda *a, **k: None)
    sampler = ref_shim.make_kdiff_sampler(lambda xt, sigma, cond=None: demo_denoise(xt))
    d = ref.demofusion.DemoFusion(p, sampler)
    d.window_size, d.sig = c["window"], c["sig"]
    if jitter_seed is not None:
        random.seed(jitter_seed)       # the reference draws from Python's global `random` (demofusion.py:122-132)
    d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
    d.sampler_forward = position_aware_denoise(d) if jitter_seed is not None else (lambda xt, sigma, cond=None: demo_denoise(xt))
    d.repeat_3 = False
    d.cosine_factor = odf.cosine_factor(p.current_step, p.t_enc)
    cond = {"c_crossattn": [torch.zeros(c["N"], 77, 8)], "c_concat": [torch.zeros(c["N"], 5, 1, 1)]}
    return d, x, cond


def vae_case_inputs(is_decoder: bool, H: int, W: int):
    """Tiny ldm-shaped net (4 resolutions, like SD) + platform-stable input for the VAE fixtures."""
    from . import ldm_vae
    if is_decoder:
        net = ldm_vae.seeded_init(ldm_vae.Decoder(ch=32, ch_mult=(1, 1, 2, 2), num_res_blocks=1), 1)
        z = synth.latent(5, (1, 4, H, W), torch.float32)
    else:
        net = ldm_vae.seeded_init(ldm_vae.Encoder(ch=32, ch_mult=(1, 1, 2, 2), num_res_blocks=1), 2)
        z = synth.latent(6, (1, 3, H, W), torch.float32)
    net.eval()
    net.original_forward = net.forward
    return net, z


def _bits(t: torch.Tensor) -> np.ndarray:
    t = t.contiguous()
    if t.dtype == torch.float32:
        return t.numpy().view(np.uint32)
    return t.view(torch.int16).numpy().view(np.uint16)


def sha(t: torch.Tensor) -> str:
    return hashlib.sha256(_bits(t).tobytes()).hexdigest()


def run_reference_step(ref, method: str, x: torch.Tensor, W, H, tw, th, ov, bs):
    """One hooked denoiser call of the reference on latent x; fake UNet = synth.fake_denoise."""
    N = x.shape[0]
    p = ref_shim.make_p(W * 8, H * 8)
    cond = {"c_crossattn": [torch.zeros(N, 2, 4)], "c_concat": [torch.zeros(N, 5, 1, 1)]}
    state = {}

    def unet(x_tile, sigma, cond=None):
        return synth.fake_denoise(x_tile, state["bboxes"], N)

    sampler = ref_shim.make_kdiff_sampler(unet)
    cls = ref.multidiffusion.MultiDiffusion if method == "md" else ref.mixtureofdiffusers.MixtureOfDiffusers
    d = cls(p, sampler)
    d.init_grid_bbox(tw, th, ov, bs)
    d.init_done()
    d.pbar.disable = True
    # the reference hands `bboxes` to repeat_func only; capture them for the fake UNet
    if method == "md":
        def repeat_func(x_tile, bboxes):
            state["bboxes"] = bboxes
            return unet(x_tile, None)
        out = d.sample_one_step(x, None, repeat_func, None)
    else:
        batches = iter(d.batched_bboxes)

        def apply_model(x_tile, t, c):
            state["bboxes"] = next(batches)
            return unet(x_tile, None)
        ref.shared.sd_model.apply_model = apply_model
        d.hook()
        try:
            out = ref.shared.sd_model.apply_model(x, torch.ones(N), cond)
        finally:
            d.unhook()
        out = out.clone()
    return d, out


def main():
    if not ref_shim.available():
        sys.exit("reference tree not found: set TD_REFERENCE_ROOT to a checkout of the original extension")
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    ref = ref_shim.load()
    torch.set_num_threads(1)
    if "region" in sys.argv[1:]:      # regenerate only region_small.npz
        gen_region(ref)
        return
    if "jitter" in sys.argv[1:]:      # regenerate only demofusion_jitter.npz
        gen_demofusion_jitter(ref)
        return

    # 1. split_bboxes sweep (utils.py:160-177) ------------------------------------
    cases, counts, flat = [], [], []
    for (w, h, tw, th, ov) in BBOX_SWEEP:
        tw_, th_ = min(tw, w), min(th, h)
        ov_ = max(0, min(ov, min(tw, th) - 4))
        if tw_ <= ov_ or th_ <= ov_:
            continue
        bbs, _ = ref.utils.split_bboxes(w, h, tw_, th_, ov_, 1.0)
        cases.append((w, h, tw_, th_, ov_))
        counts.append(len(bbs))
        flat += [(b.x, b.y, b.w, b.h) for b in bbs]
    splitable = [(w * 8, h * 8, tw, th, ov, int(ref.utils.splitable(w * 8, h * 8, tw, th, ov)))
                 for (w, h, tw, th, ov) in BBOX_SWEEP if tw > 4 and th > 4]
    np.savez_compressed(os.path.join(GOLDEN_DIR, "bboxes.npz"), cases=np.array(cases, np.int32),
                        counts=np.array(counts, np.int32), xywh=np.array(flat, np.int32),
                        splitable=np.array(splitable, np.int32))

    # 2. gaussian weights (utils.py:180-194) --------------------------------------
    g = {f"g_{tw}x{th}": ref.utils.gaussian_weights(tw, th).numpy() for (tw, th) in
         [(96, 96), (64, 48), (128, 128), (16, 24), (24, 16), (33, 17), (192, 192)]}
    np.savez_compressed(os.path.join(GOLDEN_DIR, "gaussian.npz"), **g)

    # 3. init_grid_bbox state (abstractdiffusion.py:172-186) + MoD rescale -------
    out = {}
    for i, (W, H, tw, th, ov, bs) in enumerate(GRID_CASES):
        for method in ("md", "mod"):
            p = ref_shim.make_p(W * 8, H * 8)
            s = ref_shim.make_kdiff_sampler(lambda *a, **k: None)
            cls = ref.multidiffusion.MultiDiffusion if method == "md" else ref.mixtureofdiffusers.MixtureOfDiffusers
            d = cls(p, s)
            d.init_grid_bbox(tw, th, ov, bs)
            d.init_done()
            d.pbar.disable = True
            key = f"{i}_{method}"
            out[key + "_scalars"] = np.array([d.tile_w, d.tile_h, d.num_tiles, d.num_batches, d.tile_bs], np.int32)
            out[key + "_bboxes"] = np.array([(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb], np.int32)
            out[key + "_batch_sizes"] = np.array([len(bb) for bb in d.batched_bboxes], np.int32)
            if W * H <= 128 * 128:
                out[key + "_weights"] = d.weights[0, 0].numpy()
                if method == "mod":
                    out[key + "_rescale"] = d.rescale_factor[0, 0].numpy()
            else:
                out[key + "_weights_sha"] = np.frombuffer(sha(d.weights).encode(), np.uint8)
    out["cases"] = np.array(GRID_CASES, np.int32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "grid_plans.npz"), **out)

    # 4. one sampler step, small canvases, full outputs --------------------------
    out = {"cases": np.array([c[1:] for c in BLEND_CASES], np.int32), "names": np.array([c[0] for c in BLEND_CASES])}
    for (name, N, C, W, H, tw, th, ov, bs) in BLEND_CASES:
        for dn, dt in DTYPES.items():
            x = synth.latent(synth.case_seed(name, dn), (N, C, H, W), dt)
            for method in ("md", "mod"):
                _, o = run_reference_step(ref, method, x, W, H, tw, th, ov, bs)
                out[f"{name}_{dn}_{method}"] = _bits(o)
                out[f"{name}_{dn}_{method}_dtype"] = np.array(str(o.dtype))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "blend_small.npz"), **out)

    # 5. full-size configs, hash only ---------------------------------------------
    out = {"cases": np.array([c[1:] for c in HASH_CASES], np.int32), "names": np.array([c[0] for c in HASH_CASES])}
    for (name, N, C, W, H, tw, th, ov, bs) in HASH_CASES:
        for dn, dt in DTYPES.items():
            if name == "cfg1" and dn != "f16":
                continue
            x = synth.latent(synth.case_seed(name, dn), (N, C, H, W), dt)
            for method in ("md", "mod"):
                _, o = run_reference_step(ref, method, x, W, H, tw, th, ov, bs)
                out[f"{name}_{dn}_{method}"] = np.array(sha(o))
                out[f"{name}_{dn}_{method}_dtype"] = np.array(str(o.dtype))
    np.savez_compressed(os.path.join(GOLDEN_DIR, "blend_hashes.npz"), **out)

    # 6. tiled VAE geometry (scripts/tilevae.py:390-462), exact ------------------------------
    hook_cls = ref.tilevae.VAEHook
    geo = {}
    cases = []
    for (h, w, ts, dec) in itertools.product([40, 97, 128, 200, 333, 1024], [52, 64, 300, 1024], [16, 64, 96, 512, 1536], [1, 0]):
        hk = hook_cls(None, ts, bool(dec), True, True, False)
        ib, ob = hk.split_tiles(h, w)
        geo[f"in_{len(cases)}"] = np.array(ib, np.int32)
        geo[f"out_{len(cases)}"] = np.array(ob, np.int32)
        cases.append((h, w, ts, dec))
    geo["cases"] = np.array(cases, np.int32)
    geo["cfg4_dec"] = np.array(hook_cls(None, 96, True, True, True, False).split_tiles(1024, 1024)[0], np.int32)
    geo["cfg4_enc"] = np.array(hook_cls(None, 1536, False, True, True, False).split_tiles(8192, 8192)[0], np.int32)
    best = [(lo, up, hook_cls(None, 64, True, True, True, False).get_best_tile_size(lo, up)) for lo in range(1, 200, 7) for up in (lo, lo + 5, lo + 31, 256)]
    geo["best_tile"] = np.array(best, np.int32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "vae_geometry.npz"), **geo)

    # 7. tiled VAE forward of the reference on a tiny ldm-shaped net (sub-sampled outputs) --
    from . import ldm_vae
    out = {}
    for name, is_dec, fast, cf, H, W, tile in VAE_CASES:
        net, z = vae_case_inputs(is_dec, H, W)
        hook = hook_cls(net, tile, is_dec, fast_decoder=fast, fast_encoder=fast, color_fix=cf)
        with torch.no_grad():
            y = hook(z)
        out[name] = y[:, :, ::VAE_SUBSAMPLE, ::VAE_SUBSAMPLE].contiguous().numpy()
        out[name + "_shape"] = np.array(y.shape, np.int32)
        out[name + "_absmax"] = np.array(float(y.abs().max()), np.float32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "vae_small.npz"), **out)

    # 8. DemoFusion sample_one_step of the reference (tile_methods/demofusion.py:219-324), jitter off -------
    out = {}
    for name, dn, mixture in DEMO_CASES:
        d, x, cond = demofusion_reference_case(ref, DTYPES[dn], mixture)
        y = d.sample_one_step(x, torch.ones(x.shape[0]), cond)
        out[name] = _bits(y)
        out[name + "_dtype"] = np.array(str(y.dtype))
        out[name + "_local"] = np.array([(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb], np.int32)
        out[name + "_tile_bs"] = np.array([d.tile_bs, d.global_tile_bs, d.global_num_tiles], np.int32)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "demofusion_small.npz"), **out)

    gen_region(ref)
    gen_demofusion_jitter(ref)

    for f in sorted(os.listdir(GOLDEN_DIR)):
        print(f, os.path.getsize(os.path.join(GOLDEN_DIR, f)))


if __name__ == "__main__":
    main()
