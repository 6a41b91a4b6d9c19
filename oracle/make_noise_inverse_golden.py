"""TEST INFRASTRUCTURE -- fixture of tiled noise inversion from the UNMODIFIED reference.

Runs the reference's `sample_img2img` replacement (tile_methods/abstractdiffusion.py:604-742 + multidiffusion.py:220-243)
on CPU under oracle/ref_shim.py for the job defined in tests/noise_inverse_job.py and writes tests/golden/noise_inverse.npz
(inverted latent, combined noise, per mode).  The gpu test replays the same job on our delegate with the real kernels.
Usage: TD_REFERENCE_ROOT=<checkout of the original extension> python -m oracle.make_noise_inverse_golden
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    from oracle import ref_shim
    import noise_inverse_job as job
    if not ref_shim.available():
        sys.exit("reference tree not found: set TD_REFERENCE_ROOT to a checkout of the original extension")
    ref = ref_shim.load()
    out = {}
    for mode in job.MODES:
        ref.shared.state.sampling_step = 0
        ref.shared.sd_model.apply_model = job.fake_apply_model
        if hasattr(ref.shared.sd_model, "apply_model_original_md"):
            del ref.shared.sd_model.apply_model_original_md
        with_regions, bg = mode != "grid", mode != "regions_only"
        settings = {i: ref.utils.BBoxSettings(*r) for i, r in enumerate(job.ROWS)}
        d, sampler, p, cache = job.make_job(ref.multidiffusion.MultiDiffusion, settings, bg, with_regions, ref.KDiffusionSampler,
                                            ref.utils.NoiseInverseCache, torch.device("cpu"))
        res = sampler.sample_img2img(p, job.x0(), job.noise(), None, None)
        out[f"{mode}_xt"] = cache["v"].xt.numpy()
        out[f"{mode}_noise"] = res[2].numpy()
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "noise_inverse.npz"), **out)
    print("wrote tests/golden/noise_inverse.npz", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
