"""The oracle against the unmodified reference: one hooked denoiser step and the tile scatter, compared with what the
reference computed on the same inputs (`reference_traces` below, stored in tests/golden/reference_traces.npz)."""
import numpy as np
import pytest
import torch

from helpers import DTYPES, assert_trace, digest, reference_trace
from oracle import blend, synth, tiling

N, C, W, H, TW, TH, OV, BS = 2, 4, 88, 56, 32, 24, 10, 3


def reference_traces(ref):
    """The reference's side of the tests below (oracle/make_reference_traces.py)."""
    from oracle.make_golden import run_reference_step
    out = {}
    for method in ("md", "mod"):
        for dn in DTYPES:
            d, want = run_reference_step(ref, method, synth.latent(11, (N, C, H, W), DTYPES[dn]), W, H, TW, TH, OV, BS)
            out[f"oracle_step_{method}_{dn}"] = [digest(want)]
        out[f"oracle_step_{method}_bboxes"] = np.array([(b.x, b.y, b.w, b.h) for bb in d.batched_bboxes for b in bb], np.int32)
    x = synth.latent(5, (2, 4, 64, 80), torch.float16)
    bbs, _ = ref.utils.split_bboxes(80, 64, 24, 16, 6, 1.0)
    out["scatter_bboxes"] = np.array([(b.x, b.y, b.w, b.h) for b in bbs], np.int32)
    out["scatter_cat"] = [digest(torch.cat([x[b.slicer] for b in bbs], dim=0))]
    return out


@pytest.mark.parametrize("method", ["md", "mod"])
@pytest.mark.parametrize("dn", list(DTYPES))
def test_step_matches_reference(method, dn):
    x = synth.latent(11, (N, C, H, W), DTYPES[dn])
    plan = tiling.GridPlan(W, H, TW, TH, OV, BS, method == "mod")
    assert plan.bboxes == [tuple(int(v) for v in b) for b in reference_trace(f"oracle_step_{method}_bboxes")]
    den = lambda t, bb: synth.fake_denoise(t, bb, N)
    if method == "md":
        got = blend.multidiffusion_step(x, plan.batched_bboxes, plan.weights, den)
    else:
        got = blend.mixture_step(x, plan.batched_bboxes, plan.tile_weights, plan.rescale_factor, den)
    assert_trace([digest(got)], f"oracle_step_{method}_{dn}")


def test_scatter_matches_reference_cat():
    x = synth.latent(5, (2, 4, 64, 80), torch.float16)
    bbs = [tuple(int(v) for v in b) for b in reference_trace("scatter_bboxes")]
    assert_trace([digest(blend.scatter_tiles(x, bbs))], "scatter_cat")
