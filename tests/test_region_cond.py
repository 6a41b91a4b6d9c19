"""Region prompt control, conditioning side: `kdiff_custom_forward` / `ddim_custom_forward` must hand the UNet exactly
the rows, sigmas and cond tensors the reference hands it, for every way the k-diffusion CFG wrapper slices a batch.

Our delegate runs under the stub WebUI of oracle/ref_shim.py (with its deterministic stand-in for the WebUI prompt
parser); the UNet calls it makes must equal those the UNMODIFIED reference made under the same stub (`reference_traces`
below, stored in tests/golden/reference_traces.npz).
"""
import itertools
import types

import pytest
import torch

from helpers import assert_trace, digest, reference_trace, stub_webui

W, H = 64, 48
ROWS = [(True, 0.1, 0.2, 0.5, 0.4, "a cat", "", "Background", 0.2, -1),
        (True, 0.4, 0.3, 0.45, 0.6, "a very long region prompt that spills into a second chunk of tokens", "ugly", "Foreground", 0.3, 5)]
SHORT, LONG = "a photo", "a photo of something described with so many words that the encoder needs two chunks"


@pytest.fixture()
def hosts(monkeypatch):
    from multidiffusion_upscaler_for_automatic1111_b200 import host
    with stub_webui(monkeypatch) as ref:
        yield ref, host


def _p(prompt, neg, batch_size):
    return types.SimpleNamespace(width=W * 8, height=H * 8, sampler_name="Euler a", disable_extra_networks=True,
                                 batch_size=batch_size, steps=20, styles=None,
                                 all_prompts=[f"{prompt} {i}" for i in range(batch_size)],
                                 all_negative_prompts=[f"{neg} {i}" for i in range(batch_size)])


def _delegate(cls, settings, prompt, neg, batch_size, edit):
    """A delegate of `cls` with the regions of ROWS, on CPU."""
    from oracle import ref_shim
    sampler = ref_shim.make_kdiff_sampler(lambda x, s, cond=None: x)
    d = cls(_p(prompt, neg, batch_size), sampler)
    d.init_grid_bbox(16, 16, 8, 4)
    d.init_custom_bbox(settings, True, False)
    d.init_done()
    if getattr(d, "pbar", None) is not None:
        d.pbar.disable = True
    d.is_edit_model = edit
    return d


def _ours(prompt, neg, batch_size, edit):
    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    return _delegate(MultiDiffusion, {i: r for i, r in enumerate(ROWS)}, prompt, neg, batch_size, edit)


def _reference(ref, prompt, neg, batch_size, edit):
    return _delegate(ref.multidiffusion.MultiDiffusion, {i: ref.utils.BBoxSettings(*r) for i, r in enumerate(ROWS)}, prompt, neg, batch_size, edit)


class _Recorder:
    def __init__(self):
        self.calls = []

    def __call__(self, x, sigma, cond=None):
        tc = cond["c_crossattn"][0]
        ic = cond["c_concat"][0]
        self.calls += [digest(x), digest(sigma), digest(tc), digest(ic)]
        return x * 2 + tc.mean() + sigma.view(-1, 1, 1, 1)


def _drive(d, chunks, steps=(0, 1)):
    """Feed every region the virtual batch in `chunks` (row counts), for two sampler steps: digests of the UNet calls,
    then of the outputs."""
    rec = _Recorder()
    outs = []
    rows = sum(chunks)
    for step in steps:
        d.sampler.model_wrap_cfg.step = step
        for bbox_id, bbox in enumerate(d.custom_bboxes):
            x_full = torch.arange(rows * 4 * bbox.h * bbox.w, dtype=torch.float32).view(rows, 4, bbox.h, bbox.w) / 1000.0 + step
            sigma = torch.arange(rows, dtype=torch.float32) + 1
            cond = {"c_crossattn": [torch.zeros(rows, 77, 8)], "c_concat": [torch.full((rows, 5, 1, 1), 0.5)]}
            lo = 0
            for n in chunks:
                outs.append(digest(d.kdiff_custom_forward(x_full[lo:lo + n], sigma[lo:lo + n], cond, bbox_id, bbox, rec)))
                lo += n
    return rec.calls + outs


def _drive_ddim(d):
    """Digests of the UNet calls `ddim_custom_forward` makes at step 3, then of its outputs."""
    d.sampler.model_wrap_cfg.step = 3
    calls, outs = [], []

    def fwd(x, cond, ts, unconditional_conditioning=None):
        calls.extend(digest(t) for t in (x, ts, cond["c_crossattn"][0], unconditional_conditioning["c_crossattn"][0], cond["c_concat"][0]))
        return x + 1
    for bbox in d.custom_bboxes:
        x = torch.ones(1, 4, bbox.h, bbox.w)
        cond_in = {"c_crossattn": [torch.zeros(1, 77, 8)], "c_concat": [torch.arange(5 * H * W, dtype=torch.float32).view(1, 5, H, W)]}
        outs.append(digest(d.ddim_custom_forward(x, cond_in, bbox, torch.tensor([7]), fwd)))
    return calls + outs


SCENARIOS = []
for batch_size, (prompt, neg), edit, bcu in itertools.product([1, 2], [(SHORT, SHORT), (LONG, SHORT)], [False, True], [True, False]):
    rows = batch_size * (3 if edit else 2)
    splits = {(rows,), tuple([1] * rows), (batch_size,) * (rows // batch_size)}
    if rows >= 3:
        splits.add((rows - 1, 1))
        splits.add((1, rows - 1))
    for chunks in sorted(splits):
        if bcu and len(chunks) > 1:
            continue                      # with batch_cond_uncond the wrapper always sends the whole batch at once
        SCENARIOS.append((batch_size, prompt, neg, edit, bcu, chunks))
SCENARIO_IDS = [f"bs{s[0]}_{'long' if s[1] is LONG else 'short'}_{'edit' if s[3] else 'std'}_{'bcu' if s[4] else 'seq'}_{'-'.join(map(str, s[5]))}"
                for s in SCENARIOS]
DDIM_PROMPTS = [(SHORT, SHORT), (LONG, SHORT), (SHORT, LONG)]


def reference_traces(ref):
    """The reference's side of the tests below (oracle/make_reference_traces.py)."""
    out = {}
    keep = ref.shared.batch_cond_uncond
    for name, (batch_size, prompt, neg, edit, bcu, chunks) in zip(SCENARIO_IDS, SCENARIOS):
        ref.shared.batch_cond_uncond = bcu
        try:
            out[f"region_cond_kdiff_{name}"] = _drive(_reference(ref, prompt, neg, batch_size, edit), chunks)
        except Exception as e:       # slicings the reference itself cannot serve
            out[f"region_cond_kdiff_{name}_raises"] = type(e).__name__
    ref.shared.batch_cond_uncond = keep
    for i, (prompt, neg) in enumerate(DDIM_PROMPTS):
        out[f"region_cond_ddim_{i}"] = _drive_ddim(_reference(ref, prompt, neg, 1, False))
    return out


@pytest.mark.parametrize("name,sc", list(zip(SCENARIO_IDS, SCENARIOS)), ids=SCENARIO_IDS)
def test_kdiff_custom_forward_feeds_the_unet_like_the_reference(hosts, name, sc):
    ref, host = hosts
    batch_size, prompt, neg, edit, bcu, chunks = sc
    raised = reference_trace(f"region_cond_kdiff_{name}_raises")
    if raised is not None:           # slicings the reference itself cannot serve (it raises): nothing to compare
        pytest.skip(f"reference raises {raised} here")
    ref.shared.batch_cond_uncond = bcu
    assert_trace(_drive(_ours(prompt, neg, batch_size, edit), chunks), f"region_cond_kdiff_{name}")


@pytest.mark.parametrize("prompt,neg", DDIM_PROMPTS)
def test_ddim_custom_forward_like_the_reference(hosts, prompt, neg):
    assert_trace(_drive_ddim(_ours(prompt, neg, 1, False)), f"region_cond_ddim_{DDIM_PROMPTS.index((prompt, neg))}")
