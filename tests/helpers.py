"""Shared helpers for the parity tests (bit views, oracle plans)."""
import contextlib
import hashlib
import os

import numpy as np
import torch

DTYPES = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}
REFERENCE_TRACES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_traces.npz")


def digest(t: torch.Tensor) -> int:
    """First 8 bytes of the sha256 of a tensor's dtype, shape and bit pattern: what tests/golden/reference_traces.npz
    (oracle/make_reference_traces.py) keeps of every tensor the reference handed out.  Some traces start from seeded
    `torch.randn` draws, which are the same on every host where ATen runs its AVX2 or AVX-512 kernels."""
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.reshape(-1).view(torch.uint8).numpy().tobytes())
    return int.from_bytes(h.digest()[:8], "little")


def reference_trace(key: str):
    """The stored reference trace `key` (uint64 digests, int32 boxes or a string), or None if the reference has none."""
    with np.load(REFERENCE_TRACES) as g:
        return g[key] if key in g.files else None


def assert_trace(got, key: str):
    """`got`: digests of our tensors, in the order the reference's were recorded under `key`."""
    want = reference_trace(key)
    assert want is not None, f"{key}: no reference trace stored (oracle/make_reference_traces.py)"
    want = [int(v) for v in want]
    assert len(got) == len(want), f"{key}: {len(got)} tensors vs the reference's {len(want)}"
    bad = [i for i, (a, b) in enumerate(zip(got, want)) if a != b]
    assert not bad, f"{key}: tensors {bad} (of {len(want)}) differ from the reference's"


@contextlib.contextmanager
def stub_webui(monkeypatch):
    """Our delegate under the stub WebUI the reference traces were recorded in (oracle/ref_shim.py: `modules.*`
    stand-ins, deterministic prompt parser), with its buffers on the host as on a machine without a GPU."""
    from multidiffusion_upscaler_for_automatic1111_b200 import host
    from oracle import ref_shim
    ns = ref_shim.install()
    host._a1111_cache.clear()
    monkeypatch.setattr(host, "device", lambda: torch.device("cpu"))
    try:
        yield ns
    finally:
        ref_shim.uninstall()
        host._a1111_cache.clear()


def bits(t: torch.Tensor) -> np.ndarray:
    t = t.detach().cpu().contiguous()
    if t.dtype == torch.float32:
        return t.numpy().view(np.uint32)
    return t.view(torch.int16).numpy().view(np.uint16)


def sha(t: torch.Tensor) -> str:
    return hashlib.sha256(bits(t).tobytes()).hexdigest()


def assert_bit_equal(a: torch.Tensor, b: torch.Tensor, what: str = "", allow_signed_zero: bool = False):
    """Bit patterns must match (sign of zero and NaN payloads included).  `allow_signed_zero=True` is an explicit
    opt-out for comparisons whose two sides legitimately differ in the sign of a zero (say why at the call site)."""
    assert a.dtype == b.dtype, f"{what}: dtype {a.dtype} vs {b.dtype}"
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    ba, bb = bits(a), bits(b)
    if np.array_equal(ba, bb):
        return
    fa, fb = a.detach().cpu().float(), b.detach().cpu().float()
    bad = ~((fa == fb) | (fa.isnan() & fb.isnan()))
    n = int(bad.sum())
    assert n == 0, f"{what}: {n} mismatching elements, max abs diff {(fa - fb).abs().max().item()}"
    if not allow_signed_zero:
        nz = int((ba != bb).sum())
        raise AssertionError(f"{what}: values equal but {nz} elements differ in bit pattern (sign of zero / NaN payload)")


def region_composite_reference(x_buffer, weights, regions, out=None):
    """The reference's tensor expressions (multidiffusion.py:187-216, mixtureofdiffusers.py:145-175) on CPU tensors:
    what td_region_composite fuses on the device."""
    N, C, H, W = x_buffer.shape
    buf = x_buffer.clone()
    fb = fm = fc = None
    for (x, y, w, h, mode, r_out, aux) in regions:
        sl = (slice(None), slice(None), slice(y, y + h), slice(x, x + w))
        if mode == 0:
            buf[sl] += r_out if aux is None else r_out * aux
        else:
            if fb is None:
                fb, fm, fc = torch.zeros_like(buf), torch.zeros((1, 1, H, W)), torch.zeros((1, 1, H, W))
            fb[sl] += r_out
            fm[sl] += aux
            fc[sl] += 1
    res = buf
    if weights is not None:
        wv = weights.view(1, 1, H, W)
        res = torch.where(wv > 1, buf / wv, buf)
    if fb is not None:
        fb = torch.where(fc > 1, fb / fc, fb)
        fm = torch.where(fc > 1, fm / fc, fm)
        res = torch.where(fc > 0, res * (1 - fm) + fb * fm, res)
    return res.float()



def install_demofusion_stand_ins(set_attr=setattr):
    """Swap every device entry point DemoFusion.sample_one_step uses for torch-CPU stand-ins (the kernels themselves are
    pinned by the gpu tests): what remains under test is the delegate's plumbing -- window / view order, the mixture
    halves, jitter offsets, batching."""
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion, engine
    from oracle import blend
    from oracle import demofusion as odf

    def bbs(g):
        return [tuple(int(v) for v in r) for r in engine.grid_bboxes_xywh(g)]

    def scatter_tiles(g, x, out=None, tile_begin=0, tile_end=None, flags=0):
        return blend.scatter_tiles(x, bbs(g)[tile_begin:tile_end])

    def blend_multidiffusion(g, outs, N, C, tile_bs, weights, acc_dtype, x_buffer=None, flags=0, out=None, rcp_weights=None):
        buf = torch.zeros((N, C, g.H, g.W), dtype=acc_dtype)
        blend.accumulate_md(buf, torch.cat(list(outs), dim=0), bbs(g), N)
        return buf.float() / weights.view(1, 1, g.H, g.W)

    def dilated_gather(x, x_second, view_bx, view_by, view_second, s, out_h, out_w):
        return torch.cat([(x_second if sec else x)[:, :, by:by + out_h * s:s, bx:bx + out_w * s:s]
                          for bx, by, sec in zip(view_bx, view_by, view_second)], dim=0)

    def demofusion_combine(x_local, view_outs, views_per_batch, n_views, s, out_h, out_w, offset, end_y, end_x, mixture, c2, one_minus_c2):
        N = x_local.shape[0]
        allv = torch.cat(list(view_outs), dim=0)
        xg = torch.zeros_like(x_local)
        for v in range(n_views):
            by, bx = (v % (s * s)) // s, v % s
            xg[:, :, offset + by:end_y:s, offset + bx:end_x:s] += allv[v * N:(v + 1) * N]
        if mixture:
            xg = xg / 2
        return x_local * one_minus_c2 + xg * c2

    def scatter_bboxes(x, origins_dev, origins_host, n_tiles, tile_h, tile_w, out=None):
        o = origins_dev.view(-1, 2).tolist()
        return torch.cat([x[:, :, oy:oy + tile_h, ox:ox + tile_w] for ox, oy in o], dim=0)

    def blend_bboxes(batch_outs, tile_bs, origins_dev, origins_host, n_tiles, N, C, H, W, tile_h, tile_w):
        o = origins_dev.view(-1, 2).tolist()
        allt = torch.cat(list(batch_outs), dim=0)
        buf = torch.zeros((N, C, H, W), dtype=allt.dtype)
        cnt = torch.zeros((N, C, H, W), dtype=torch.float32)
        for t, (ox, oy) in enumerate(o):
            buf[:, :, oy:oy + tile_h, ox:ox + tile_w] += allt[t * N:(t + 1) * N]
            cnt[:, :, oy:oy + tile_h, ox:ox + tile_w] += 1
        return buf.float() / cnt.clamp_(min=1)

    for name, fn in dict(scatter_tiles=scatter_tiles, blend_multidiffusion=blend_multidiffusion, dilated_gather=dilated_gather,
                         demofusion_combine=demofusion_combine, scatter_bboxes=scatter_bboxes, blend_bboxes=blend_bboxes).items():
        set_attr(engine, name, fn)
    set_attr(DemoFusion, "_check_input", lambda self, x: x.contiguous())
    set_attr(DemoFusion, "gaussian_filter", lambda self, latents, kernel_size=3, sigma=1.0: odf.gaussian_filter(latents, kernel_size, sigma))
    set_attr(DemoFusion, "_renormalise", lambda self, g_, x_in: (g_ - g_.mean()) / g_.std() * x_in.std() + x_in.mean())
