#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on the B200-native tiled-diffusion hot path.

Workload (config.workload): BASELINE configs[1] -- SD1.5 4096x4096 txt2img, MultiDiffusion,
96x96 latent tiles, overlap 48 (the UI default), 50 sampler steps: latent [N=2, C=4, 512, 512]
fp16, T = 100 tiles.  One bench "step" = one sampler step of the hot path:

    td_scatter_tiles (latent -> [T*N,4,96,96] tile batch)  ->  [UNet: the host application's, stubbed]
    ->  td_blend_multidiffusion (tile outputs -> blended fp32 latent)

`value` = megapixels of final image per second = 16.777216 MP / (50 * seconds_per_step), inputs
resident in HBM.  The UNet is NOT part of the path (SURVEY.md section 8): its outputs are
pre-generated synthetic tensors (25 batch tensors of 4 tiles), rotated over enough buffer sets that
every launch reads cold (HBM-resident, not L2-resident) data.

`e2e` = the same metric through the reference-facing class (MultiDiffusion.kdiff_forward, identity
denoiser) with the step's latent copied from pinned host memory and the blended result copied back.

`--impl reference` / `cpu_baseline` = the op-for-op restatement of the reference's `sample_one_step` (oracle/blend.py,
bit-identical to the reference; `kind: "port"`) on the host cores at the thread count that runs it fastest, identity
denoiser.

`--dump-outputs DIR` (single GPU) writes what the last timed step computed, as float32 .npy files: cfg2 / cfg3 the tile
batch td_scatter_tiles hands the UNet (`tiles.npy`) and the blended latent (`latent.npy`); cfg4 the decoded image at 2^21
pixel positions drawn with a fixed seed (`image_sample.npy` [3, 2^21], positions y * W + x in `image_sample_index.npy`,
float64); cfg5 the step's latent (`latent.npy`).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.  `--steps` is used exactly as given.

Other BASELINE configs (same JSON contract, DESIGN.md section 6):
    --config cfg3   Mixture of Diffusers step (td_blend_mixture heads the roofline object)
    --config cfg4   tiled VAE decode only, z [1,4,1024,1024] -> 8192 x 8192 RGB through tilevae.VAEHook (one step = one decode;
                    roofline.bound = "tensor": the dominant tcgen05 convolution + the whole-decode TFLOP/s); --vae-slow
    --config cfg5   one DemoFusion.sample_one_step at the x4 phase of an SDXL 6144^2 upscale (latent [2,4,768,768])
    --gpus N        under torchrun: row-strip tile shard for cfg2 (weak scaling by default, strong rides along, in-run
                    parity_ok), tile round-robin for cfg4, window / view shard for cfg5
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

IMAGE_MP = 4096 * 4096 / 1e6
SAMPLER_STEPS = 50
CFG = dict(N=2, C=4, H=512, W=512, tile=96, overlap=48, tile_bs=4)
METRIC = "megapixels/sec final image (SD1.5 4K MultiDiffusion)"
METRIC_MOD = "megapixels/sec final image (SD1.5 4K Mixture of Diffusers, gaussian tile weights)"


def mp_per_s(sec_per_step: float) -> float:
    return IMAGE_MP / (SAMPLER_STEPS * sec_per_step)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampler running while the GPU is under load (recipe in B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU arm
def cpu_reference_step_fn(method: str = "md"):
    """One sampler step of the reference's PyTorch tile path on the host cores, identity denoiser: the oracle
    restatement, which executes the reference's exact op sequence (`x_buffer[slicer] += tile` in the latent dtype,
    `torch.where(weights > 1, x_buffer / weights, x_buffer)`; oracle/blend.py, bit-identical outputs, same speed within
    noise as the unmodified reference: 4.2 vs 4.2 ms on one host) -- kind "port"."""
    from oracle import blend, synth, tiling
    c = CFG
    x = synth.latent(0, (c["N"], c["C"], c["H"], c["W"]), torch.float16)
    if method == "mod":      # Mixture of Diffusers: op-for-op restatement (mixtureofdiffusers.py:61-179 grid part)
        plan = tiling.GridPlan(c["W"], c["H"], c["tile"], c["tile"], c["overlap"], c["tile_bs"], True)
        return (lambda: blend.mixture_step(x, plan.batched_bboxes, plan.tile_weights, plan.rescale_factor, lambda t, bb: t)), "port"
    plan = tiling.GridPlan(c["W"], c["H"], c["tile"], c["tile"], c["overlap"], c["tile_bs"], False)
    return (lambda: blend.multidiffusion_step(x, plan.batched_bboxes, plan.weights, lambda t, bb: t)), "port"


def eager_cuda_baseline(method: str = "md", steps: int = 20):
    """The reference's op sequence (oracle restatement: per-tile slice copies, `x_buffer[slicer] += tile`, where / divide) in
    stock torch EAGER on this GPU, device-resident tensors, identity denoiser -- what the unmodified reference does on a
    CUDA device (SURVEY.md section 8(d): "the kernel to beat").  Part of the cpu_baseline leg; None without a GPU."""
    if not torch.cuda.is_available():
        return None
    from oracle import blend, synth, tiling
    c = CFG
    x = synth.latent(0, (c["N"], c["C"], c["H"], c["W"]), torch.float16).cuda()
    plan = tiling.GridPlan(c["W"], c["H"], c["tile"], c["tile"], c["overlap"], c["tile_bs"], method == "mod")
    if method == "mod":
        step = lambda: blend.mixture_step(x, plan.batched_bboxes, plan.tile_weights, plan.rescale_factor, lambda t, bb: t)
    else:
        step = lambda: blend.multidiffusion_step(x, plan.batched_bboxes, plan.weights, lambda t, bb: t)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3) / steps
    return {"ms_per_step": ms, "value": mp_per_s(ms / 1e3), "unit": "MP/s",
            "what": "reference op sequence, stock torch eager on this GPU (device-resident, identity denoiser, host launch overhead included)"}


def pick_cpu_threads(step) -> int:
    """Use the thread count at which the reference path is FASTEST on this host (tiny per-tile ops
    get slower with too many OpenMP threads); the count used is reported as `cores`."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (1, 4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = 1, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        elif dt > 3 * best_t:
            break
    return best


def run_cpu(steps: int, warmup: int, budget_s: float = None, method: str = "md"):
    step, kind = cpu_reference_step_fn(method)
    threads = pick_cpu_threads(step)
    torch.set_num_threads(threads)
    for _ in range(max(warmup, 1)):
        step()
    t0 = time.perf_counter()
    done = 0
    while done < steps:
        step()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = (time.perf_counter() - t0) / done
    return dt, done, threads, kind


def reference_arm(args, rank):
    if rank != 0:
        return
    mod = args.config == "cfg3"
    dt, done, threads, kind = run_cpu(args.steps, args.warmup, method="mod" if mod else "md")
    v = mp_per_s(dt)
    line = {
        "impl": "reference", "metric": METRIC_MOD if mod else METRIC, "value": v, "unit": "MP/s", "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": workload_config(),
        "cpu_baseline": {"value": v, "unit": "MP/s", "cores": threads, "kind": kind,
                         "sample": f"{done} sampler steps of cfg2 (scatter+blend+normalise, identity denoiser), torch CPU, "
                                   "op-for-op restatement of the reference's sample_one_step"},
        "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config():
    c = CFG
    return {"workload": "SD1.5 4096x4096 txt2img MultiDiffusion: latent [2,4,512,512] fp16, 96x96 tiles, overlap 48 "
                        "(T=100, 25 batches of 4), 50 sampler steps; hot path = scatter + blend/normalise per step",
            "denoiser": "stubbed (UNet belongs to the host application; tile outputs are pre-generated synthetic tensors)",
            "l2": "inputs larger than L2: buffer sets rotate (see buffer_sets / set_mb)",
            **{k: c[k] for k in ("N", "C", "H", "W", "tile", "overlap", "tile_bs")}}


def synthetic_latent(seed: int, shape, dtype=torch.float16) -> torch.Tensor:
    """Bell-shaped synthetic latent k/256 (sum of three PCG64 uniforms): platform-stable, exact in fp16.
    (Same construction as the fixtures' inputs; kept here so the GPU arm needs nothing from oracle/.)"""
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(seed))
    k = rng.integers(-341, 342, size=(3,) + tuple(shape), dtype=np.int32).sum(axis=0)
    return torch.from_numpy(k.astype(np.float32) / 256.0).to(dtype)


# ----------------------------------------------------------------------------- GPU arm
def canvas_for(world: int, scaling: str):
    """Latent canvas (H, W).  strong: BASELINE cfg2's 512 x 512 whatever N.  weak: N x the cfg2 area -- every rank keeps a
    cfg2-sized share of the tiles (more GPUs = larger upscale, the regime tile sharding exists for)."""
    if scaling == "strong" or world == 1:
        return CFG["H"], CFG["W"]
    return {2: (1024, 512), 4: (2048, 512), 8: (2048, 1024)}.get(world, (512 * min(world, 4), 512 * max(1, world // 4)))


class StripWorkload:
    """N > 1: row-strip tile shard with halo-only exchange (parallel.StripShard / StripExchange).  One step of rank r =
    scatter its tiles -> [UNet: stubbed, outputs pre-generated in the exchange's own-tile buffer] -> push the overlapping
    tile rows to the next rank(s) + signal -> blend its strip (waits in-kernel for the halos) -> push the latent halo
    rows back + signal + wait."""

    def __init__(self, device, rank, world, scaling):
        from multidiffusion_upscaler_for_automatic1111_b200 import _cabi, engine, parallel
        self.cabi, self.engine, self.parallel = _cabi, engine, parallel
        c = CFG
        self.dev, self.rank, self.world, self.scaling = device, rank, world, scaling
        self.N, self.C = c["N"], c["C"]
        self.H, self.W = canvas_for(world, scaling)
        self.g = engine.make_grid(self.W, self.H, c["tile"], c["tile"], c["overlap"], c["tile_bs"])
        g = self.g
        self.T = g.num_tiles
        w_host = engine.grid_weights(g)
        self.weights = torch.from_numpy(w_host).to(device)
        self.rcp_weights = torch.from_numpy(engine.exact_reciprocals(w_host)).to(device)
        self.shard = parallel.StripShard(list(g.ys[:g.rows]), g.cols, g.tile_h, g.H, rank, world)
        self.ex = parallel.StripExchange(self.shard, self.N, self.C, g.tile_w, g.W, torch.float16, device)
        self.t0, self.t1 = self.shard.tile_range()
        self.x = synthetic_latent(rank, (self.N, self.C, g.H, g.W), torch.float16).to(device)
        own = self.ex.own_tiles()
        own.copy_((torch.randn(own.shape, device=device, dtype=torch.float32) * 0.8).half())
        self.tiles_in = torch.empty_like(own)
        self.stream = ctypes.c_void_p(0)
        es = 2
        lo, hi = self.shard.strip()
        self.bytes_scatter = (self.N * self.C * (self.shard.scatter_rows()[1] - self.shard.scatter_rows()[0]) * g.W + own.numel()) * es
        halo_rows = sum(v1 - v0 for (_, _, v0, v1) in self.shard.halo_in())
        self.bytes_blend = (own.numel() + halo_rows * g.cols * self.N * self.C * g.tile_w) * es + self.N * self.C * (hi - lo) * g.W * 4 + (hi - lo) * g.W * 4
        self.halo_bytes_out = sum((v1 - v0) for (_, _, v0, v1) in self.shard.halo_out()) * g.cols * self.N * self.C * g.tile_w * es + \
            sum(b - a for (_, a, b) in self.shard.x_out()) * g.W * self.N * self.C * 4
        self.nsets, self.set_mb = 1, (self.x.numel() * 2 + 2 * own.numel() * 2 + self.N * self.C * g.H * g.W * 4) / 1e6
        self.exchange_mode = "strip"

    def set_stream(self):
        self.stream = self.cabi.current_stream_ptr(self.dev)

    def scatter(self, s=0, flags=0):
        c = self.cabi
        if self.t1 > self.t0:
            c.check(c.lib.td_scatter_tiles(ctypes.byref(self.g), self.x.data_ptr(), self.tiles_in.data_ptr(), self.N, self.C, c.TD_F16,
                                           self.t0, self.t1, flags, self.stream))

    def step(self, i):
        self.scatter()
        self.ex.push_tile_halos()
        self.ex.blend(self.g, self.weights, self.rcp_weights)
        self.ex.push_x_halos_and_wait()

    def launches_per_step(self):
        sh = self.shard
        return 4          # scatter, tile-halo push (+ signal), strip blend (+ in-kernel wait), latent-halo push (+ signal + wait)

    def parity(self):
        """One more step, then: every rank's strip == the single-GPU blend of ALL ranks' tile outputs (computed on every
        rank from the gathered outputs; compared on the gathered latent).  Bit patterns."""
        import torch.distributed as dist
        g, sh = self.g, self.shard
        # fresh tile outputs first: a halo left over from the timed steps (same values every step) must not pass
        own_now = self.ex.own_tiles()
        own_now.copy_((torch.randn(own_now.shape, device=self.dev, dtype=torch.float32) * 0.8 + 0.1 * (self.rank + 1)).half())
        torch.cuda.synchronize()
        dist.barrier()
        self.step(0)
        torch.cuda.synchronize()
        full = self.ex.gather_latent(self.ex.x_out)
        per_band = g.cols * self.N
        nb = max(len(sh.bands(r)) for r in range(self.world))
        own = self.ex.own_tiles()
        pad = torch.zeros((nb * per_band,) + tuple(own.shape[1:]), dtype=own.dtype, device=self.dev)
        pad[:own.shape[0]] = own
        allo = torch.empty((self.world,) + tuple(pad.shape), dtype=own.dtype, device=self.dev)
        dist.all_gather_into_tensor(allo.view(-1), pad.view(-1))
        outs = []
        for r in range(self.world):
            for k, _ in enumerate(sh.bands(r)):
                outs.append(allo[r][k * per_band:(k + 1) * per_band])
        want = self.engine.blend_multidiffusion(g, outs, self.N, self.C, g.cols, self.weights, torch.float16, rcp_weights=self.rcp_weights)
        torch.cuda.synchronize()
        ok = torch.equal(full.view(torch.int32), want.view(torch.int32))
        t = torch.tensor([1 if ok else 0], device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def close(self):
        self.ex.close()


class Workload:
    def __init__(self, device, rank, world, nsets, exchange="peer"):
        from multidiffusion_upscaler_for_automatic1111_b200 import _cabi, engine
        self.cabi, self.engine = _cabi, engine
        c = CFG
        self.dev, self.rank, self.world = device, rank, world
        self.N, self.C = c["N"], c["C"]
        self.g = engine.make_grid(c["W"], c["H"], c["tile"], c["tile"], c["overlap"], c["tile_bs"])
        g = self.g
        self.T = g.num_tiles
        w_host = engine.grid_weights(g)
        self.weights = torch.from_numpy(w_host).to(device)
        self.rcp_weights = torch.from_numpy(engine.exact_reciprocals(w_host)).to(device)   # MultiDiffusion weights are integers
        # tile shard of this rank (contiguous chunk of the row-major tile list)
        self.chunk = -(-self.T // world)
        self.t0 = min(rank * self.chunk, self.T)
        self.t1 = min(self.t0 + self.chunk, self.T)
        self.nsets = nsets
        base = synthetic_latent(0, (self.N, self.C, g.H, g.W), torch.float16).to(device)
        tile_shape = (self.N, self.C, g.tile_h, g.tile_w)
        self.x, self.tiles_in, self.outs, self.x_out, self.gathered = [], [], [], [], []
        for s in range(nsets):
            self.x.append(base.roll(s, 3).contiguous())
            self.tiles_in.append(torch.empty(((self.t1 - self.t0) * self.N,) + tile_shape[1:], dtype=torch.float16, device=device))
            if world == 1:
                outs = []
                for b in range(g.num_batches):
                    nt = min(g.tile_bs, self.T - b * g.tile_bs)
                    outs.append((torch.randn((nt * self.N,) + tile_shape[1:], device=device, dtype=torch.float32) * 0.8).half())
                self.outs.append(outs)
            else:
                self.outs.append([(torch.randn((self.chunk * self.N,) + tile_shape[1:], device=device) * 0.8).half()])
                self.gathered.append(torch.empty((world * self.chunk * self.N,) + tile_shape[1:], dtype=torch.float16, device=device))
            self.x_out.append(torch.empty((self.N, self.C, g.H, g.W), dtype=torch.float32, device=device))
        es = 2
        self.bytes_scatter = (self.N * self.C * g.H * g.W + (self.t1 - self.t0) * self.N * self.C * g.tile_h * g.tile_w) * es
        self.bytes_blend = self.T * self.N * self.C * g.tile_h * g.tile_w * es + self.N * self.C * g.H * g.W * 4 + g.H * g.W * 4
        # Mixture of Diffusers: tiles + x_buffer in the latent dtype + rescale canvas + gaussian tile weights
        self.bytes_blend_mod = self.T * self.N * self.C * g.tile_h * g.tile_w * es + self.N * self.C * g.H * g.W * es + g.H * g.W * 4 + g.tile_h * g.tile_w * 4
        self.set_mb = (self.x[0].numel() * 2 + self.tiles_in[0].numel() * 2 + sum(o.numel() for o in self.outs[0]) * 2 +
                       self.x_out[0].numel() * 4 + (self.gathered[0].numel() * 2 if self.gathered else 0)) / 1e6
        self.stream = ctypes.c_void_p(0)
        self.exchange_mode = exchange if world > 1 else "none"
        self.method = "md"
        self.peer = None
        self.step_no = 0
        if self.exchange_mode == "peer":
            from multidiffusion_upscaler_for_automatic1111_b200 import parallel
            self.parallel = parallel
            self.shard = parallel.TileShard(self.T, rank, world)
            self.peer = parallel.PeerExchange(self.chunk * self.N * self.C * g.tile_h * g.tile_w * es, device)
        self._tables = []
        for s in range(nsets):
            if world == 1:
                ts = self.outs[s]
                self._tables.append(((ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts]), len(ts), g.tile_bs))
            else:
                stride = self.chunk * self.N * self.C * g.tile_h * g.tile_w * es
                basep = self.gathered[s].data_ptr()
                nb = -(-self.T // self.chunk)
                self._tables.append(((ctypes.c_void_p * nb)(*[basep + b * stride for b in range(nb)]), nb, self.chunk))

    def set_stream(self):
        self.stream = self.cabi.current_stream_ptr(self.dev)

    def scatter(self, s, flags=0):
        c = self.cabi
        c.check(c.lib.td_scatter_tiles(ctypes.byref(self.g), self.x[s].data_ptr(), self.tiles_in[s].data_ptr(), self.N, self.C,
                                       c.TD_F16, self.t0, self.t1, flags, self.stream))

    def exchange(self, s):
        if self.exchange_mode == "nccl":
            torch.distributed.all_gather_into_tensor(self.gathered[s], self.outs[s][0])

    def blend(self, s, flags=0):
        c = self.cabi
        ptrs, nb, tbs = self._tables[s]
        c.check(c.lib.td_blend_multidiffusion(ctypes.byref(self.g), ptrs, nb, tbs, self.N, self.C, c.TD_F16, c.TD_F16,
                                              self.weights.data_ptr(), None if (flags & 0x200) else self.rcp_weights.data_ptr(),
                                              self.x_out[s].data_ptr(), None, flags & 0x5ff, self.stream))

    def blend_mod(self, s, flags=0):
        """Mixture of Diffusers blend on the same tile outputs (BASELINE config 3's method)."""
        c = self.cabi
        if not hasattr(self, "_mod"):
            from multidiffusion_upscaler_for_automatic1111_b200.tile_utils import utils
            tw = utils.gaussian_weights_np(self.g.tile_w, self.g.tile_h)
            w = self.engine.grid_weights(self.g, tw)
            self._mod = (torch.from_numpy(tw).to(self.dev), torch.from_numpy(self.engine.rescale_factor(w)).to(self.dev),
                         [torch.empty((self.N, self.C, self.g.H, self.g.W), dtype=torch.float16, device=self.dev) for _ in range(self.nsets)])
        twt, rs, bufs = self._mod
        ptrs, nb, tbs = self._tables[s]
        c.check(c.lib.td_blend_mixture(ctypes.byref(self.g), ptrs, nb, tbs, self.N, self.C, c.TD_F16, c.TD_F16, twt.data_ptr(),
                                       rs.data_ptr(), bufs[s].data_ptr(), flags, self.stream))

    def empty(self, s):
        c = self.cabi
        c.check(c.lib.td_debug_launch_empty(1024, 128, self.stream))

    def outputs(self, s):
        """What a step on buffer set `s` hands on: the tile batch for the UNet and the blended latent (fp32 for
        MultiDiffusion, the latent dtype for Mixture of Diffusers)."""
        return {"tiles": self.tiles_in[s], "latent": self._mod[2][s] if self.method == "mod" else self.x_out[s]}

    def step(self, i):
        s = i % self.nsets
        self.scatter(s)
        if self.exchange_mode == "peer":
            # UNet output -> IPC-shared exchange buffer (double-buffered by step parity), publish the step
            # counter, then ONE kernel waits for the peers and blends while reading their tiles over NVLink
            self.step_no += 1
            parity = self.step_no & 1
            n = (self.t1 - self.t0) * self.N
            if n > 0:
                buf = self.peer.local_buffer(parity, torch.float16)[:self.outs[s][0][:n].numel()].view_as(self.outs[s][0][:n])
                buf.copy_(self.outs[s][0][:n])
            self.peer.signal()
            self.parallel.blend_multidiffusion_peer(self.g, self.peer, parity, self.shard, self.N, self.C, self.weights,
                                                    torch.float16, out=self.x_out[s])
            return
        self.exchange(s)
        if self.method == "mod":
            self.blend_mod(s)
        else:
            self.blend(s)


def vae_kernel_rooflines(dev, stream, peak):
    """Tiled-VAE streaming kernels at BASELINE cfg4's level-0 decoder tile: [1,128,944,944] fp16 (228 MB)."""
    from multidiffusion_upscaler_for_automatic1111_b200 import tilevae
    x = (torch.randn((1, 128, 944, 944), device=dev, dtype=torch.float32) * 0.7).half()
    y = torch.empty_like(x)
    gamma = torch.ones(128, device=dev)
    beta = torch.zeros(128, device=dev)
    nbytes = x.numel() * 2
    var, mean = tilevae.get_var_mean(x, 32)
    reps = 20
    t_stats = event_time_ms(lambda: [tilevae.get_var_mean(x, 32) for _ in range(reps)], stream) / reps * 1e-3
    def apply():
        for _ in range(reps):
            tilevae.check(tilevae.lib.td_gn_apply(x.data_ptr(), y.data_ptr(), 1, 128, 944 * 944, 0, 32, mean.data_ptr(), var.data_ptr(), 0,
                                                  gamma.data_ptr(), beta.data_ptr(), 1e-6, 1, tilevae.current_stream_ptr(dev)))
    apply()
    t_apply = event_time_ms(apply, stream) / reps * 1e-3
    return {"workload": "decoder level-0 tile [1,128,944,944] fp16 (BASELINE cfg4: 8192^2 RGB, tile 96)",
            "gn_stats": {"algorithmic_bytes": nbytes, "avg_launch_us": t_stats * 1e6, "achieved": nbytes / t_stats / 1e9,
                         "frac": nbytes / t_stats / 1e9 / peak, "note": "two launches (partials + finaliser) per call, 228 MB read > L2"},
            "gn_apply_silu": {"algorithmic_bytes": 2 * nbytes, "avg_launch_us": t_apply * 1e6, "achieved": 2 * nbytes / t_apply / 1e9,
                              "frac": 2 * nbytes / t_apply / 1e9 / peak}}


def timed_graph_loop(fn_step, steps, stream, chunk=1024):
    """Capture `steps` hot-path steps into CUDA graphs (chunks of <= `chunk`) and return a replay closure."""
    graphs = []
    done = 0
    while done < steps:
        n = min(chunk, steps - done)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            for i in range(done, done + n):
                fn_step(i)
        graphs.append(g)
        done += n

    def replay():
        for g in graphs:
            g.replay()
    return replay


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each tensor of `arrays` as <out_dir>/<name>.npy, float64 kept, everything else as float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), (t if t.dtype == torch.float64 else t.float()).cpu().numpy())


def event_time_ms(fn, stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def gpu_arm(args, rank, world, local_rank):
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    peak, peak_src = load_peaks()
    nsets = args.buffer_sets
    torch.manual_seed(0)      # the synthetic tile outputs are the same in every run
    if world > 1:   # peer exchange is double-buffered by step parity: keep every launch group even (odd --steps refused in main)
        args.warmup = max(args.warmup, 4) + (max(args.warmup, 4) & 1)
    wl = Workload(dev, rank, world, nsets, args.exchange)
    mod = args.config == "cfg3"
    if mod:
        if world > 1:
            sys.exit("--config cfg3 is measured on one GPU (the Mixture-of-Diffusers delegate shards by all-gather: see tests/test_multi_rank.py)")
        wl.method = "mod"
        wl.blend_mod(0)
    stream = torch.cuda.Stream(dev)
    sampler = ClockSampler(local_rank).start() if rank == 0 else None

    def barrier():
        if world > 1:
            torch.distributed.barrier()

    with torch.cuda.stream(stream):
        wl.set_stream()
        for i in range(max(args.warmup, 3) + (max(args.warmup, 3) & 1 if world > 1 else 0)):   # eager warm-up steps
            wl.step(i)
        torch.cuda.synchronize()
        use_graph = not args.no_graph
        if use_graph:
            replay = timed_graph_loop(wl.step, args.steps, stream)
            replay()                                   # extra untimed warm-up of the instantiated graphs
        else:
            def replay():
                for i in range(args.steps):
                    wl.step(i)
        torch.cuda.synchronize()
        barrier()
        ms = event_time_ms(replay, stream)             # EXACTLY args.steps steps
        barrier()
        t = torch.tensor([ms], device=dev)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
        sec_per_step = ms / 1e3 / args.steps
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, wl.outputs((args.steps - 1) % nsets))

        # --- per-kernel duration for the roofline (same buffers, same stream, CUDA events) -------------
        roof = None
        if rank == 0:
            reps = max(args.steps, 2000)
            def only(fn):
                r = timed_graph_loop(lambda i: fn(i % nsets), reps, stream)
                r()
                return event_time_ms(r, stream) / reps * 1e-3
            t_blend = only(wl.blend)
            t_scatter = only(wl.scatter)
            wl.blend_mod(0)
            t_mod = only(lambda s: wl.blend_mod(s, 0))
            t_blend_ser = only(lambda s: wl.blend(s, 32))      # TD_FLAG_NO_PDL: fully serialised launches
            t_scatter_ser = only(lambda s: wl.scatter(s, 32))
            if args.variants:
                tbl = {"empty_1024x128": only(wl.empty)}
                tbl["blend_rows"] = only(lambda s: wl.blend(s, 0x400))
                tbl["blend_rows_L2hot"] = only(lambda s: wl.blend(0, 0x400))
                tbl["blend_rows_no_tiles"] = only(lambda s: wl.blend(s, 0x100 | 0x400))
                tbl["blend_rows_no_pdl"] = only(lambda s: wl.blend(s, 32 | 0x400))
                tbl["blend_rows_ieee_div"] = only(lambda s: wl.blend(s, 0x200 | 0x400))
                tbl["scatter_rows"] = only(lambda s: wl.scatter(s, 0x400))
                tbl["scatter_rows_L2hot"] = only(lambda s: wl.scatter(0, 0x400))
                tbl["scatter_rows_no_pdl"] = only(lambda s: wl.scatter(s, 32 | 0x400))
                wl.blend_mod(0)
                tbl["blend_mixture_rows"] = only(lambda s: wl.blend_mod(s, 0x400))
                tbl["blend_mixture_rows_L2hot"] = only(lambda s: wl.blend_mod(0, 0x400))
                tbl["blend_async_one_plane"] = only(lambda s: wl.blend(s, 64))
                tbl["blend_async_ieee_div"] = only(lambda s: wl.blend(s, 0x200))
                wl.blend_mod(0)
                tbl["blend_mixture_async"] = only(lambda s: wl.blend_mod(s, 0))
                tbl["blend_mixture_reg"] = only(lambda s: wl.blend_mod(s, 2))
                for name, fl in (("async", 0), ("pipe", 8), ("tma", 4), ("reg", 2)):
                    tbl[f"blend_{name}"] = only(lambda s, fl=fl: wl.blend(s, fl))
                    tbl[f"blend_{name}_no_tiles"] = only(lambda s, fl=fl: wl.blend(s, fl | 0x100))
                    tbl[f"blend_{name}_L2hot"] = only(lambda s, fl=fl: wl.blend(0, fl))
                    tbl[f"scatter_{name}"] = only(lambda s, fl=fl: wl.scatter(s, fl))
                    tbl[f"scatter_{name}_L2hot"] = only(lambda s, fl=fl: wl.scatter(0, fl))
                print("VARIANTS(us): " + json.dumps({k: round(v * 1e6, 2) for k, v in tbl.items()}), file=sys.stderr, flush=True)
            roof = {
                "bound": "hbm", "kernel": "blend_md_async_kernel<half> (td_blend_multidiffusion, cp.async-staged)",
                "achieved": wl.bytes_blend / t_blend / 1e9, "peak": peak, "unit": "GB/s",
                "frac": wl.bytes_blend / t_blend / 1e9 / peak, "traffic": load_traffic("blend"),
                "peak_source": peak_src, "algorithmic_bytes": wl.bytes_blend, "avg_launch_us": t_blend * 1e6,
                "avg_launch_us_no_pdl": t_blend_ser * 1e6,
                "scatter": {"kernel": "scatter_tma_kernel<half> (td_scatter_tiles, TMA-staged)", "achieved": wl.bytes_scatter / t_scatter / 1e9,
                            "frac": wl.bytes_scatter / t_scatter / 1e9 / peak, "algorithmic_bytes": wl.bytes_scatter,
                            "avg_launch_us": t_scatter * 1e6, "avg_launch_us_no_pdl": t_scatter_ser * 1e6,
                            "traffic": load_traffic("scatter")},
                "mixture": {"kernel": "blend_mod_async_kernel<half> (td_blend_mixture, Mixture of Diffusers, BASELINE cfg3's method)",
                            "achieved": wl.bytes_blend_mod / t_mod / 1e9, "frac": wl.bytes_blend_mod / t_mod / 1e9 / peak,
                            "algorithmic_bytes": wl.bytes_blend_mod, "avg_launch_us": t_mod * 1e6},
                "note": "back-to-back launches inside a CUDA graph, programmatic dependent launch on (the next launch becomes "
                        "resident while this one drains; every global access still waits for completion); avg includes the "
                        "inter-kernel gap; *_no_pdl = same loop with plain stream serialisation",
            }
            roof["mixture"]["traffic"] = load_traffic("blend_mixture")
            if mod:      # cfg3: the step's dominant kernel is the Mixture-of-Diffusers blend -- it heads the roofline object
                md = {k: roof[k] for k in ("kernel", "achieved", "frac", "traffic", "algorithmic_bytes", "avg_launch_us", "avg_launch_us_no_pdl")}
                for k, v in roof["mixture"].items():
                    roof[k] = v
                roof["multidiffusion"] = md
                del roof["mixture"]
            try:
                roof["vae"] = vae_kernel_rooflines(dev, stream, peak)
            except Exception as e:   # never let the side measurement break the headline line
                roof["vae"] = {"error": repr(e)[:200]}

        # --- e2e through the public class API with host buffers ----------------------------------------
        e2e = e2e_arm(args, dev, stream, world, rank) if world == 1 else None
    clocks = sampler.stop() if sampler else None

    if rank == 0:
        cpu_dt, cpu_done, cpu_threads, cpu_kind = run_cpu(10 ** 9, 2, budget_s=args.cpu_budget, method="mod" if mod else "md")
        line = {
            "metric": METRIC_MOD if mod else METRIC, "value": mp_per_s(sec_per_step), "unit": "MP/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {**workload_config(), "buffer_sets": nsets, "set_mb": round(wl.set_mb, 1),
                       "cuda_graph": use_graph,
                       "parallelism": "single GPU" if world == 1 else (
                           f"tile-shard over {world} ranks; tile outputs exchanged through IPC-mapped peer buffers and read over "
                           "NVLink inside the blend kernel (td_peer_signal + td_blend_multidiffusion_peer), replicated deterministic blend"
                           if wl.exchange_mode == "peer" else
                           f"tile-shard over {world} ranks, NCCL all-gather of tile outputs, replicated blend")},
            "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * (2 if world == 1 else (4 if wl.exchange_mode == "peer" else 2)),
            "roofline": roof,
            "cpu_baseline": {"value": mp_per_s(cpu_dt), "unit": "MP/s", "cores": cpu_threads, "kind": cpu_kind,
                             "ms_per_step": cpu_dt * 1e3,
                             "sample": f"{cpu_done} sampler steps of the same workload (op-for-op restatement of the "
                                       f"reference's sample_one_step, identity denoiser, torch CPU, {cpu_threads} threads)",
                             "eager_cuda": eager_cuda_baseline("mod" if mod else "md") if world == 1 and args.cpu_budget > 1.0 else None},
            "impl": "b200",
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        sys.stdout.flush()
        torch.distributed.barrier()
        if wl.peer is not None:
            wl.peer.close()
            torch.distributed.destroy_process_group()
        else:
            os._exit(0)   # NCCL communicators captured in CUDA graphs can block a clean teardown; the line is out


def strip_arm(args, rank, world, local_rank):
    """N > 1 (default exchange): row-strip tile shard, halo-only exchange.  Prints the weak-scaling line (per-rank work
    fixed: the canvas grows with N) with the strong-scaling numbers (BASELINE cfg2's 512 x 512 canvas split over the
    ranks) in `strong`; both with an in-run parity check of the gathered latent against the single-GPU blend."""
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    torch.distributed.init_process_group("nccl", device_id=dev)
    dist = torch.distributed
    peak, peak_src = load_peaks()
    stream = torch.cuda.Stream(dev)
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    results = {}
    for scaling in (["weak", "strong"] if args.scaling == "weak" else ["strong"]):
        wl = StripWorkload(dev, rank, world, scaling)
        with torch.cuda.stream(stream):
            wl.set_stream()
            for i in range(max(args.warmup, 3)):
                wl.step(i)
            torch.cuda.synchronize()
            dist.barrier()
            use_graph = not args.no_graph
            if use_graph:
                replay = timed_graph_loop(wl.step, args.steps, stream)
                replay()
            else:
                def replay():
                    for i in range(args.steps):
                        wl.step(i)
            torch.cuda.synchronize()
            dist.barrier()
            ms = event_time_ms(replay, stream)             # EXACTLY args.steps steps
            dist.barrier()
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item()) / 1e3 / args.steps
            ok = wl.parity()
            if args.variants:      # where the step goes: graphs of growing prefixes of the step (every rank replays the same prefix)
                def prefix(n):
                    def run(i):
                        wl.scatter()
                        if n >= 2: wl.ex.push_tile_halos()
                        if n >= 3: wl.ex.blend(wl.g, wl.weights, wl.rcp_weights)
                        if n >= 4: wl.ex.push_x_halos_and_wait()
                        else: wl.ex.join_side()
                    return run
                table = {}
                # (a prefix that pushes tile halos without the closing latent-halo push leaves the blend's expect counter behind:
                # the blend of later replays would not wait -- so the blend is only timed inside the full step)
                for n, name in ((4, "full step"), (1, "scatter"), (2, "scatter+push_tiles")):
                    torch.cuda.synchronize(); dist.barrier()
                    rp = timed_graph_loop(prefix(n), 500, stream)
                    rp(); torch.cuda.synchronize(); dist.barrier()
                    tt = torch.tensor([event_time_ms(rp, stream)], device=dev)
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    table[name] = round(float(tt.item()) / 500 * 1e3, 2)
                if rank == 0:
                    print(f"[strip variants {scaling}] us/step: {table}", file=sys.stderr, flush=True)
            e2e = strip_e2e(args, dev, stream, world, rank) if scaling == "strong" else None
        mp_img = wl.H * wl.W * 64 / 1e6
        results[scaling] = {"value": mp_img / (SAMPLER_STEPS * sec), "ms_per_step": sec * 1e3, "canvas": [wl.H, wl.W], "tiles": wl.T,
                            "tiles_this_rank": wl.t1 - wl.t0, "strip_rows": list(wl.shard.strip()), "halo_bytes_out_per_step": wl.halo_bytes_out,
                            "launches_per_step": wl.launches_per_step(), "parity_ok": ok, "cuda_graph": use_graph, "e2e": e2e}
        dist.barrier()
        wl.close()
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        cpu_dt, cpu_done, cpu_threads, cpu_kind = run_cpu(10 ** 9, 2, budget_s=args.cpu_budget)
        head = results["weak" if args.scaling == "weak" else "strong"]
        line = {
            "metric": METRIC, "value": head["value"], "unit": "MP/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {**workload_config(), "canvas_latent": head["canvas"], "tiles": head["tiles"], "cuda_graph": head["cuda_graph"],
                       "l2": "one buffer set (L2-resident tile outputs): the N > 1 step is bound by launch and NVLink signal latency, not HBM",
                       "parallelism": f"row-strip tile shard over {world} ranks: each rank denoises a run of tile rows and blends the canvas "
                                      "rows it owns; per step only the overlapping tile rows go down the ranks and the scattered-from "
                                      "latent rows come back (pushed into CUDA-IPC peer buffers over NVLink, release/acquire flags, no NCCL "
                                      "on the data path)" + (f"; weak scaling: the canvas grows with N ({head['canvas'][0]} x {head['canvas'][1]} "
                                      "latent), per-rank tile count fixed" if args.scaling == "weak" else "")},
            "clocks": clocks, "parity_ok": head["parity_ok"], "e2e": results.get("strong", {}).get("e2e"),
            "gpu_launches": args.steps * head["launches_per_step"],
            "strip": head, "strong": results.get("strong") if args.scaling == "weak" else None,
            "roofline": None,
            "cpu_baseline": {"value": mp_per_s(cpu_dt), "unit": "MP/s", "cores": cpu_threads, "kind": cpu_kind, "ms_per_step": cpu_dt * 1e3,
                             "sample": f"{cpu_done} sampler steps of BASELINE cfg2 on the host cores, identity denoiser, torch CPU, {cpu_threads} threads"},
            "impl": "b200",
        }
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    dist.barrier()
    dist.destroy_process_group()


def strip_e2e(args, dev, stream, world, rank):
    """The metric through MultiDiffusion.kdiff_forward on the strip shard (BASELINE cfg2 canvas): every step copies the
    latent from pinned host memory, runs the hooked forward (identity denoiser on this rank's tiles) and reads this
    rank's rows of the result back."""
    import types

    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    c = CFG
    inner = types.SimpleNamespace(forward=lambda x, sigma, cond=None: x)
    sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None))
    p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a")
    d = MultiDiffusion(p, sampler)
    d.init_grid_bbox(c["tile"], c["tile"], c["overlap"], c["tile_bs"])
    d.init_done()
    d.init_tile_shard(None, fused=True)
    d.hook()
    fwd = sampler.model_wrap_cfg.inner_model.forward
    lo, hi = d._strip.strip()
    x_host = synthetic_latent(0, (c["N"], c["C"], c["H"], c["W"]), torch.float16).pin_memory()
    out_host = torch.empty((c["N"], c["C"], max(hi - lo, 1), c["W"]), dtype=torch.float32).pin_memory()
    x_dev = torch.empty_like(x_host, device=dev)
    sigma = torch.ones(c["N"], device=dev, dtype=torch.float16)
    cond = {"c_crossattn": [torch.zeros(c["N"], 77, 768, device=dev, dtype=torch.float16)],
            "c_concat": [torch.zeros(c["N"], 5, 1, 1, device=dev, dtype=torch.float16)]}

    def step():
        x_dev.copy_(x_host, non_blocking=True)
        out = fwd(x_dev, sigma, cond=cond)
        if hi > lo:
            out_host.copy_(out[:, :, lo:hi], non_blocking=True)

    n = 50
    for _ in range(5):
        step()
    torch.cuda.synchronize()
    torch.distributed.barrier()
    t0 = time.perf_counter()
    ms = event_time_ms(lambda: [step() for _ in range(n)], stream)
    wall = time.perf_counter() - t0
    t = torch.tensor([max(ms / 1e3, wall) / n], device=dev)
    torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    sec = float(t.item())
    torch.distributed.barrier()
    d._strip_exchange.close()
    return {"value": mp_per_s(sec), "unit": "MP/s", "h2d_bytes_per_step": x_host.numel() * 2, "d2h_bytes_per_step": out_host.numel() * 4,
            "ms_per_step": sec * 1e3, "steps": n,
            "api": "MultiDiffusion.kdiff_forward on the row-strip shard (per rank: full latent in, own rows out), identity denoiser"}


def load_traffic(kernel: str):
    """dram bytes per launch from the committed ncu --set full capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def e2e_arm(args, dev, stream, world, rank):
    """Same metric through MultiDiffusion.kdiff_forward with pinned-host input and host read-back each step."""
    import types

    from multidiffusion_upscaler_for_automatic1111_b200 import MultiDiffusion
    c = CFG
    inner = types.SimpleNamespace(forward=lambda x, sigma, cond=None: x)  # identity denoiser
    sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None))
    p = types.SimpleNamespace(width=c["W"] * 8, height=c["H"] * 8, sampler_name="Euler a")
    d = MultiDiffusion(p, sampler)
    d.init_grid_bbox(c["tile"], c["tile"], c["overlap"], c["tile_bs"])
    d.init_done()
    d.hook()
    fwd = sampler.model_wrap_cfg.inner_model.forward
    x_host = synthetic_latent(0, (c["N"], c["C"], c["H"], c["W"]), torch.float16).pin_memory()
    out_host = torch.empty((c["N"], c["C"], c["H"], c["W"]), dtype=torch.float32).pin_memory()
    x_dev = torch.empty_like(x_host, device=dev)
    sigma = torch.ones(c["N"], device=dev, dtype=torch.float16)
    cond = {"c_crossattn": [torch.zeros(c["N"], 77, 768, device=dev, dtype=torch.float16)],
            "c_concat": [torch.zeros(c["N"], 5, 1, 1, device=dev, dtype=torch.float16)]}

    def step():
        x_dev.copy_(x_host, non_blocking=True)
        out = fwd(x_dev, sigma, cond=cond)
        out_host.copy_(out, non_blocking=True)

    n = max(20, min(args.steps, 200))
    for _ in range(5):
        step()
    torch.cuda.synchronize()
    if args.profile_e2e:
        import cProfile
        import pstats
        pr = cProfile.Profile()
        pr.enable()
        for _ in range(20):
            step()
        torch.cuda.synchronize()
        pr.disable()
        pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(25)
    t0 = time.perf_counter()
    ms = event_time_ms(lambda: [step() for _ in range(n)], stream)
    wall = time.perf_counter() - t0
    sec = max(ms / 1e3, wall) / n   # host-bound loops are charged wall time
    return {"value": mp_per_s(sec), "unit": "MP/s", "h2d_bytes_per_step": x_host.numel() * 2,
            "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": sec * 1e3, "steps": n,
            "api": "MultiDiffusion.kdiff_forward (hooked inner_model.forward), identity denoiser, 25 tile batches"}


# ----------------------------------------------------------------------------- cfg4: tiled VAE decode
VAE_METRIC = "megapixels/sec final image (tiled VAE decode only, 8192x8192 RGB)"


def _sd_vae_half(is_decoder: bool, seed: int):
    """Random-init network with the published Stable-Diffusion autoencoder layout (ch 128, ch_mult (1,2,4,4), 2 res
    blocks, GroupNorm(32, eps 1e-6), single-head attention in the mid block) and the attribute names the reference
    walks (scripts/tilevae.py:107-195): synthetic weights, as BASELINE.json asks."""
    import torch.nn as nn
    import torch.nn.functional as F

    def norm(c):
        return nn.GroupNorm(32, c, eps=1e-6, affine=True)

    class Res(nn.Module):
        def __init__(self, cin, cout):
            super().__init__()
            self.in_channels, self.out_channels, self.use_conv_shortcut = cin, cout, False
            self.norm1, self.conv1 = norm(cin), nn.Conv2d(cin, cout, 3, 1, 1)
            self.norm2, self.conv2 = norm(cout), nn.Conv2d(cout, cout, 3, 1, 1)
            if cin != cout:
                self.nin_shortcut = nn.Conv2d(cin, cout, 1, 1, 0)

        def forward(self, x):
            h = self.conv2(F.silu(self.norm2(self.conv1(F.silu(self.norm1(x))))))
            return (self.nin_shortcut(x) if self.in_channels != self.out_channels else x) + h

    class Attn(nn.Module):
        def __init__(self, c):
            super().__init__()
            self.norm = norm(c)
            self.q, self.k, self.v, self.proj_out = (nn.Conv2d(c, c, 1) for _ in range(4))

    class Up(nn.Module):
        def __init__(self, c):
            super().__init__()
            self.with_conv, self.conv = True, nn.Conv2d(c, c, 3, 1, 1)

    class Down(nn.Module):
        def __init__(self, c):
            super().__init__()
            self.with_conv, self.conv = True, nn.Conv2d(c, c, 3, 2, 0)

    ch, mult, nres = 128, (1, 2, 4, 4), 2
    net = nn.Module()
    net.num_resolutions, net.num_res_blocks = len(mult), nres
    net.mid = nn.Module()
    if is_decoder:
        net.give_pre_end, net.tanh_out = False, False
        cur = ch * mult[-1]
        net.conv_in = nn.Conv2d(4, cur, 3, 1, 1)
        net.mid.block_1, net.mid.attn_1, net.mid.block_2 = Res(cur, cur), Attn(cur), Res(cur, cur)
        ups = []
        for lvl in reversed(range(len(mult))):
            lv = nn.Module()
            blocks = []
            for _ in range(nres + 1):
                blocks.append(Res(cur, ch * mult[lvl]))
                cur = ch * mult[lvl]
            lv.block = nn.ModuleList(blocks)
            if lvl != 0:
                lv.upsample = Up(cur)
            ups.insert(0, lv)
        net.up = nn.ModuleList(ups)
        net.norm_out, net.conv_out = norm(cur), nn.Conv2d(cur, 3, 3, 1, 1)
    else:
        net.conv_in = nn.Conv2d(3, ch, 3, 1, 1)
        cur = ch
        downs = []
        for lvl in range(len(mult)):
            lv = nn.Module()
            blocks = []
            for _ in range(nres):
                blocks.append(Res(cur, ch * mult[lvl]))
                cur = ch * mult[lvl]
            lv.block = nn.ModuleList(blocks)
            if lvl != len(mult) - 1:
                lv.downsample = Down(cur)
            downs.append(lv)
        net.down = nn.ModuleList(downs)
        net.mid.block_1, net.mid.attn_1, net.mid.block_2 = Res(cur, cur), Attn(cur), Res(cur, cur)
        net.norm_out, net.conv_out = norm(cur), nn.Conv2d(cur, 8, 3, 1, 1)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, prm in net.named_parameters():
            if prm.dim() == 4:
                fan_in = prm.shape[1] * prm.shape[2] * prm.shape[3]
                prm.copy_((torch.rand(prm.shape, generator=g) * 2 - 1) * (3.0 / fan_in) ** 0.5)
            elif name.endswith("weight"):
                prm.copy_(1.0 + 0.25 * (torch.rand(prm.shape, generator=g) * 2 - 1))
            else:
                prm.copy_(0.1 * (torch.rand(prm.shape, generator=g) * 2 - 1))
    net.eval()
    net.original_forward = None
    return net


def vae_decode_flops(hook, height, width):
    """Algorithmic FLOPs of one tiled decode: 2 * Cin * Cout * k^2 * output pixels per convolution, 4 * T^2 * C for the
    attention's QK^T and PV (+ the 1x1 projections), summed over the tiles the hook splits the latent into."""
    from multidiffusion_upscaler_for_automatic1111_b200 import vae_engine as ve
    prog = ve.compile_program(hook.net, hook.is_decoder)
    in_bboxes, _ = hook.split_tiles(height, width)
    total = 0.0
    for b in in_bboxes:
        h, w = b[3] - b[2], b[1] - b[0]
        for op in prog.ops:
            if isinstance(op, ve.Conv):
                if op.upsample_first:
                    h, w = 2 * h, 2 * w
                if op.downsample:
                    h, w = (h - 2) // 2 + 1, (w - 2) // 2 + 1
                m = op.module
                total += 2.0 * m.in_channels * m.out_channels * m.kernel_size[0] * m.kernel_size[1] * h * w
            elif isinstance(op, ve.Skip) and op.module is not None:
                m = op.module
                total += 2.0 * m.in_channels * m.out_channels * m.kernel_size[0] * m.kernel_size[1] * h * w
            elif isinstance(op, ve.Attention):
                c, t = op.module.q.in_channels, h * w
                total += 4 * 2.0 * c * c * t + 2 * 2.0 * t * t * c
    return total


def vae_arm(args, rank, world, local_rank):
    """BASELINE cfg4: tiled VAE decode only, z [1,4,1024,1024] fp16 -> 8192 x 8192 RGB, decoder tile 96 (121 tiles),
    fast mode (the UI default) unless --vae-slow.  One bench step = one whole decode through `VAEHook`."""
    from multidiffusion_upscaler_for_automatic1111_b200 import tilevae, vae_engine as ve, vae_ops
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    lat = args.vae_latent
    net = _sd_vae_half(True, 1).to(dev).half()
    hook = tilevae.VAEHook(net, 96, True, fast_decoder=not args.vae_slow, fast_encoder=True, color_fix=False)
    if world > 1:
        hook.init_tile_shard(None)
    g = torch.Generator().manual_seed(7)
    z_host = torch.randn((1, 4, lat, lat), generator=g).half().pin_memory()
    z = z_host.to(dev)
    out_host = torch.empty((1, 3, lat * 8, lat * 8), dtype=torch.float16).pin_memory()
    mp = (lat * 8) ** 2 / 1e6
    stream = torch.cuda.current_stream(dev)
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    steps, warm = args.steps, max(1, min(args.warmup, 2))
    for _ in range(warm):
        y = hook(z)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    last = {}

    def timed():
        for _ in range(steps):
            last["y"] = hook(z)
    ms = event_time_ms(timed, stream)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    sec = float(t.item()) / 1e3 / steps
    if args.dump_outputs:      # the 8192^2 image is 805 MB in fp32: a fixed, seeded sample of 2^21 pixels, with their positions
        img = last["y"].reshape(last["y"].shape[1], -1)
        idx = torch.randint(img.shape[1], (min(1 << 21, img.shape[1]),), generator=torch.Generator().manual_seed(0))
        dump_outputs(args.dump_outputs, {"image_sample": img[:, idx.to(dev)], "image_sample_index": idx.double()})

    def e2e_step():
        zd = z_host.to(dev, non_blocking=True)
        out_host.copy_(hook(zd), non_blocking=True)
    e2e_step(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_ms = event_time_ms(lambda: [e2e_step() for _ in range(steps)], stream)
    e2e_sec = max(e2e_ms / 1e3, time.perf_counter() - t0) / steps
    clocks = sampler.stop() if sampler else None
    # in-run parity (every rank: the sharded hook's calls are collective): the same fp16 network on a 160 x 160 corner of the
    # latent, tensor-core backend vs module backend
    zc = z[:, :, :160, :160].contiguous()
    a_tc = hook(zc).float()
    orig = ve.pick_backend
    ve.pick_backend = lambda program, device, dtype: ve.ModuleBackend(program, device, dtype)
    try:
        a_mod = hook(zc).float()
    finally:
        ve.pick_backend = orig
    if rank != 0:
        if world > 1:
            torch.distributed.barrier()
        return

    flops = vae_decode_flops(hook, lat, lat)
    tf_burst, tf_sust = 1661.3, 1404.6
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        tf_burst, tf_sust, peak_src = float(pk["bf16_tflops"]), float(pk["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json, cuBLAS bf16)"
    except Exception:
        tf_burst, tf_sust, peak_src = 1590.0, 1400.0, "fallback (B200_PROFILING.md)"
    # dominant kernel: the level-0 128 -> 128 3x3 convolution of a full tile (944 x 944), timed alone
    x = (torch.randn((1, 944, 944, 128), device=dev) * 0.5).half()
    w = (torch.randn((9, 128, 128), device=dev) * 0.03).half()
    b = torch.zeros(128, device=dev)
    yb = torch.empty_like(x)
    conv = lambda: vae_ops.conv2d_nhwc(x, w, b, ksize=3, pad=(1, 1), out=yb)
    conv(); torch.cuda.synchronize()
    t_conv = event_time_ms(lambda: [conv() for _ in range(20)], stream) / 20 * 1e-3
    conv_flops = 2.0 * 944 * 944 * 128 * 128 * 9
    scale = a_mod.abs().max().item()
    diff = (a_tc - a_mod).abs()
    line = {
        "metric": VAE_METRIC, "value": mp / sec, "unit": "MP/s", "n_gpus": world, "steps": steps, "warmup": warm,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"BASELINE cfg4: tiled VAE decode only, z [1,4,{lat},{lat}] fp16 -> {lat * 8}x{lat * 8} RGB, decoder tile 96, "
                               f"{len(hook.split_tiles(lat, lat)[0])} tiles, {'slow (GroupNorm barrier per site)' if args.vae_slow else 'fast'} mode, "
                               "random-init SD-shaped decoder (ch 128, mult 1-2-4-4)",
                   "backend": hook.backend_name, "l2": "activations of one tile (228 MB at level 0) exceed L2",
                   "parallelism": "single GPU" if world == 1 else f"VAE tiles round-robin over {world} ranks, all-gather of the output regions"},
        "clocks": clocks,
        "e2e": {"value": mp / e2e_sec, "unit": "MP/s", "h2d_bytes_per_step": z_host.numel() * 2, "d2h_bytes_per_step": out_host.numel() * 2,
                "ms_per_step": e2e_sec * 1e3, "api": "VAEHook.__call__ (hooked decoder forward), pinned-host latent in, pinned-host image out"},
        "gpu_launches": None,
        "roofline": {"bound": "tensor", "kernel": "conv_gemm_kernel (td_conv2d_nhwc, tcgen05 implicit GEMM), 128->128 3x3 on [1,944,944,128]",
                     "achieved": conv_flops / t_conv / 1e12, "peak": tf_burst, "unit": "TFLOP/s", "frac": conv_flops / t_conv / 1e12 / tf_burst,
                     "traffic": load_traffic("conv_944_128_128"), "peak_source": peak_src + ", burst (kernel timed alone)", "algorithmic_flops": conv_flops,
                     "avg_launch_us": t_conv * 1e6,
                     "whole_decode": {"algorithmic_flops": flops, "achieved": flops / sec / 1e12, "peak": tf_sust,
                                      "frac": flops / sec / 1e12 / tf_sust, "peak_source": "sustained (inside a long step)"}},
        "parity": {"what": "tcgen05 / channels-last backend vs cuDNN-module backend, same fp16 weights, z[:, :, :160, :160] (4 tiles)",
                   "mean_rel": diff.mean().item() / scale, "max_rel": diff.max().item() / scale},
        "impl": "b200",
    }
    cpu = vae_cpu_baseline(args.cpu_budget)
    line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()


def vae_cpu_baseline(budget_s: float, steps: int = 1):
    """The reference's tiled VAE algorithm on the host cores (oracle restatement, fp32 torch CPU) on a bounded sample:
    `steps` decodes of a 48 / 64 / 96-pixel latent (384^2 .. 768^2 px image) in 4 tiles, fast mode; thread count and sample
    size are chosen from a short probe so that one decode stays within about 2.5 x --cpu-budget seconds."""
    if budget_s <= 1.0:      # measurement runs that only want the GPU numbers
        return {"value": None, "unit": "MP/s", "cores": 0, "kind": "port", "seconds": 0.0, "sample": "skipped (--cpu-budget <= 1)"}
    from oracle import ldm_vae, vae
    net = ldm_vae.seeded_init(ldm_vae.Decoder(), 1).eval()
    zp = torch.randn((1, 4, 24, 24), generator=torch.Generator().manual_seed(8))

    def probe():      # one small untiled decode: which thread count suits this host's convolutions
        with torch.no_grad():
            net(zp)
    torch.set_num_threads(pick_cpu_threads(probe))
    t0 = time.perf_counter()
    probe()
    t_probe = time.perf_counter() - t0
    # bounded sample: the largest of three tiled decodes (4 tiles of (L/2 + 22)^2 latent pixels each + the estimator pass)
    # whose predicted time stays within ~2.5 x the budget (default 12 s -> <= 30 s of host work)
    L = 48
    for cand in (64, 96):
        if t_probe * 4 * (cand // 2 + 22) ** 2 / 24 ** 2 * 1.15 <= 2.5 * budget_s:
            L = cand
    z = torch.randn((1, 4, L, L), generator=torch.Generator().manual_seed(7))
    t0 = time.perf_counter()
    with torch.no_grad():
        for _ in range(steps):
            vae.vae_hook_call(net, z, L // 2, True, True, False)
    dt = time.perf_counter() - t0
    return {"value": (L * 8) ** 2 / 1e6 / (dt / steps), "unit": "MP/s", "cores": torch.get_num_threads(), "kind": "port", "seconds": dt,
            "steps": steps, "sample": f"{steps} tiled decode(s) of a {L}x{L} latent ({L * 8}x{L * 8} px, decoder tile {L // 2}, fast mode: 4 tiles + estimator pass), "
                      "oracle restatement of scripts/tilevae.py on torch CPU fp32"}


def vae_reference_arm(args, rank):
    if rank != 0:
        return
    cpu = vae_cpu_baseline(args.cpu_budget, args.steps or 1)
    line = {"impl": "reference", "metric": VAE_METRIC, "value": cpu["value"], "unit": "MP/s", "n_gpus": args.gpus,
            "steps": cpu.get("steps", 0), "warmup": 0, "ms_per_step": cpu["seconds"] * 1e3 / max(cpu.get("steps", 0), 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": cpu["sample"]}, "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- cfg5: DemoFusion dilated sampling
DEMO_METRIC = "demofusion_step_throughput"
DEMO = dict(N=2, C=4, lat=768, window=128, overlap=64, scale=4, tile_bs=8, tile_bs_g=4, sig=0.6, cs1=3.0, cs2=1.0, cs3=1.0,
            current_step=10, t_enc=40)


def _demo_job(dev, dtype, mixture, jitter):
    """A DemoFusion delegate at BASELINE cfg5's final phase (SDXL, 6144^2 px = latent 768^2, x4 over the 1536^2 base:
    current_scale_num 4, window 128 = SDXL's 1024 px) with an identity UNet stand-in: the step is the hot path alone."""
    import types
    from multidiffusion_upscaler_for_automatic1111_b200 import DemoFusion
    c = DEMO
    p = types.SimpleNamespace(width=c["lat"] * 8, height=c["lat"] * 8, sampler_name="Euler a", current_scale_num=c["scale"], mixture=mixture,
                              gaussian_filter=True, random_jitter=jitter, cosine_scale_1=c["cs1"], cosine_scale_2=c["cs2"],
                              cosine_scale_3=c["cs3"], current_step=c["current_step"], steps=50, t_enc=c["t_enc"], sd_model=None)
    calls = [0]

    def fwd(x_tile, sigma, cond=None):
        calls[0] += 1
        return x_tile
    inner = types.SimpleNamespace(forward=fwd)
    sampler = types.SimpleNamespace(model_wrap_cfg=types.SimpleNamespace(inner_model=inner, image_cfg_scale=None, forward=None))
    d = DemoFusion(p, sampler)
    d.window_size, d.sig = c["window"], c["sig"]
    return d, fwd, calls


def demofusion_arm(args, rank, world, local_rank):
    """BASELINE cfg5: one DemoFusion `sample_one_step` at the x4 phase of an SDXL 6144^2 upscale: latent [2,4,768,768] fp16,
    121 local windows of 128^2 (stride 64) count-blended, 7x7 gaussian blur + renormalise, 32 dilated global views (mixture),
    add-back + cosine mix.  UNet stand-in = identity, so the timed region is the tile path only.  N>1: windows and views
    sharded over the ranks (all-gather form, DemoFusion.init_tile_shard)."""
    import math
    import random
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    c = DEMO
    d, fwd, calls = _demo_job(dev, torch.float16, True, False)
    if world > 1:
        d.init_tile_shard(None)
    d.get_views(c["overlap"], c["tile_bs"], c["tile_bs_g"])
    d.sampler_forward = fwd
    d.cosine_factor = 0.5 * (1 + math.cos(math.pi * (c["t_enc"] - c["current_step"]) / c["t_enc"]))
    N, C, L = c["N"], c["C"], c["lat"]
    x_host = synthetic_latent(11, (N, C, L, L)).pin_memory()
    x = x_host.to(dev)
    out_host = torch.empty_like(x_host).pin_memory()
    sigma = torch.ones(N, device=dev)
    cond = {"c_crossattn": [torch.zeros(N, 77, 2048, device=dev, dtype=torch.float16)], "c_concat": [torch.zeros(N, 5, 1, 1, device=dev, dtype=torch.float16)]}
    stream = torch.cuda.current_stream(dev)
    steps, warm = args.steps, max(3, min(args.warmup, 10))
    sampler = ClockSampler(local_rank).start() if rank == 0 else None
    for _ in range(warm):
        y = d.sample_one_step(x, sigma, cond)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    calls[0] = 0
    last = {}

    def timed():
        for _ in range(steps):
            last["y"] = d.sample_one_step(x, sigma, cond)
    ms = event_time_ms(timed, stream)
    unet_calls = calls[0] // steps
    t = torch.tensor([ms], device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    sec = float(t.item()) / 1e3 / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latent": last["y"]})

    def e2e_step():
        xd = x_host.to(dev, non_blocking=True)
        out_host.copy_(d.sample_one_step(xd, sigma, cond), non_blocking=True)
    e2e_step(); torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    e2e_ms = event_time_ms(lambda: [e2e_step() for _ in range(steps)], stream)
    te = torch.tensor([max(e2e_ms / 1e3, time.perf_counter() - t0)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(te, op=torch.distributed.ReduceOp.MAX)
    e2e_sec = float(te.item()) / steps
    clocks = sampler.stop() if sampler else None

    # property checks at full size (the oracle comparison at this size is tests/test_demofusion.py::test_cfg5_size):
    #  * identity UNet + count-normalised blend: the local result equals the input wherever fp16 (sum/count) is exact, i.e.
    #    everywhere (count*x/count rounds back to x for count in {1,2,4}); so out = (1-c2)*x + c2*(global add-back)/2
    #  * all ranks hold the same bits
    y = d.sample_one_step(x, sigma, cond)
    digest = torch.tensor([float(y.float().sum().item()), float(y.float().abs().max().item())], device=dev, dtype=torch.float64)
    same = True
    if world > 1:
        lo, hi = digest.clone(), digest.clone()
        torch.distributed.all_reduce(lo, op=torch.distributed.ReduceOp.MIN)
        torch.distributed.all_reduce(hi, op=torch.distributed.ReduceOp.MAX)
        same = bool(torch.equal(lo, hi))
    finite = bool(torch.isfinite(y).all().item())
    if rank != 0:
        if world > 1:
            torch.distributed.barrier()
        return
    peak, peak_src = load_peaks()
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs_sustained"])
        peak_src = "measured (MEASURED_PEAKS.json, sustained copy: the step is many kernels back to back)"
    except Exception:
        pass
    esz = 2
    canvas = N * C * L * L * esz
    windows = d.num_tiles * N * C * c["window"] ** 2 * esz
    views = d.global_num_tiles * canvas // (c["scale"] ** 2)
    # scatter: canvas in, windows out | blend: windows in, canvas out | blur: canvas in/out | stats: 2 x canvas in |
    # affine: canvas in/out | gather: x + x_g in, views out | combine: views + x_local in, canvas out
    algo = (canvas + windows) + (windows + canvas) + 2 * canvas + 2 * canvas + 2 * canvas + (2 * canvas + views) + (views + canvas + canvas)
    mp = (L * 8) ** 2 / 1e6
    line = {
        "metric": DEMO_METRIC, "value": mp / sec, "unit": "MP/s", "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"BASELINE cfg5: SDXL-shaped 6144x6144 img2img x4 upscale, DemoFusion final phase: latent [{N},{C},{L},{L}] fp16, "
                               f"{d.num_tiles} local windows {c['window']}^2 stride {c['window'] - c['overlap']} (batches of {d.tile_bs}), scale {c['scale']}, "
                               f"{d.global_num_tiles} dilated views (mixture), gaussian filter k={2 * c['scale'] - 1}, identity UNet stand-in "
                               f"({unet_calls} calls / step)",
                   "l2": f"{algo / 1e6:.0f} MB of algorithmic traffic per step (> the 126 MB L2); every intermediate is written once and read once",
                   "parallelism": "single GPU" if world == 1 else f"windows + views sharded over {world} ranks, two all-gathers per step (NCCL)"},
        "clocks": clocks,
        "e2e": {"value": mp / e2e_sec, "unit": "MP/s", "h2d_bytes_per_step": canvas, "d2h_bytes_per_step": canvas, "ms_per_step": e2e_sec * 1e3,
                "api": "DemoFusion.sample_one_step, pinned-host latent in, pinned-host latent out"},
        "gpu_launches": None,
        "roofline": {"bound": "hbm", "kernel": "whole step (scatter_tma, blend_md_async, depthwise_conv2d, gn_stats, affine_clamp, "
                                               "dilated_gather, demofusion_combine): eager launches, host-launch bound",
                     "achieved": algo / sec / 1e9, "peak": peak, "unit": "GB/s", "frac": algo / sec / 1e9 / peak,
                     "traffic": None, "algorithmic_bytes": algo, "peak_source": peak_src},
        "parity": {"finite": finite, "ranks_identical": same,
                   "full_size_oracle_check": "tests/test_demofusion.py::test_demofusion_cfg5_size_matches_oracle"},
        "impl": "b200",
    }
    line["cpu_baseline"] = demofusion_cpu_baseline(args.cpu_budget)
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()


def demofusion_cpu_baseline(budget_s: float, steps: int = None):
    """The reference's DemoFusion step (oracle restatement, torch CPU) on the cfg5 latent in fp32, identity UNet stand-in:
    `steps` steps, or as many as fit in `budget_s` seconds (at most 50) when `steps` is None."""
    if budget_s <= 1.0:
        return {"value": None, "unit": "MP/s", "cores": 0, "kind": "port", "seconds": 0.0, "sample": "skipped (--cpu-budget <= 1)"}
    from oracle import demofusion as odf
    from oracle import tiling
    c = DEMO
    L = c["lat"]
    x = synthetic_latent(11, (c["N"], c["C"], L, L)).float()
    local, _, _ = tiling.demofusion_views(L, L, c["window"], c["overlap"])
    nb = -(-len(local) // c["tile_bs"]); tbs = -(-len(local) // nb)
    lb = [local[i * tbs:(i + 1) * tbs] for i in range(nb)]
    views = odf.global_views(c["scale"], True)
    gnb = -(-len(views) // c["tile_bs_g"]); gtbs = -(-len(views) // gnb)
    gb = [views[i * gtbs:(i + 1) * gtbs] for i in range(gnb)]
    cf = odf.cosine_factor(c["current_step"], c["t_enc"])
    ident = lambda t, b: t

    def one():
        with torch.no_grad():
            odf.sample_one_step(x, lb, gb, c["scale"], True, True, c["sig"], cf, c["cs2"], c["cs3"], ident, ident)
    torch.set_num_threads(pick_cpu_threads(one))      # the thread count at which the host runs this step fastest
    n, t0 = 0, time.perf_counter()
    with torch.no_grad():
        while True:
            one()
            n += 1
            if n == steps or steps is None and (time.perf_counter() - t0 > budget_s or n >= 50):
                break
    dt = (time.perf_counter() - t0) / n
    return {"value": (L * 8) ** 2 / 1e6 / dt, "unit": "MP/s", "cores": torch.get_num_threads(), "kind": "port", "seconds": dt * n,
            "steps": n, "sample": f"{n} whole cfg5 steps (latent [2,4,{L},{L}], fp32 on the host cores), oracle restatement of tile_methods/demofusion.py:219-324"}


def demofusion_reference_arm(args, rank):
    if rank != 0:
        return
    cpu = demofusion_cpu_baseline(max(args.cpu_budget, 5.0), args.steps)
    line = {"impl": "reference", "metric": DEMO_METRIC, "value": cpu["value"], "unit": "MP/s", "n_gpus": args.gpus, "steps": cpu["steps"],
            "warmup": 0, "ms_per_step": cpu["seconds"] / cpu["steps"] * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": cpu["sample"]}, "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps, used exactly as given (default: 2000 for cfg2 / cfg3, 5 "
                    "decodes for cfg4, 200 for cfg5; the cfg4 / cfg5 reference arms: 1 decode / as many steps as --cpu-budget allows)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--buffer-sets", type=int, default=8)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--exchange", default="strip", choices=["strip", "peer", "nccl"],
                    help="N>1: strip = row-strip shard with halo-only exchange (default); peer / nccl = round-1 replicate-all forms")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N>1 strip shard: weak = canvas grows with N (per-rank work fixed; the strong numbers ride along), strong = cfg2 canvas split")
    ap.add_argument("--profile-e2e", action="store_true")
    ap.add_argument("--variants", action="store_true", help="print a table of per-kernel micro-timings to stderr")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"], help="BASELINE.json config: cfg2 = MultiDiffusion hot path "
                    "(default, the headline), cfg3 = Mixture of Diffusers hot path, cfg4 = tiled VAE decode only, cfg5 = DemoFusion step")
    ap.add_argument("--vae-latent", type=int, default=1024, help="cfg4: latent edge (1024 -> 8192^2 image)")
    ap.add_argument("--vae-slow", action="store_true", help="cfg4: slow mode (GroupNorm statistics merged over all tiles at every site)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="single GPU: write what the last timed step computed to DIR/<name>.npy "
                    "(float32; cfg4: a fixed, seeded sample of the image)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps is None:
        if args.impl == "b200" or args.config in ("cfg2", "cfg3"):
            args.steps = {"cfg2": 2000, "cfg3": 2000, "cfg4": 5, "cfg5": 200}[args.config]
    elif args.steps < 1:
        ap.error("--steps must be at least 1")
    elif args.steps & 1 and world > 1 and args.impl == "b200" and args.config in ("cfg2", "cfg3") and args.exchange != "strip":
        ap.error("--steps must be even for the peer / nccl exchange (its buffers alternate by step parity)")
    if args.dump_outputs and (args.impl != "b200" or world > 1):
        ap.error("--dump-outputs is for the single-GPU runs of the GPU arm")
    if args.impl == "reference":
        {"cfg4": vae_reference_arm, "cfg5": demofusion_reference_arm}.get(args.config, reference_arm)(args, rank)
        return
    if args.config == "cfg5":
        demofusion_arm(args, rank, world, local_rank)
        return
    if args.config == "cfg4":
        vae_arm(args, rank, world, local_rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        sys.exit(f"--gpus {args.gpus} needs torchrun (WORLD_SIZE={world})")
    if world > 1 and args.exchange == "strip":
        strip_arm(args, rank, world, local_rank)
        return
    gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
