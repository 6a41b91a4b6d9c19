"""TEST INFRASTRUCTURE -- CPU oracle for the tiled-diffusion / tiled-VAE hot path.

This package is a plain CPU restatement (Python ints/floats, numpy, torch-CPU) of
the reference algorithms listed in SURVEY.md section 8(a).  It is the CHECKER for the
CUDA path, never the product:

  * only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` /
    `--impl reference` legs of `bench.py` may import it;
  * nothing under `multidiffusion_upscaler_for_automatic1111_b200/` imports it,
    and the product path raises if the CUDA library is missing (no CPU fallback).

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so the
oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF, produced by importing the
unmodified reference under the stub host in `oracle/ref_shim.py`
(`oracle/make_golden.py`, `oracle/make_reference_traces.py` -> `tests/golden/*.npz`,
committed together with the generating scripts).
"""
