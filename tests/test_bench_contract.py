"""bench.py's reference arm runs on host cores only, so its JSON line can be checked without a GPU: the keys the
driver reads, the metric / config naming shared with the GPU arm, and the oracle-only import rule of the GPU arm.
On the GPU: `--steps` is the number of timed steps of every config, and `--dump-outputs` writes the last timed step's
outputs, the same in every run."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _bench(*args, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["metric"].startswith("megapixels/sec") and d["unit"] == "MP/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and abs(d["value"] - 16.777216 / (d["ms_per_step"] * 1e-3 * 50)) / d["value"] < 1e-6   # 4096^2 image, 50 steps
    assert d["vs_baseline"] is None and d["data"].startswith("synthetic")
    assert d["e2e"] == {"value": d["value"], "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port"      # the oracle's op-for-op restatement of the reference's step
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["config"]["workload"].startswith("SD1.5 4096x4096") and (d["config"]["H"], d["config"]["W"], d["config"]["tile"]) == (512, 512, 96)


def test_demofusion_reference_arm_runs_the_steps_it_is_given():
    d = _bench("--impl", "reference", "--config", "cfg5", "--steps", "2", timeout=600)
    assert d["impl"] == "reference" and d["steps"] == 2 and d["cpu_baseline"]["steps"] == 2


@pytest.mark.gpu
@pytest.mark.parametrize("config,extra", [("cfg2", []), ("cfg3", []), ("cfg4", ["--vae-latent", "128"]), ("cfg5", [])])
def test_dump_outputs_are_the_last_timed_step_and_repeat_exactly(tmp_path, config, extra):
    runs = []
    for r in range(2):
        out_dir = tmp_path / f"run{r}"
        d = _bench("--config", config, "--steps", "3", "--warmup", "1", "--cpu-budget", "1", "--dump-outputs", str(out_dir), *extra)
        assert d["steps"] == 3
        files = sorted(out_dir.glob("*.npy"))
        assert files and sum(f.stat().st_size for f in files) <= 64 << 20
        runs.append({f.stem: np.load(f) for f in files})
        assert all(a.dtype in (np.float32, np.float64) for a in runs[-1].values())
    assert runs[0].keys() == runs[1].keys()
    for name in runs[0]:
        assert np.array_equal(runs[0][name], runs[1][name]), f"{config} {name}: two runs with the same arguments differ"
    if config in ("cfg2", "cfg3"):
        # the last of 3 timed steps ran on buffer set 2: its latent is the base latent rolled by 2 columns
        import bench
        from oracle import blend, tiling
        c = bench.CFG
        x = bench.synthetic_latent(0, (c["N"], c["C"], c["H"], c["W"])).roll(2, 3)
        plan = tiling.GridPlan(c["W"], c["H"], c["tile"], c["tile"], c["overlap"], c["tile_bs"], False)
        assert np.array_equal(runs[0]["tiles"], blend.scatter_tiles(x, plan.bboxes).float().numpy())


def test_gpu_arm_takes_nothing_from_the_oracle():
    """Only the cpu_baseline / reference legs may execute oracle/ (they ARE the CPU restatement being timed)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    for m in re.finditer(r"from oracle import [^\n]+", src):
        head = src[:m.start()]
        fn = re.findall(r"\ndef (\w+)\(", head)[-1]
        assert fn in ("cpu_reference_step_fn", "eager_cuda_baseline", "vae_cpu_baseline", "demofusion_cpu_baseline"), f"`{m.group(0)}` inside {fn}(): the GPU arm must not use the oracle"
    assert "import oracle" not in src
