"""TEST INFRASTRUCTURE -- generate tests/golden/reference_traces.npz FROM THE UNMODIFIED REFERENCE.

The CPU tests that hold our delegate against the reference's host-side code (tests/test_oracle_vs_reference.py,
test_region_cond.py, test_side_inputs.py, test_noise_inverse.py, test_demofusion.py) each define
`reference_traces(ref)`: the drivers they run our delegate through, run on the reference's own classes under the stub
host of `oracle/ref_shim.py`.  This script stores what those return -- per tensor the digest of tests/helpers.py,
boxes as int32, strings -- and the tests compare our delegate with it.  Usage:

    TD_REFERENCE_ROOT=<checkout of the original extension> python -m oracle.make_reference_traces
"""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")
MODULES = ("test_oracle_vs_reference", "test_region_cond", "test_side_inputs", "test_noise_inverse", "test_demofusion")


def main():
    from oracle import ref_shim
    if not ref_shim.available():
        sys.exit("reference tree not found: set TD_REFERENCE_ROOT to a checkout of the original extension")
    sys.path.insert(0, TESTS)
    ref = ref_shim.load()
    out = {}
    for name in MODULES:
        for key, v in importlib.import_module(name).reference_traces(ref).items():
            assert key not in out, key
            out[key] = np.array(v, np.uint64) if isinstance(v, list) else np.asarray(v)
    path = os.path.join(TESTS, "golden", "reference_traces.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} traces, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
