"""Soak run of the mixed-primitive fuzz (tests/test_gpu_parity.py::test_fuzz_mixed_primitives) over many
seeds and frame sizes on the GPU box: `python tools/fuzz_soak.py 60`.  Prints the failing seeds, if any.
`python tools/fuzz_soak.py 150 opaque`: only the all-opaque variant (one-kernel and two-kernel opaque stage).
`python tools/fuzz_soak.py 20 shapes`: the batch-size sweep of tests/test_gpu_launch_shapes.py (every raster
work-item shape) over more seeds, frame sizes, densities, raster paths and ids off / on."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import test_gpu_parity as t  # noqa: E402
import test_gpu_round2 as t2  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 40
family = sys.argv[2] if len(sys.argv) > 2 else "mixed"
only_opaque = family == "opaque"
rng = np.random.default_rng(77)
bad = []
if family == "shapes":
    import test_gpu_launch_shapes as ts  # noqa: E402
    for seed in range(1, 1 + n):
        # partial last tile column and row, and fewer tiles per frame than a B200 has SMs
        size = (int(rng.integers(2, 10)) * 64 + int(rng.integers(1, 64)), int(rng.integers(2, 12)) * 32 + int(rng.integers(1, 32)))
        density = str(rng.choice(["sparse", "dense"]))
        path = str(rng.choice(sorted(ts.PATHS)))
        ids = bool(rng.integers(0, 2))
        try:
            ts.check_sweep(size, density, path, ids, seed)
        except AssertionError as e:
            bad.append((seed, size, density, path, ids, str(e)[:120]))
            print("FAIL shapes", seed, size, density, path, ids, str(e)[:200], flush=True)
    print(f"shapes soak: {n} seeds, {len(bad)} failures", bad)
    sys.exit(1 if bad else 0)
for seed in range(100, 100 + n):
    size = (int(rng.integers(3, 1400)), int(rng.integers(3, 900)))
    try:
        if not only_opaque:
            t.test_fuzz_mixed_primitives(True, seed, size)
    except AssertionError as e:
        bad.append((seed, size, str(e)[:120]))
        print("FAIL", seed, size, str(e)[:200], flush=True)
    try:  # the all-opaque variant: the same calls through the one-kernel and the two-kernel opaque stage
        t2.test_fuzz_opaque_passes_take_the_deferred_stage(True, seed, size)
    except AssertionError as e:
        bad.append(("opaque", seed, size, str(e)[:120]))
        print("FAIL opaque", seed, size, str(e)[:200], flush=True)
print(f"fuzz soak: {n} seeds x {1 if only_opaque else 2} kinds, {len(bad)} failures", bad)
sys.exit(1 if bad else 0)
