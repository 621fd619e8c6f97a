"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step computed (small scene, side blocks off).  Two runs with the
same arguments dump the same values, and `--steps` is the number of steps that really ran before the dump: warm-up 4 + 1 timed
step ends where warm-up 3 + 2 timed steps do, warm-up 3 + 1 timed step one optimiser step earlier."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, warmup, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--points", "20000", "--width", "208", "--height", "128", "--global-batch", "2", "--render-frames", "0",
           "--no-raster-only", "--no-c5", "--no-launcher-path", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    return {os.path.basename(f)[:-4]: np.load(f) for f in glob.glob(os.path.join(str(out), "*.npy"))}


def _frac_changed(a, b):
    """Fraction of elements that differ by more than float32 accumulation-order noise."""
    return float((np.abs(a.astype(np.float64) - b) > 1e-6 * (1.0 + np.abs(b))).mean())


def test_dump_outputs(tmp_path):
    a = _bench(tmp_path / "a", 3, 2)
    assert {"loss", "_xyz", "_features_dc", "_features_rest", "_opacity", "_scaling", "_rotation", "viewspace_grad",
            "max_radii"} <= set(a)
    assert any(".grids." in n for n in a) and any("deform" in n and n.endswith("weight") for n in a)
    assert all(x.dtype in (np.float32, np.float64) and np.isfinite(x).all() for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["_xyz"].shape == (20000, 3) and a["loss"].shape == (1,) and a["loss"][0] > 0
    # same arguments, same inputs: every array agrees file by file (up to the order of float atomics in the backward)
    again = _bench(tmp_path / "again", 3, 2)
    same_total = _bench(tmp_path / "same_total", 4, 1)
    one_less = _bench(tmp_path / "one_less", 3, 1)
    for other in (again, same_total):
        assert set(other) == set(a)
        for n in a:
            assert other[n].shape == a[n].shape, n
            assert _frac_changed(other[n], a[n]) < 1e-2, (n, _frac_changed(other[n], a[n]))
        assert abs(float(other["loss"][0]) - float(a["loss"][0])) <= 1e-5 * float(a["loss"][0])
    # one optimiser step fewer: the parameters and the loss are visibly elsewhere
    assert _frac_changed(one_less["_xyz"], a["_xyz"]) > 0.5
    assert float(one_less["loss"][0]) != float(a["loss"][0])
