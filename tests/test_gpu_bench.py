"""bench.py on the device at a small batch: `--steps` sets the timed steps of the device-resident and the end-to-end
loops, and `--dump-outputs` writes the filters the timed steps designed (B200 only)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_filters_of_the_timed_batch(tmp_path):
    import bench
    import emagls_b200 as em
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0",
                        "--orient", "8", "--no-render", "--no-cpu-baseline", "--no-spot-check",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2
    assert sorted(os.listdir(out)) == ["wL.npy", "wR.npy"]
    pr = bench.problem(0, 8)
    wL, wR = em.getEMagLs2Filters(pr["hL"], pr["hR"], pr["az"], pr["ze"], pr["r"], pr["maz"], pr["mze"], bench.ORDER,
                                  pr["fs"], bench.LEN, rotations=pr["R"])
    for name, ref in (("wL", wL), ("wR", wR)):
        got = np.load(out / f"{name}.npy")
        assert got.dtype == np.float64 and got.shape == (8, 32, bench.LEN)      # the whole batch: 8 < DUMP_SETS
        ref = ref.transpose(2, 1, 0)
        assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max(), name
