"""bench.py --dump-outputs: the dump is what the last timed step left in its buffer.  It is the same from run to run, and
it equals the oracle's cascade over the same sequence of steps (warm-up, then --steps timed steps on the rotating buffers,
filter state carried), so no step is missing.  One extra timed step would process another buffer and leave the dump as it
is; the launch count of the timed window (one cascade launch per step) shows that there is none."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FS = 96000.0
CN, T, WARMUP = 512, 384, 3                 # small enough that the dump holds every channel


def _bench(out_dir, arith, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--arith", arith, "--channels", str(CN), "--frames", str(T),
           "--steps", str(steps), "--warmup", str(WARMUP), "--no-e2e", "--no-cpu", "--no-extras", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == steps
    return np.load(os.path.join(out_dir, "eq_out.npy"))


def _oracle_run(oracle, arith, steps):
    from dspi_b200 import api, workloads as W
    q = arith == "q28"
    bq = api.compute_coefficients(W.eq_params_fast("B" if q else "A", CN, fs=FS, seed=1), q28=q, fs=FS)
    nbuf = max(2, min(4, steps))
    x = (W.inputs_q28 if q else W.inputs_f32)(CN, nbuf * T)
    bufs = [x[:, b * T:(b + 1) * T].copy() for b in range(nbuf)]
    for i in list(range(WARMUP)) + list(range(steps)):
        oracle.eq_many(arith, bq, bufs[i % nbuf], 10, 96)
    return bufs[(steps - 1) % nbuf]


@pytest.mark.parametrize("arith,steps", [("f32f", 2), ("q28", 3)])
def test_dump_is_the_last_timed_step(tmp_path, oracle, arith, steps):
    got = _bench(tmp_path / "a", arith, steps)
    assert got.dtype == (np.float64 if arith == "q28" else np.float32) and got.shape == (CN, T)
    want = _oracle_run(oracle, arith, steps)
    if arith == "q28":
        assert np.array_equal(got, want.astype(np.float64))
    else:
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    again = _bench(tmp_path / "b", arith, steps)
    assert np.array_equal(got.view(np.uint8), again.view(np.uint8))
