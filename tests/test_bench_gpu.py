"""bench.py's CUDA arm at a small size: `--steps` sets the number of timed steps and `--dump-outputs` writes the result point
of the last timed step of each timed loop (scalars resident, host scalars, host scalars prefetched).  The scalar set of
that step depends on warmup + steps, so the closed form of its inputs checks both."""
import json
import os
import subprocess
import sys

import pytest

import bench
from montgomery_b200 import inputs
from tests.helpers import OracleCurve, dumped_point

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cuda_arm_steps_and_dumped_outputs(tmp_path):
    logn, steps, warmup = 12, 3, 1
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--logn", str(logn), "--steps", str(steps),
                          "--warmup", str(warmup), "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, env=env)
    assert res.returncode == 0, res.stderr[-4000:]
    line = json.loads(res.stdout.strip())
    assert line["steps"] == steps and line["parity_ok"]
    n = 1 << logn
    last = (warmup + steps - 1) % min(4, warmup + steps)           # bench.py rotates over min(4, warmup + steps) scalar sets
    O = OracleCurve("bls12-377")
    k = inputs.dot_known_dlogs(inputs.random_scalars(O.q, n, bench.SEED_SCALARS + last), inputs.known_dlogs(bench.SEED_POINTS, n))
    expect = O.result_of(O.scale(k % O.q, O.G))
    assert sorted(os.listdir(tmp_path)) == ["msm.npy", "msm_e2e.npy", "msm_e2e_pipelined.npy"]
    for f in os.listdir(tmp_path):
        assert dumped_point(tmp_path / f, 48) == expect, f
