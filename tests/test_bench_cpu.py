"""CPU checks of bench.py's contract for the reference arm (`--impl reference`: the CPU restatement of the reference
algorithm, oracle/msm_cpu.cpp, timed on the host cores): one JSON line with the keys the driver reads, the same `config`
/ metric / unit as the CUDA arm prints for the same arguments, rank 0 alone working under a multi-rank launch.  The
CUDA arm itself needs a GPU (tests/test_gpu_*.py, profiles/r02_bench*.json)."""
import json
import os
import subprocess
import sys

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, *args):
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--logn", "11", "--steps", "2", "--warmup", "1", *args],
                          capture_output=True, text=True, timeout=300, env=env)


def test_reference_arm_prints_the_contract_line():
    res = _run()
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "msm_points_per_s" and line["unit"] == "points/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 1
    assert line["value"] > 0 and abs(line["value"] - (1 << 11) / (line["ms_per_step"] * 1e-3)) < 1e-6 * line["value"]
    # the driver compares the two arms' config: it is built by the same function from the same arguments
    assert line["config"] == bench.workload_config("bls12-377", 11, 1)
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == line["value"] and "2^11" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["vs_baseline"] is None


def test_reference_arm_dumps_the_last_step(tmp_path):
    """--dump-outputs: the result of the last timed step (set (warmup + steps - 1) mod 3 of the seeded scalar sets against
    the seeded known-dlog points), which must be the closed form of those inputs"""
    from montgomery_b200 import inputs
    from tests.helpers import OracleCurve, dumped_point
    res = _run(None, "--dump-outputs", str(tmp_path / "out"))
    assert res.returncode == 0, res.stderr[-2000:]
    assert os.listdir(tmp_path / "out") == ["msm.npy"]
    O = OracleCurve("bls12-377")
    n = 1 << 11
    k = inputs.dot_known_dlogs(inputs.random_scalars(O.q, n, bench.SEED_SCALARS + 2), inputs.known_dlogs(bench.SEED_POINTS, n))
    assert dumped_point(tmp_path / "out" / "msm.npy", 48) == O.result_of(O.scale(k % O.q, O.G))


def test_reference_arm_under_a_multi_rank_launch():
    """torchrun starts one process per GPU; rank 0 alone runs and prints, the others exit 0 without work"""
    quiet = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert quiet.returncode == 0 and quiet.stdout.strip() == ""
    lead = _run({"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"}, "--gpus", "2")
    assert lead.returncode == 0, lead.stderr[-2000:]
    line = json.loads(lead.stdout.strip())
    assert line["n_gpus"] == 2 and line["config"] == bench.workload_config("bls12-377", 11, 2)
