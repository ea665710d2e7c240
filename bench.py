#!/usr/bin/env python3
"""Benchmark of the MSM hot path (BASELINE.json: BLS12-377 G1, N = 2^20 points per GPU).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port)

A "step" is one complete MSM over one batch of synthetic input: fresh seeded scalars (a different
pre-generated set every step, as scripts/msm-weierstrass.ts:28-35 draws fresh scalars per run) against
a fixed seeded point set (known-dlog points a_i*G, the construction class of randomPointsFast,
src/curve-random.ts:24-92), result returned to the host as the canonical affine point.

  value   points/s with the scalars already resident in HBM (mgb_msm_device), whole job over all ranks
  e2e     the same through mgb_msm with HOST scalars in pinned memory: H2D of the scalars and D2H of
          the result inside the timed region.  The points stay resident, as they do in the
          reference (its `pointPtr` lives in wasm memory across calls; conversion is excluded from
          its timing, doc/zprize23.md:74).
  N > 1   one process per GPU (torchrun); points/scalars sharded contiguously, 2^20 pairs per GPU
          (weak scaling); each rank computes a partial sum, the partial accumulators are all-gathered
          with NCCL and every rank adds them and normalises (SURVEY.md 8e).

--steps K sets the timed steps of every block of the line; the inputs depend only on the arguments.
--dump-outputs DIR writes the result point of the last timed step of every timed loop as DIR/<name>.npy:
float64 [x limbs, y limbs, isZero], x and y in little-endian 32-bit limbs (exact in float64).  Names:
`msm` (scalars resident, the headline), `msm_e2e` (host scalars), `msm_e2e_pipelined` (host scalars,
prefetched), the same three per `configs` entry and for `strong_2p24` (`<block>`, `<block>_e2e`, ...);
the reference arm writes `msm`.  Two builds run with the same arguments can be compared file by file.

The oracle (oracle/) is used here only for `cpu_baseline` and `--impl reference`.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOGN_DEFAULT = 20
SEED_POINTS = 0x6D6F6E74
SEED_SCALARS = 0x6D6F6E74 ^ 3          # "seed xor config index" (config 4 = index 3)
ALGO_FIELD_MULTS_PER_POINT = 108.6     # SURVEY 8d, BLS12-377 2^20 at the reference's c = 18
MADS_PER_FIELD_MULT = 288              # 2 * 12^2 32x32->64 multiply-accumulates
# The other BASELINE.json configs, reported as `extra` blocks beside the headline (SURVEY 8d table: field
# multiplications per input point at the reference's window size, 32x32->64 MADs per multiplication = 2 * limbs^2)
EXTRA_CONFIGS = {
    "bls377_2p16": {"curve": "bls12-377", "logn": 16, "mults_per_point": 139.0, "mads_per_mult": 288, "seed_index": 0},
    "ed377_2p18": {"curve": "ed-on-bls12-377", "logn": 18, "mults_per_point": 188.0, "mads_per_mult": 128, "seed_index": 1},
    "pallas_2p18": {"curve": "pallas", "logn": 18, "mults_per_point": 142.0, "mads_per_mult": 128, "seed_index": 2},
}
STRONG_LOGN = 24                       # BASELINE config 5: 2^24 pairs in total, sharded over the GPUs of the run
STRONG_MULTS_PER_POINT = 107.5


def workload_config(curve, logn, world):
    """`config` of BOTH arms (the driver compares them): what one step computes."""
    return {"workload": "%s G1 MSM, 2^%d points per GPU, 4 rotating pre-generated scalar sets (a different one every step), points resident" % (curve, logn),
            "l2": "inputs larger than L2 (point table %d MB + scalars %d MB per GPU)" % ((1 << logn) * 144 >> 20, (1 << logn) * 32 >> 20),
            "parallelism": "points sharded x%d, one NCCL all-gather of the partial sums" % world}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--logn", type=int, default=LOGN_DEFAULT, help="log2 of the points per GPU")
    ap.add_argument("--curve", default="bls12-377")
    ap.add_argument("--c", type=int, default=0, help="window bits (0 = engine default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `configs` / `strong_2p24` blocks (the other BASELINE configs)")
    ap.add_argument("--cpu-logn", type=int, default=0,
                    help="log2 size of the CPU baseline sample (0 = the whole workload when the host has >= 8 cores, else 2^18)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result point of the last timed step of every timed loop to DIR/<name>.npy (float64 32-bit limbs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def result_limbs(res, coord_bytes):
    """{x, y, isZero} -> float64 [x limbs, y limbs, isZero], x and y as little-endian 32-bit limbs."""
    limbs = [(v >> (32 * i)) & 0xFFFFFFFF for v in (res["x"], res["y"]) for i in range(coord_bytes // 4)]
    return np.array(limbs + [int(res["isZero"])], dtype=np.float64)


def dump_outputs(out_dir, results):
    """results: {name: (result point, coordinate bytes)} -> out_dir/<name>.npy"""
    os.makedirs(out_dir, exist_ok=True)
    for name, (res, coord_bytes) in results.items():
        np.save(os.path.join(out_dir, name + ".npy"), result_limbs(res, coord_bytes))


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def wait_first_sample(self, timeout=3.0):
        """nvidia-smi takes ~0.1 s to initialise NVML (and holds driver locks meanwhile): the sampler is started before
        the warm-up steps and the timed region only begins once it is in its steady 100 ms polling loop."""
        t_end = time.perf_counter() + timeout
        while self.proc and not self.lines and time.perf_counter() < t_end:
            time.sleep(0.005)

    def stop(self, t0=None, t1=None):
        """Summary of the samples taken in [t0, t1] (perf_counter values bracketing the timed region)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if t1 is not None and not any(t0 <= t <= t1 + 0.1 for t, _ in self.lines):
            time.sleep(0.15)            # region shorter than one polling period: take the sample right after it
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        inside = [ln for t, ln in self.lines if t0 is None or t0 <= t <= t1 + 0.1]
        for ln in inside or [ln for _, ln in self.lines[-1:]]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _measured_peak(key):
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh).get(key)
    except Exception:
        return None


def cpu_sample_logn(args):
    """The CPU arm runs the WHOLE per-GPU workload (one 2^20 MSM is ~2 s on 16 cores, ~30 core-seconds) unless the
    host is too small for that to stay within the bench's time budget."""
    if args.cpu_logn:
        return min(args.logn, args.cpu_logn)
    return args.logn if (os.cpu_count() or 1) >= 8 else min(args.logn, 18)


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel, from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by scripts/summarize_ncu.py traffic); None when absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


def dist_setup(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU BEFORE any pinned host buffer is
    allocated, so that the scalar buffers of the end-to-end path are first-touched on the GPU's own NUMA node (with
    several ranks on one host the uploads otherwise cross the socket interconnect and contend with each other:
    round 1 lost 12 % end to end at 8 GPUs).  Best effort: returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = (cpus & allowed) or allowed
        os.sched_setaffinity(0, cpus)
        return {"bound": True, "cpus": len(cpus), "of": ncpu}
    except Exception as e:      # no NVML, container without the capability, ...
        return {"bound": False, "why": str(e)[:80]}


def cpu_reference_msm(label, points_bytes, scalars, n, threads):
    from oracle import cpu_ref
    res, ms = cpu_ref.msm(label, scalars, points_bytes, n, threads=threads)
    return res, ms


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle/msm_cpu.cpp, a native restatement --
    the reference's own Wasm needs Node, which this image does not have) on all host cores."""
    rank, world, local = dist_setup(args)
    if rank != 0:
        return
    from montgomery_b200 import curves, inputs
    curve = curves.BY_LABEL[args.curve]
    cl = cpu_sample_logn(args)
    n = 1 << cl
    # same seeded known-dlog point set as the GPU arm, generated on the CPU (untimed, like the
    # reference's randomPointsFast before its timed loop); no GPU code runs in this arm
    from oracle import cpu_ref
    threads = os.cpu_count() or 1
    pts = cpu_ref.known_dlog_points(args.curve, SEED_POINTS, n, threads)
    sets = [inputs.random_scalars(curve.q, n, SEED_SCALARS + i) for i in range(min(4, args.steps + args.warmup))]
    times = []
    for i in range(args.warmup + args.steps):
        res, ms = cpu_reference_msm(args.curve, pts, sets[i % len(sets)], n, threads)
        if i >= args.warmup:
            times.append(ms)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"msm": (res, curve.coord_bytes)})
    ms_step = float(np.mean(times))
    value = n / (ms_step * 1e-3)
    sample = ("one MSM of 2^%d points per step (the whole per-GPU workload), %d threads" % (cl, threads)) if cl == args.logn else (
        "one MSM of 2^%d points per step (the first 2^%d of the 2^%d-per-GPU workload), %d threads" % (cl, cl, args.logn, threads))
    line = {
        "impl": "reference", "metric": "msm_points_per_s", "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 limbs (native restatement; the reference computes in 29-bit limbs in i64)", "data": "synthetic",
        "config": workload_config(args.curve, args.logn, args.gpus),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_b200(args):
    import torch
    import montgomery_b200 as m
    from montgomery_b200 import _native, inputs
    import ctypes

    rank, world, local = dist_setup(args)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node = --gpus"
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"bound": False, "why": "single rank"}
    torch.cuda.set_device(local)
    dist = None
    # stdout carries exactly one JSON line: NCCL prints its version banner with a plain printf when a communicator
    # is created (torch's and the engine's own), so file descriptor 1 points at stderr until the line is printed
    sys.stdout.flush()
    saved_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
        torch.cuda.synchronize()
    from montgomery_b200.distributed import ShardedMsm
    from tests.helpers import OracleCurve       # the oracle is the checker of `parity_ok`, never the thing timed

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_ints(v):
        """exact Python ints from every rank -> list on every rank"""
        if not dist:
            return [v]
        out = [None] * world
        dist.all_gather_object(out, v)
        return out

    def measure(label, logn_local, seed_points, seed_scalars, steps, warmup, sampler=None, c=None, nsets=4):
        """Weak-scaling-shaped run of one configuration: 2^logn_local pairs on every rank.  Returns device-resident and
        end-to-end timings, the phase breakdown, and the parity verdict against the closed form over all shards."""
        curve = m.curves.BY_LABEL[label]
        n = 1 << logn_local
        sharded = ShardedMsm(curve, local, n)
        sharded.random_points(n, seed_points)       # rank r: seed + r -> this rank's shard of the global point set
        nsets = min(nsets, steps + warmup)
        np_sets = [inputs.random_scalars(curve.q, n, seed_scalars + 1000 * rank + i) for i in range(nsets)]
        host_sets = [torch.from_numpy(a).pin_memory() for a in np_sets]
        dev_sets = [h.cuda(non_blocking=False) for h in host_sets]
        torch.cuda.synchronize()

        def step(i, e2e, pipelined=False):
            k = i % nsets
            if pipelined:       # the NEXT step's scalars start travelling before this step's MSM is launched
                sharded.prefetch(host_sets[(i + 1) % nsets], n)
            return sharded.msm(host_sets[k] if e2e else dev_sets[k], n, on_device=not e2e, c=c)

        def timed(e2e, smp=None, pipelined=False):
            if smp:
                smp.start()
                smp.wait_first_sample()
            if pipelined:
                sharded.prefetch(host_sets[0], n)
            for i in range(warmup):
                step(i, e2e, pipelined)
            gc.collect()
            gc.disable()                # no collector pauses inside the timed region
            barrier()
            t0 = time.perf_counter()
            phases, launches, res, tm = {}, 0, None, None
            for i in range(steps):
                res, tm = step(warmup + i, e2e, pipelined)
                launches += tm["n_launches"]
                for key in ("h2d_scalars", "decompose_slice", "sort", "accumulate", "reduce", "final_sum", "total"):
                    phases[key] = phases.get(key, 0.0) + tm[key] / steps
            barrier()
            el = time.perf_counter() - t0
            gc.enable()
            clocks = smp.stop(t0, t0 + el) if smp else None
            if pipelined:       # the set uploaded during the last timed step: consume it, so that no prefetch slot stays occupied
                step(warmup + steps, e2e, False)
            t = torch.tensor([el, phases["total"]], dtype=torch.float64, device="cuda")
            if dist:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0].item()), float(t[1].item()), phases, launches, res, tm, clocks

        el, dev_ms_max, phases, launches, res, tm, clocks = timed(False, sampler)
        el_e2e, _, phases_e2e, _, res_e2e, _, _ = timed(True)
        el_pipe, res_pipe, phases_pipe = None, None, None
        if nsets >= 2:          # software-pipelined end to end: the upload of step i + 1 overlaps the MSM of step i
            el_pipe, _, phases_pipe, _, res_pipe, _, _ = timed(True, pipelined=True)
        # parity: the closed form over every rank's shard, for the scalar set of the LAST step of each timed loop
        last = (warmup + steps - 1) % nsets
        ks = gather_ints(inputs.dot_known_dlogs(np_sets[last], inputs.known_dlogs(seed_points + rank, n)))
        O = OracleCurve(label)
        expect = O.result_of(O.scale(sum(ks) % O.q, O.G))
        parity_ok = bool(res == expect and res_e2e == expect and (res_pipe is None or res_pipe == expect))
        out = {"curve": curve, "n": n, "el": el, "el_e2e": el_e2e, "el_pipe": el_pipe, "phases_pipe": phases_pipe, "dev_ms_max": dev_ms_max, "phases": phases, "phases_e2e": phases_e2e,
               "launches": launches, "res": res, "res_e2e": res_e2e, "res_pipe": res_pipe, "tm": tm, "clocks": clocks, "parity_ok": parity_ok,
               "sharded": sharded, "host_sets": host_sets}
        return out

    outputs = {}        # --dump-outputs: the last timed step's result of every timed loop

    def keep_outputs(block, r):
        cb = r["curve"].coord_bytes
        outputs[block] = (r["res"], cb)
        outputs[block + "_e2e"] = (r["res_e2e"], cb)
        if r["res_pipe"] is not None:
            outputs[block + "_e2e_pipelined"] = (r["res_pipe"], cb)

    sampler = ClockSampler(local) if rank == 0 else None
    head = measure(args.curve, args.logn, SEED_POINTS, SEED_SCALARS, args.steps, args.warmup, sampler, c=args.c or None)
    keep_outputs("msm", head)
    curve, n, phases, tm, sharded = head["curve"], head["n"], head["phases"], head["tm"], head["sharded"]
    eng = sharded.engine
    parity_ok = head["parity_ok"]
    ms_step = head["el"] / args.steps * 1e3
    total_points = n * world
    value = total_points / (head["el"] / args.steps)
    e2e_value = total_points / (head["el_e2e"] / args.steps)

    # ---- roofline denominator: the integer-multiply pipe, measured live (BASELINE.md section 2)
    lib = _native.lib()
    ops = ctypes.c_double()
    msb = ctypes.c_float()
    lib.mgb_microbench(local, 3, 2, 1024, 2000, ctypes.byref(ops), ctypes.byref(msb))    # carry-chained IMAD.WIDE.U32.X = one full 32x32+64->64 MAD
    peak_mads = ops.value
    lib.mgb_microbench(local, 0, 2, 1024, 2000, ctypes.byref(ops), ctypes.byref(msb))    # plain IMAD (mad.lo.u32) issue rate
    peak_imad_lo = ops.value
    lib.mgb_microbench(local, 6, 4, 256, 2000, ctypes.byref(ops), ctypes.byref(msb))     # Fp377 Montgomery products, 8 warps per scheduler
    peak_fp377_mults = ops.value

    # ---- the other BASELINE configs (the named size on every GPU of the run, like the headline: weak scaling; the CPU port
    # beside them at N = 1) and config 5 (2^24 in total, every N)
    extra_steps, extra_warm = args.steps, 3
    configs = {}
    cpu_host_threads = os.cpu_count() or 1
    if args.logn == LOGN_DEFAULT and args.curve == "bls12-377" and not args.no_extras:
        sharded.close()
        for name, cfg in EXTRA_CONFIGS.items():
            r = measure(cfg["curve"], cfg["logn"], SEED_POINTS ^ (cfg["seed_index"] + 1), 0x6D6F6E74 ^ cfg["seed_index"], extra_steps, extra_warm)
            keep_outputs(name, r)
            nn = r["n"]
            dev_ms = r["dev_ms_max"]            # slowest rank (= this rank's phases["total"] at N = 1)
            where = "1 GPU" if world == 1 else "per GPU on %d GPUs (weak: %d x 2^%d pairs in total, one all-gather of the partial sums)" % (world, world, cfg["logn"])
            blk = {"workload": "%s MSM, 2^%d points, %s" % (cfg["curve"], cfg["logn"], where), "n_gpus": world, "ms_device": dev_ms,
                   "ms_per_step": r["el"] / extra_steps * 1e3, "points_per_s": nn * world / (r["el"] / extra_steps),
                   "e2e_ms_per_step": r["el_e2e"] / extra_steps * 1e3, "e2e_points_per_s": nn * world / (r["el_e2e"] / extra_steps),
                   "e2e_pipelined_ms_per_step": r["el_pipe"] and r["el_pipe"] / extra_steps * 1e3,
                   "roofline_frac": cfg["mults_per_point"] * cfg["mads_per_mult"] * nn / (dev_ms * 1e-3) / peak_mads,
                   "window_bits": r["tm"]["c"], "windows": r["tm"]["K"], "tree_rounds": r["tm"]["rounds"], "kernels_per_msm": r["tm"]["n_launches"],
                   "phases_ms": r["phases"], "parity_ok": r["parity_ok"]}
            if world == 1 and not args.no_cpu_baseline:
                pts, _ = r["sharded"].engine.get_points(0, nn)
                cres, cms = cpu_reference_msm(cfg["curve"], pts, r["host_sets"][0].numpy(), nn, cpu_host_threads)
                gres, _ = r["sharded"].engine.msm(r["host_sets"][0].numpy(), n=nn)
                blk["cpu_port_ms"] = cms
                blk["cpu_port_cores"] = cpu_host_threads
                blk["cpu_port_agrees_with_gpu"] = bool(cres == gres)
            r["sharded"].close()
            configs[name] = blk
        head_engine_closed = True
    else:
        head_engine_closed = False
    strong = None
    if args.logn == LOGN_DEFAULT and args.curve == "bls12-377" and not args.no_extras and STRONG_LOGN - (world.bit_length() - 1) >= 10 and (world & (world - 1)) == 0:
        if not head_engine_closed:
            sharded.close()
            head_engine_closed = True
        ln = STRONG_LOGN - (world.bit_length() - 1)
        ssteps = args.steps
        r = measure("bls12-377", ln, SEED_POINTS ^ 0x5A5A, 0x6D6F6E74 ^ 4, ssteps, 2, nsets=2)
        keep_outputs("strong_2p24", r)
        tot = (1 << ln) * world
        strong = {"workload": "bls12-377 G1 MSM, 2^%d points in total = 2^%d per GPU on %d GPU(s) (BASELINE config 5)" % (STRONG_LOGN, ln, world),
                  "scaling": "strong", "n_gpus": world, "ms_per_step": r["el"] / ssteps * 1e3, "ms_device_max": r["dev_ms_max"],
                  "points_per_s": tot / (r["el"] / ssteps), "e2e_ms_per_step": r["el_e2e"] / ssteps * 1e3, "e2e_points_per_s": tot / (r["el_e2e"] / ssteps),
                  "e2e_pipelined_ms_per_step": r["el_pipe"] and r["el_pipe"] / ssteps * 1e3,
                  "roofline_frac": STRONG_MULTS_PER_POINT * MADS_PER_FIELD_MULT * (1 << ln) / (r["dev_ms_max"] * 1e-3) / peak_mads,
                  "window_bits": r["tm"]["c"], "windows": r["tm"]["K"], "tree_rounds": r["tm"]["rounds"], "steps": ssteps, "parity_ok": r["parity_ok"]}
        r["sharded"].close()
        parity_ok = parity_ok and r["parity_ok"]
    parity_ok = parity_ok and all(b["parity_ok"] for b in configs.values())

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    algo_mads = ALGO_FIELD_MULTS_PER_POINT * MADS_PER_FIELD_MULT * n        # per GPU per step (reference op counts)
    acc_ms = phases["accumulate"]
    traffic = ncu_traffic() if (args.logn == LOGN_DEFAULT and args.curve == "bls12-377") else None
    achieved = algo_mads / (phases["total"] * 1e-3)
    executed_mults_per_s = 6.0 * tm["n_pairs"] / (acc_ms * 1e-3)
    roofline = {
        "bound": "imad", "achieved": achieved / 1e12, "peak": peak_mads / 1e12, "unit": "T 32x32->64 MAD/s",
        "frac": achieved / peak_mads, "traffic": traffic and traffic.get("bytes_per_launch"),
        "traffic_note": traffic and traffic.get("note"),
        "note": "integer-multiply roofline of BASELINE.md: ALGORITHMIC MADs (the reference's operation count at its own window size: 108.6 field "
                "mults/point x 288) / device time of the whole MSM (CUDA events on the engine's stream) / measured rate of carry-chained "
                "IMAD.WIDE.U32.X (one full 32x32+64->64 MAD per lane) on this GPU; plain IMAD (mad.lo) issues at %.2f T/s, i.e. a full MAD costs "
                "two IMAD slots, as SURVEY 8d assumed.  `dominant_kernel` reports the work the engine actually EXECUTES instead" % (peak_imad_lo / 1e12),
        "dominant_kernel": {"name": "k_batch_add", "phase_ms": acc_ms, "share_of_step": acc_ms / phases["total"],
                            "pairs_per_step": int(tm["n_pairs"]), "executed_field_mults_per_s": executed_mults_per_s,
                            "fp377_mult_peak_per_s": peak_fp377_mults, "frac_of_mult_peak": executed_mults_per_s / peak_fp377_mults,
                            "executed_mads_frac_of_imad_peak": executed_mults_per_s * MADS_PER_FIELD_MULT / peak_mads,
                            "note": "6 field multiplications per affine addition executed by the tree rounds (exact pair count from the engine) against the "
                                    "live-measured throughput of the same Montgomery multiplication with 8 warps per scheduler"},
    }
    # HBM side of the path (north star: "HBM GB/s for the sort and gather phases").  The sort no longer copies points:
    # per sorted entry the scatter reads digit + rank (8 B) and the bucket's offset + count (8 B, L2-resident) and writes
    # a 4-byte point reference (+ half a byte of tree depth); the 96-byte gather of every point happens inside round 0 of
    # k_batch_add, straight from the point table (2 x 96 B read + 96 B written per addition of round 0).
    ent_bytes = 8 + 8 + 4 + 0.5
    hbm = {"sort_scatter_gbs": tm["n_pairs"] and (n * 2 * tm["K"] * ent_bytes) / (phases["sort"] * 1e-3) / 1e9,
           "sort_ms": phases["sort"], "hbm_peak_gbs": _measured_peak("hbm_gbs"),
           "note": "sort = 3 scan kernels + scatter of 4-byte references; latency/atomic-bound, not bandwidth-bound at this size"}
    line = {
        "metric": "msm_points_per_s", "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (12 x 32-bit Montgomery)", "data": "synthetic",
        "config": workload_config(args.curve, args.logn, world),
        "engine": {"window_bits": tm["c"], "windows": tm["K"], "tree_rounds": tm["rounds"], "kernels_per_msm": tm["n_launches"]},
        "parity_ok": parity_ok, "parity": "closed form [(sum s_i a_i) mod q] G over every rank's shard (known-dlog points), checked on the "
                                          "results of the last device-timed and the last end-to-end step of every configuration in this line",
        "msm_ms": ms_step, "msm_ms_device": phases["total"], "phases_ms": phases, "result_x": hex(head["res"]["x"]),
        "e2e": {"value": e2e_value, "unit": "points/s", "ms_per_step": head["el_e2e"] / args.steps * 1e3,
                "h2d_bytes_per_step": n * 32 * world, "d2h_bytes_per_step": (2 * curve.coord_bytes + 4) * world, "phases_ms": head["phases_e2e"],
                "mode": "one blocking call per step: upload this step's scalars (pinned host memory, 4 chunks overlapped with the digit kernel), "
                        "MSM, read the point back",
                "pipelined": head["el_pipe"] and {
                    "value": total_points / (head["el_pipe"] / args.steps), "unit": "points/s", "ms_per_step": head["el_pipe"] / args.steps * 1e3, "phases_ms": head["phases_pipe"],
                    "note": "the same steps with mgb_msm_prefetch: every step still uploads its own scalar set and reads its own result back, but "
                            "the upload of step i+1 is started before the MSM call of step i and overlaps it (what a prover committing to "
                            "several polynomials does)"}},
        "gpu_launches": head["launches"], "clocks": head["clocks"], "roofline": roofline, "hbm_phases": hbm,
        "host_affinity": numa,
    }
    if configs:
        line["configs"] = configs
    if strong:
        line["strong_2p24"] = strong
    if world == 1 and not args.no_cpu_baseline:
        cl = cpu_sample_logn(args)
        ncpu = 1 << cl
        ceng = m.MsmEngine(curve, local, ncpu) if head_engine_closed else eng
        if head_engine_closed:
            ceng.random_points(ncpu, SEED_POINTS)
        pts, _ = ceng.get_points(0, ncpu)
        sc = head["host_sets"][0].numpy()[:ncpu]
        cres, cms = cpu_reference_msm(args.curve, pts, sc, ncpu, cpu_host_threads)
        gres, _ = ceng.msm(sc, n=ncpu)
        line["cpu_baseline"] = {"value": ncpu / (cms * 1e-3), "unit": "points/s", "cores": cpu_host_threads, "kind": "port",
                                "sample": ("one MSM of the whole 2^%d-point workload, %.0f ms" if cl == args.logn else
                                           "one MSM of the first 2^%d points of the workload, %.0f ms") % (cl, cms),
                                "agrees_with_gpu": cres == gres}
        ceng.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    sys.stdout.flush()
    os.dup2(saved_fd, 1)
    os.close(saved_fd)
    print(json.dumps(line))
    sys.stdout.flush()
    if dist:
        dist.destroy_process_group()
    assert parity_ok, "parity check failed: the engine's result differs from the closed form"


def main():
    sys.dont_write_bytecode = True      # the tree bench.py runs from may be read-only: no bytecode caches in it
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
