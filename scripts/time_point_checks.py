"""Cost of checked point ingestion: mgb_set_points against mgb_set_points_checked, and the k_check_points kernel.

    python scripts/time_point_checks.py [--out FILE.jsonl]              wall clock of the blocking calls
    python scripts/time_point_checks.py --profile [--out FILE.jsonl]    k_check_points kernel time (torch.profiler)

Wall clock: per curve at 2^20 points (BLS12-377 also at 2^22), both calls alternately from the same pageable bytes
(made by mgb_random_points + mgb_get_points), 2 warm-ups, then 7 repeats each; the median is reported.  The profile run is
separate (tracing slows the host) and reports the device time of k_check_points against the measured product peak of
profiles/r01_microbench.jsonl.  Products per point are counted from the chains (montgomery_b200/gen_constants.py).
Every line printed is one JSON record; the first names the card, its power limit and its maximum SM clock.
"""
import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import montgomery_b200 as m  # noqa: E402

# field products of the group-law pieces (ec.cuh): XYZZ doubling 9, mixed XYZZ + affine addition 10; twisted Edwards
# unified addition / doubling 9, mixed addition 7
W_DBL, W_MADD, TE_ADD, TE_MADD = 9, 10, 9, 7
Z = {"bls12-377": (0x8508C00000000001, True), "bls12-381": (0xD201000000010000, False)}


def products_per_point(label):
    spec = importlib.util.spec_from_file_location("gen_constants", os.path.join(ROOT, "montgomery_b200", "gen_constants.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    if label == "pallas":
        return 3                                        # y^2, x^2, x^3: the curve equation only (cofactor 1)
    if label == "ed-on-bls12-377":
        pos, neg = gen.naf_masks(m.curves.ED_ON_BLS12_377.q)
        top = pos.bit_length() - 1
        adds = bin(pos).count("1") + bin(neg).count("1") - 1
        return 4 + 1 + top * TE_ADD + adds * TE_MADD    # curve equation, T = xy, 250 doublings + 87 mixed additions
    z, beta_sq = Z[label]
    z2 = z * z
    chain = (z2.bit_length() - 1) * W_DBL + (bin(z2).count("1") - 1) * W_MADD
    return 3 + chain + W_MADD + (1 if beta_sq else 0) + 2   # curve equation, [z^2] P, - P, beta', two cross products


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                              # noqa: BLE001 -- reported, not hidden
        return {"gpu": "unknown (%s)" % e}


def peaks():
    """measured product rates (products per second) of profiles/r01_microbench.jsonl: Fp377 (12 limbs), Fr377 (8 limbs)"""
    rates = {}
    with open(os.path.join(ROOT, "profiles", "r01_microbench.jsonl")) as fh:
        for line in fh:
            r = json.loads(line)
            if r.get("mode") in (4, 5):
                rates[12 if r["mode"] == 4 else 8] = r["ops_per_s"]
    return rates


CASES = [("bls12-377", 20), ("bls12-377", 22), ("pallas", 20), ("ed-on-bls12-377", 20), ("bls12-381", 20)]


def emit(rec, fh):
    line = json.dumps(rec)
    print(line, flush=True)
    if fh:
        fh.write(line + "\n")


def wall_clock(fh):
    for label, logn in CASES:
        cv = m.curves.BY_LABEL[label]
        n = 1 << logn
        eng = m.MsmEngine(cv, 0, n)
        eng.random_points(n, seed=1)
        xy, z = eng.get_points(0, n)
        xy = xy.reshape(-1).copy()                      # pageable host bytes
        t = {False: [], True: []}
        for rep in range(9):
            for check in (False, True):
                t0 = time.perf_counter()
                eng.set_points(xy, z, check=check)
                dt = (time.perf_counter() - t0) * 1e3
                if rep >= 2:
                    t[check].append(dt)
        eng.close()
        plain, checked = statistics.median(t[False]), statistics.median(t[True])
        emit({"label": label, "n": n, "set_points_ms": round(plain, 2), "set_points_checked_ms": round(checked, 2),
              "extra_ms": round(checked - plain, 2), "products_per_point": products_per_point(label), "repeats": 7}, fh)


def profile(fh):
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity
    rates = peaks()
    for label, logn in CASES:
        cv = m.curves.BY_LABEL[label]
        n = 1 << logn
        eng = m.MsmEngine(cv, 0, n)
        eng.random_points(n, seed=1)
        xy, z = eng.get_points(0, n)
        eng.set_points(xy, z, check=True)               # warm-up
        with torch.profiler.profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                eng.set_points(xy, z, check=True)
        eng.close()
        times = [e.time_range.elapsed_us() for e in prof.events() if "k_check_points" in e.name and e.device_type == DeviceType.CUDA]
        assert len(times) == 3, [e.name for e in prof.events()][:20]
        us = statistics.median(times)
        prod = products_per_point(label) * n
        nl = cv.coord_bytes // 4
        rate = prod / (us * 1e-6)
        emit({"label": label, "n": n, "k_check_points_ms": round(us / 1e3, 3), "products": prod,
              "products_per_s": round(rate / 1e9, 2), "unit": "G/s",
              "share_of_measured_product_peak": round(rate / rates[12 if nl == 12 else 8], 3),
              "peak_G_per_s": round(rates[12 if nl == 12 else 8] / 1e9, 1)}, fh)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    fh = open(a.out, "a") if a.out else None
    emit(dict(card(), run="profile" if a.profile else "wall_clock"), fh)
    (profile if a.profile else wall_clock)(fh)
    if fh:
        fh.close()


if __name__ == "__main__":
    main()
