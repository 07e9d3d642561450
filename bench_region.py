"""Region queries on the config-2 cube (3652 days x 32^3 = 1.2e8 cells, 3 float32 measures with status
planes): the region kernel (olap_region_sum / olap_region_copy) against the compositions of existing kernels
that compute the same thing, timed alternately in the same process.

  sum:  region/sum                vs  dice + total (one total_kernel pass gives the sum AND the count of set
                                      cells, which the NaN-default rule needs: sum + (R - count) * default)
  copy: region/copy               vs  dice + load (scatter of the diced region back into the target)

Workloads: (a) one month of days, (b) g1 filtered to 16 of 32 items in shuffled order, (c) the innermost g3
filtered to every other item, (d) no filter.  Kernel times come from olap_last_op_ms() (CUDA events around the
kernels of one call, table uploads excluded), medians over --reps alternated repetitions after --warmup; the
wall time is a host clock around the whole call (lowering, allocation, synchronisation).  Bytes are what the
region needs: 4R read for the sum, 4R read + 5R written for the copy; share of peak against the 6544 GB/s
measured HBM peak of the B200 (profiles/membw_r02.json).  The 480 MB plane is larger than the 126 MB L2.

The per-cell host loop the kernel replaced is timed on (a) only (--host-loop); the other workloads say
"not measured"."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PEAK_GBS = 6544.0


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def build_cube(days_end):
    from olap_in_memory_b200 import Cube, GenericDimension, TimeDimension

    dims = [TimeDimension("time", "day", "2001-01-01", days_end)] + [
        GenericDimension(g, "item", [f"{g}_{i}" for i in range(32)]) for g in ("g1", "g2", "g3")]
    cube = Cube(dims)
    rng = np.random.default_rng(11)
    for k, default in enumerate((0, float("nan"), 0)):
        name = f"m{k}"
        cube.createStoredMeasure(name, {}, "float32", default)
        v = rng.standard_normal(cube.storeSize, dtype=np.float32)
        v[rng.random(cube.storeSize, dtype=np.float32) < 0.3] = default
        cube.storedMeasures[name].set_data_f32(v)
    return cube


def workloads(cube):
    rng = np.random.default_rng(5)
    days = cube.dimensions[0].getItems()
    g1 = [f"g1_{i}" for i in rng.permutation(32)[:16]]
    return {
        "a_one_month": {"time": [d for d in days if d.startswith(days[0][:7])]},
        "b_g1_16_shuffled": {"g1": g1},
        "c_g3_every_other": {"g3": [f"g3_{i}" for i in range(0, 32, 2)]},
        "d_no_filter": {},
    }


def timed(fn):
    from olap_in_memory_b200 import _native as N

    t0 = time.perf_counter()
    out = fn()
    return out, (time.perf_counter() - t0) * 1e3, N.lib().olap_last_op_ms()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--days-end", default="2010-12-31", help="last day of the time axis (2010-12-31: 3652 days)")
    ap.add_argument("--host-loop", action="store_true", help="also time the per-cell host loop on (a)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from olap_in_memory_b200 import _native as N
    from olap_in_memory_b200.cube import _region
    from olap_in_memory_b200.store import GpuStore

    N.init(0)
    cube = build_cube(args.days_end)
    src, other, dst = (cube.storedMeasures[m] for m in ("m0", "m1", "m2"))
    result = {"card": card(), "cells": cube.storeSize, "peak_gbs": PEAK_GBS, "reps": args.reps, "workloads": {}}

    for name, f in workloads(cube).items():
        lens, keep = _region(cube.dimensions, f, lambda: None)
        R = int(np.prod([n if k is None else len(k) for n, k in zip(lens, keep)]))
        dice_keep = [list(range(n)) if k is None else k.tolist() for n, k in zip(lens, keep)]

        def region_sum():
            return other.regionSum(lens, keep)

        def composed_sum():  # dice + one total_kernel pass (sum and count of set cells)
            ms = 0.0
            diced, _, t = timed(lambda: GpuStore.dice_lowered([other], lens, dice_keep)[0])
            ms += t
            total, _, t = timed(lambda: diced.total)
            ms += t
            return total, ms

        def region_copy():
            dst.regionCopy(src, lens, keep)

        def composed_copy():  # dice + load back into the target
            ms = 0.0
            diced, _, t = timed(lambda: GpuStore.dice_lowered([src], lens, dice_keep)[0])
            ms += t
            _, _, t = timed(lambda: dst.load_lowered(diced, lens, [len(k) for k in dice_keep], dice_keep))
            ms += t
            return ms

        copy_too = name in ("b_g1_16_shuffled", "d_no_filter")
        rows = {"region_sum": [], "compose_sum": [], "region_sum_wall": [], "compose_sum_wall": [],
                "region_copy": [], "compose_copy": [], "region_copy_wall": [], "compose_copy_wall": []}
        bits = set()
        for rep in range(args.warmup + args.reps):
            s, wall, ms = timed(region_sum)
            bits.add(np.float64(s).view(np.uint64).item())
            t0 = time.perf_counter()
            _, cms = composed_sum()
            cwall = (time.perf_counter() - t0) * 1e3
            if rep >= args.warmup:
                rows["region_sum"].append(ms); rows["region_sum_wall"].append(wall)
                rows["compose_sum"].append(cms); rows["compose_sum_wall"].append(cwall)
            if copy_too:
                _, wall, ms = timed(region_copy)
                t0 = time.perf_counter()
                cms = composed_copy()
                cwall = (time.perf_counter() - t0) * 1e3
                if rep >= args.warmup:
                    rows["region_copy"].append(ms); rows["region_copy_wall"].append(wall)
                    rows["compose_copy"].append(cms); rows["compose_copy_wall"].append(cwall)
        med = {k: statistics.median(v) for k, v in rows.items() if v}
        spread = {k: [min(v), max(v)] for k, v in rows.items() if v}
        entry = {"cells": R, "median_ms": med, "min_max_ms": spread,
                 "same_bits_every_call": len(bits) == 1}
        sum_bytes = 4 * R
        entry["sum_bytes"] = sum_bytes
        entry["region_sum_gbs"] = sum_bytes / med["region_sum"] / 1e6
        entry["region_sum_frac_peak"] = entry["region_sum_gbs"] / PEAK_GBS
        entry["compose_sum_frac_peak_of_region_bytes"] = sum_bytes / med["compose_sum"] / 1e6 / PEAK_GBS
        if name == "c_g3_every_other":
            # every other cell of the innermost axis: the kernel touches every 32-byte sector of the plane
            entry["physical_bytes"] = 4 * cube.storeSize
            entry["region_sum_frac_peak_physical"] = 4 * cube.storeSize / med["region_sum"] / 1e6 / PEAK_GBS
        if copy_too:
            entry["copy_bytes"] = 9 * R
            entry["region_copy_frac_peak"] = 9 * R / med["region_copy"] / 1e6 / PEAK_GBS
        entry["host_loop_ms"] = "not measured"
        result["workloads"][name] = entry
        print(name, json.dumps(entry), flush=True)

    if args.host_loop:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from test_region_queries import loop_getTotalForDimensionItems

        f = workloads(cube)["a_one_month"]
        t0 = time.perf_counter()
        want = loop_getTotalForDimensionItems(cube, "m0", f)
        loop_ms = (time.perf_counter() - t0) * 1e3
        got = cube.getTotalForDimensionItems("m0", f)
        result["workloads"]["a_one_month"]["host_loop_ms"] = loop_ms
        result["workloads"]["a_one_month"]["host_loop_matches"] = (got != got and want != want) or abs(got - want) <= 1e-9 * max(1, abs(want))
        print("host loop (a):", loop_ms, "ms", flush=True)

    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
