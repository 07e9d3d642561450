"""Computed measures in region queries and status accessors, on the config-2 cube (3652 days x 32^3 = 1.2e8
cells, the stored measures m_sum, m_average, m_highest with status planes) and the computed measure
(m_sum + m_average) / m_highest.  Workloads (a)-(d) are those of bench_region.py.

  region/eval-sum   olap_region_eval_sum      vs  the host path (getData of the whole cube, numpy sum of the region)
                                              vs  evaluateToStore + regionSum (rounds to float32: speed reference only)
  region/eval-copy  into a float32 target on (b) and (d)
  status/merge      getStatus of the computed measure        vs  the host merge (a Python OR per cell and input)
  status/map        getStatusMap of the computed measure     vs  the host loop (dict work per cell and store)

Kernel times come from olap_last_op_ms() (CUDA events around the kernels of one call), medians over --reps
alternated repetitions after --warmup; wall times are a host clock around the whole call.  Bytes come from
shapes: eval-sum 4kR, eval-copy 4kR + 5R (k inputs, R region cells), merge S*N + N (S bytes per cell of the
inputs' planes), map 2*4*M*N + 17 B per key (M stores: two passes over their values).  Share of peak against
the 6544 GB/s measured HBM peak of the B200 (profiles/membw_r02.json).  The data keep every region sum
finite, so each workload also checks the fused sum against the host path within 1e-12 * sum|v|.  The host
paths are slow: they are run --host-reps times, and the status accessors' host code on a cube of --host-days
days only (the JSON says which size)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from bench_region import PEAK_GBS, card, timed, workloads  # noqa: E402

FORMULA = "(m_sum + m_average) / m_highest"


def build_cube(days_end, store_cls=None):
    from olap_in_memory_b200 import Cube, GenericDimension, TimeDimension

    dims = [TimeDimension("time", "day", "2001-01-01", days_end)] + [
        GenericDimension(g, "item", [f"{g}_{i}" for i in range(32)]) for g in ("g1", "g2", "g3")]
    cube = Cube(dims, store_cls)
    rng = np.random.default_rng(11)
    # m_sum is 30% unset; m_average (NaN default) and the divisor m_highest (>= 1) are set everywhere, so that
    # every region sum of the formula is finite and the fused and host paths can be compared value for value
    for name, default, unset in (("m_sum", 0, 0.3), ("m_average", float("nan"), 0.0), ("m_highest", 0, 0.0)):
        cube.createStoredMeasure(name, {}, "float32", default)
        v = rng.standard_normal(cube.storeSize, dtype=np.float32)
        if name == "m_highest":
            v = 1.0 + np.abs(v)
        v[rng.random(cube.storeSize, dtype=np.float32) < unset] = default
        cube.storedMeasures[name].set_data_f32(v)
    cube.createStoredMeasure("m_target", {}, "float32", 0)
    cube.createComputedMeasure("ratio", FORMULA)
    return cube


def host_path_cls():
    from olap_in_memory_b200.store import GpuStore

    class HostPath(GpuStore):  # Cube keeps its host code for a store class without the device members
        regionEvalSum = regionEvalCopy = statusMerge = statusMap = None

    return HostPath


def med(rows):
    return {k: statistics.median(v) for k, v in rows.items() if v}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-reps", type=int, default=1)
    ap.add_argument("--days-end", default="2010-12-31", help="last day of the time axis (2010-12-31: 3652 days)")
    ap.add_argument("--host-days-end", default="2001-01-31", help="cube on which the status host code is timed")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from olap_in_memory_b200 import _native as N
    from olap_in_memory_b200.cube import _region
    from olap_in_memory_b200.parser import getParser
    from olap_in_memory_b200.store import GpuStore

    N.init(0)
    cube = build_cube(args.days_end)
    host = build_cube(args.days_end, host_path_cls())
    stores = [cube.storedMeasures[m] for m in ("m_sum", "m_average", "m_highest")]
    abs_expr = getParser().parse(f"abs({FORMULA})")
    k = len(stores)
    result = {"card": card(), "cells": cube.storeSize, "formula": FORMULA, "peak_gbs": PEAK_GBS, "reps": args.reps,
              "host_reps": args.host_reps, "workloads": {}}

    for name, f in workloads(cube).items():
        lens, keep = _region(cube.dimensions, f, lambda: None)
        R = int(np.prod([n if q is None else len(q) for n, q in zip(lens, keep)]))

        def composed_sum():  # evaluateToStore + regionSum (the value is rounded to float32 on the way)
            s, _, t1 = timed(lambda: cube.evaluateToStore("ratio"))
            total, _, t2 = timed(lambda: s.regionSum(lens, keep))
            return total, t1 + t2

        copy_too = name in ("b_g1_16_shuffled", "d_no_filter")
        rows = {k_: [] for k_ in ("eval_sum", "eval_sum_wall", "compose_sum", "compose_sum_wall", "eval_copy",
                                  "eval_copy_wall")}
        bits = set()
        for rep in range(args.warmup + args.reps):
            s, wall, ms = timed(lambda: cube.getTotalForDimensionItems("ratio", f))
            assert N.lib().olap_last_op_path().decode() == "region/eval-sum"
            bits.add(np.float64(s).view(np.uint64).item())
            t0 = time.perf_counter()
            _, cms = composed_sum()
            cwall = (time.perf_counter() - t0) * 1e3
            if rep >= args.warmup:
                rows["eval_sum"].append(ms); rows["eval_sum_wall"].append(wall)
                rows["compose_sum"].append(cms); rows["compose_sum_wall"].append(cwall)
            if copy_too:
                _, wall, ms = timed(lambda: cube.copyMeasureData("ratio", "m_target", f))
                assert N.lib().olap_last_op_path().decode() == "region/eval-copy"
                if rep >= args.warmup:
                    rows["eval_copy"].append(ms); rows["eval_copy_wall"].append(wall)
        host_wall, host_value = [], None
        for _ in range(args.host_reps):
            t0 = time.perf_counter()
            host_value = host.getTotalForDimensionItems("ratio", f)
            host_wall.append((time.perf_counter() - t0) * 1e3)
        # sum |v| over the region (one more fused sum) scales the agreement test of the two paths
        abs_sum = GpuStore.regionEvalSum(abs_expr, ["m_sum", "m_average", "m_highest"], stores, lens, keep)
        m = med(rows)
        entry = {"cells": R, "median_ms": m, "min_max_ms": {k_: [min(v), max(v)] for k_, v in rows.items() if v},
                 "same_bits_every_call": len(bits) == 1, "host_path_wall_ms": statistics.median(host_wall),
                 "host_path_sum": host_value, "eval_sum": s, "sum_abs": abs_sum,
                 "host_path_agrees": abs(host_value - s) <= 1e-12 * abs_sum}
        entry["eval_sum_bytes"] = 4 * k * R
        entry["eval_sum_frac_peak"] = 4 * k * R / m["eval_sum"] / 1e6 / PEAK_GBS
        entry["compose_sum_frac_peak_of_eval_bytes"] = 4 * k * R / m["compose_sum"] / 1e6 / PEAK_GBS
        if copy_too:
            entry["eval_copy_bytes"] = 4 * k * R + 5 * R
            entry["eval_copy_frac_peak"] = (4 * k * R + 5 * R) / m["eval_copy"] / 1e6 / PEAK_GBS
        result["workloads"][name] = entry
        print(name, json.dumps(entry), flush=True)

    # ---- status accessors: the device at full size, the host code on a small cube (and the device there too)
    N_cells = cube.storeSize
    rows = {"merge": [], "merge_wall": [], "map": [], "map_wall": []}
    merged = np.empty(N_cells, dtype=np.uint8)
    handles = N.store_array([s._h for s in stores])
    n_keys = 0
    for rep in range(args.warmup + args.reps):
        t0 = time.perf_counter()
        N.check(N.lib().olap_status_merge(handles, k, merged.ctypes.data, N_cells))
        wall = (time.perf_counter() - t0) * 1e3
        ms = N.lib().olap_last_op_ms()
        t0 = time.perf_counter()
        keys, _, _ = GpuStore.statusMap_arrays(list(cube.storedMeasures.values()))
        mwall = (time.perf_counter() - t0) * 1e3
        mms = N.lib().olap_last_op_ms()
        n_keys = int(keys.size)
        if rep >= args.warmup:
            rows["merge"].append(ms); rows["merge_wall"].append(wall)
            rows["map"].append(mms); rows["map_wall"].append(mwall)
    m = med(rows)
    M = len(cube.storedMeasures)
    merge_bytes = k * N_cells + N_cells  # every input has a status plane (1 byte per cell)
    map_bytes = 2 * 4 * M * N_cells + 17 * n_keys
    status = {"cells": N_cells, "median_ms": m, "merge_bytes": merge_bytes,
              "merge_frac_peak": merge_bytes / m["merge"] / 1e6 / PEAK_GBS, "map_stores": M, "map_keys": n_keys,
              "map_bytes": map_bytes, "map_frac_peak": map_bytes / m["map"] / 1e6 / PEAK_GBS}

    small, small_host = build_cube(args.host_days_end), build_cube(args.host_days_end, host_path_cls())
    sw = {"merge_device": [], "merge_host": [], "map_device": [], "map_host": []}
    for _ in range(args.host_reps):
        for key, fn in (("merge_device", lambda: small.getStatus("ratio")), ("merge_host", lambda: small_host.getStatus("ratio")),
                        ("map_device", lambda: small.getStatusMap("ratio")), ("map_host", lambda: small_host.getStatusMap("ratio"))):
            t0 = time.perf_counter()
            out = fn()
            sw[key].append((time.perf_counter() - t0) * 1e3)
            sw.setdefault(key + "_len", len(out))
    status["host_code_size"] = {"cells": small.storeSize, "days_end": args.host_days_end,
                                "wall_ms": {k_: statistics.median(v) for k_, v in sw.items() if isinstance(v, list)},
                                "same_result": small.getStatus("ratio") == small_host.getStatus("ratio")
                                and list(small.getStatusMap("ratio")) == list(small_host.getStatusMap("ratio"))}
    result["status"] = status
    print("status", json.dumps(status), flush=True)

    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
