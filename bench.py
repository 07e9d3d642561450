#!/usr/bin/env python
"""bench.py — drillUp throughput of the cube-transform hot path on B200.

A "step" is one pass of the hot path over one batch of synthetic input: the config-2
cube of BASELINE.json (time day x3652, 3 generic dims x32 -> 119 668 736 cells, 3 stored
measures with time rules sum / average / highest, 1 computed measure) is drilled up
day -> month (one batched olap_drill_up call for the 3 measures) and the computed
measure `(m_sum + m_avg) / m_max` is evaluated on the result by the JIT-fused kernel.

  value   : measure-cells/s (M x N_in / t) with the cube resident in HBM
  e2e     : the same metric through the public Cube API with HOST buffers: every step
            uploads the 3 measures from pinned host memory, runs the step and downloads
            the 4 result planes
  roofline: the drillUp kernel's algorithmic bytes / its CUDA-event duration, against
            the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline / --impl reference: the reference's algorithm (oracle/olap_oracle.c, a
            plain-C restatement of src/store/in-memory.js) on the host cores, on a
            bounded sample of the same workload.

Launch:  python bench.py [--gpus N --steps K --warmup W].  N = 1 runs config 2 (the
configuration the metric is quoted on).  For N > 1, under torchrun with one rank per GPU,
the step is config 4 of BASELINE.json: ONE univac-style cube (10 dimensions x 10 items =
1e10 cells, 3 stored measures) sharded by rows of (dim0, dim1) across the N ranks — strong
scaling, fixed total cells — and a step rolls up an inner dimension (dim9 -> all, shard-local,
HBM-bound) AND the sharded dimension (dim0 -> all: every rank computes its own output rows,
reading the child rows out of its peers' stores over NVLink inside the rollup kernel).  A
sharded-vs-single-cube parity guard runs on the devices before anything is timed.

  --dump-outputs DIR (N = 1): after the timed steps, the 4 result planes of the last one go to
  DIR/<name>.npy, so that two builds can be compared output for output on identical inputs."""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TIME_START, TIME_END = "2010-01-01", "2019-12-31"
GENERIC = 32
METHODS = ("sum", "average", "highest")
SHARDED_METHODS = ("sum", "average", "highest")  # rules of the three measures of the N > 1 cube, on every dimension
NVLINK_GBS = 770.0  # B200_PROFILING.md: measured peer copy per direction per GPU (900 nominal)
FORMULA = "(m_sum + m_avg) / m_max"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


# ------------------------------------------------------------------ synthetic data
def splitmix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def synth(out, seed, measure, start=0):
    """SURVEY.md §8d generator: float32 values uniform in [1, 1000), never 0 / NaN."""
    n = out.size
    chunk = 1 << 24
    with np.errstate(over="ignore"):
        for lo in range(0, n, chunk):
            hi = min(n, lo + chunk)
            idx = np.arange(start + lo, start + hi, dtype=np.uint64)
            h = splitmix64(idx ^ np.uint64(seed) ^ (np.uint64(measure) << np.uint64(40)))
            out[lo:hi] = (1.0 + (h >> np.uint64(40)).astype(np.float64) * (999.0 / (1 << 24))).astype(np.float32)
    return out


class Clocks(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML every ~2 ms while the
    timed regions run (the nvidia-smi CLI is too slow for sub-second regions)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.reasons, self.max_mhz = index, [], 0, None
        self.stop_flag = threading.Event()
        self.busy = threading.Event()  # set while a timed region is running

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception:
            return
        while not self.stop_flag.is_set():
            if self.busy.is_set():
                try:
                    self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    self.reasons |= int(get_reasons(h))
                except Exception:
                    pass
            time.sleep(0.002)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=2)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                "hw_power_brake_slowdown": 0x80}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": self.max_mhz, "reasons": [k for k, v in bits.items() if self.reasons & v],
                "samples": len(sm)}


# ------------------------------------------------------------------ CPU arm (oracle port)
def cpu_port_run(steps, warmup, threads, inner):
    """The reference's drillUp algorithm on host cores: each thread owns an independent
    sub-cube [3652 days x inner] per measure and rolls it up day -> month.  inner = 4096
    gives 14.96 M cells per measure, just under the 2^24-entry limit of the JS Map the
    reference keeps its cells in (SURVEY.md F5)."""
    from olap_in_memory_b200 import TimeDimension
    from oracle.c_oracle import COracleStore

    day = TimeDimension("time", "day", TIME_START, TIME_END)
    month_map = np.asarray(day.getGroupIndexFromRootIndexMap("month"), dtype=np.int32)
    C, P, I = day.numItems, 120, inner
    n = C * I
    ident = np.arange(I, dtype=np.int32)
    stores = []
    for t in range(threads):
        per = []
        for m, _ in enumerate(METHODS):
            s = COracleStore(n, "float32", 0.0)
            s.set_data_f32(synth(np.empty(n, np.float32), 1 + t, m))
            per.append(s)
        stores.append(per)

    def work(t):
        for s, method in zip(stores[t], METHODS):
            s.drillUp_lowered([C, I], [P, I], [month_map, ident], method)

    def one_step():
        ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()

    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = (time.perf_counter() - t0) / max(1, steps)
    cells = threads * len(METHODS) * n
    sample = (f"drillUp day->month of [3652 x {I}] cells x {len(METHODS)} measures (sum/average/highest) per thread, "
              f"{threads} independent sub-cubes, C port of in-memory.js:265-334 (ordered hash map)")
    return cells / dt, dt * 1e3, sample


REFERENCE_THREADS = 16  # fixed, so that BENCH and SCALE boxes (16 / 32 host threads) time the same baseline


def cpu_port_run_univac(steps, warmup, threads, ndims=6):
    """The reference's algorithm on the N > 1 workload: each thread owns a univac-style sub-cube
    (ndims dimensions x 10 items) x 3 measures and rolls up its innermost dimension and dim0."""
    from oracle.c_oracle import COracleStore

    lens = [10] * ndims
    n = 10 ** ndims
    ident = [np.arange(10, dtype=np.int32) for _ in lens]
    zeros = np.zeros(10, dtype=np.int32)
    stores = []
    for t in range(threads):
        per = []
        for m, _ in enumerate(SHARDED_METHODS):
            st = COracleStore(n, "float32", 0.0)
            st.set_data_f32(synth(np.empty(n, np.float32), 1 + t, m))
            per.append(st)
        stores.append(per)

    def work(t):
        for st, method in zip(stores[t], SHARDED_METHODS):
            st.drillUp_lowered(lens, lens[:-1] + [1], ident[:-1] + [zeros], method)
            st.drillUp_lowered(lens, [1] + lens[1:], [zeros] + ident[1:], method)

    def one_step():
        ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()

    for _ in range(warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = (time.perf_counter() - t0) / max(1, steps)
    cells = 2 * threads * len(SHARDED_METHODS) * n
    sample = (f"drillUp dim{ndims - 1}->all and dim0->all of a [10]^{ndims} = {n}-cell cube x {len(SHARDED_METHODS)} measures "
              f"({'/'.join(SHARDED_METHODS)}) per thread, {threads} independent sub-cubes, C port of in-memory.js:265-334 "
              f"(ordered hash map)")
    return cells / dt, dt * 1e3, sample


def run_reference(args, rank):
    """The reference's own algorithm (C port of in-memory.js, oracle/) on the host cores, on a
    bounded SAMPLE of this arm's workload — the sample, not the full config, is what
    `config.workload` names.  Warm-up as asked (at least one step, so that first-touch page
    faults stay out of the timed region); the thread count is fixed and printed."""
    if rank != 0:
        return
    threads = max(1, min(os.cpu_count() or 1, REFERENCE_THREADS))
    warmup = max(1, args.warmup)
    steps = max(1, args.steps)
    if args.gpus > 1:
        value, ms, sample = cpu_port_run_univac(steps, warmup, threads)
        config = sharded_config(args.gpus)
    else:
        value, ms, sample = cpu_port_run(steps, warmup, threads, 512)
        config = workload_config()
    config = dict(config)
    config["full_workload"] = config["workload"]
    config["workload"] = "SAMPLE of the arm's workload (the reference keeps cells in a JS Map capped at 2^24 entries): " + sample
    line = {
        "impl": "reference", "metric": "drillUp input measure-cells/s", "value": value, "unit": "cells/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config,
        "cpu_baseline": {"value": value, "unit": "cells/s", "cores": threads, "kind": "port", "sample": sample,
                         "host_threads_available": os.cpu_count()},
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config():
    return {"workload": "config 2: cube [time day x3652, g1 x32, g2 x32, g3 x32] = 119668736 cells, 3 stored float32 "
                        "measures (time rules sum/average/highest) + 1 computed measure; drillUp time day->month "
                        "-> 3932160 cells; per-measure status plane (5 B/cell)",
            "cells_in": 3652 * GENERIC ** 3, "cells_out": 120 * GENERIC ** 3, "measures": 3, "computed": FORMULA,
            "l2": "inputs (2.4 GB) exceed the 126 MB L2, no flush needed", "sharding": "single GPU"}


def sharded_config(world, ndims=None):
    ndims = ndims or int(os.environ.get("OLAP_BENCH_NDIMS", "10"))
    n = 10 ** ndims
    return {"workload": f"config 4: univac-style cube of {ndims} dimensions x 10 items = {n} cells, 3 stored float32 measures "
                        f"(rules {'/'.join(SHARDED_METHODS)} on every dimension), per-measure status plane (5 B/cell), ONE cube "
                        f"sharded by rows of (dim0, dim1) across {world} GPUs; a step = drillUp dim{ndims - 1}->all (shard-local) + "
                        f"drillUp dim0->all (the sharded dimension: peer-memory pull over NVLink inside the rollup kernel)",
            "cells_in": n, "measures": 3, "ops_per_step": 2, "ndims": ndims,
            "l2": "per-GPU inputs exceed the 126 MB L2, no flush needed",
            "sharding": f"strong scaling: fixed {n}-cell cube, rows of (dim0, dim1) split over {world} ranks",
            "note": "N = 1 runs config 2 (the metric's own configuration); compare the N = 2, 4, 8 lines with one another"}


def dump_outputs(directory, arrays):
    """--dump-outputs: DIR/<name>.npy for every array the timed step hands its caller.  The inputs
    come from synth() with fixed seeds, so two builds run with the same arguments can be compared
    file by file.  Config 2 gives 4 float32 planes of 120 x 32^3 cells: 62.9 MB in all, written whole."""
    os.makedirs(directory, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), arr)


# ------------------------------------------------------------------ GPU arm
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from olap_in_memory_b200 import Cube, GenericDimension, TimeDimension
    from olap_in_memory_b200 import _native as N

    torch.cuda.set_device(local_rank)
    N.init(local_rank)
    lib = N.lib()
    stream = torch.cuda.Stream()
    N.check(lib.olap_set_stream(stream.cuda_stream))

    dims = [TimeDimension("time", "day", TIME_START, TIME_END)] + [
        GenericDimension(f"g{k}", "root", [f"g{k}-{i}" for i in range(GENERIC)]) for k in (1, 2, 3)]
    cube = Cube(dims)
    names = ["m_sum", "m_avg", "m_max"]
    for name, rule in zip(names, METHODS):
        cube.createStoredMeasure(name, {"time": rule}, "float32", 0)
    cube.createComputedMeasure("ratio", FORMULA)
    n_in = cube.storeSize
    n_out = 120 * GENERIC ** 3

    # pinned host buffers (the e2e path copies from / to these every step)
    import ctypes as C

    def pinned(n_floats):
        p = C.c_void_p()
        N.check(lib.olap_host_alloc(n_floats * 4, C.byref(p)))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(n_floats,)), p

    host_in, host_out, keep = [], [], []
    for m, name in enumerate(names):
        arr, p = pinned(n_in)
        synth(arr, 1 + rank, m)
        host_in.append(arr)
        keep.append(p)
        cube.setData(name, arr)
    for _ in range(4):
        arr, p = pinned(n_out)
        host_out.append(arr)
        keep.append(p)

    def step_device():
        rolled = cube.drillUp("time", "month")
        ms_up = None
        if step_device.measure:
            ms_up = lib.olap_last_op_ms()
            step_device.path = lib.olap_last_op_path().decode()
        ratio = rolled.evaluateToStore("ratio")
        return rolled, ratio, ms_up

    step_device.measure = False

    def step_e2e():
        for name, arr in zip(names, host_in):
            cube.setData(name, arr)
        rolled, ratio, _ = step_device()
        for name, out in zip(names, host_out):
            N.check(lib.olap_store_download_f32(rolled.storedMeasures[name]._h, out.ctypes.data, n_out))
        N.check(lib.olap_store_download_f32(ratio._h, host_out[3].ctypes.data, n_out))
        return float(host_out[3][0])

    clocks = Clocks(local_rank)
    clocks.start()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        timed.launches = lib.olap_kernel_launches()
        clocks.busy.set()
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps - 1):
                fn()
            timed.last = fn()  # the last step's results, for --dump-outputs
            e1.record(stream)
        barrier()
        clocks.busy.clear()
        timed.launches = lib.olap_kernel_launches() - timed.launches
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # correctness guard before timing: month sums of one column against numpy (float64)
    rolled, ratio, _ = step_device()
    col = host_in[0].reshape(3652, -1)[:, 12345].astype(np.float64)
    month_map = np.asarray(dims[0].getGroupIndexFromRootIndexMap("month"))
    want = np.zeros(120)
    np.add.at(want, month_map, col)
    got = rolled.storedMeasures["m_sum"].data_f32().reshape(120, -1)[:, 12345]
    assert np.array_equal(got, want.astype(np.float32)), "bench: drillUp result does not match the float64 reference"
    del rolled, ratio

    N.check(lib.olap_set_async(1))
    ms_value = timed(step_device, args.steps, args.warmup)
    launches = timed.launches  # kernels of libolapgpu.so launched inside the timed region
    N.check(lib.olap_set_async(0))
    if args.dump_outputs:
        rolled, ratio, _ = timed.last
        outputs = {name: rolled.storedMeasures[name].data_f32() for name in names}
        outputs["ratio"] = ratio.data_f32()
        dump_outputs(args.dump_outputs, outputs)
        del rolled, ratio, outputs
    timed.last = None

    # per-launch duration of the dominant kernel, CUDA events on the launching stream
    step_device.measure = True
    ups = []
    for _ in range(max(3, args.steps)):
        _, _, ms_up = step_device()
        ups.append(ms_up)
    step_device.measure = False
    up_ms = float(np.mean(ups))
    path = step_device.path

    ms_e2e = timed(step_e2e, max(1, min(args.steps, 5)), 1)
    clk = clocks.summary()

    measures = len(names)
    cells_per_step = measures * n_in
    value = world * cells_per_step / (ms_value * 1e-3)
    e2e_value = world * cells_per_step / (ms_e2e * 1e-3)
    # float32 cell + status byte per measure; the status plane of a store filled by setData follows from its
    # values (olap_store_status_derived), so the rollup never reads it: 4 bytes per input cell, 5 per output cell
    derived = all(cube.storedMeasures[name].status_derived for name in names)
    algo_bytes = measures * ((4 if derived else 5) * n_in + 5 * n_out)
    achieved = algo_bytes / (up_ms * 1e-3) / 1e9
    peak, peak_src = FALLBACK_HBM_GBS, "fallback"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        peak_src = "measured"
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "drillup_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        pass

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            threads = 1
            v, _, sample = cpu_port_run(1, 0, threads, GENERIC * GENERIC * 4)
            cpu = {"value": v, "unit": "cells/s", "cores": threads, "kind": "port", "sample": sample}
        line = {
            "metric": "drillUp input measure-cells/s", "value": value, "unit": "cells/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_value, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(),
            "e2e": {"value": e2e_value, "unit": "cells/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": world * measures * n_in * 4, "d2h_bytes_per_step": world * 4 * n_out * 4},
            "gpu_launches": int(launches), "clocks": clk,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": path, "kernel_ms": up_ms, "algorithmic_bytes": algo_bytes,
                         "bytes_per_cell": {"input": 4 if derived else 5, "output": 5,
                                            "why": "input status planes are derived from the values (set by setData) and not read" if derived
                                                   else "value + status byte"},
                         "peak_source": peak_src},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm, N > 1: one sharded cube
def univac_dims(ndims):
    from olap_in_memory_b200 import GenericDimension

    dims = []
    for k in range(ndims):
        d = GenericDimension(f"dim{k}", "root", [str(i) for i in range(10)])
        d.addAttribute("root", "parity", lambda item: "even" if int(item) % 2 == 0 else "odd")
        dims.append(d)
    return dims


def sharded_parity_guard(dist, rank, world):
    """Hardware parity proof of the multi-GPU path, run before anything is timed: small sharded
    cubes against ONE single-GPU cube of the same data (itself held bit-equal to the CPU oracle by
    tests/).  Pull exchange: bit-exact, every method, both defaults, mixed-sign data whose float32
    partial sums would cancel badly; NCCL exchange: rel 1e-6 (float32 partials); plus the paths
    that had only ever run over gloo: prefix-deepening rollups, the re-partitioning
    reorderDimensions, sharded computed measures.  Returns a summary for the JSON line."""
    import math

    from olap_in_memory_b200 import Cube
    from olap_in_memory_b200 import sharded as SH
    from olap_in_memory_b200.sharded import ShardedCube

    rules = ("sum", "average", "highest", "lowest", "first", "last")
    nd = 6
    n = 10 ** nd
    mismatches, cases, timed_path_mismatches = [], 0, 0
    default_mode = SH.EXCHANGE
    min_deep, SH.MIN_DEEP_INNER = SH.MIN_DEEP_INNER, 64  # let the small cubes take the balance-driven deepening too

    def same_bits(a, b):
        a = np.asarray(a, dtype=np.float64).astype(np.float32)
        b = np.asarray(b, dtype=np.float64).astype(np.float32)
        return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))

    for default in (0.0, math.nan):
        for kind in ("uniform", "sparse mixed-sign"):
            rng = np.random.default_rng(17)
            sc, ref = ShardedCube(univac_dims(nd), prefix=2), Cube(univac_dims(nd))
            for m, rule in enumerate(rules):
                if kind == "uniform":
                    data = rng.uniform(1.0, 1000.0, n).astype(np.float32)
                else:
                    data = (rng.uniform(-1e6, 1e6, n) * rng.choice([1.0, 1e-6], n)).astype(np.float32)
                    data[rng.random(n) < 0.4] = default
                for c in (sc, ref):
                    c.createStoredMeasure(f"m_{rule}", {f"dim{k}": rule for k in range(nd)}, "float32", default)
                    c.setData(f"m_{rule}", data)
            for c in (sc, ref):
                c.createComputedMeasure("ratio", "(m_sum + m_average) / m_highest")
            ops = [("dim0", "all"), ("dim0", "parity"), ("dim1", "all"), (f"dim{nd - 1}", "all")]
            for mode in ("pull", "pull2", "nccl"):
                SH.EXCHANGE = mode
                for dim, attr in ops:
                    a, b = sc.drillUp(dim, attr), ref.drillUp(dim, attr)
                    exchanged = dim in ("dim0", "dim1")
                    for rule in rules:
                        got, want = a.getData(f"m_{rule}"), b.getData(f"m_{rule}")
                        cases += 1
                        if mode == "pull" or not exchanged or rule not in ("sum", "average"):
                            ok = same_bits(got, want)  # pull reads the children themselves; order-only rules are exact in every mode
                        elif kind != "uniform":
                            continue  # float32 partial sums under cancellation: outside the stated tolerance of pull2 / nccl
                        else:
                            ok = np.allclose(got, np.asarray(want, dtype=np.float64), rtol=1e-6, atol=0, equal_nan=True)
                        if not ok:
                            mismatches.append(f"{mode} default={default} {kind} drillUp({dim},{attr}) m_{rule}")
                            timed_path_mismatches += mode == default_mode and (dim, attr) in (("dim0", "all"), (f"dim{nd - 1}", "all"))
                    if mode == "pull" and attr == "all":
                        cases += 1
                        if not np.allclose(a.getData("ratio"), np.asarray(b.getData("ratio"), dtype=np.float64), rtol=1e-6, atol=0, equal_nan=True):
                            mismatches.append(f"computed measure after drillUp({dim},{attr}) default={default} {kind}")
            SH.EXCHANGE = default_mode
            # the re-partitioning reorder (cube.js:757-783) on a prefix-1 cube, then a rollup of the new sharded axis
            if kind == "uniform":
                s1 = ShardedCube(univac_dims(nd), prefix=1)
                for rule in ("sum", "first"):
                    s1.createStoredMeasure(f"m_{rule}", {f"dim{k}": rule for k in range(nd)}, "float32", default)
                    s1.setData(f"m_{rule}", np.asarray(ref.getData(f"m_{rule}"), dtype=np.float32))
                order = ["dim2", "dim0"] + [f"dim{k}" for k in range(nd - 1, 0, -1) if k != 2]
                try:
                    ra, rb = s1.reorderDimensions(order), ref.reorderDimensions(order)
                    for rule in ("sum", "first"):
                        cases += 2
                        if not same_bits(ra.getData(f"m_{rule}"), rb.getData(f"m_{rule}")):
                            mismatches.append(f"reorderDimensions m_{rule} default={default}")
                        if not same_bits(ra.drillUp("dim2", "all").getData(f"m_{rule}"), rb.drillUp("dim2", "all").getData(f"m_{rule}")):  # default exchange: pull
                            mismatches.append(f"reorderDimensions then drillUp(dim2,all) m_{rule} default={default}")
                except Exception as exc:  # reported, not fatal: not on the timed path
                    mismatches.append(f"reorderDimensions raised {type(exc).__name__}: {exc}")
    import torch

    SH.MIN_DEEP_INNER = min_deep
    t = torch.tensor([len(mismatches), timed_path_mismatches], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"cases": cases, "mismatches": int(t[0].item()), "first_mismatches": mismatches[:5], "timed_path_mismatches": int(t[1].item()),
            "what": "small sharded cubes vs ONE single-GPU cube on the same data: pull exchange bit-exact (6 methods, 0 / NaN default, "
                    "mixed-sign sparse data), NCCL exchange rel 1e-6, deepened prefixes, re-partitioning reorder, computed measures"}


def run_sharded(args, rank, world, local_rank):
    import ctypes as C

    import torch
    import torch.distributed as dist

    from olap_in_memory_b200 import _native as N
    from olap_in_memory_b200 import interop
    from olap_in_memory_b200 import sharded as SH
    from olap_in_memory_b200.sharded import ShardedCube, _exchange_costs

    torch.cuda.set_device(local_rank)
    N.init(local_rank)
    lib = N.lib()
    stream = torch.cuda.Stream()
    N.check(lib.olap_set_stream(stream.cuda_stream))
    guard = sharded_parity_guard(dist, rank, world)
    assert guard["timed_path_mismatches"] == 0, f"bench: the sharded rollups do not match the single-GPU cube: {guard}"

    cfg = sharded_config(world)
    ndims = cfg["ndims"]
    dims = univac_dims(ndims)
    cube = ShardedCube(dims, prefix=2)
    names = ["m_sum", "m_avg", "m_max"]
    with torch.cuda.stream(stream):
        for name, rule in zip(names, SHARDED_METHODS):
            cube.createStoredMeasure(name, {d.id: rule for d in dims}, "float32", 0)
            interop.values_tensor(cube.storedMeasures[name]).uniform_(1.0, 1000.0)
    torch.cuda.synchronize()
    for name in names:  # planes written through raw pointers: canonicalise values, derive the status plane from them
        cube.storedMeasures[name].canonicalise()
    n_total, n_local, measures = cube.storeSize, cube.localSize, len(names)
    last = f"dim{ndims - 1}"

    def op_inner():
        return cube.drillUp(last, "all")

    def op_outer():
        return cube.drillUp("dim0", "all")

    def step_device():
        return op_inner(), op_outer()

    clocks = Clocks(local_rank)
    clocks.start()

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        timed.launches = lib.olap_kernel_launches()
        clocks.busy.set()
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                fn()
            e1.record(stream)
        barrier()
        clocks.busy.clear()
        timed.launches = lib.olap_kernel_launches() - timed.launches
        t = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def max_over_ranks(x):
        t = torch.tensor([float(x)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # full-size property before timing: a sum rollup preserves the grand total
    total_before = cube.getTotal("m_sum")
    rolled = op_outer()
    total_after = rolled.getTotal("m_sum")
    assert abs(total_after - total_before) <= 1e-6 * abs(total_before), "bench: dim0 -> all lost cells"
    deep = rolled.prefix
    out_bounds = list(rolled.row_bounds)
    exchange = getattr(rolled, "last_exchange", SH.EXCHANGE)
    exchange_setting = SH.EXCHANGE
    del rolled

    N.check(lib.olap_set_async(1))
    ms_value = timed(step_device, args.steps, args.warmup)
    launches = timed.launches
    N.check(lib.olap_set_async(0))
    ms_inner = timed(op_inner, max(3, min(args.steps, 10)), 1)
    ms_outer = timed(op_outer, max(3, min(args.steps, 10)), 1)
    # kernel-only brackets (CUDA events inside the library, on its stream)
    k_inner, k_outer = [], []
    for _ in range(3):
        op_inner()
        k_inner.append(lib.olap_last_op_ms())
        path_inner = lib.olap_last_op_path().decode()
        res = op_outer()
        k_outer.append(getattr(res, "last_pull_ms", None) or lib.olap_last_op_ms())  # the pull kernel itself
        path_outer = "drillup/pull-peers" if getattr(res, "last_pull_ms", None) else lib.olap_last_op_path().decode()
        pull_derived = bool(getattr(res, "last_pull_derived", False))  # status planes derived from the values: not read over NVLink
        del res
    k_inner_ms, k_outer_ms = max_over_ranks(np.mean(k_inner)), max_over_ranks(np.mean(k_outer))

    # the partial-based exchange modes on the same rollup (opt-in: float32 partials, rel 1e-6), a few repetitions each
    alternatives = {}
    free_b = torch.tensor([float(torch.cuda.mem_get_info()[0])], device="cuda")
    dist.all_reduce(free_b, op=dist.ReduceOp.MIN)
    room = float(free_b.item()) > 2 * 5 * 4 * (n_total // 10) + (8 << 30)  # partial planes + receive buffers, every rank
    for mode in ("pull2", "push", "nccl"):
        if mode == exchange or not room or os.environ.get("OLAP_BENCH_ALTERNATIVES", "1") == "0":
            continue
        SH.EXCHANGE = mode
        try:
            alternatives[mode] = timed(op_outer, 3, 1)
        except Exception as exc:  # an alternative that cannot run here (memory for receive buffers) is reported, not fatal
            alternatives[mode] = f"{type(exc).__name__}: {exc}"[:200]
        SH.EXCHANGE = exchange_setting
    # bytes that cross NVLink into this GPU during dim0 -> all: the remote children of my output rows
    view = cube
    while view.prefix < deep:
        view = view._deepened()
    full_map = view._row_map(0, np.zeros(10, dtype=np.int32), [1] + [10] * (deep - 1), all_rows=True)
    direct_rows, partial_rows, _, _, _ = _exchange_costs(full_map, view.row_bounds, out_bounds)
    planes = measures + sum(1 for m in SHARDED_METHODS if m == "average")  # `average` partials travel as (sum, count)
    cell_bytes = 4 if (exchange == "pull" and pull_derived) else 5
    nvlink_in = float(direct_rows * cell_bytes * measures * view.inner if exchange == "pull" else partial_rows * 5 * planes * view.inner)
    pulled = path_outer == "drillup/pull-peers" or exchange == "pull2"

    # ---- e2e: host buffers -> sharded cube -> both rollups -> host
    def pinned(n_floats):
        p = C.c_void_p()
        N.check(lib.olap_host_alloc(max(1, n_floats) * 4, C.byref(p)))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(max(1, n_floats),)), p

    host_in, keep_in = pinned(n_local)
    block = synth(np.empty(min(n_local, 1 << 24), np.float32), 1 + rank, 0)
    for lo in range(0, n_local, block.size):
        hi = min(n_local, lo + block.size)
        host_in[lo:hi] = block[: hi - lo]
    a, b = step_device()
    out_cells = max(next(iter(a.storedMeasures.values())).size, next(iter(b.storedMeasures.values())).size)
    d2h_local = measures * (next(iter(a.storedMeasures.values())).size + next(iter(b.storedMeasures.values())).size) * 4
    del a, b
    host_out, keep_out = pinned(out_cells)

    def step_e2e():
        for name in names:
            cube.setLocalData(name, host_in[:n_local])
        a, b = step_device()
        for res in (a, b):
            for name in names:
                st = res.storedMeasures[name]
                N.check(lib.olap_store_download_f32(st._h, host_out.ctypes.data, st.size))
        return float(host_out[0])

    ms_e2e = timed(step_e2e, max(1, min(args.steps, 2)), 1)
    clk = clocks.summary()
    t = torch.tensor([float(d2h_local)], device="cuda")
    dist.all_reduce(t)
    d2h_total = int(t.item())

    peak, peak_src = FALLBACK_HBM_GBS, "fallback"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        peak_src = "measured"
    except Exception:
        pass
    cells_per_step = 2 * measures * n_total
    value = cells_per_step / (ms_value * 1e-3)
    # the shard-local rollup reads 4 bytes per input cell when the status planes follow from the values, 5 otherwise
    in_cell = 4 if all(cube.storedMeasures[name].status_derived for name in names) else 5
    inner_bytes = measures * (in_cell * n_local + 5 * (n_local // 10))
    nv_gbs = nvlink_in / (k_outer_ms * 1e-3) / 1e9
    if rank == 0:
        line = {
            "metric": "drillUp input measure-cells/s", "value": value, "unit": "cells/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_value, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "e2e": {"value": cells_per_step / (ms_e2e * 1e-3), "unit": "cells/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": measures * n_total * 4, "d2h_bytes_per_step": d2h_total,
                    "note": "every rank uploads its shard of the 3 measures from one pinned host buffer, runs both rollups, downloads the 6 result planes"},
            "gpu_launches": int(launches), "clocks": clk,
            "roofline": {"bound": "nvlink", "achieved": nv_gbs, "peak": NVLINK_GBS, "unit": "GB/s", "frac": nv_gbs / NVLINK_GBS,
                         "traffic": None, "kernel": path_outer, "kernel_ms": k_outer_ms, "algorithmic_bytes": nvlink_in,
                         "peak_source": "B200_PROFILING.md measured peer copy per direction per GPU",
                         "what": "bytes the busiest GPU reads from its peers during drillUp dim0 -> all (pull: the remote children of its "
                                 "output rows x 5 B x 3 measures; pull2: the peers' partial rows x 5 B x 4 planes) / device time of the "
                                 "pull kernel, max over ranks"},
            "sharded": {
                "exchange": exchange, "exchange_setting": exchange_setting,
                "alternative_exchanges_ms": alternatives, "pulled_over_peer_memory": pulled, "prefix_after_rollup": deep,
                "rows_per_rank_out": [out_bounds[r + 1] - out_bounds[r] for r in range(world)],
                "inner_rollup": {"op": f"drillUp {last}->all (shard-local)", "ms": ms_inner, "kernel_ms": k_inner_ms, "kernel": path_inner,
                                 "bytes_per_input_cell": in_cell, "hbm_GBs_per_gpu": inner_bytes / (k_inner_ms * 1e-3) / 1e9,
                                 "hbm_frac": inner_bytes / (k_inner_ms * 1e-3) / 1e9 / peak, "hbm_peak": peak, "peak_source": peak_src},
                "sharded_rollup": {"op": "drillUp dim0->all (sharded dimension)", "ms": ms_outer, "kernel_ms": k_outer_ms, "kernel": path_outer,
                                   "nvlink_bytes_in_per_gpu": nvlink_in, "bytes_per_cell_over_nvlink": cell_bytes, "nvlink_GBs_per_gpu": nv_gbs, "nvlink_frac_of_770": nv_gbs / NVLINK_GBS,
                                   "bound_ms": nvlink_in / (NVLINK_GBS * 1e9) * 1e3},
                "parity_guard": guard,
            },
            "cpu_baseline": None,
        }
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the result planes of the last timed step (m_sum, m_avg, m_max, ratio) as DIR/<name>.npy "
                         "(float32); single GPU only")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours on a single GPU")
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if world > 1:
            run_sharded(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
