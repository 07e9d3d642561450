"""getTotalForDimensionItems, getDistribution and copyMeasureData against the per-cell host loops they
replaced (kept below, verbatim, as the reference): results, errors and their messages, on Cube with the
CPU oracle store and on ShardedCube over gloo (2 and 3 ranks) against one oracle Cube."""
import math
import os
import socket
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

from olap_in_memory_b200 import Cube, GenericDimension, TimeDimension  # noqa: E402
from region_stores import RegionOracleShardStore, RegionOracleStore  # noqa: E402


# ---- the reference: the host loops of Cube as they stood before the region kernels ------------------
def _loop_options(cube, dimensionsFilter):
    options = {k: ([v] if isinstance(v, str) else v) for k, v in (dimensionsFilter or {}).items()}
    for d in cube.dimensionIds:
        if d not in options:
            options[d] = cube.getDimension(d).getItems()
    return options


def loop_values(cube, measureId, dimensionsFilter=None):
    return [cube.getSingleData(measureId, c) for c in cube._combinations(_loop_options(cube, dimensionsFilter))]


def loop_getTotalForDimensionItems(cube, measureId, dimensionsFilter=None):
    options = _loop_options(cube, dimensionsFilter)
    return sum((cube.getSingleData(measureId, c) for c in cube._combinations(options)), 0)


def loop_getDistribution(cube, measureId, dimensionsFilter=None):
    space = loop_getTotalForDimensionItems(cube, measureId, dimensionsFilter)
    total = cube.getTotal(measureId)
    return space if total == 0 else space / total


def loop_copyMeasureData(cube, sourceMeasureId, targetMeasureId, dimensionsFilter=None):
    options = _loop_options(cube, dimensionsFilter)
    for combination in cube._combinations(options):
        cube.setSingleData(targetMeasureId, combination, cube.getSingleData(sourceMeasureId, combination))


# ---- comparison rules ----------------------------------------------------------------------------
def outcome(fn):
    try:
        return ("ok", fn())
    except AttributeError:  # a store lacking a protocol member is a broken test, not a result
        raise
    except Exception as e:  # noqa: BLE001 - the exception IS the result being compared
        return ("error", type(e), str(e))


def assert_same_sum(got, values):
    """|got - fsum| <= 1e-12 * sum|v|; NaN and +-inf exactly as the loop's sum."""
    want = sum(values, 0)
    if not math.isfinite(want):
        assert (math.isnan(got) and math.isnan(want)) or got == want, (got, want)
        return
    exact = math.fsum(values)
    assert abs(got - exact) <= 1e-12 * math.fsum(abs(v) for v in values), (got, exact)


def assert_same_outcome(got, want, values=None):
    assert got[0] == want[0], (got, want)
    if got[0] == "error":
        assert got[1:] == want[1:], (got, want)
    elif values is not None:
        assert_same_sum(got[1], values)
    else:
        g, w = got[1], want[1]
        assert (math.isnan(g) and math.isnan(w)) or abs(g - w) <= 1e-12 * max(1.0, abs(w)), (g, w)


# ---- seeded cases --------------------------------------------------------------------------------
def make_cube(seed, store_cls, ndim=None):
    """1-4 generic dimensions of 1-5 items, stored measures of both defaults and several types, dense or sparse
    (a set NaN under a zero default included), and computed measures (one with an `x__total` variable)."""
    rng = np.random.default_rng(seed)
    ndim = ndim or 1 + seed % 4
    dims = [GenericDimension(f"d{k}", "item", [f"i{j}" for j in range(int(rng.integers(1, 6)))]) for k in range(ndim)]
    cube = Cube(dims, store_cls)
    density = (0.2, 0.7, 1.0)[seed % 3]
    for name, type_, default in (("m_zero", "float32", 0), ("m_nan", "float32", math.nan),
                                 ("m_int", "int32", 0), ("m_nint", "uint32", math.nan)):
        cube.createStoredMeasure(name, {}, type_, default)
        data = rng.integers(-40, 40, cube.storeSize).astype(np.float64) * (0.25 if type_ == "float32" else 1.0)
        if type_ == "uint32":
            data = np.abs(data)
        data[rng.random(cube.storeSize) >= density] = default
        if name == "m_zero" and seed % 5 == 0:
            data[int(rng.integers(cube.storeSize))] = math.nan  # a set NaN under a zero default
        cube.setData(name, data.tolist())
    cube.createComputedMeasure("c_sum", "m_zero + m_int * 2")
    cube.createComputedMeasure("c_share", "m_zero / m_zero__total")
    return cube


def make_filters(cube, seed):
    rng = np.random.default_rng(1000 + seed)
    filters = [None, {}]
    for _ in range(8):
        f = {}
        for d in cube.dimensions:
            r = rng.random()
            items = d.getItems()
            if r < 0.3:
                continue
            if r < 0.5:
                f[d.id] = str(items[int(rng.integers(len(items)))])
            else:  # any order, repeats allowed
                f[d.id] = [str(items[int(i)]) for i in rng.integers(0, len(items), int(rng.integers(1, 2 * len(items) + 1)))]
        if rng.random() < 0.3:
            f["not_a_dim"] = ["x", "y", "z"][: int(rng.integers(1, 4))]
        if rng.random() < 0.15:
            f["also_not"] = "w"
        # shuffle the key order (the loop's product order follows it)
        keys = list(f)
        rng.shuffle(keys)
        filters.append({k: f[k] for k in keys})
    d0 = cube.dimensions[0]
    filters += [
        {d0.id: []},                                    # empty list: empty region
        {"not_a_dim": []},                              # empty extra key: empty region
        {d0.id: list(reversed(d0.getItems())) * 2},     # unordered, every item twice
    ]
    return filters


MEASURES = ("m_zero", "m_nan", "m_int", "m_nint", "c_sum", "c_share", "no_such")


@pytest.mark.parametrize("seed", range(24))
def test_total_and_distribution_match_the_loop(seed):
    cube = make_cube(seed, RegionOracleStore)
    for f in make_filters(cube, seed):
        for m in MEASURES:
            values = outcome(lambda: loop_values(cube, m, f))
            got = outcome(lambda: cube.getTotalForDimensionItems(m, f))
            want = outcome(lambda: loop_getTotalForDimensionItems(cube, m, f))
            assert_same_outcome(got, want, values[1] if values[0] == "ok" else None)
            assert_same_outcome(outcome(lambda: cube.getDistribution(m, f)), outcome(lambda: loop_getDistribution(cube, m, f)))


PAIRS = (("m_zero", "m_nan"), ("m_nan", "m_zero"), ("m_nan", "m_int"), ("m_zero", "m_zero"), ("m_nint", "m_nan"),
         ("c_sum", "m_nan"), ("c_share", "m_zero"), ("no_such", "m_zero"), ("m_zero", "c_sum"), ("m_zero", "no_such"))


def _maps(cube):
    return {m: dict(s._dataMap) for m, s in cube.storedMeasures.items()}


def _same_maps(a, b):
    assert a.keys() == b.keys()
    for m in a:
        assert a[m].keys() == b[m].keys(), m
        for k in a[m]:
            x, y = a[m][k], b[m][k]
            assert (x != x and y != y) or x == y, (m, k, x, y)


@pytest.mark.parametrize("seed", range(16))
def test_copy_matches_the_loop(seed):
    for f in make_filters(make_cube(seed, RegionOracleStore), seed):
        for src, dst in PAIRS:
            mine, ref = make_cube(seed, RegionOracleStore), make_cube(seed, RegionOracleStore)
            got = outcome(lambda: mine.copyMeasureData(src, dst, f))
            want = outcome(lambda: loop_copyMeasureData(ref, src, dst, f))
            assert got[0] == want[0] and got[1:] == want[1:] if got[0] == "error" else got == want, (got, want)
            if got[0] == "ok":
                _same_maps(_maps(mine), _maps(ref))


# ---- each rule of the loop, pinned -----------------------------------------------------------------
def _small():
    cube = Cube([GenericDimension("a", "x", ["a0", "a1", "a2"]), GenericDimension("b", "x", ["b0", "b1"])], RegionOracleStore)
    cube.createStoredMeasure("m_a", {}, "float32", 0)
    cube.setData("m_a", [1.0, 2.0, 0.0, 4.0, 8.0, 16.0])
    cube.createStoredMeasure("m_n", {}, "float32", math.nan)
    cube.setData("m_n", [1.0, math.nan, 3.0, 4.0, 5.0, 6.0])
    cube.createStoredMeasure("m_z", {}, "float32", 0)
    cube.createComputedMeasure("c_t", "m_a / m_a__total")
    return cube


def test_items_repeats_and_extra_keys():
    cube = _small()
    assert cube.getTotalForDimensionItems("m_a") == 31
    assert cube.getTotalForDimensionItems("m_a", {"a": "a1"}) == 4
    assert cube.getTotalForDimensionItems("m_a", {"a": ["a2", "a0", "a2"]}) == 1 + 2 + 2 * (8 + 16)
    assert cube.getTotalForDimensionItems("m_a", {"zz": ["p", "q", "r"], "b": "b1"}) == 3 * (2 + 4 + 16)
    assert cube.getTotalForDimensionItems("m_a", {"zz": []}) == 0
    assert cube.getTotalForDimensionItems("no_such", {"zz": []}) == 0  # empty region: no error
    assert cube.getTotalForDimensionItems("m_a", {"a": ["nope"], "b": []}) == 0


def test_unset_cells_read_as_the_default():
    cube = _small()
    assert math.isnan(cube.getTotalForDimensionItems("m_n"))
    assert cube.getTotalForDimensionItems("m_n", {"b": "b0"}) == 1 + 3 + 5
    cube.setSingleData("m_a", {"a": "a0", "b": "b0"}, math.nan)  # a set NaN under a zero default
    assert math.isnan(cube.getTotalForDimensionItems("m_a"))


def test_distribution_with_a_zero_total_is_the_region_total():
    cube = _small()
    assert cube.getDistribution("m_z", {"a": "a1"}) == 0
    assert cube.getDistribution("m_a", {"a": "a1"}) == 4 / 31
    with pytest.raises(KeyError):
        cube.getDistribution("c_t")  # the region total is fine, getTotal of a computed measure is not


@pytest.mark.parametrize("f", [
    {"a": ["a0", "nope"]}, {"a": ["a0", ""]}, {"b": [None]}, {"a": ["nope"], "b": [""]},
    {"b": ["b0", "nope"], "a": ["a1", "bad"]}, {"zz": ["u", "v"], "a": ["a0", "a9"]}, {"a": "", "b": "nope"},
])
@pytest.mark.parametrize("measure", ["m_a", "no_such", "c_t"])
def test_errors_are_those_of_the_first_failing_combination(f, measure):
    cube = _small()
    got = outcome(lambda: cube.getTotalForDimensionItems(measure, f))
    want = outcome(lambda: loop_getTotalForDimensionItems(cube, measure, f))
    assert got[0] == "error" and got == want
    got = outcome(lambda: cube.copyMeasureData(measure, "m_z", f))
    want = outcome(lambda: loop_copyMeasureData(_small(), measure, "m_z", f))
    assert got[0] == "error" and got == want
    assert cube.storedMeasures["m_z"]._dataMap == {}  # validated before anything is written


def test_total_variable_in_a_computed_measure_raises_key_error():
    cube = _small()
    with pytest.raises(KeyError, match="m_a__total"):
        cube.getTotalForDimensionItems("c_t")
    with pytest.raises(KeyError, match="m_a__total"):
        cube.copyMeasureData("c_t", "m_z")


def test_copy_status_across_defaults():
    cube = _small()
    cube.copyMeasureData("m_n", "m_z", {"b": "b1"})  # the NaN default's unset cell becomes a set NaN
    data = cube.getData("m_z")
    assert data[0] == 0 and math.isnan(data[1]) and data[3] == 4 and data[5] == 6
    assert cube.getStatus("m_z") == [0x1, 0x2, 0x1, 0x2, 0x1, 0x2]
    cube.copyMeasureData("m_a", "m_a", {"a": ["a1", "a1"]})
    assert cube.getData("m_a") == [1.0, 2.0, 0.0, 4.0, 8.0, 16.0]


# ---- ShardedCube over gloo ---------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_dims():
    region = GenericDimension("region", "city", [f"c{i}" for i in range(7)])
    product = GenericDimension("product", "sku", [f"p{i}" for i in range(5)])
    time = TimeDimension("time", "month", "2010-01", "2010-12")
    return [region, product, time]


SHARDED_FILTERS = [
    None,
    {"region": ["c6", "c0", "c6"], "time": ["2010-03", "2010-01"]},
    {"product": "p2", "extra": ["e0", "e1"]},
    {"time": "2010-07", "region": "c3"},
    {"product": ["p4", "p0"], "region": ["c1", "c2", "c5"]},
    {"extra": []},
    {"region": ["c0", "nope"]},
    {"time": [""], "product": ["p1"]},
]
SHARDED_MEASURES = ("m_zero", "m_nan", "c_sum", "c_share", "no_such")


def _sharded_fill(cube, seed):
    rng = np.random.default_rng(seed)
    for name, default in (("m_zero", 0), ("m_nan", math.nan), ("m_target", 0), ("m_ntarget", math.nan)):
        cube.createStoredMeasure(name, {}, "float32", default)
        data = rng.integers(-20, 20, 7 * 5 * 12).astype(np.float64)
        data[rng.random(data.size) < 0.4] = default
        cube.setData(name, data.tolist())
    cube.createComputedMeasure("c_sum", "m_zero * 3 + m_target")
    cube.createComputedMeasure("c_share", "m_zero / m_zero__total")


def _sharded_collect(cube, diced):
    if diced:
        cube = cube.dice("region", "city", ["c0", "c2", "c3", "c5", "c6"])
    results = {}
    for i, f in enumerate(SHARDED_FILTERS):
        for m in SHARDED_MEASURES:
            results[("total", i, m)] = outcome(lambda: cube.getTotalForDimensionItems(m, f))
            results[("dist", i, m)] = outcome(lambda: cube.getDistribution(m, f))
    for i, f in enumerate(SHARDED_FILTERS):
        for src, dst in (("m_nan", "m_target"), ("m_zero", "m_ntarget"), ("c_sum", "m_target"), ("no_such", "m_target"),
                         ("m_zero", "c_sum")):
            results[("copy", i, src, dst)] = outcome(lambda: cube.copyMeasureData(src, dst, f))
        for m in ("m_target", "m_ntarget"):
            results[("data", i, m)] = np.asarray(cube.getData(m), dtype=np.float64)
    return results


def _sharded_worker(rank, world, port, prefix, diced, queue):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from olap_in_memory_b200.sharded import ShardedCube
        cube = ShardedCube(_sharded_dims(), prefix=prefix, store_cls=RegionOracleShardStore)
        _sharded_fill(cube, 5)
        results = _sharded_collect(cube, diced)
        queue.put((rank, results))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,prefix,diced", [(2, 1, False), (2, 2, True), (3, 1, True), (3, 2, False)])
def test_sharded_region_queries_match_one_cube(world, prefix, diced):
    ctx = mp.get_context("spawn")
    queue = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_sharded_worker, args=(r, world, port, prefix, diced, queue)) for r in range(world)]
    for p in procs:
        p.start()
    by_rank = dict(queue.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    one = Cube(_sharded_dims(), RegionOracleStore)
    _sharded_fill(one, 5)
    want = _sharded_collect(one, diced)
    for rank, got in by_rank.items():
        assert got.keys() == want.keys()
        for key in want:
            g, w = got[key], want[key]
            if key[0] == "data":
                assert np.array_equal(g, w, equal_nan=True), (rank, key)
            elif key[0] == "copy":
                assert g == w, (rank, key, g, w)
            else:
                assert_same_outcome(g, w)
