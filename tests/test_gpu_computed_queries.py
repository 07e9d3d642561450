"""Computed measures in region queries and status accessors on the device: getTotalForDimensionItems /
getDistribution (olap_region_eval_sum), copyMeasureData from a computed source (olap_region_eval_copy), getStatus
(olap_status_merge) and getStatusMap (olap_status_map_export).  The reference is the host code kept in cube.py,
reached through a GpuStore subclass that hides the four members, on identically seeded cubes; at a size larger
than L2 it is numpy on the downloaded planes."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_region_queries as R  # noqa: E402
from test_gpu_region import BRANCHES, _lists, _store  # noqa: E402
from olap_in_memory_b200 import Cube, GenericDimension  # noqa: E402
from olap_in_memory_b200 import _native as N  # noqa: E402
from olap_in_memory_b200 import cube as cube_mod  # noqa: E402
from olap_in_memory_b200.parser import getParser  # noqa: E402
from olap_in_memory_b200.store import GpuStore  # noqa: E402

MEMBERS = ("regionEvalSum", "regionEvalCopy", "statusMerge", "statusMap")


class HostPathStore(GpuStore):
    """GpuStore without the four members: Cube keeps its host code (the reference)."""


class NoPlaneStore(GpuStore):
    WITH_STATUS = False


class NoPlaneHostPathStore(NoPlaneStore):
    pass


for _m in MEMBERS:
    setattr(HostPathStore, _m, None)
    setattr(NoPlaneHostPathStore, _m, None)

# formulas over the stored measures of R.make_cube, every operator and helper of the lowering
FORMULAS = {
    "f_arith": "(m_zero - m_nan) * 3 / (m_int % 7) + m_nint ^ 2",
    "f_coalesce": "m_nan || m_nint",
    "f_cond": "isNaN(m_nan) ? m_zero : max(m_int, m_nint, 1.5)",
    "f_minmax": "min(m_zero, m_int) - max(m_nan, 0)",
    "c_int": "m_int * 2 - m_nint",
}


def _path():
    return N.lib().olap_last_op_path().decode()


def _launches():
    return N.lib().olap_kernel_launches()


def _cube(seed, store_cls):
    cube = R.make_cube(seed, store_cls)
    for name, formula in FORMULAS.items():
        cube.createComputedMeasure(name, formula)
    return cube


def _region_values(cube, measureId, f):
    region = cube_mod._region(cube.dimensions, f, lambda: None)
    if region is None:
        return []
    lens, keep = region
    data = np.asarray(cube.getData(measureId), dtype=np.float64)
    return data.reshape(lens)[np.ix_(*cube_mod._region_lists(lens, keep))].ravel().tolist()


def _bits(x):
    return np.float64(x).view(np.uint64)


@pytest.mark.parametrize("seed", range(8))
def test_region_sums_match_the_host_path(seed):
    mine, ref = _cube(seed, GpuStore), _cube(seed, HostPathStore)
    for f in R.make_filters(mine, seed):
        for m in ("c_sum",) + tuple(FORMULAS) + ("c_share",):
            before = _launches()
            got = R.outcome(lambda: mine.getTotalForDimensionItems(m, f))
            launched, path = _launches() - before, _path()
            want = R.outcome(lambda: ref.getTotalForDimensionItems(m, f))
            assert got[0] == want[0], (m, f, got, want)
            if got[0] == "error":
                assert got[1:] == want[1:], (m, f, got, want)
                continue
            values = _region_values(mine, m, f)
            R.assert_same_sum(got[1], values)
            if values:
                assert path == "region/eval-sum" and launched == 1, (m, f, path, launched)
                assert _bits(mine.getTotalForDimensionItems(m, f)) == _bits(got[1])
            else:
                assert got[1] == 0
            R.assert_same_outcome(R.outcome(lambda: mine.getDistribution(m, f)),
                                  R.outcome(lambda: ref.getDistribution(m, f)))


@pytest.mark.parametrize("branch", list(BRANCHES))
@pytest.mark.parametrize("default", [0.0, math.nan])
def test_region_sum_branches_against_numpy(branch, default):
    lens, keep = BRANCHES[branch]
    size = int(np.prod(lens))
    a, b = _store(size, default, 3), _store(size, 0.0, 4)
    expression = getParser().parse("a * 2 + b / 3")
    got = GpuStore.regionEvalSum(expression, ["a", "b"], [a, b], lens, keep)
    path = _path()
    plane = GpuStore.evaluate_f64(expression, ["a", "b"], [a, b], {}, size)
    sel = plane.reshape(lens)[np.ix_(*_lists(lens, keep))].ravel()
    if sel.size:
        assert path == "region/eval-sum"
    if np.isnan(sel).any():
        assert math.isnan(got)
    else:
        assert abs(got - math.fsum(sel)) <= 1e-12 * np.abs(sel).sum(), (got, math.fsum(sel))
    assert _bits(GpuStore.regionEvalSum(expression, ["a", "b"], [a, b], lens, keep)) == _bits(got)


@pytest.mark.parametrize("branch", list(BRANCHES))
@pytest.mark.parametrize("dst_default", [0.0, math.nan])
def test_region_copy_branches_against_numpy(branch, dst_default):
    """GpuStore.regionEvalCopy straight through the C ABI, every lowering branch (the empty region included):
    the region's cells get the formula's value as setValue stores it, every other cell keeps its bits."""
    lens, keep = BRANCHES[branch]
    size = int(np.prod(lens))
    a, b, dst = _store(size, math.nan, 3), _store(size, 0.0, 4), _store(size, dst_default, 5)
    expression = getParser().parse("a * 2 + b / 3")
    before_v, before_st = dst.data_f32(), _status_np(dst)
    n0 = _launches()
    GpuStore.regionEvalCopy(dst, expression, ["a", "b"], [a, b], lens, keep)
    launched = _launches() - n0
    ix = np.ix_(*_lists(lens, keep))
    want_v, want_st = before_v.copy().reshape(lens), before_st.copy().reshape(lens)
    x = GpuStore.evaluate_f64(expression, ["a", "b"], [a, b], {}, size).astype(np.float32).reshape(lens)[ix]
    x[np.isnan(x)] = np.float32(np.nan)
    if dst_default == 0:
        x[x == 0] = 0.0
    want_v[ix] = x
    want_st[ix] = np.where(np.isnan(x) if dst_default != dst_default else x == 0, 1, 2)
    assert launched == (1 if x.size else 0), (branch, launched)
    assert np.array_equal(dst.data_f32().view(np.uint32), want_v.ravel().view(np.uint32)), branch
    assert np.array_equal(_status_np(dst), want_st.ravel()), branch


COPY_PAIRS = (("c_sum", "m_nan"), ("c_sum", "m_zero"), ("c_sum", "m_int"), ("c_int", "m_int"), ("c_int", "m_nint"),
              ("f_coalesce", "m_nan"), ("f_cond", "m_nint"), ("f_arith", "m_zero"), ("c_share", "m_zero"))


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("planes", [True, False])
def test_copies_match_the_host_path(seed, planes):
    cls, ref_cls = (GpuStore, HostPathStore) if planes else (NoPlaneStore, NoPlaneHostPathStore)
    for f in R.make_filters(_cube(seed, cls), seed)[:8] + [{"d0": ["i0", "i0"], "not_a_dim": ["x", "y"]}]:
        for src, dst in COPY_PAIRS:
            mine, ref = _cube(seed, cls), _cube(seed, ref_cls)
            before_v, before_st = mine.storedMeasures[dst].data_f32(), mine.storedMeasures[dst].status
            n0 = _launches()
            got = R.outcome(lambda: mine.copyMeasureData(src, dst, f))
            launched, path = _launches() - n0, _path()
            want = R.outcome(lambda: ref.copyMeasureData(src, dst, f))
            assert got == want, (src, dst, f, got, want)
            target = mine.storedMeasures[dst]
            if got[0] == "error":
                # refused before anything was written
                assert np.array_equal(target.data_f32().view(np.uint32), before_v.view(np.uint32))
                assert target.status == before_st
                continue
            if _region_values(mine, src, f) and src != "c_share":
                assert path == "region/eval-copy", (src, dst, path)
                assert launched == (2 if target._type in ("int32", "uint32") else 1), (src, dst, launched)
            for m in mine.storedMeasureIds:
                a, b = mine.storedMeasures[m], ref.storedMeasures[m]
                assert np.array_equal(a.data_f32().view(np.uint32), b.data_f32().view(np.uint32)), (src, dst, f, m)
                assert a.status == b.status, (src, dst, f, m)


def test_fractional_value_into_an_integer_target_names_the_first_cell():
    dims = [GenericDimension("a", "x", ["a0", "a1", "a2"]), GenericDimension("b", "x", ["b0", "b1", "b2", "b3"])]
    results = []
    for cls in (GpuStore, HostPathStore):
        cube = Cube(dims, cls)
        cube.createStoredMeasure("m_f", {}, "float32", 0)
        cube.setData("m_f", [4.0, 8.0, 1.0, 2.0, 6.0, 3.0, 12.0, 0.0, 3.0, 9.0, 5.0, 6.0])
        cube.createStoredMeasure("m_i", {}, "int32", 0)
        cube.setData("m_i", [1.0] * 12)
        cube.createComputedMeasure("c_x", "m_f / 10 + m_i")  # 0.1 has no Float32 cell
        before = cube.storedMeasures["m_i"].data_f32()
        out = R.outcome(lambda: cube.copyMeasureData("c_x", "m_i", {"b": ["b3", "b1", "b1"], "a": ["a2", "a0"]}))
        assert np.array_equal(cube.storedMeasures["m_i"].data_f32(), before)
        results.append(out)
    assert results[0][0] == "error" and results[0] == results[1], results


def _status_cube(store_cls, stores, measures, formula):
    cube = Cube([GenericDimension("a", "x", [f"a{i}" for i in range(stores[0].size)])], store_cls)
    for name, store in zip(measures, stores):
        cube.storedMeasures[name] = store
        cube.storedMeasuresRules[name] = {}
    cube.createComputedMeasure("c_x", formula)
    return cube


def _seeded(size, seed, default, planes):
    rng = np.random.default_rng(seed)
    v = (rng.integers(-4, 4, size) * 0.5).astype(np.float32)
    v[rng.random(size) < 0.4] = default
    s = (GpuStore if planes else NoPlaneStore)(size, "float32", default)
    s.set_data_f32(v)
    return s


@pytest.mark.parametrize("planes", [(True, True), (False, False), (True, False)])
def test_get_status_matches_the_host_merge(planes):
    stores = [_seeded(37, 1, 0.0, planes[0]), _seeded(37, 2, math.nan, planes[1])]
    mine = _status_cube(GpuStore, stores, ["m_a", "m_b"], "m_a * m_b")
    ref = _status_cube(HostPathStore, stores, ["m_a", "m_b"], "m_a * m_b")
    n0 = _launches()
    got = mine.getStatus("c_x")
    assert _path() == "status/merge" and _launches() - n0 == 1
    assert got == ref.getStatus("c_x")
    assert mine.getStatus("m_a") == stores[0].status


def test_get_status_after_drill_up_and_drill_down():
    stores = [_seeded(24, 3, 0.0, True), _seeded(24, 4, math.nan, True)]
    up = GpuStore.drillUp_lowered(stores, [6, 4], [2, 4], [[0, 0, 1, 1, 0, 1], None], ["sum", "highest"])
    down = GpuStore.drillDown_lowered(stores, [6, 4], [12, 4], [[0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5], list(range(4))],
                                      ["sum", "sum"])
    seen = set()
    for result in (up, down):
        # a third input without a status plane contributes SET / UNSET from its values
        flat = list(result) + [_seeded(result[0].size, 5, 0.0, False)]
        mine = _status_cube(GpuStore, flat, ["m_a", "m_b", "m_c"], "m_a + m_b - m_c")
        ref = _status_cube(HostPathStore, flat, ["m_a", "m_b", "m_c"], "m_a + m_b - m_c")
        got = mine.getStatus("c_x")
        assert got == ref.getStatus("c_x")
        seen.update(got)
    assert 0x3 in seen and any(b & 0x4 for b in seen), sorted(seen)


SPECIALS = np.array([0.0, -0.0, math.nan, math.inf, -math.inf, 0.5, -2.75, -7.0, 2.0 ** 31, 2.0 ** 32 + 512, 3e38, 1.0,
                     3.0, -1.0, 1e-3, 6.0], dtype=np.float64)


def _same_items(got, want):
    assert len(got) == len(want)
    for (kg, vg), (kw, vw) in zip(got, want):
        assert kg == kw and type(vg) is type(vw), (kg, kw, vg, vw)
        if isinstance(vw, float) and vw != vw:
            assert vg != vg
        else:
            assert vg == vw and math.copysign(1, vg) == math.copysign(1, vw), (kg, vg, vw)


@pytest.mark.parametrize("n_stores", [1, 2, 3, 4])
@pytest.mark.parametrize("seed", range(3))
def test_get_status_map_matches_the_host_loop(n_stores, seed):
    rng = np.random.default_rng(seed)
    size = 48
    stores = []
    for k in range(n_stores):
        default = (0.0, math.nan)[(k + seed) % 2]
        v = SPECIALS[rng.integers(0, SPECIALS.size, size)]
        v[rng.random(size) < 0.3] = default
        s = GpuStore(size, "float32", default)
        s.set_data_f32(v.astype(np.float32))
        stores.append(s)
    names = [f"m_{k}" for k in range(n_stores)]
    mine = _status_cube(GpuStore, stores, names, names[0] + " * 2")
    ref = _status_cube(HostPathStore, stores, names, names[0] + " * 2")
    got = mine.getStatusMap("c_x")
    assert _path() == "status/map"
    _same_items(list(got.items()), list(ref.getStatusMap("c_x").items()))


def _status_np(store):
    out = np.empty(store.size, dtype=np.uint8)
    N.check(N.lib().olap_store_status(store._h, out.ctypes.data, store.size))
    return out


def _to_int32(x):
    ok = np.abs(x) < 2.0 ** 63
    r = np.zeros(x.shape, dtype=np.int64)
    r[ok] = x[ok].astype(np.int64)
    return (r & 0xFFFFFFFF).astype(np.uint32).view(np.int32)


def test_cube_larger_than_l2_against_numpy():
    """50 x 1000 x 1000 = 5e7 cells (200 MB a plane, larger than the 126 MB L2)."""
    lens = [50, 1000, 1000]
    size = int(np.prod(lens))
    rng = np.random.default_rng(11)
    defaults = (0.0, math.nan, 0.0)
    stores, planes = [], []
    for k, default in enumerate(defaults):
        v = (rng.standard_normal(size, dtype=np.float32) * 100).round()
        v[rng.random(size) < 0.3] = default
        s = (GpuStore if k < 2 else NoPlaneStore)(size, "float32", default)
        s.set_data_f32(v)
        stores.append(s)
        planes.append(s.data_f32().astype(np.float64))
    # regions of 1e6..5e7 cells: far more work items than the grid has threads, so every lane of every thread and
    # the grid-stride step run (VEC 4 and, with the innermost axis filtered, VEC 1)
    regions = ([list(range(3, 40, 2)), None, None], [None, rng.permutation(1000)[:300].tolist(), None],
               [None, None, list(range(0, 1000, 2))], [None, None, None])
    # a finite formula (b's NaN cells are skipped by ||, no divisor is 0): the sums are compared value for value
    finite = getParser().parse("(a || b) * 2 - c / 4")
    cells = np.where(np.isnan(planes[1]), planes[0], planes[0] + planes[1]) * 2 - planes[2] / 4
    assert np.isfinite(cells).all()
    for keep in regions:
        got = GpuStore.regionEvalSum(finite, ["a", "b", "c"], stores, lens, keep)
        sel = cells.reshape(lens)[np.ix_(*_lists(lens, keep))]
        want = float(np.sum(sel))  # pairwise: within a few 1e-15 * sum|v| of the exact sum
        assert abs(got - want) <= 1e-12 * float(np.abs(sel).sum()), (keep[:2], got, want)
    # NaN propagates: (a + b) / c is NaN wherever b is unset or a + b = c = 0
    ratio = getParser().parse("(a + b) / c")
    assert math.isnan(GpuStore.regionEvalSum(ratio, ["a", "b", "c"], stores, lens, regions[1]))
    # copies of the finite formula into a float32 target, bit for bit (a repeated item, the innermost axis filtered)
    target = GpuStore(size, "float32", 0.0)
    want_v = np.zeros(size, dtype=np.float32)
    for keep in ([None, regions[1][1] + regions[1][1][:7], None], [[4, 9, 4], None, regions[2][2]]):
        GpuStore.regionEvalCopy(target, finite, ["a", "b", "c"], stores, lens, keep)
        assert _path() == "region/eval-copy"
        x = cells.astype(np.float32)
        x[x == 0] = 0.0  # -0 -> +0 under a zero default
        want_v.reshape(lens)[np.ix_(*_lists(lens, keep))] = x.reshape(lens)[np.ix_(*_lists(lens, keep))]
        assert np.array_equal(target.data_f32().view(np.uint32), want_v.view(np.uint32)), keep[0]
    assert np.array_equal(_status_np(target), np.where(want_v != 0, 2, 1).astype(np.uint8))
    # getStatus
    merged = np.empty(size, dtype=np.uint8)
    N.check(N.lib().olap_status_merge(N.store_array([s._h for s in stores]), 3, merged.ctypes.data, size))
    assert np.array_equal(merged, _status_np(stores[0]) | _status_np(stores[1]) | _status_np(stores[2]))
    # getStatusMap arrays
    keys, values, is_int = GpuStore.statusMap_arrays(stores)
    present = [~np.isnan(p) if d != d else p != 0 for p, d in zip(planes, defaults)]
    group = np.full(size, -1, dtype=np.int64)
    for k in reversed(range(3)):
        group[present[k]] = k
    assert np.array_equal(keys, np.concatenate([np.flatnonzero(group == k) for k in range(3)]))
    val = np.zeros(size)
    flag = np.zeros(size, dtype=np.uint8)
    have = np.zeros(size, dtype=bool)
    for k in range(3):
        x = planes[k]
        first = present[k] & ~have
        val[first] = x[first]
        later = present[k] & have
        truthy = later & (val == val) & (val != 0)
        val[truthy] = (_to_int32(val[truthy]) | _to_int32(x[truthy])).astype(np.float64)
        flag[truthy] = 1
        other = later & ~truthy
        val[other] = x[other]
        flag[other] = 0
        have |= present[k]
    assert np.array_equal(values, val[keys], equal_nan=True) and np.array_equal(is_int, flag[keys])


def test_single_rank_sharded_cube_matches_the_cube():
    from olap_in_memory_b200.sharded import ShardedCube

    for prefix in (1, 2):
        sharded, one = ShardedCube(R._sharded_dims(), prefix=prefix), Cube(R._sharded_dims(), GpuStore)
        for c in (sharded, one):
            R._sharded_fill(c, 5)
        for f in R.SHARDED_FILTERS:
            got = R.outcome(lambda: sharded.getTotalForDimensionItems("c_sum", f))
            want = R.outcome(lambda: one.getTotalForDimensionItems("c_sum", f))
            R.assert_same_outcome(got, want)
            for dst in ("m_target", "m_ntarget"):
                got = R.outcome(lambda: sharded.copyMeasureData("c_sum", dst, f))
                want = R.outcome(lambda: one.copyMeasureData("c_sum", dst, f))
                assert got == want, (f, dst, got, want)
                a = np.asarray(sharded.getData(dst), dtype=np.float64)
                b = np.asarray(one.getData(dst), dtype=np.float64)
                assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), (prefix, f, dst)


def test_no_write_lands_in_a_guard_region(monkeypatch):
    monkeypatch.setenv("OLAP_GUARD", "1")
    script = (
        "import sys, gc, math; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import test_gpu_computed_queries as T\n"
        "from olap_in_memory_b200 import _native as N\n"
        "T.test_copies_match_the_host_path(1, True)\n"
        "T.test_copies_match_the_host_path(2, False)\n"
        "for b in T.BRANCHES:\n"
        "    T.test_region_sum_branches_against_numpy(b, math.nan)\n"
        "    T.test_region_copy_branches_against_numpy(b, 0.0)\n"
        "T.test_get_status_map_matches_the_host_loop(3, 0)\n"
        "T.test_get_status_matches_the_host_merge((True, False))\n"
        "gc.collect()\n"
        "print('guard_violations', N.lib().olap_guard_violations())\n"
    ) % (ROOT, os.path.join(ROOT, "tests"))
    proc = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
    assert "guard_violations 0" in proc.stdout, proc.stdout[-500:]
