"""Region queries on the device (olap_region_sum / olap_region_copy behind Cube.getTotalForDimensionItems,
getDistribution and copyMeasureData): the seeded cases of test_region_queries.py through GpuStore against the
host loop, every lowering branch of the region kernel against numpy on the downloaded planes, a cube larger
than L2, and the guard regions."""
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
from olap_in_memory_b200 import _native as N  # noqa: E402
from olap_in_memory_b200.store import GpuStore  # noqa: E402


def _path():
    return N.lib().olap_last_op_path().decode()


@pytest.mark.parametrize("seed", range(8))
def test_total_and_distribution_match_the_loop(seed):
    cube = R.make_cube(seed, GpuStore)
    for f in R.make_filters(cube, seed):
        for m in R.MEASURES:
            values = R.outcome(lambda: R.loop_values(cube, m, f))
            got = R.outcome(lambda: cube.getTotalForDimensionItems(m, f))
            want = R.outcome(lambda: R.loop_getTotalForDimensionItems(cube, m, f))
            R.assert_same_outcome(got, want, values[1] if values[0] == "ok" else None)
            R.assert_same_outcome(R.outcome(lambda: cube.getDistribution(m, f)),
                                  R.outcome(lambda: R.loop_getDistribution(cube, m, f)))


@pytest.mark.parametrize("seed", range(6))
def test_copy_matches_the_loop(seed):
    for f in R.make_filters(R.make_cube(seed, GpuStore), seed)[:6]:
        for src, dst in R.PAIRS:
            mine, ref = R.make_cube(seed, GpuStore), R.make_cube(seed, GpuStore)
            got = R.outcome(lambda: mine.copyMeasureData(src, dst, f))
            want = R.outcome(lambda: R.loop_copyMeasureData(ref, src, dst, f))
            assert got == want, (got, want)
            if got[0] == "ok":
                for m in mine.storedMeasureIds:
                    a, b = mine.storedMeasures[m], ref.storedMeasures[m]
                    assert np.array_equal(a.data_f32().view(np.uint32), b.data_f32().view(np.uint32)), m
                    assert a.status == b.status, m


def _store(size, default, seed, density=0.6):
    rng = np.random.default_rng(seed)
    v = (rng.integers(-1000, 1000, size) * 0.125).astype(np.float32)
    v[rng.random(size) >= density] = default
    s = GpuStore(size, "float32", default)
    s.set_data_f32(v)
    return s


def _lists(lens, keep):
    return [np.arange(n) if k is None else np.asarray(k, dtype=np.int64) for n, k in zip(lens, keep)]


# every lowering branch of plan_region / region_vec: (lens, keep)
BRANCHES = {
    "whole run, length % 4 == 0": ([8, 64], [[1, 5, 2, 5], None]),
    "whole run, length % 4 != 0": ([8, 30], [[3, 1], None]),
    "filtered innermost axis": ([6, 10], [None, [9, 0, 3, 3]]),
    "every axis filtered": ([5, 6, 7], [[4, 1], [0, 5, 5], [6, 2]]),
    "one cell": ([5, 6, 7], [[2], [3], [4]]),
    "empty region": ([5, 6, 7], [[], None, None]),
    "whole store": ([5, 6, 8], [None, None, None]),
    "multiplicity axis": ([1, 5, 6, 8], [[0, 0, 0], [3], None, [7, 1]]),
}


@pytest.mark.parametrize("branch", list(BRANCHES))
@pytest.mark.parametrize("default", [0.0, math.nan])
def test_region_sum_branches_against_numpy(branch, default):
    lens, keep = BRANCHES[branch]
    s = _store(int(np.prod(lens)), default, 3)
    got = s.regionSum(lens, keep)
    assert _path() == "region/sum"
    sel = s.data_f32().astype(np.float64).reshape(lens)[np.ix_(*_lists(lens, keep))].ravel()
    if np.isnan(sel).any():
        assert math.isnan(got)
    else:
        assert abs(got - math.fsum(sel)) <= 1e-12 * np.abs(sel).sum(), (got, math.fsum(sel))
    again = s.regionSum(lens, keep)
    assert np.float64(again).view(np.uint64) == np.float64(got).view(np.uint64)


def _emulate_copy(dst_v, src_v, lens, keep, dst_default):
    """setValue(i, src[i]) on the host: canonical value and status byte by the target's rule."""
    out = dst_v.copy().reshape(lens)
    st = np.where(np.isnan(dst_v) if dst_default != dst_default else dst_v == 0, 1, 2).astype(np.uint8).reshape(lens)
    ix = np.ix_(*_lists(lens, keep))
    x = src_v.reshape(lens)[ix].copy()
    x[np.isnan(x)] = np.float32(np.nan)
    if dst_default == 0:
        x[x == 0] = 0.0  # -0 -> +0
    out[ix] = x
    st[ix] = np.where(np.isnan(x) if dst_default != dst_default else x == 0, 1, 2)
    return out.ravel(), st.ravel()


@pytest.mark.parametrize("branch", list(BRANCHES))
@pytest.mark.parametrize("src_default,dst_default", [(math.nan, 0.0), (0.0, math.nan), (0.0, 0.0)])
def test_region_copy_branches_against_numpy(branch, src_default, dst_default):
    lens, keep = BRANCHES[branch]
    size = int(np.prod(lens))
    src, dst = _store(size, src_default, 4), _store(size, dst_default, 5)
    before = dst.data_f32()
    want_v, want_st = _emulate_copy(before, src.data_f32(), lens, keep, dst_default)
    dst.regionCopy(src, lens, keep)
    assert _path() == "region/copy"
    got = dst.data_f32()
    # canonical NaN bits, cells outside the region bit-identical
    assert np.array_equal(got.view(np.uint32), want_v.view(np.uint32))
    assert np.array_equal(np.asarray(dst.status, dtype=np.uint8), want_st)


def test_copy_into_itself_changes_nothing():
    lens, keep = [6, 8, 12], [[5, 0, 5], None, None]
    s = _store(6 * 8 * 12, math.nan, 9)
    before, status = s.data_f32(), s.status
    s.regionCopy(s, lens, keep)
    assert np.array_equal(s.data_f32().view(np.uint32), before.view(np.uint32)) and s.status == status


def test_argument_errors():
    s = _store(24, 0.0, 1)
    with pytest.raises(N.OlapValueError, match="dimensions describe 20 cells, store has 24"):
        s.regionSum([4, 5], [None, None])
    with pytest.raises(N.OlapValueError, match="lists item 6, outside"):
        s.regionSum([4, 6], [None, [6]])
    with pytest.raises(N.OlapValueError, match="stores of 24 and 12 cells"):
        s.regionCopy(_store(12, 0.0, 2), [4, 6], [None, None])


def test_config2_sized_cube_against_numpy():
    """3652 days x 32^3 = 1.2e8 cells (480 MB, larger than the 126 MB L2): the four workloads of bench_region.py."""
    lens = [3652, 32, 32, 32]
    size = int(np.prod(lens))
    rng = np.random.default_rng(2)
    v = rng.standard_normal(size, dtype=np.float32)
    s = GpuStore(size, "float32", 0)
    s.set_data_f32(v)
    plane = s.data_f32().astype(np.float64).reshape(lens)
    g1 = rng.permutation(32)[:16].tolist()
    for keep in ([list(range(31, 61)), None, None, None], [None, g1, None, None], [None, None, None, list(range(0, 32, 2))],
                 [None, None, None, None]):
        got = s.regionSum(lens, keep)
        sel = plane[np.ix_(*_lists(lens, keep))]
        want = float(np.sum(sel, dtype=np.float64))
        assert abs(got - want) <= 1e-12 * float(np.abs(sel).sum()) + 1e-9, (keep[:2], got, want)


def test_no_write_lands_in_a_guard_region(monkeypatch):
    monkeypatch.setenv("OLAP_GUARD", "1")
    script = (
        "import sys, gc, math; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import test_gpu_region as T\n"
        "from olap_in_memory_b200 import _native as N\n"
        "for b in T.BRANCHES:\n"
        "    for sd, dd in ((math.nan, 0.0), (0.0, math.nan)):\n"
        "        T.test_region_copy_branches_against_numpy(b, sd, dd)\n"
        "gc.collect()\n"
        "print('guard_violations', N.lib().olap_guard_violations())\n"
    ) % (ROOT, os.path.join(ROOT, "tests"))
    proc = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
    assert "guard_violations 0" in proc.stdout, proc.stdout[-500:]
