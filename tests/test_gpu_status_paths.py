"""Status bytes and kernel paths of drillUp, drillDown, dice, reorder and load, on every kernel path of
csrc/olap_gpu.cu.

Every entry of the ledgers below names the path (`olap_last_op_path()`) its shape must take with default settings,
so a planner change that reroutes a shape fails here.  Each entry runs under a zero and a NaN default, with and
without status planes, and with input planes that are derived (set by an upload), read (a mutable pointer was handed
out, same content) or read with 0x4 ORed into a third of the set cells (a kernel that re-derives instead of reading
is caught).  Per run: values bit-exact against the C oracle, status bytes equal to tests/status_model.py, a plane the
library calls derived equals derive(values), and a derived and a read plane of identical content give identical
results."""
import math
import re
from pathlib import Path

import numpy as np
import pytest

import cases
import status_model as sm
from oracle.c_oracle import COracleStore

pytestmark = pytest.mark.gpu

ident = cases.identity
PLANES = ("derived", "read", "read4", "mixed")  # mixed: even measures derived, odd ones read4
F32 = ("float32", "sum")


def _G():
    from olap_in_memory_b200.store import GpuStore

    return GpuStore


def _path():
    from olap_in_memory_b200 import _native as N

    return N.lib().olap_last_op_path().decode()


def _mono(rng, n, m):
    return cases.random_map(rng, n, m, True)


def _any(rng, n, m):
    """A non-monotone map that reaches every one of the m targets (n >= m)."""
    out = np.concatenate([np.arange(m), rng.integers(0, m, n - m)]).astype(np.int32)
    return out[rng.permutation(n)]


def _few(rng, n, m):
    """n distinct targets out of m > n: targets without a source (parents without children)."""
    return np.sort(rng.choice(m, n, replace=False)).astype(np.int32)


# (name, old_len, new_len, maps(rng), measures, path); drillUp maps old item -> new item.  A path given as a pair
# (derived, read) names the path of runs without a plane or with derived ones, then of runs that read a plane.
UP = [
    ("mid-vec4", [6, 40, 64], [6, 5, 64], lambda r: [ident(6), _any(r, 40, 5), ident(64)], None, "drillup/mid-vec4"),
    ("mid-vec2-many", [16, 40, 66], [16, 5, 66], lambda r: [ident(16), _any(r, 40, 5), ident(66)], None, "drillup/mid-vec2"),
    ("mid-vec2-few", [1, 1600, 66], [1, 2, 66], lambda r: [ident(1), _any(r, 1600, 2), ident(66)], None, "drillup/mid-vec2"),
    ("mid-scalar-33-many", [2, 1600, 33], [2, 100, 33], lambda r: [ident(2), _any(r, 1600, 100), ident(33)], None, "drillup/mid-scalar"),
    ("i33-few", [1, 1600, 33], [1, 2, 33], lambda r: [ident(1), _mono(r, 1600, 2), ident(33)], None, "drillup/long"),
    ("mid-scalar-129", [2, 40, 129], [2, 5, 129], lambda r: [ident(2), _any(r, 40, 5), ident(129)], None, "drillup/mid-scalar"),
    ("tile", [4096, 40], [4096, 5], lambda r: [ident(4096), _mono(r, 40, 5)], None, "drillup/tile"),
    # rows longer than a shared-memory tile (C * I * 5 bytes > 200 KiB), with and without status planes; the lanes
    # kernel takes derived planes only, a plane that has to be read goes to the long kernel
    ("lanes", [64, 52000], [64, 4], lambda r: [ident(64), _any(r, 52000, 4)], None, ("drillup/lanes", "drillup/long")),
    ("long", [3, 60001], [3, 4], lambda r: [ident(3), _any(r, 60001, 4)], None, "drillup/long"),
    ("generic", [5, 6, 7], [2, 6, 3], lambda r: [_any(r, 5, 2), ident(6), _mono(r, 7, 3)], None, "drillup/generic"),
    ("parent-without-child", [4, 3], [3, 3], lambda r: [np.array([0, 0, 2, 2], np.int32), ident(3)], None, "drillup/tile"),
    ("empty", [0, 3], [1, 3], lambda r: [np.zeros(0, np.int32), ident(3)], None, "drillup/empty"),
    ("20-measures", [16, 40, 66], [16, 5, 66], lambda r: [ident(16), _any(r, 40, 5), ident(66)],
     [("float32", cases.METHODS[k % 7]) for k in range(20)], "drillup/mid-vec2"),
]
UP_MEASURES = [("float32", "sum"), ("float32", "highest"), ("float32", "average")]

# (name, old_len, new_len, maps(rng), measures, path, distributions); drillDown maps new item -> old item
MIXED = [("float32", "sum"), ("int32", "sum"), ("float32", "average")]
DOWN = [
    ("mid-vec4-float", [3, 40, 300], [3, 130, 300], lambda r: [ident(3), _mono(r, 130, 40), ident(300)], [F32], "drilldown/mid-vec4", None),
    ("mid-vec4-mixed", [3, 40, 300], [3, 130, 300], lambda r: [ident(3), _any(r, 130, 40), ident(300)], MIXED, "drilldown/mid-vec4", None),
    ("mid-vec2-float", [3, 40, 258], [3, 130, 258], lambda r: [ident(3), _mono(r, 130, 40), ident(258)], [F32], "drilldown/mid-vec2", None),
    ("mid-scalar-float", [3, 40, 257], [3, 130, 257], lambda r: [ident(3), _any(r, 130, 40), ident(257)], [F32], "drilldown/mid-scalar", None),
    ("mid-int-spread", [2, 30, 64], [2, 100, 64], lambda r: [ident(2), _any(r, 100, 30), ident(64)],
     [("int32", "sum"), ("uint32", "sum")], "drilldown/mid-vec4", None),
    ("inner-rows-vec4-ragged", [500, 12], [500, 40], lambda r: [ident(500), _any(r, 40, 12)], MIXED + [("uint32", "sum")],
     "drilldown/inner-rows", None),
    ("inner-rows-c37", [300, 10], [300, 37], lambda r: [ident(300), _any(r, 37, 10)], MIXED, "drilldown/inner-rows", None),
    ("block-rows-vec4-ragged", [120, 6, 8], [120, 20, 8], lambda r: [ident(120), _any(r, 20, 6), ident(8)],
     [F32, ("float32", "average")], "drilldown/block-rows", None),
    ("block-rows-i3", [200, 5, 3], [200, 17, 3], lambda r: [ident(200), _mono(r, 17, 5), ident(3)], [F32], "drilldown/block-rows", None),
    ("gather-scalar-c9000", [3, 100], [3, 9000], lambda r: [ident(3), _mono(r, 9000, 100)], MIXED, "gather/scalar", None),
    ("gather-rows-two-axes", [4, 6, 5], [9, 6, 11], lambda r: [_any(r, 9, 4), ident(6), _any(r, 11, 5)], MIXED, "gather/rows", None),
    ("gather-vec4-two-axes", [4, 5, 8], [9, 12, 8], lambda r: [_mono(r, 9, 4), _any(r, 12, 5), ident(8)], MIXED, "gather/vec4", None),
    ("gather-rows-dist", [2, 1], [2, 3], lambda r: [ident(2), np.zeros(3, np.int32)], [F32, ("float32", "average")], "gather/rows",
     [0.5, 0.3, 0.2, 0.1, 0.1, 0.8]),
    ("gather-vec4-dist", [4, 1, 8], [4, 3, 8], lambda r: [ident(4), np.zeros(3, np.int32), ident(8)], [F32, ("int32", "sum")],
     "gather/vec4", [0.25, 0.5, 0.25]),
    # the block kernel's shared memory (RB * P * I * 14 + 8 * C + 16 bytes) above its 160 KiB opt-in limit
    ("smem-4096x2", [2, 4096, 2], [2, 8192, 2], lambda r: [ident(2), _mono(r, 8192, 4096), ident(2)], [F32], "gather/rows", None),
    ("smem-1024x8", [2, 1024, 8], [2, 8192, 8], lambda r: [ident(2), _mono(r, 8192, 1024), ident(8)], [F32], "gather/vec4", None),
    ("smem-8000", [3, 8000], [3, 8192], lambda r: [ident(3), _mono(r, 8192, 8000)], [F32], "gather/scalar", None),
    ("smem-7200", [3, 7200], [3, 8192], lambda r: [ident(3), _any(r, 8192, 7200)], [F32], "gather/scalar", None),
    ("smem-parents-without-children", [64, 8000], [64, 100], lambda r: [ident(64), _few(r, 100, 8000)], MIXED, "gather/rows", None),
    ("empty", [3, 2], [3, 0], lambda r: [ident(3), np.zeros(0, np.int32)], [F32], "drilldown/empty", None),
    ("empty-source", [0, 2], [0, 5], lambda r: [np.zeros(0, np.int32), _mono(r, 5, 2)], [F32], "drilldown/empty", None),
]

# (name, op, old_len, arg(rng), path): dice arg = keep lists, reorder arg = new_to_old
MOVE = [
    ("dice-empty", "dice", [8, 4], lambda r: [np.zeros(0, np.int32), ident(4)], "dice/empty"),
    ("dice-inner-flat", "dice", [1000, 10], lambda r: [ident(1000), np.arange(0, 10, 2, dtype=np.int32)], "gather/inner-flat"),
    ("dice-rows", "dice", [10, 15], lambda r: [r.permutation(10)[:4].astype(np.int32), ident(15)], "gather/rows"),
    ("dice-vec4", "dice", [64, 40, 64], lambda r: [ident(64), np.arange(0, 40, 2, dtype=np.int32), ident(64)], "gather/vec4"),
    ("reorder-flat-to-front", "reorder", [300, 7, 10], lambda r: [2, 0, 1], "gather/flat-to-front"),
    ("reorder-planes-to-inner", "reorder", [10, 5004], lambda r: [1, 0], "gather/planes-to-inner"),
    ("reorder-pair", "reorder", [64, 40, 64], lambda r: [2, 1, 0], "reorder/pair-transpose"),
    ("reorder-box", "reorder", [63, 40, 65], lambda r: [2, 1, 0], "reorder/box-transpose"),
    ("reorder-empty", "reorder", [0, 3], lambda r: [1, 0], "reorder/empty"),
]

# (name, my_len, his_len, his_to_mine(rng), path)
LOAD = [
    ("vec4", [6, 12], [3, 8], lambda r: [[None, 4, 1], [4 + j for j in range(8)]], "load/scatter-vec4"),
    ("vec4-folded", [5, 4, 8], [3, 4, 8], lambda r: [[2, None, 0], list(range(4)), list(range(8))], "load/scatter-vec4"),
    ("rows-m0-3", [5, 10], [4, 6], lambda r: [[3, None, 0, 4], [3 + j for j in range(6)]], "load/scatter-rows"),
    ("rows-table", [4, 6], [3, 5], lambda r: [[1, 3, None], [5, None, 0, 2, 3]], "load/scatter-rows"),
    ("rows-folded-odd", [6, 3, 5], [4, 3, 5], lambda r: [[5, 0, None, 2], list(range(3)), list(range(5))], "load/scatter-rows"),
    ("scalar-store", [], [], lambda r: [], "load/scatter"),
]


def _data(rng, n, type, method, default):
    if method == "product":
        return cases.make_data(rng, n, default, 0.7, "small")
    d = cases.make_data(rng, n, default, rng.choice([1.0, 0.7, 0.2]), "int" if type != "float32" or rng.random() < 0.5 else "real")
    if type == "uint32":
        d = np.abs(d)
    if type == "float32" and n:
        # the smallest subnormal: divided by two or more siblings it underflows to 0 (unset under a zero default)
        tiny = rng.random(n) < 0.05
        d[tiny] = np.float32(1.4e-45) * np.where(rng.random(int(tiny.sum())) < 0.5, -1, 1).astype(np.float32)
    return d


def _input_planes(data, default, plane, k):
    """(model bytes, kind) of measure k's input plane for one plane variant."""
    st = sm.derive(data, default)
    kind = plane if plane != "mixed" else ("derived" if k % 2 == 0 else "read4")
    if kind == "read4":
        st[(np.arange(st.size) % 3 == 0) & (st == sm.SET)] |= sm.INTERPOLATED
    return st, kind


def _gpu_store(data, type, default, with_status, kind=None, st=None):
    from olap_in_memory_b200 import interop

    s = _G()(len(data), type, default, with_status=with_status)
    s.set_data_f32(data)
    if with_status and kind in ("read", "read4"):
        import torch

        t = interop.status_tensor(s)  # a mutable pointer handed out: the library no longer calls the plane derived
        if kind == "read4" and t is not None and t.numel():
            t.copy_(torch.from_numpy(st).to(t.device))
    return s


def _oracle(data, type, default):
    o = COracleStore(len(data), type, default)
    o.set_data_f32(data)
    return o


def _cells(values, default):
    """The oracle's doubles as a float32 store holds them: rounded, and -0 (a quotient that underflowed below a
    negative parent) canonicalised to the default +0 under a zero default."""
    v = np.asarray(values).astype(np.float32)
    if default == default:
        v[v == 0] = 0.0
    return v


def _check_out(out, want_values, want_status, with_status, what):
    got = out.data_f32()
    assert cases.bits_equal(got, want_values), f"{what}: values"
    if not with_status:
        return None
    st = np.asarray(out.status, np.uint8)
    if out.status_derived:
        bad = np.flatnonzero(st != sm.derive(got, out._defaultValue))
        assert not bad.size, (f"{what}: a plane marked derived differs from derive(values) at {bad[:8]}: "
                              f"values {got[bad[:8]]}, bytes {st[bad[:8]]}")
    bad = np.flatnonzero(st != want_status)
    assert not bad.size, f"{what}: status bytes at {bad[:8]}\n got  {st[bad[:8]]}\n want {want_status[bad[:8]]}"
    return got.view(np.uint32).tolist(), st.tolist()


def _run_transform(op, stores, entry, methods, dists):
    G = _G()
    if op == "up":
        return G.drillUp_lowered(stores, entry["old"], entry["new"], entry["maps"], methods)
    if op == "down":
        return G.drillDown_lowered(stores, entry["old"], entry["new"], entry["maps"], methods, dists)
    if op == "dice":
        return G.dice_lowered(stores, entry["old"], entry["arg"])
    return G.reorder_lowered(stores, entry["old"], entry["arg"])


def _oracle_transform(op, o, entry, method, dist):
    if op == "up":
        return o.drillUp_lowered(entry["old"], entry["new"], entry["maps"], method)
    if op == "down":
        return o.drillDown_lowered(entry["old"], entry["new"], entry["maps"], method, dist)
    if op == "dice":
        return o.dice_lowered(entry["old"], entry["arg"])
    return o.reorder_lowered(entry["old"], entry["arg"])


def _model(op, st, vin, vout, entry, default):
    if op == "up":
        return sm.drill_up(st, entry["old"], entry["new"], entry["maps"])
    if op == "down":
        return sm.drill_down(st, vin, vout, entry["old"], entry["new"], entry["maps"], default)
    if op == "dice":
        return sm.dice(st, entry["old"], entry["arg"])
    return sm.reorder(st, entry["old"], entry["arg"])


def _check_entry(op, entry, measures, path, dist=None, seed=0):
    wrong = set()
    for default in (0.0, math.nan):
        rng = np.random.default_rng(seed)
        n = int(np.prod(entry["old"]))
        datas = [_data(rng, n, t, m, default) for t, m in measures]
        methods = [m for _, m in measures]
        oracle_in = [_oracle(d, t, default) for d, (t, _) in zip(datas, measures)]
        vins = [o.data_f64() for o in oracle_in]
        wants = [_cells(_oracle_transform(op, o, entry, m, dist).data_f64(), default) for o, m in zip(oracle_in, methods)]
        for with_status in (False, True):
            results = {}
            for plane in PLANES if with_status else (None,):
                stores, planes = [], []
                for k, (d, (t, _)) in enumerate(zip(datas, measures)):
                    st, kind = _input_planes(vins[k], default, plane or "derived", k)
                    stores.append(_gpu_store(d, t, default, with_status, kind, st))
                    planes.append(st)
                outs = _run_transform(op, stores, entry, methods, [dist] * len(measures) if dist else None)
                want_path = path if isinstance(path, str) else path[plane in ("read", "read4", "mixed")]
                if _path() != want_path:
                    wrong.add((plane, _path()))
                results[plane] = [
                    _check_out(out, want, _model(op, st, vin, want, entry, default), with_status,
                               f"{op} {entry['name']} {measures[k]} default={default} status={with_status} plane={plane}")
                    for k, (out, want, st, vin) in enumerate(zip(outs, wants, planes, vins))
                ]
            if with_status:
                assert results["derived"] == results["read"], f"{op} {entry['name']}: a read plane of derived content changes the result"
    assert not wrong, f"{op} {entry['name']}: (plane, path) {sorted(wrong, key=str)}, ledger says {path}"


@pytest.mark.parametrize("name,old,new,maps,measures,path", UP, ids=[e[0] for e in UP])
def test_drillup_status_and_path(name, old, new, maps, measures, path):
    entry = dict(name=name, old=old, new=new, maps=maps(np.random.default_rng(5)))
    _check_entry("up", entry, measures or UP_MEASURES, path, seed=len(name))


@pytest.mark.parametrize("name,old,new,maps,measures,path,dist", DOWN, ids=[e[0] for e in DOWN])
def test_drilldown_status_and_path(name, old, new, maps, measures, path, dist):
    entry = dict(name=name, old=old, new=new, maps=maps(np.random.default_rng(6)))
    _check_entry("down", entry, measures, path, dist, seed=len(name))


@pytest.mark.parametrize("name,old,new,maps,path,dist", [(e[0], e[1], e[2], e[3], e[5], e[6]) for e in DOWN if e[6]],
                         ids=[e[0] for e in DOWN if e[6]])
def test_drilldown_distribution_missing(name, old, new, maps, path, dist):
    """A NaN weight where a truthy parent needs one: both the oracle and the store refuse, on either gather."""
    G = _G()
    m = maps(np.random.default_rng(6))
    holed = list(dist)
    holed[1] = None
    data = np.arange(1, int(np.prod(old)) + 1, dtype=np.float32)
    with pytest.raises(ValueError, match="distribution missing"):
        _oracle(data, "float32", 0.0).drillDown_lowered(old, new, m, "sum", holed)
    with pytest.raises(Exception, match="distribution missing"):
        G.drillDown_lowered([_gpu_store(data, "float32", 0.0, True)], old, new, m, ["sum"], [holed])
    assert _path() == path


@pytest.mark.parametrize("name,op,old,arg,path", MOVE, ids=[e[0] for e in MOVE])
def test_dice_reorder_status_and_path(name, op, old, arg, path):
    entry = dict(name=name, old=old, arg=arg(np.random.default_rng(7)))
    _check_entry(op, entry, [("float32", "sum"), ("float32", "sum")], path, seed=len(name))


@pytest.mark.parametrize("name,my_len,his_len,his_to_mine,path", LOAD, ids=[e[0] for e in LOAD])
def test_load_status_and_path(name, my_len, his_len, his_to_mine, path):
    """load for the four default pairs, source and target each without a plane, derived, read and read4."""
    maps = his_to_mine(np.random.default_rng(8))
    seen = set()
    for my_default in (0.0, math.nan):
        for his_default in (0.0, math.nan):
            rng = np.random.default_rng(len(name))
            mine = cases.make_data(rng, int(np.prod(my_len)), my_default, 0.6, "int")
            his = cases.make_data(rng, int(np.prod(his_len)), his_default, 0.6, "int")
            if his.size:
                his[::5] = 0.0  # unset under a zero default, set under a NaN one: the cross-default cells
            o = _oracle(mine, "float32", my_default)
            o_src = _oracle(his, "float32", his_default)
            o.load_lowered(o_src, my_len, his_len, maps)
            want = _cells(o.data_f64(), my_default)
            his_canon = o_src.data_f64()
            results = {}
            for src_plane in (None, "derived", "read", "read4"):
                for dst_plane in (None, "derived", "read", "read4"):
                    src_st, _ = _input_planes(his_canon, his_default, src_plane or "derived", 0)
                    dst_st, _ = _input_planes(_oracle(mine, "float32", my_default).data_f64(), my_default, dst_plane or "derived", 0)
                    src = _gpu_store(his, "float32", his_default, src_plane is not None, src_plane, src_st)
                    dst = _gpu_store(mine, "float32", my_default, dst_plane is not None, dst_plane, dst_st)
                    dst.load_lowered(src, my_len, his_len, maps)
                    seen.add(_path())
                    model = sm.load(dst_st, src_st if src_plane else None, his_canon, my_len, his_len, maps, my_default)
                    what = f"load {name} my_default={my_default} his_default={his_default} src={src_plane} dst={dst_plane}"
                    results[(src_plane, dst_plane)] = _check_out(dst, want, model, dst_plane is not None, what)
            for a, b in (("derived", "read"),):
                for other in (None, "derived"):
                    assert results[(a, other)] == results[(b, other)], (name, a, b, other)
                    assert results[(other, a)] == results[(other, b)], (name, other, a, b)
    assert seen == {path}, f"load {name}: paths {seen}, ledger says {path}"


def test_shared_status_plane_drilldown():
    """Three measures on ONE status plane (olap_store_create_batch(..., shared_status=1)) through one drillDown call:
    the plane is written once, by the first measure's rule; the values of every measure match the oracle."""
    import ctypes as C

    from olap_in_memory_b200 import _native as N

    G = _G()
    lib = N.lib()
    old, new = [3, 40, 300], [3, 130, 300]
    maps = [ident(3), _any(np.random.default_rng(9), 130, 40), ident(300)]
    n, size = 3, int(np.prod(old))
    for default, kind in ((0.0, 0), (math.nan, 1)):
        handles = (C.c_void_p * n)()
        N.check(lib.olap_store_create_batch(n, size, (C.c_int * n)(2, 2, 2), (C.c_int * n)(kind, kind, kind), 1, 1, handles))
        stores = [G._wrap(handles[k]) for k in range(n)]
        base = _data(np.random.default_rng(10), size, "float32", "sum", default)
        datas = [base * (k + 1) for k in range(n)]  # one fill pattern: the shared plane is exact for every measure
        for s, d in zip(stores, datas):
            s.set_data_f32(d)
        methods = ["sum", "average", "sum"]
        outs = G.drillDown_lowered(stores, old, new, maps, methods)
        assert _path() == "drilldown/mid-vec4"
        assert len({lib.olap_store_status_ptr(o._h) for o in outs}) == 1
        vin = _oracle(datas[0], "float32", default).data_f64()
        for d, m, out in zip(datas, methods, outs):
            want = _cells(_oracle(d, "float32", default).drillDown_lowered(old, new, maps, m).data_f64(), default)
            assert cases.bits_equal(out.data_f32(), want), (default, m)
        want0 = _cells(_oracle(datas[0], "float32", default).drillDown_lowered(old, new, maps, "sum").data_f64(), default)
        model = sm.drill_down(sm.derive(vin, default), vin, want0, old, new, maps, default)
        assert np.array_equal(np.asarray(outs[0].status, np.uint8), model), default


# path literals no ledger entry can reach on one GPU with default settings, and where they are covered instead
EXCLUDED = {
    "gather/vec4-big": "needs more than 2^31 cells: tests/test_gpu_fullsize.py",
    "gather/scalar-big": "needs more than 2^31 cells: tests/test_gpu_fullsize.py",
    "drillup/mid-rows-p2p": "needs peer GPUs: tests/test_gpu_sharded.py",
    "drillup/pull-peers": "needs peer GPUs: tests/test_gpu_pull.py",
    "reorder/tma-transpose": "opt-in: tests/test_gpu_parity.py::test_tma_transpose",
    "reorder/pair-async": "opt-in: tests/test_gpu_parity.py::test_async_pair_transpose",
}


def test_every_path_literal_has_a_ledger_entry():
    """A kernel path added to olap_gpu.cu without an entry above fails here."""
    src = (Path(__file__).resolve().parents[1] / "olap_in_memory_b200" / "csrc" / "olap_gpu.cu").read_text()
    literals = set(re.findall(r'"((?:drillup|drilldown|dice|reorder|gather|load)/[a-z0-9\-]+)"', src))
    assert EXCLUDED.keys() <= literals, sorted(EXCLUDED.keys() - literals)
    ledger = {e[5] for e in DOWN} | {e[-1] for e in MOVE} | {e[-1] for e in LOAD}
    for e in UP:
        ledger |= {e[-1]} if isinstance(e[-1], str) else set(e[-1])
    assert ledger <= literals, sorted(ledger - literals)
    assert not literals - EXCLUDED.keys() - ledger, sorted(literals - EXCLUDED.keys() - ledger)
