"""Reference model of the status plane (DESIGN.md §2 "Status byte"), in plain numpy and independent of the
kernels: 0x1 not set, 0x2 set, 0x4 interpolated.

Every transform takes the input plane as bytes and the lowered arguments the store ABI takes (tests/cases.py);
drillDown and load also need cell values, because whether an output cell is set depends on them.  The values
come from the caller (the C oracle's result, or the source data), never from the device store under test."""
from __future__ import annotations

import numpy as np

UNSET, SET, INTERPOLATED = 0x1, 0x2, 0x4


def present(values, default):
    """A cell is set iff its value differs from the default: under a NaN default any non-NaN value (0 included),
    under a zero default any non-zero value (NaN included)."""
    v = np.asarray(values, dtype=np.float64)
    return ~np.isnan(v) if default != default else v != 0


def derive(values, default):
    """The plane a store has after upload / fill / eval: SET where the value is present, else UNSET."""
    return np.where(present(values, default), SET, UNSET).astype(np.uint8)


def _flat(maps, lens_out):
    """Flat index into the grid `lens_out` of every cell of the grid len(maps[0]) x len(maps[1]) x ...,
    cell (i0, i1, ...) going to (maps[0][i0], maps[1][i1], ...).  A negative map entry poisons the index."""
    idx = np.zeros((), dtype=np.int64)
    bad = np.zeros((), dtype=bool)
    for m, n in zip(maps, lens_out):
        m = np.asarray([-1 if x is None else x for x in m], dtype=np.int64)
        idx = idx[..., None] * int(n) + m
        bad = bad[..., None] | (m < 0)
    return idx.ravel(), bad.ravel()


def drill_up(st, old_len, new_len, maps):
    """maps[d][old item] = new item.  A parent is the OR of all its children's bytes, set or not; a parent
    without any child is UNSET."""
    out = np.zeros(int(np.prod(new_len)), dtype=np.uint8)
    target, _ = _flat([np.arange(n) if m is None else m for m, n in zip(maps, old_len)], new_len)
    np.bitwise_or.at(out, target, np.asarray(st, dtype=np.uint8))
    out[out == 0] = UNSET
    return out


def drill_down(st, parent_values, child_values, old_len, new_len, maps, default):
    """maps[d][new item] = old item.  A child is `parent byte | 0x4` when its parent is truthy (the reference
    skips falsy parents: `if (!oldValue) continue`) and its own value is set; every other child is UNSET
    (integer spreading that lands on 0 under a zero default, a float quotient that underflows, falsy
    parents)."""
    src, _ = _flat(maps, old_len)
    pv = np.asarray(parent_values, dtype=np.float64)[src]
    pb = np.asarray(st, dtype=np.uint8)[src]
    truthy = (pv != 0) & ~np.isnan(pv)
    ok = truthy & present(child_values, default)
    return np.where(ok, pb | INTERPOLATED, UNSET).astype(np.uint8)


def dice(st, old_len, keep):
    """keep[d][new item] = old item: a gather of the bytes."""
    src, _ = _flat(keep, old_len)
    return np.asarray(st, dtype=np.uint8)[src]


def reorder(st, old_len, new_to_old):
    return np.asarray(st, dtype=np.uint8).reshape(old_len).transpose(new_to_old).ravel()


def load(dst_st, src_st, src_values, my_len, his_len, his_to_mine, my_default):
    """his_to_mine[d][his item] = my item, or None / -1 when I lack it (the cell is dropped).  Cells nobody
    writes keep their bytes.  A written cell is UNSET when the value is unset under MY default; when it is set
    it takes the source's byte if that byte has 0x2, else SET (a source without a plane counts as SET).  So a
    set cell is never UNSET-only, whatever the source's default said."""
    out = np.array(dst_st, dtype=np.uint8, copy=True)
    target, drop = _flat(his_to_mine, my_len)
    keep = ~drop
    v = np.asarray(src_values, dtype=np.float64)
    sb = np.full(v.size, SET, np.uint8) if src_st is None else np.asarray(src_st, dtype=np.uint8)
    set_ = present(v, my_default)
    byte = np.where(set_, np.where(sb & SET, sb, SET), UNSET).astype(np.uint8)
    out[target[keep]] = byte[keep]
    return out
