"""The status-byte reference model (tests/status_model.py) against the C oracle and the hand-derived vectors.

The oracle has no status plane, only presence (a cell is set iff it differs from the default), so what can be
pinned against it is the SET bit on inputs whose planes are derived from their values.  The OR, 0x4 and load
rules are pinned by the README vectors below and, on the device, by tests/test_gpu_status_paths.py."""
import itertools
import math

import numpy as np
import pytest

import cases
import status_model as sm
from oracle.c_oracle import COracleStore

ALL = list(itertools.chain(cases.drillup_cases(), cases.drillup_long_cases(), cases.drilldown_cases(), cases.dice_cases(),
                           cases.reorder_cases(), cases.load_cases(), cases.load_linear_cases()))


def _oracle(data, type, default):
    s = COracleStore(len(data), type, default)
    s.set_data_f32(np.asarray(data, np.float32))
    return s


def _model_of_case(case):
    """(model bytes, oracle result store) of one case, its input planes derived from its values."""
    op = case["op"]
    if op == "load":
        dst = _oracle(case["my_data"], "float32", case["my_default"])
        src = _oracle(case["his_data"], "float32", case["his_default"])
        dst_st = sm.derive(dst.data_f64(), case["my_default"])
        src_st = sm.derive(src.data_f64(), case["his_default"])
        dst.load_lowered(src, case["my_len"], case["his_len"], case["his_to_mine"])
        return sm.load(dst_st, src_st, src.data_f64(), case["my_len"], case["his_len"], case["his_to_mine"],
                       case["my_default"]), dst
    src = _oracle(case["data"], case["type"], case["default"])
    vin = src.data_f64()
    st = sm.derive(vin, case["default"])
    if op == "drillUp":
        out = src.drillUp_lowered(case["old_len"], case["new_len"], case["maps"], case["method"])
        return sm.drill_up(st, case["old_len"], case["new_len"], case["maps"]), out
    if op == "drillDown":
        out = src.drillDown_lowered(case["old_len"], case["new_len"], case["maps"], case["method"], case["distributions"])
        return sm.drill_down(st, vin, out.data_f64(), case["old_len"], case["new_len"], case["maps"], case["default"]), out
    if op == "dice":
        return sm.dice(st, case["old_len"], case["keep"]), src.dice_lowered(case["old_len"], case["keep"])
    return sm.reorder(st, case["old_len"], case["new_to_old"]), src.reorder_lowered(case["old_len"], case["new_to_old"])


@pytest.mark.parametrize("case", ALL, ids=[f"{i}-{c['op']}" for i, c in enumerate(ALL)])
def test_set_bit_matches_oracle_presence(case):
    model, out = _model_of_case(case)
    presence = np.asarray(out.status) == sm.SET
    set_bit = (model & sm.SET) != 0
    assert model.dtype == np.uint8 and model.size == out.size
    assert not (model & ~np.uint8(0x7)).any() and (model != 0).all()
    if case["op"] == "drillUp":
        # flags are ORed from the children whatever the aggregate is: a parent with a set child whose aggregate
        # lands on the default (5 + -5 under a zero default, inf + -inf under a NaN one) keeps 0x2
        values = out.data_f64()
        lands_on_default = set_bit & ~presence
        assert not (presence & ~set_bit).any(), cases.describe(case)
        assert (~sm.present(values[lands_on_default], case["default"])).all()
        assert case["method"] in ("sum", "average", "product") or not lands_on_default.any(), cases.describe(case)
    else:
        assert np.array_equal(set_bit, presence), cases.describe(case)


def test_drillup_or_keeps_set_on_a_cancelling_sum():
    st = sm.derive([5.0, -5.0, 0.0], 0.0)
    assert sm.drill_up(st, [3], [1], [np.zeros(3, np.int32)]).tolist() == [3]
    out = _oracle([5.0, -5.0, 0.0], "float32", 0.0).drillUp_lowered([3], [1], [np.zeros(3, np.int32)], "sum")
    assert out.status == [1]  # the value is the default; the flags still say "incomplete"


def test_hand_derived_status_plane_semantics():
    """The vectors of tests/test_gpu_parity.py::test_status_plane_semantics."""
    nan = math.nan
    values = [1, nan, 3, nan, nan, 4]
    st = sm.derive(values, nan)
    assert st.tolist() == [2, 1, 2, 1, 1, 2]
    up = sm.drill_up(st, [3, 2], [3, 1], [cases.identity(3), np.zeros(2, np.int32)])
    assert up.tolist() == [3, 3, 3]
    assert sm.drill_up(st, [3, 2], [1, 2], [np.zeros(3, np.int32), cases.identity(2)]).tolist() == [3, 3]
    parents = [1.0, 3.0, 4.0]
    children = [0.5, 0.5, 1.5, 1.5, 2.0, 2.0]
    dn = sm.drill_down(up, parents, children, [3], [6], [np.repeat(np.arange(3, dtype=np.int32), 2)], nan)
    assert dn.tolist() == [7] * 6


def test_readme_only_status_examples():
    """The vectors of tests/test_gpu_parity.py::test_readme_only_status_examples, lowered."""
    nan = math.nan
    # months rolled up to quarters: Q1 has no month set, Q2 one of three, Q3 all three
    st = sm.derive([nan, nan, nan, 1, nan, nan, 0.5, 0.5, 1], nan)
    q = sm.drill_up(st, [9], [3], [np.repeat(np.arange(3, dtype=np.int32), 3)])
    assert [(s & 3) for s in q.tolist()] == [1, 3, 2] and not (q & 4).any()
    # every cell set and raw; a drillDown quarter -> month interpolates and stays complete
    quarters = [33.0, 7.0, 33.0, 7.0]
    st = sm.derive(quarters, nan)
    assert st.tolist() == [2] * 4
    to_month = [cases.identity(2), np.repeat(np.arange(2, dtype=np.int32), 3)]
    months = _oracle(quarters, "float32", nan).drillDown_lowered([2, 2], [2, 6], to_month, "sum")
    assert months.data_f64()[:3].tolist() == [11.0] * 3
    dn = sm.drill_down(st, quarters, months.data_f64(), [2, 2], [2, 6], to_month, nan)
    assert dn.tolist() == [6] * 12
    # hydrateFromCube copies the flags between cubes
    target = sm.derive([nan] * 12, nan)
    loaded = sm.load(target, dn, months.data_f64(), [2, 6], [2, 6], [list(range(2)), list(range(6))], nan)
    assert loaded.tolist() == [6] * 12


def test_load_rule_across_defaults():
    """A zero-default source's unset cell (0, byte 0x1) is a SET cell of a NaN-default target: it becomes 0x2,
    not 0x1.  A NaN-default source's set 0 is unset under a zero default: 0x1.  Dropped items and cells nobody
    writes keep their bytes."""
    nan = math.nan
    dst = np.array([6, 1, 2, 1], np.uint8)
    src_vals = [0.0, 7.0, 0.0]
    got = sm.load(dst, sm.derive(src_vals, 0.0), src_vals, [4], [3], [[0, 1, None]], nan)
    assert got.tolist() == [2, 2, 2, 1]
    got = sm.load(dst, sm.derive(src_vals, nan), src_vals, [4], [3], [[3, 2, 0]], 0.0)
    assert got.tolist() == [1, 1, 2, 1]
    got = sm.load(dst, np.array([1, 6, 3], np.uint8), src_vals, [4], [3], [[0, 1, 2]], nan)
    assert got.tolist() == [2, 6, 3, 1]
    got = sm.load(dst, None, src_vals, [4], [3], [[1, 2, 3]], nan)  # a source without a plane
    assert got.tolist() == [6, 2, 2, 2]
