"""Cube orchestrator (host side).  Same public API and query semantics as
/root/reference/src/cube.js:34-1186 (method names kept verbatim so a user of
the reference finds the calls they know); every O(cells) step is delegated to
the store — by default the device-resident GpuStore behind the C ABI.

Differences from the reference, all on the store side of the boundary:
* one store call covers ALL stored measures of the cube (`*_many` batched
  entry points) instead of one call per measure (cube.js:1012-1020), so index
  maps are uploaded once per query and one launch serves every measure;
* computed measures are evaluated by one fused device kernel instead of a
  per-cell tree walk (cube.js:353-360).
There is no CPU fallback: without the CUDA library every store call raises."""
from __future__ import annotations

import copy

import numpy as np
import itertools
import re

from . import formatter
from .dimension.catch_all import CatchAll
from .dimension.timeslot import TimeSlot
from .parser import getParser

_MEASURE_ID = re.compile(r"^[a-z][_a-z0-9]+$|^[_a-z0-9]+__total$", re.IGNORECASE)


def _default_store_cls():
    from .store import GpuStore

    return GpuStore


def _to_int32(x):
    """JS ToInt32: NaN / infinities -> 0, truncation toward zero, wrap modulo 2^32 into [-2^31, 2^31)."""
    if x != x or x in (float("inf"), float("-inf")):
        return 0
    n = int(x) & 0xFFFFFFFF
    return n - (1 << 32) if n >= (1 << 31) else n


def _js_or(a, b):
    return _to_int32(a) | _to_int32(b)


def _check_measure_id(measureId):
    if not _MEASURE_ID.match(measureId):
        raise ValueError(f"Invalid measureId: {measureId}")


def _check_coords(dimensions, who, coords):
    ids = [d.id for d in dimensions]
    if any(not coords.get(d) for d in ids):
        raise ValueError(f"{who}: no value for all dimensions. Dimensions: {','.join(ids)}, Coords: {coords}")


def _position(dimensions, coords):
    position = 0
    for dimension in dimensions:
        if dimension.id not in coords:
            raise ValueError(f"getPosition: no such dimension {dimension.id}. Coords: {coords}")
        index = dimension.getRootIndexFromRootItem(coords[dimension.id])
        if index == -1:
            raise ValueError(f"getPosition: no such item {coords[dimension.id]}. Dimension items: {dimension.getItems()}")
        position = position * dimension.numItems + index
    return position


def _check_readable(storedMeasures, computedMeasures, measureId):
    """What getSingleData(measureId, coords) raises for a measure, once the coordinates are valid."""
    if measureId in storedMeasures:
        return
    if measureId in computedMeasures:
        for name in computedMeasures[measureId].variables():
            if name not in storedMeasures:
                raise KeyError(name)  # an `x__total` variable: the per-cell evaluation has no such store
        return
    raise KeyError(f"getSingleData: no such measure {measureId}")


def _region(dimensions, dimensionsFilter, check_measures):
    """The combinations of getTotalForDimensionItems / copyMeasureData (cube.js) as one region of the store:
    (lens, keep), keep[d] = item indices of dimension d in filter order, repeats kept, or None for a dimension
    the filter does not name.  A filter key that is not a dimension multiplies every combination by the length
    of its list: a leading axis of one item listed that many times.  None when there is no combination.

    Raises what the loop raises on its first failing combination, in its order (filter keys in dict order,
    then the other dimensions, last key fastest); `check_measures` raises what every valid combination would."""
    options = {k: ([v] if isinstance(v, str) else list(v)) for k, v in (dimensionsFilter or {}).items()}
    for d in dimensions:
        if d.id not in options:
            options[d.id] = None
    keys = list(options)
    by_id = {d.id: d for d in dimensions}
    if any((by_id[k].numItems if v is None else len(v)) == 0 for k, v in options.items()):
        return None

    def bad(key, item):
        return key in by_id and (not item or by_id[key].getRootIndexFromRootItem(item) == -1)

    def first_item(key):
        return options[key][0] if options[key] is not None else by_id[key].getItems()[0]

    def fail(combination):
        _check_coords(dimensions, "getSingleData", combination)
        _position(dimensions, combination)

    first = {k: first_item(k) for k in keys}
    if any(bad(k, v) for k, v in first.items()):
        fail(first)
    check_measures()
    # the first failing combination differs from the first one in ONE key: the fastest-varying key that has a bad item
    for k in reversed(keys):
        if options[k] is None:
            continue
        for item in options[k]:
            if bad(k, item):
                fail({**first, k: item})
    lens, keep = [d.numItems for d in dimensions], []
    for d in dimensions:
        items = options[d.id]
        keep.append(None if items is None else np.array([d.getRootIndexFromRootItem(i) for i in items], dtype=np.int32))
    multiplicity = 1
    for k in keys:
        if k not in by_id:
            multiplicity *= len(options[k])
    if multiplicity != 1:
        lens, keep = [1] + lens, [np.zeros(multiplicity, dtype=np.int32)] + keep
    return lens, keep


def _formula_inputs(store_cls, member, computedMeasures, storedMeasures, measureId):
    """(expression, cell names, their stores) of a computed measure when the store class has `member` (the device
    forms of the region queries and status accessors) and the formula reads at least one cell; else None, and the
    caller keeps its host code.  Formulas with an `x__total` variable were rejected by _check_readable before."""
    if getattr(store_cls, member, None) is None:
        return None
    expression = computedMeasures[measureId]
    cell_names = [n for n in expression.variables() if "__total" not in n]
    if not cell_names:
        return None
    return expression, cell_names, [storedMeasures[n] for n in cell_names]


def _region_lists(lens, keep):
    return [np.arange(n) if k is None else np.asarray(k, dtype=np.int64) for n, k in zip(lens, keep)]


def _region_sum_f64(data, lens, keep):
    """Region sum of a computed measure evaluated on the host (doubles)."""
    return float(data.reshape(lens)[np.ix_(*_region_lists(lens, keep))].sum())


def _region_set_f64(store, data, lens, keep):
    """store.setValue(i, data[i]) for every cell i of the region (a computed source): one batched call."""
    index = np.ravel_multi_index(np.ix_(*_region_lists(lens, keep)), lens).ravel() if lens else np.zeros(1, np.int64)
    if hasattr(store, "setValues"):
        store.setValues(index, data[index])
    else:
        for i in index.tolist():
            store.setValue(i, float(data[i]))


class Cube:
    def __init__(self, dimensions, store_cls=None):
        self.dimensions = list(dimensions)
        self.storedMeasures = {}
        self.storedMeasuresRules = {}
        self.computedMeasures = {}
        self._store_cls = store_cls or _default_store_cls()

    # ------------------------------------------------------------------ sizes
    @property
    def storeSize(self):
        size = 1
        for d in self.dimensions:
            size *= d.numItems
        return size

    @property
    def byteLength(self):
        return sum(store.byteLength for store in self.storedMeasures.values())

    @property
    def dimensionIds(self):
        return [d.id for d in self.dimensions]

    @property
    def storedMeasureIds(self):
        return list(self.storedMeasures.keys())

    @property
    def computedMeasureIds(self):
        return list(self.computedMeasures.keys())

    def getDimension(self, dimensionId):
        for d in self.dimensions:
            if d.id == dimensionId:
                return d
        return None

    def getDimensionIndex(self, dimensionId):
        for i, d in enumerate(self.dimensions):
            if d.id == dimensionId:
                return i
        return -1

    # --------------------------------------------------------------- measures
    def clone(self, measures=()):
        out = Cube(copy.deepcopy(self.dimensions), self._store_cls)
        keep = (lambda ids: list(ids)) if not measures else (lambda ids: [m for m in ids if m in measures])
        for m in keep(self.computedMeasureIds):
            out.computedMeasures[m] = self.computedMeasures[m]
        for m in keep(self.storedMeasureIds):
            out.storedMeasures[m] = self.storedMeasures[m].clone()
            out.storedMeasuresRules[m] = copy.deepcopy(self.storedMeasuresRules[m])
        return out

    def createComputedMeasure(self, measureId, formula):
        _check_measure_id(measureId)
        if measureId in self.storedMeasures or measureId in self.computedMeasures:
            raise ValueError(f"This measure already exists {measureId}")
        # formulas may reference other computed measures: inline them (cube.js:107-121)
        for other in self.computedMeasureIds:
            pattern = re.compile(rf"\b{re.escape(other)}\b")
            if pattern.search(formula):
                formula = pattern.sub(f"({self.computedMeasures[other].toString()})", formula)
        expression = getParser().parse(formula)
        known = set(self.storedMeasureIds) | {f"{m}__total" for m in self.storedMeasureIds}
        unknown = [v for v in expression.variables() if v not in known]
        if unknown:
            raise ValueError(f"Unknown measure(s): {','.join(unknown)}")
        self.computedMeasures[measureId] = expression

    def copyStoredMeasure(self, measureId, copyMeasureId):
        _check_measure_id(copyMeasureId)
        if measureId not in self.storedMeasures:
            raise ValueError(f"This measure does not exists: {measureId}")
        if copyMeasureId in self.storedMeasures:
            raise ValueError(f"This measure already exists: {copyMeasureId}")
        self.storedMeasures[copyMeasureId] = self.storedMeasures[measureId].clone()
        self.storedMeasuresRules[copyMeasureId] = copy.deepcopy(self.storedMeasuresRules[measureId])

    def createStoredMeasure(self, measureId, rules=None, type="float32", defaultValue=0):
        _check_measure_id(measureId)
        if measureId in self.storedMeasures:
            raise ValueError(f"This measure already exists: {measureId}")
        self.storedMeasures[measureId] = self._store_cls(self.storeSize, type, defaultValue)
        self.storedMeasuresRules[measureId] = {} if rules is None else rules

    def cloneStoredMeasure(self, originCube, measureId):
        _check_measure_id(measureId)
        if measureId in self.storedMeasures:
            raise ValueError(f"This measure already exists: {measureId}")
        if measureId not in originCube.storedMeasures:
            raise ValueError(f"This measure does not exists in originCube: {measureId}")
        self.storedMeasuresRules[measureId] = dict(originCube.storedMeasuresRules[measureId])
        origin = originCube.storedMeasures[measureId]
        self.storedMeasures[measureId] = self._store_cls(self.storeSize, origin._type, origin._defaultValue)

    def copyToStoredMeasure(self, computedMeasureId, storedMeasureId, rules=None, type="float32", defaultValue=0):
        data = self.getData(computedMeasureId)
        self.createStoredMeasure(storedMeasureId, rules, type, defaultValue)
        self.setData(storedMeasureId, data)

    def convertToStoredMeasure(self, measureId, rules=None, type="float32", defaultValue=0):
        if measureId not in self.computedMeasures:
            raise ValueError(f"convertToStoredMeasure: no such computed measure: {measureId}")
        data = self.getData(measureId)
        self.dropMeasure(measureId)
        self.createStoredMeasure(measureId, rules, type, defaultValue)
        self.setData(measureId, data)

    def renameMeasure(self, oldMeasureId, newMeasureId):
        if oldMeasureId == newMeasureId:
            return
        if oldMeasureId in self.computedMeasures:
            self.computedMeasures[newMeasureId] = self.computedMeasures.pop(oldMeasureId)
        elif oldMeasureId in self.storedMeasures:
            self.storedMeasures[newMeasureId] = self.storedMeasures.pop(oldMeasureId)
            self.storedMeasuresRules[newMeasureId] = self.storedMeasuresRules.pop(oldMeasureId)
            for cid, expression in list(self.computedMeasures.items()):
                if oldMeasureId in expression.variables():
                    self.computedMeasures[cid] = expression.substitute(oldMeasureId, newMeasureId)
        else:
            raise ValueError(f"renameMeasure: no such measure {oldMeasureId} -> {newMeasureId}")

    def replaceStoredMeasure(self, toKeep, toDrop):
        for m in (toKeep, toDrop):
            if m not in self.storedMeasures:
                raise ValueError(f"replaceStoredMeasure: no such measure {m}")
        for cid, expression in list(self.computedMeasures.items()):
            if toDrop in expression.variables():
                self.computedMeasures[cid] = expression.substitute(toDrop, toKeep)
        self.dropMeasure(toDrop)

    def dropMeasure(self, measureId):
        if measureId in self.computedMeasures:
            del self.computedMeasures[measureId]
        elif measureId in self.storedMeasures:
            del self.storedMeasures[measureId]
            del self.storedMeasuresRules[measureId]
            for cid in [c for c, e in self.computedMeasures.items() if measureId in e.variables()]:
                del self.computedMeasures[cid]
        else:
            raise ValueError(f"dropMeasure: no such measure: {measureId}")

    def dropMeasures(self, measureIds):
        for m in measureIds:
            self.dropMeasure(m)

    def keepMeasure(self, measureId):
        self.keepMeasures([measureId])

    def keepMeasures(self, measureIds):
        for m in self.computedMeasureIds + self.storedMeasureIds:
            if m not in measureIds and (m in self.computedMeasures or m in self.storedMeasures):
                self.dropMeasure(m)

    def updateStoredMeasureRules(self, measureId, cb):
        self.storedMeasuresRules[measureId] = cb(self.storedMeasuresRules[measureId])

    # ------------------------------------------------------------ data access
    def getData(self, measureId):
        if measureId in self.storedMeasures:
            return self.storedMeasures[measureId].data
        if measureId in self.computedMeasures:
            expression = self.computedMeasures[measureId]
            names = expression.variables()
            cell_names = [n for n in names if "__total" not in n]
            totals = {n: self.storedMeasures[n.replace("__total", "")].total for n in names if "__total" in n}
            return self._store_cls.evaluate(
                expression, cell_names, [self.storedMeasures[n] for n in cell_names], totals, self.storeSize
            )
        raise KeyError(f"getData: no such measure {measureId}")

    def evaluateToStore(self, measureId, type="float32", defaultValue=0):
        """getData(computedId) kept on the device as a new store — the device-side half
        of copyToStoredMeasure (cube.js:205-215), without the host round trip."""
        expression = self.computedMeasures[measureId]
        names = expression.variables()
        cell_names = [n for n in names if "__total" not in n]
        totals = {n: self.storedMeasures[n.replace("__total", "")].total for n in names if "__total" in n}
        return self._store_cls.evaluate_to_store(
            expression, cell_names, [self.storedMeasures[n] for n in cell_names], totals, type, defaultValue
        )

    def getStatusMap(self, measureId):
        """Map cell index -> value of the cells that are set (cube.js:368-389)."""
        if measureId in self.storedMeasures:
            return self.storedMeasures[measureId]._dataMap
        if measureId in self.computedMeasures:
            status_map = getattr(self._store_cls, "statusMap", None)
            if status_map is not None:
                return status_map(list(self.storedMeasures.values())) if self.storedMeasures else {}
            # cube.js:374-386: union of the stored measures' keys in first-seen order; a key seen before
            # with a truthy value gets  previous | value  (JS ToInt32 bitwise OR), else the value itself
            result = {}
            for store in self.storedMeasures.values():
                for key, value in store._dataMap.items():
                    previous = result.get(key)
                    if previous is not None and previous == previous and previous != 0:
                        result[key] = _js_or(previous, value)
                    else:
                        result[key] = value
            return result
        raise KeyError(f"getStatusMap: no such measure {measureId}")

    def getStatus(self, measureId):
        """Status byte of every cell, in getData() order (README.md:694-721:
        0x1 not set, 0x2 set, 0x4 interpolated; drillUp ORs its children)."""
        if measureId in self.storedMeasures:
            return self.storedMeasures[measureId].status
        if measureId in self.computedMeasures:
            fused = _formula_inputs(self._store_cls, "statusMerge", self.computedMeasures, self.storedMeasures, measureId)
            if fused is not None:
                return self._store_cls.statusMerge(fused[2], self.storeSize)
            merged = None
            for name in self.computedMeasures[measureId].variables():
                if "__total" in name:
                    continue
                status = self.storedMeasures[name].status
                merged = status if merged is None else [a | b for a, b in zip(merged, status)]
            return merged if merged is not None else [0x2] * self.storeSize
        raise KeyError(f"getStatus: no such measure {measureId}")

    def fillData(self, measureId, value):
        if measureId not in self.storedMeasures:
            raise ValueError(f"fillData can only be called on stored measures: {measureId}")
        self.storedMeasures[measureId].fill(value)

    def setData(self, measureId, values):
        if measureId not in self.storedMeasures:
            raise ValueError(f"setData can only be called on stored measures: {measureId}")
        self.storedMeasures[measureId].data = values

    def getNestedArray(self, measureId):
        return formatter.toNestedArray(self.getData(measureId), None, self.dimensions)

    def setNestedArray(self, measureId, values):
        self.setData(measureId, formatter.fromNestedArray(values, self.dimensions))

    def getNestedObject(self, measureId, withTotals=False):
        if not withTotals or len(self.dimensions) == 0:
            return formatter.toNestedObject(self.getData(measureId), None, self.dimensions)
        return self.getNestedObjects([measureId], True)[measureId]

    def _totals_lattice(self):
        """Every sub-cube of cube.js:429-439 / 454-462 (dimension i rolled up to 'all' iff bit
        i of the mask is set), each computed ONCE: the reference rebuilds mask j from the full
        cube (D * 2^(D-1) store passes); its chain for j is the chain for j without its highest
        bit followed by one more drillUp, so walking the masks as a tree gives the same
        operations in the same order with 2^D - 1 passes over ever smaller stores."""
        def walk(cube, mask, start):
            yield mask, cube
            for i in range(start, len(self.dimensions)):
                yield from walk(cube.drillUp(self.dimensions[i].id, "all"), mask | (1 << i), i + 1)

        return walk(self, 0, 0)

    def getNestedObjects(self, measureIds, withTotals=False):
        if not withTotals or len(self.dimensions) == 0:
            return {m: formatter.toNestedObject(self.getData(m), None, self.dimensions) for m in measureIds}
        parts = {mask: {m: sub.getNestedObject(m, False) for m in measureIds} for mask, sub in self._totals_lattice()}
        result = {}
        for mask in sorted(parts):  # merge in the reference's order (ascending mask)
            _deep_merge(result, parts[mask])
        return result

    def setNestedObject(self, measureId, value):
        self.setData(measureId, formatter.fromNestedObject(value, self.dimensions))

    def hydrateFromSparseNestedObject(self, measureId, obj, offset=0, dimOffset=0):
        """cube.js:472-491.  The reference calls setValue per leaf; here the leaves are
        collected first and written with ONE batched store call when the store has one."""
        store = self.storedMeasures[measureId]
        indexes, values = [], []
        self._collect_sparse(obj, offset, dimOffset, indexes, values)
        if hasattr(store, "setValues") and len(indexes) > 1:
            d = float(store._defaultValue)
            store.setValues(indexes, [d if v is None else v for v in values])
        else:
            for index, value in zip(indexes, values):
                store.setValue(index, value)

    def _collect_sparse(self, obj, offset, dimOffset, indexes, values):
        if dimOffset == len(self.dimensions):
            indexes.append(offset)
            values.append(obj)
            return
        dimension = self.dimensions[dimOffset]
        for key, child in obj.items():
            item_offset = dimension.getRootIndexFromRootItem(key)
            if item_offset != -1:
                self._collect_sparse(child, offset * dimension.numItems + item_offset, dimOffset + 1, indexes, values)

    def _check_coords(self, who, coords):
        _check_coords(self.dimensions, who, coords)

    def setSingleData(self, measureId, coords, value):
        self._check_coords("setSingleData", coords)
        if measureId not in self.storedMeasures:
            raise ValueError(f"setSingleData: no such stored measure {measureId}")
        self.storedMeasures[measureId].setValue(self.getPosition(coords), value)

    def getSingleData(self, measureId, coords):
        self._check_coords("getSingleData", coords)
        position = self.getPosition(coords)
        if measureId in self.storedMeasures:
            return self.storedMeasures[measureId].getValue(position)
        if measureId in self.computedMeasures:
            expression = self.computedMeasures[measureId]
            params = {m: self.storedMeasures[m].getValue(position) for m in expression.variables()}
            return expression.evaluate(params)
        raise KeyError(f"getSingleData: no such measure {measureId}")

    def getPosition(self, coords):
        return _position(self.dimensions, coords)

    def getTotal(self, measureId):
        return self.storedMeasures[measureId].total

    def getDimensionItemsMap(self, dimensionIds=None):
        ids = self.dimensionIds if dimensionIds is None else [d for d in self.dimensionIds if d in dimensionIds]
        return {d: self.getDimension(d).getItems() for d in ids}

    def _combinations(self, options):
        keys = list(options.keys())
        return [dict(zip(keys, combo)) for combo in itertools.product(*[options[k] for k in keys])]

    # getTotalForDimensionItems / copyMeasureData: the reference loops over every combination of the
    # filter's items with getSingleData / setSingleData.  Here the combinations are one region of the
    # store (per-dimension item lists, _region) and one store call covers it; results and errors are
    # those of the loop.
    def getTotalForDimensionItems(self, measureId, dimensionsFilter=None):
        region = _region(self.dimensions, dimensionsFilter,
                         lambda: _check_readable(self.storedMeasures, self.computedMeasures, measureId))
        if region is None:
            return 0
        lens, keep = region
        if measureId in self.storedMeasures:
            return self.storedMeasures[measureId].regionSum(lens, keep)
        fused = _formula_inputs(self._store_cls, "regionEvalSum", self.computedMeasures, self.storedMeasures, measureId)
        if fused is not None:
            return self._store_cls.regionEvalSum(*fused, lens, keep)
        return _region_sum_f64(np.asarray(self.getData(measureId), dtype=np.float64), lens, keep)

    def getDistribution(self, measureId, dimensionsFilter=None):
        space = self.getTotalForDimensionItems(measureId, dimensionsFilter)
        total = self.getTotal(measureId)
        return space if total == 0 else space / total

    def copyMeasureData(self, sourceMeasureId, targetMeasureId, dimensionsFilter=None):
        def check():
            _check_readable(self.storedMeasures, self.computedMeasures, sourceMeasureId)
            if targetMeasureId not in self.storedMeasures:
                raise ValueError(f"setSingleData: no such stored measure {targetMeasureId}")

        region = _region(self.dimensions, dimensionsFilter, check)
        if region is None:
            return
        lens, keep = region
        target = self.storedMeasures[targetMeasureId]
        if sourceMeasureId in self.storedMeasures:
            target.regionCopy(self.storedMeasures[sourceMeasureId], lens, keep)
            return
        fused = _formula_inputs(self._store_cls, "regionEvalCopy", self.computedMeasures, self.storedMeasures, sourceMeasureId)
        if fused is not None:
            self._store_cls.regionEvalCopy(target, *fused, lens, keep)
        else:
            _region_set_f64(target, np.asarray(self.getData(sourceMeasureId), dtype=np.float64), lens, keep)

    def scan(self, dimensionIds, cb):
        for combination in self._combinations(self.getDimensionItemsMap(dimensionIds)):
            cb(self.diceByDimensionItems(combination), combination)

    def iterateOverDimension(self, dimension, cb):
        others = [d for d in self.dimensionIds if d != dimension]
        if len(others) == len(self.dimensionIds):
            raise ValueError(f"Cube has no {dimension} dimension. Dimensions: {self.dimensionIds}")
        if not others:
            cb(self, {})
            return
        self.scan(others, lambda diced, items: cb(diced.aggregateByDimensions([dimension]), items))

    # ------------------------------------------------- the cube-transform path
    def _derive(self, newDimensions, storedIds=None, computedIds=None, rules="share"):
        """New cube over `newDimensions` carrying computed measures and rules."""
        out = Cube(newDimensions, self._store_cls)
        for m in self.computedMeasureIds if computedIds is None else computedIds:
            out.computedMeasures[m] = self.computedMeasures[m]
        ids = self.storedMeasureIds if storedIds is None else storedIds
        for m in ids:
            rule = self.storedMeasuresRules[m]
            out.storedMeasuresRules[m] = rule if rules == "share" else copy.deepcopy(rule)
        return out, ids

    def _apply(self, out, ids, op, *args):
        """Run one store transform over every stored measure in `ids` (batched)."""
        stores = [self.storedMeasures[m] for m in ids]
        many = getattr(self._store_cls, op + "_many", None)
        if many is not None:
            results = many(stores, *args) if stores else []
        else:
            per_store = [a for a in args]
            results = []
            for k, store in enumerate(stores):
                call_args = [a[k] if isinstance(a, _PerMeasure) else a for a in per_store]
                results.append(getattr(store, op)(*call_args))
        for m, store in zip(ids, results):
            out.storedMeasures[m] = store
        return out

    def drillUp(self, dimensionId, attribute):
        """Aggregate one dimension by a coarser attribute (cube.js:995-1023)."""
        dimIdx = self.getDimensionIndex(dimensionId)
        if self.dimensions[dimIdx].rootAttribute == attribute:
            return self
        newDimensions = list(self.dimensions)
        newDimensions[dimIdx] = newDimensions[dimIdx].drillUp(attribute)
        if newDimensions[dimIdx] is self.dimensions[dimIdx]:
            return self
        out, ids = self._derive(newDimensions)
        methods = _PerMeasure([self.storedMeasuresRules[m].get(dimensionId) or "sum" for m in ids])
        return self._apply(out, ids, "drillUp", self.dimensions, newDimensions, methods)

    def drillDown(self, dimensionId, attribute):
        """Split one dimension into a finer attribute (cube.js:966-989)."""
        dimIdx = self.getDimensionIndex(dimensionId)
        if self.dimensions[dimIdx].rootAttribute == attribute:
            return self
        newDimensions = list(self.dimensions)
        newDimensions[dimIdx] = newDimensions[dimIdx].drillDown(attribute)
        if newDimensions[dimIdx] is self.dimensions[dimIdx]:
            return self
        out, ids = self._derive(newDimensions)
        methods = _PerMeasure([self.storedMeasuresRules[m].get(dimensionId) or "sum" for m in ids])
        return self._apply(out, ids, "drillDown", self.dimensions, newDimensions, methods, _PerMeasure([None] * len(ids)))

    def addDimension(self, newDimension, aggregation=None, index=None, distributions=None):
        """cube.js:910-948: insert a one-item placeholder then drill it down."""
        aggregation = aggregation or {}
        distributions = distributions or {}
        at = len(self.dimensions) if index is None else index
        oldDimensions = list(self.dimensions)
        oldDimensions.insert(at, CatchAll(newDimension.id, newDimension))
        newDimensions = list(oldDimensions)
        newDimensions[at] = newDimension
        out, ids = self._derive(newDimensions, rules="copy")
        for m in out.storedMeasuresRules:
            out.storedMeasuresRules[m][newDimension.id] = aggregation.get(m)
        methods = _PerMeasure([aggregation.get(m) or "sum" for m in ids])
        dists = _PerMeasure([distributions.get(m) for m in ids])
        return self._apply(out, ids, "drillDown", oldDimensions, newDimensions, methods, dists)

    def removeDimension(self, dimensionId):
        """cube.js:950-964: drillUp to 'all', then forget the dimension."""
        rolled = self.drillUp(dimensionId, "all")
        out = Cube([d for d in self.dimensions if d.id != dimensionId], self._store_cls)
        out.storedMeasures = dict(rolled.storedMeasures)
        out.computedMeasures.update(self.computedMeasures)
        out.storedMeasuresRules = copy.deepcopy(self.storedMeasuresRules)
        for rule in out.storedMeasuresRules.values():
            rule.pop(dimensionId, None)
        return out

    def dice(self, dimensionId, attribute, items, reorder=False):
        """Keep some items of one dimension (cube.js:834-857)."""
        dimIdx = self.getDimensionIndex(dimensionId)
        newDimensions = list(self.dimensions)
        newDimensions[dimIdx] = newDimensions[dimIdx].dice(attribute, items, reorder)
        if newDimensions[dimIdx] is self.dimensions[dimIdx]:
            return self
        out, ids = self._derive(newDimensions)
        return self._apply(out, ids, "dice", self.dimensions, newDimensions)

    def diceRange(self, dimensionId, attribute, start, end):
        dimIdx = self.getDimensionIndex(dimensionId)
        newDimensions = list(self.dimensions)
        newDimensions[dimIdx] = newDimensions[dimIdx].diceRange(attribute, start, end)
        if newDimensions[dimIdx] is self.dimensions[dimIdx]:
            return self
        out, ids = self._derive(newDimensions)
        return self._apply(out, ids, "dice", self.dimensions, newDimensions)

    def diceByDimensionItems(self, dimensionItemsMap, measures=(), reorder=False):
        """Dice several dimensions in ONE store pass (cube.js:595-638)."""
        newDimensions = list(self.dimensions)
        for dimensionId, items in dimensionItemsMap.items():
            dimIdx = self.getDimensionIndex(dimensionId)
            if dimIdx == -1:
                continue
            items = [items] if isinstance(items, str) else list(items)
            if dimensionId == "time":
                root = TimeSlot.fromValue(items[0]).periodicity
            else:
                root = self.dimensions[dimIdx].rootAttribute
            newDimensions[dimIdx] = newDimensions[dimIdx].dice(root, items, reorder)
        if all(n is o for n, o in zip(newDimensions, self.dimensions)):
            return self
        keep = (lambda ids: list(ids)) if not measures else (lambda ids: [m for m in ids if m in measures])
        out, ids = self._derive(
            newDimensions, keep(self.storedMeasureIds), keep(self.computedMeasureIds), rules="copy"
        )
        return self._apply(out, ids, "dice", self.dimensions, newDimensions)

    def slice(self, dimensionId, attribute, value):
        if self.getDimensionIndex(dimensionId) == -1:
            raise ValueError(f"slice: no such dimension: {dimensionId}")
        return self.dice(dimensionId, attribute, [value]).removeDimension(dimensionId)

    def collapse(self):
        """cube.js:320-324."""
        fused = self._remove_fused(self.dimensionIds)
        if fused is not None:
            return fused
        cube = self
        for d in self.dimensionIds:
            cube = cube.slice(d, "all", "all")
        return cube

    def aggregateByDimensions(self, excludeDimensionIds):
        """cube.js:560-566."""
        fused = self._remove_fused([d for d in self.dimensionIds if d not in excludeDimensionIds])
        if fused is not None:
            return fused
        cube = self
        for d in self.dimensionIds:
            if d not in excludeDimensionIds:
                cube = cube.slice(d, "all", "all")
        return cube

    # Rolling several dimensions up to 'all' (collapse, aggregateByDimensions, keepDimensions,
    # removeDimensions) is a chain of single-dimension store passes in the reference.  When
    # the order of the passes cannot matter — every stored measure aggregates ALL the removed
    # dimensions with the same order-free rule (sum under a zero default, highest, lowest) —
    # a store class that sets FUSED_ROLLUPS gets ONE pass per run of adjacent removed
    # dimensions instead: the run is presented to the store as a single merged axis rolled up
    # to one parent (the store interface already takes any lengths, in-memory.js:270-274).
    # Sums are then accumulated in double across the whole run and rounded once, which is what
    # the reference's double-valued chain does.  Anything else takes the reference's chain.
    _FUSED_MAX_CHILDREN = 1 << 24

    def _remove_fused(self, dimensionIds):
        cls = self._store_cls
        if not getattr(cls, "FUSED_ROLLUPS", False) or len(dimensionIds) < 2:
            return None
        remove = [d for d in self.dimensionIds if d in set(dimensionIds)]
        if len(remove) != len(dimensionIds) or len(remove) < 2:
            return None
        ids = self.storedMeasureIds
        methods = []
        for m in ids:
            rule = {self.storedMeasuresRules[m].get(d) or "sum" for d in remove}
            store = self.storedMeasures[m]
            default_is_nan = store._defaultValue != store._defaultValue
            if len(rule) != 1 or next(iter(rule)) not in ("sum", "highest", "lowest"):
                return None
            if next(iter(rule)) == "sum" and default_is_nan:
                return None  # the restart rule (in-memory.js:311-318) depends on the pass order
            methods.append(next(iter(rule)))
        # runs of adjacent removed dimensions, innermost run first
        lens = [d.numItems for d in self.dimensions]
        runs, i = [], 0
        while i < len(lens):
            if self.dimensions[i].id in remove:
                j = i
                while j < len(lens) and self.dimensions[j].id in remove:
                    j += 1
                runs.append((i, j))
                i = j
            else:
                i += 1
        if any(int(np.prod(lens[a:b])) > self._FUSED_MAX_CHILDREN or int(np.prod(lens[a:b])) == 0 for a, b in runs):
            return None
        stores = [self.storedMeasures[m] for m in ids]
        for a, b in reversed(runs):
            merged = int(np.prod(lens[a:b]))
            old_len = lens[:a] + [merged] + lens[b:]
            new_len = lens[:a] + [1] + lens[b:]
            # None = "unchanged", or "everything to the single new item" for the merged axis
            # (include/olap_gpu.h: no table is built or checked); other stores get real maps
            if getattr(cls, "IMPLIED_MAPS", False):
                maps = [None] * len(old_len)
            else:
                maps = [np.arange(n, dtype=np.int32) for n in old_len]
                maps[a] = np.zeros(merged, np.int32)
            if stores:
                stores = cls.drillUp_lowered_batch(stores, old_len, new_len, maps, methods)
            lens = lens[:a] + lens[b:]
        out = Cube([d for d in self.dimensions if d.id not in remove], cls)
        out.storedMeasures = dict(zip(ids, stores))
        out.computedMeasures.update(self.computedMeasures)
        out.storedMeasuresRules = copy.deepcopy(self.storedMeasuresRules)
        for rule in out.storedMeasuresRules.values():
            for d in remove:
                rule.pop(d, None)
        return out

    def reorderDimensions(self, dimensionIds):
        """Permute the axes (cube.js:757-783)."""
        if list(dimensionIds[: len(self.dimensions)]) == self.dimensionIds:
            return self
        newDimensions = [self.getDimension(d) for d in dimensionIds]
        out, ids = self._derive(newDimensions)
        return self._apply(out, ids, "reorder", self.dimensions, newDimensions)

    def swapDimensions(self, dim1, dim2):
        for d in (dim1, dim2):
            if d not in self.dimensionIds:
                raise ValueError(f"swapDimensions: no such dimension {d}")
        return self.reorderDimensions([dim2 if d == dim1 else dim1 if d == dim2 else d for d in self.dimensionIds])

    def keepDimensions(self, dimensionIds):
        """cube.js:890-899."""
        fused = self._remove_fused([d.id for d in self.dimensions if d.id not in dimensionIds])
        if fused is not None:
            return fused
        cube = self
        for dimension in self.dimensions:
            if dimension.id not in dimensionIds:
                cube = cube.removeDimension(dimension.id)
        return cube

    def removeDimensions(self, dimensionIds):
        """cube.js:901-908."""
        fused = self._remove_fused(list(dimensionIds))
        if fused is not None:
            return fused
        cube = self
        for d in dimensionIds:
            cube = cube.removeDimension(d)
        return cube

    def project(self, dimensionIds):
        return self.keepDimensions(dimensionIds).reorderDimensions(dimensionIds)

    # ------------------------------------------------------------ cube-to-cube
    def hydrateFromCube(self, otherCube):
        """cube.js:730-746: reshape the other cube onto my dimensions, then load."""
        try:
            compatible = otherCube.reshape(self.dimensions)
        except Exception:
            return  # no overlap between the cubes
        for m, store in self.storedMeasures.items():
            if m in compatible.storedMeasures:
                store.load(compatible.storedMeasures[m], self.dimensions, compatible.dimensions)

    def reshape(self, targetDims):
        """cube.js:1082-1133."""
        mine = self.dimensionIds
        cube = self.project([d.id for d in targetDims if d.id in mine])
        for i, target in enumerate(targetDims):
            actual = cube.dimensions[i] if i < len(cube.dimensions) else None
            if actual is None or actual.id != target.id:
                cube = cube.addDimension(target, {}, i)
        for i, target in enumerate(targetDims):
            actual = cube.dimensions[i]
            if actual.rootAttribute == target.rootAttribute:
                continue
            if target.rootAttribute in actual.attributes:
                cube = cube.drillUp(target.id, target.rootAttribute)
            elif actual.rootAttribute in target.attributes:
                cube = cube.drillDown(target.id, target.rootAttribute)
            else:
                raise ValueError(f"The cube dimensions '{target.id}' are not compatible.")
            cube = cube.dice(target.id, target.rootAttribute, target.getItems(), True)
        return cube

    def compose(self, otherCube, union=False, fillWith=None):
        """cube.js:1032-1080."""
        newDimensions = []
        for mine in self.dimensions:
            other = otherCube.getDimension(mine.id)
            if other is None:
                continue
            newDimensions.append(mine.union(other) if union else mine.intersect(other))
        out = Cube(newDimensions, self._store_cls)
        for source in (self, otherCube):
            for m in source.storedMeasureIds:
                store = source.storedMeasures[m]
                out.createStoredMeasure(m, source.storedMeasuresRules[m], store._type, store._defaultValue)
                if fillWith and fillWith.get(m):
                    out.fillData(m, fillWith[m])
                out.hydrateFromCube(source)
        out.computedMeasures.update(self.computedMeasures)
        out.computedMeasures.update(otherCube.computedMeasures)
        return out

    # ---------------------------------------------------------- serialization
    def serialize(self):
        """cube.js:1135-1151, byte-compatible with the reference's wire format."""
        from .serialization import toBuffer

        return toBuffer({
            "dimensions": [dim.serialize() for dim in self.dimensions],
            "storedMeasuresKeys": list(self.storedMeasures.keys()),
            "storedMeasures": [store.serialize() for store in self.storedMeasures.values()],
            "storedMeasuresRules": self.storedMeasuresRules,
            "computedMeasures": {m: e.toString() for m, e in self.computedMeasures.items()},
        })

    def serializeToBase64String(self):  # cube.js:1153-1155
        import base64

        return base64.b64encode(self.serialize()).decode("ascii")

    @classmethod
    def deserialize(cls, buffer, store_cls=None):
        """cube.js:1157-1179.  Every store is rebuilt with the cube's own cell count (the
        wire format keeps only a Float32 of it, serialization.js:71-74)."""
        from .dimension import DimensionFactory
        from .serialization import fromBuffer

        data = fromBuffer(buffer)
        cube = cls([DimensionFactory.deserialize(d) for d in data["dimensions"]], store_cls)
        cube.storedMeasuresRules = data["storedMeasuresRules"]
        for key, blob in zip(data["storedMeasuresKeys"], data["storedMeasures"]):
            cube.storedMeasures[key] = cube._store_cls.deserialize(blob, cube.storeSize)
        parser = getParser()
        cube.computedMeasures = {m: parser.parse(text) for m, text in data["computedMeasures"].items()}
        return cube

    @classmethod
    def deserializeFromBase64String(cls, serializedBase64, store_cls=None):  # cube.js:1181-1185
        import base64

        return cls.deserialize(base64.b64decode(serializedBase64), store_cls)


class _PerMeasure(list):
    """Marks an argument that holds one value per stored measure."""


def _deep_merge(dst, src):
    if not isinstance(src, dict):
        return src
    for key, value in src.items():
        if isinstance(value, dict) and isinstance(dst.get(key), dict):
            _deep_merge(dst[key], value)
        else:
            dst[key] = copy.deepcopy(value) if isinstance(value, dict) else value
    return dst
