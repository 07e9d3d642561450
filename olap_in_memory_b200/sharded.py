"""Cubes larger than one GPU: rows of the flattened outermost dimensions are split
contiguously across the ranks of a torch.distributed group (one process per GPU).

The reference has no notion of this (SURVEY.md §8e): a cube there is one JS Map.  The
contract kept here is that a ShardedCube behaves like ONE Cube whose cells happen to live
on several devices:

* transforms of a dimension inside the shard (index >= `prefix`) are shard-local store
  calls — no communication at all;
* drillUp of a sharded dimension = local partial rollup of my rows into the FULL output
  row space, one all-to-all that hands every rank the W partials of its own output rows
  (the bytes a reduce-scatter would move), then a local, ordered combine of the W
  partials with the very same drillUp kernel (`sum` of sums, `highest` of highests,
  `first`/`last` in rank order = ascending row order, `average` = sum of sums / sum of
  counts).  Presence and status merge exactly as in the single-GPU kernel because the
  partials are ordinary stores.
* `total` = local totals + one all-reduce of a double.

torch.distributed is plumbing: NCCL moves the planes (zero-copy views of the device
stores, olap_in_memory_b200/interop.py); every arithmetic step is a store call."""
from __future__ import annotations

import os

import numpy as np

from . import cube as _cube
from .cube import Cube  # noqa: F401  (re-exported for convenience)


def split_rows(total, world):
    """Contiguous, balanced row ranges: sizes differ by at most one (SURVEY.md §8e)."""
    base, extra = divmod(total, world)
    bounds = [0]
    for r in range(world):
        bounds.append(bounds[-1] + base + (1 if r < extra else 0))
    return bounds


def _prod(xs):
    p = 1
    for x in xs:
        p *= int(x)
    return p


# How a rollup of a sharded dimension moves its cells between GPUs (OLAP_SHARDED_EXCHANGE):
#   "pull" (default on GPUs): the rank that owns an output row reads its child rows straight out of
#          the peers' stores through CUDA-IPC-mapped pointers, inside ONE rollup kernel
#          (olap_drill_up_pull): no partial planes, no receive buffers, no combine pass, and the
#          result is bit-equal to the unsharded rollup (same accumulation order).
#   "push": ONE kernel per call computes the partial rollup of the local rows and stores every
#          output row into the receive buffer of the rank that owns it (olap_drill_up_rows), then an
#          ordered combine of the W partials.
#   "nccl": partial planes in local HBM, one NCCL all-to-all per plane, ordered combine (also the
#          path of the gloo / CPU tests).
#   "pull2": shard-local partial rollup into compact partial stores first, then the pull kernel
#          combines the W partials in rank order (= ascending row order).  Moves (W-1)/W of the
#          OUTPUT instead of (W-1)/W of my share of the INPUT: cheaper when every rank holds many
#          children of each parent (few ranks, long dimension); float32 partials (rel 1e-6).
#   "auto": "pull" or "pull2", whichever the byte count says is faster (_exchange_costs).
# The default is "pull": parity first — it is the only mode whose sums are the unsharded cube's bits
# (the others add float32-rounded partials: rel 1e-6 on same-sign data, not bounded under
# cancellation).  With fewer ranks than children per parent (2 GPUs, a 10-item dimension) the
# partial-based modes move fewer bytes: 2 x B200, 1e10 cells x 3 measures, dim0 -> all: pull 63 ms,
# pull2 47 ms, push 33 ms, nccl 53 ms.
EXCHANGE = os.environ.get("OLAP_SHARDED_EXCHANGE", "nccl" if os.environ.get("OLAP_SHARDED_P2P", "1") == "0" else "pull")
# planning figures of the cost model (GB/s): peer reads with both directions busy, local HBM
PLAN_NVLINK_GBS, PLAN_HBM_GBS = 600.0, 6000.0
# a rollup whose output rows would be spread unevenly (10 rows over 8 ranks: 2,2,1,1,1,1,1,1) is
# computed on a deeper row axis when the imbalance exceeds this factor
MAX_IMBALANCE = 1.02
MIN_DEEP_INNER = 4096  # ... as long as a row keeps at least this many cells (16 KB of values)


def _pull_tables(full_map, in_bounds, j0, j1):
    """Child tables of olap_drill_up_pull for the rank that owns output rows j0..j1-1.

    full_map[i] = output row of global input row i (all ranks' rows); in_bounds = row bounds of the
    input shards.  Returns (row_start, child_rank, child_row): output row j0 + j aggregates the
    children row_start[j] .. row_start[j+1]-1, listed in ascending global input row (the
    reference's iteration order, SURVEY.md F6); child c is local row child_row[c] of rank
    child_rank[c]."""
    full_map = np.asarray(full_map, dtype=np.int64)
    bounds = np.asarray(in_bounds, dtype=np.int64)
    mine = np.flatnonzero((full_map >= j0) & (full_map < j1))  # ascending global rows
    parents = full_map[mine] - j0
    order = np.argsort(parents, kind="stable")  # by output row, global row order kept inside a row
    rows, parents = mine[order], parents[order]
    row_start = np.searchsorted(parents, np.arange(j1 - j0 + 1, dtype=np.int64), side="left").astype(np.int32)
    rank = np.searchsorted(bounds[1:], rows, side="right")
    return row_start, rank.astype(np.int32), (rows - bounds[rank]).astype(np.int64)


def _peer_row_tables(bases, out_bounds, me, K, inner, plane_v, plane_s, with_status):
    """Where rank `me` stores each output row of each of its K partial planes (olap_drill_up_rows).

    Receive buffer of rank r (base address bases[r]): K value planes of `plane_v` bytes, then K
    status planes of `plane_s` bytes; inside a plane, one slot per SENDING rank holding r's
    rows_of[r] output rows of `inner` cells.  The kernel walks the output rows in table order:
    every rank starts with the rows of its RIGHT neighbour and ends with its own, so at any
    moment the W ranks store to W different receivers (rows in plain order make everybody hit
    rank 0 first, then rank 1, ...: one NVLink ingress at a time — measured on 8 B200: 76.7 ms
    for the 1e10-cell cube against 60 ms for NCCL).

    Returns (position, row_values, row_status): position[j] = table slot of output row j (int32,
    to be composed with the local-row -> output-row map), and the K x n tables of addresses
    (uint64; row_status is None without status planes)."""
    bounds = np.asarray(out_bounds, dtype=np.int64)
    W, n = len(bounds) - 1, int(bounds[-1])
    rows = np.arange(n, dtype=np.int64)
    owner = np.searchsorted(bounds[1:], rows, side="right")
    order = np.lexsort((rows, (owner - me - 1) % W))  # by distance to the right of me, then by row
    position = np.empty(n, dtype=np.int32)
    position[order] = np.arange(n, dtype=np.int32)
    r = owner[order]
    cell0 = (me * np.diff(bounds)[r] + (order - bounds[r])) * inner  # first cell of the row inside a plane of rank r
    base = np.asarray([int(b) for b in bases], dtype=np.uint64)[r]
    k = np.arange(K, dtype=np.uint64)[:, None]
    row_values = (base + (cell0 * 4).astype(np.uint64))[None, :] + k * np.uint64(plane_v)
    row_status = None
    if with_status:
        row_status = ((base + np.uint64(K * plane_v) + cell0.astype(np.uint64))[None, :] + k * np.uint64(plane_s)).reshape(-1)
    return position, row_values.reshape(-1), row_status


def _exchange_costs(full_map, in_bounds, out_bounds):
    """Rows that cross NVLink into the busiest rank for the two pull variants, and what the two-phase
    variant costs locally.  Pure function of the row map and the shard bounds, so every rank takes
    the same decision without talking.  Returns (direct_remote_rows, partial_remote_rows,
    partial_rows_max, local_rows_max, touched) with touched[s] = sorted output rows rank s holds
    children of."""
    full_map = np.asarray(full_map, dtype=np.int64)
    ib, ob = np.asarray(in_bounds, dtype=np.int64), np.asarray(out_bounds, dtype=np.int64)
    W = len(ib) - 1
    owner_in = np.searchsorted(ib[1:], np.arange(full_map.size), side="right")
    owner_out = np.searchsorted(ob[1:], full_map, side="right")
    direct = np.bincount(owner_out[owner_in != owner_out], minlength=W)
    touched = [np.unique(full_map[ib[s]:ib[s + 1]]) for s in range(W)]
    partial = np.zeros(W, dtype=np.int64)
    for s in range(W):
        dest = np.searchsorted(ob[1:], touched[s], side="right")
        cnt = np.bincount(dest, minlength=W)
        cnt[s] = 0
        partial += cnt
    return int(direct.max(initial=0)), int(partial.max(initial=0)), max((t.size for t in touched), default=0), int(np.diff(ib).max(initial=0)), touched


def _pull2_tables(touched, j0, j1):
    """Child tables of the second phase of "pull2" for the rank that owns output rows j0..j1-1:
    output row j combines the partial row of every rank that holds children of j, in ascending
    rank order; rank r's partial of j is row index(j in touched[r]) of its compact partial store."""
    ranks, rows, parents = [], [], []
    for r, t in enumerate(touched):
        lo, hi = np.searchsorted(t, [j0, j1])
        parents.append(np.asarray(t[lo:hi], dtype=np.int64) - j0)
        rows.append(np.arange(lo, hi, dtype=np.int64))
        ranks.append(np.full(hi - lo, r, dtype=np.int32))
    parents, rows, ranks = np.concatenate(parents), np.concatenate(rows), np.concatenate(ranks)
    order = np.argsort(parents, kind="stable")  # by output row; rank order kept inside a row
    row_start = np.searchsorted(parents[order], np.arange(j1 - j0 + 1, dtype=np.int64), side="left").astype(np.int32)
    return row_start, np.ascontiguousarray(ranks[order]), np.ascontiguousarray(rows[order])


class _PeerBuffers:
    """Receive buffers that every rank of the group has mapped (CUDA IPC), cached by size."""

    _cache = {}

    @classmethod
    def get(cls, comm, nbytes):
        import ctypes as C

        from . import _native as N

        # the membership of the group, not id(group): ids are reused after garbage collection
        group = comm.group if comm.group is not None else comm.dist.group.WORLD
        key = (tuple(comm.dist.get_process_group_ranks(group)), int(nbytes))
        hit = cls._cache.get(key)
        if hit is not None:
            return hit
        mine = C.c_void_p()
        handle = C.create_string_buffer(64)
        N.check(N.lib().olap_peer_alloc(int(nbytes), C.byref(mine), handle))
        handles = [None] * comm.world
        comm.dist.all_gather_object(handles, handle.raw, group=comm.group)
        ptrs = []
        for r, h in enumerate(handles):
            if r == comm.rank:
                ptrs.append(mine.value)
                continue
            p = C.c_void_p()
            N.check(N.lib().olap_peer_open(C.create_string_buffer(h, 64), C.byref(p)))
            ptrs.append(p.value)
        cls._cache[key] = ptrs
        cls._owner[key] = (comm, mine.value)
        return ptrs

    _owner = {}

    @classmethod
    def release(cls):
        """Collective: every rank closes its mappings of the peers' receive buffers, then frees its own
        (the push exchange keeps one buffer per size alive until this is called)."""
        from . import _native as N

        for key, ptrs in list(cls._cache.items()):
            comm, mine = cls._owner.pop(key)
            N.check(N.lib().olap_sync())
            for r, p in enumerate(ptrs):
                if r != comm.rank:
                    N.check(N.lib().olap_peer_close(p))
            comm.dist.barrier(group=comm.group)  # nobody maps my buffer any more
            N.check(N.lib().olap_peer_free(mine))
            del cls._cache[key]


class _Comm:
    """The three collectives the path needs, over torch.distributed (nccl on GPUs, gloo in
    the CPU tests) or as no-ops for a single rank."""

    def __init__(self, group=None):
        import torch.distributed as dist

        self.dist = dist
        self.group = group
        self.on = dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank(group) if self.on else 0
        self.world = dist.get_world_size(group) if self.on else 1

    def all_to_all(self, out, inp, out_splits, in_splits):
        if self.world == 1:
            out.copy_(inp)
            return
        if out.is_cuda:
            self.dist.all_to_all_single(out, inp, out_splits, in_splits, group=self.group)
            return
        # gloo has no all_to_all: pairwise exchange
        in_off = np.concatenate([[0], np.cumsum(in_splits)])
        out_off = np.concatenate([[0], np.cumsum(out_splits)])
        reqs = []
        for peer in range(self.world):
            src = inp[in_off[peer]:in_off[peer + 1]]
            dst = out[out_off[peer]:out_off[peer + 1]]
            if peer == self.rank:
                dst.copy_(src)
                continue
            if src.numel():
                reqs.append(self.dist.isend(src.contiguous(), peer, group=self.group))
            if dst.numel():
                reqs.append(self.dist.irecv(dst, peer, group=self.group))
        for r in reqs:
            r.wait()

    def all_to_all_many(self, pairs, out_splits, in_splits):
        """Exchange several planes that share the same split sizes.  One NCCL all-to-all per
        plane: on 8 B200 that measured FASTER (60 ms for 20 GB partials) than putting every
        send/receive of every plane into one grouped launch (73 ms) — fewer concurrent
        peer-to-peer channels contend less."""
        for out, inp in pairs:
            self.all_to_all(out, inp, out_splits, in_splits)

    def all_reduce_sum(self, value, device=None):
        if self.world == 1:
            return value
        import torch

        t = torch.tensor([value], dtype=torch.float64, device=device or "cpu")
        self.dist.all_reduce(t, group=self.group)
        return float(t.item())

    def all_gather(self, tensor, sizes):
        if self.world == 1:
            return tensor.clone()
        import torch

        parts = [torch.empty(int(s), dtype=tensor.dtype, device=tensor.device) for s in sizes]
        if len(set(int(s) for s in sizes)) == 1:
            self.dist.all_gather(parts, tensor.contiguous(), group=self.group)
        else:  # ragged: pad to the largest
            m = max(int(s) for s in sizes)
            padded = torch.zeros(m, dtype=tensor.dtype, device=tensor.device)
            padded[: tensor.numel()] = tensor
            bufs = [torch.empty(m, dtype=tensor.dtype, device=tensor.device) for _ in sizes]
            self.dist.all_gather(bufs, padded, group=self.group)
            parts = [b[: int(s)] for b, s in zip(bufs, sizes)]
        return torch.cat(parts)


class ShardedCube:
    def __init__(self, dimensions, prefix=1, store_cls=None, group=None, _row_bounds=None):
        if store_cls is None:
            from .store import GpuStore

            store_cls = GpuStore
        self.dimensions = list(dimensions)
        self.prefix = int(prefix)
        if not 1 <= self.prefix <= len(self.dimensions):
            raise ValueError("prefix must cover 1..ndim leading dimensions")
        self._store_cls = store_cls
        self.comm = _Comm(group)
        self.rank, self.world = self.comm.rank, self.comm.world
        if self.world > 1 and getattr(store_cls, "SHAREABLE_SHARDS", False):
            # this process holds one shard: whatever store it creates from now on (exchange buffers,
            # results of transforms) may become the source of a peer's pull
            from . import _native as N

            N.check(N.lib().olap_set_shareable(1))
        self.rows_total = _prod(d.numItems for d in self.dimensions[: self.prefix])
        self.inner_lens = [d.numItems for d in self.dimensions[self.prefix:]]
        self.inner = _prod(self.inner_lens)
        self.row_bounds = _row_bounds or split_rows(self.rows_total, self.world)
        self.row0, self.row1 = self.row_bounds[self.rank], self.row_bounds[self.rank + 1]
        self.storedMeasures = {}
        self.storedMeasuresRules = {}
        self.computedMeasures = {}

    # ------------------------------------------------------------------ basics
    @property
    def rows_local(self):
        return self.row1 - self.row0

    @property
    def localSize(self):
        return self.rows_local * self.inner

    @property
    def storeSize(self):
        return self.rows_total * self.inner

    @property
    def dimensionIds(self):
        return [d.id for d in self.dimensions]

    def getDimensionIndex(self, dimensionId):
        for i, d in enumerate(self.dimensions):
            if d.id == dimensionId:
                return i
        return -1

    def createStoredMeasure(self, measureId, rules=None, type="float32", defaultValue=0):
        if getattr(self._store_cls, "SHAREABLE_SHARDS", False):
            # device stores of a sharded cube live in memory the peers can map (pull exchange)
            store = self._store_cls(self.localSize, type, defaultValue, shareable=True)
        else:
            store = self._store_cls(self.localSize, type, defaultValue)
        self.storedMeasures[measureId] = store
        self.storedMeasuresRules[measureId] = {} if rules is None else rules

    def createComputedMeasure(self, measureId, formula):
        """cube.js:95-125.  Evaluation is shard-local (one fused kernel over my rows); an
        `x__total` variable is the whole-cube total: local totals + one all-reduce."""
        import re

        from .parser import getParser

        if measureId in self.storedMeasures or measureId in self.computedMeasures:
            raise ValueError(f"This measure already exists {measureId}")
        for other, expr in self.computedMeasures.items():  # formulas may use computed measures: inline them (cube.js:107-121)
            pattern = re.compile(rf"\b{re.escape(other)}\b")
            if pattern.search(formula):
                formula = pattern.sub(f"({expr.toString()})", formula)
        expression = getParser().parse(formula)
        known = set(self.storedMeasures) | {f"{m}__total" for m in self.storedMeasures}
        unknown = [v for v in expression.variables() if v not in known]
        if unknown:
            raise ValueError(f"Unknown measure(s): {','.join(unknown)}")
        self.computedMeasures[measureId] = expression

    def _evaluate_local(self, measureId):
        expression = self.computedMeasures[measureId]
        names = expression.variables()
        cell_names = [n for n in names if "__total" not in n]
        # every rank takes part in the all-reduce, whether it holds rows or not
        totals = {n: self.getTotal(n.replace("__total", "")) for n in names if "__total" in n}
        if self.localSize == 0:
            return np.empty(0, dtype=np.float64)
        stores = [self.storedMeasures[n] for n in cell_names]
        return np.asarray(self._store_cls.evaluate(expression, cell_names, stores, totals, self.localSize), dtype=np.float64)

    def getLocalStore(self, measureId, type="float32", defaultValue=0):
        """My rows of a measure as a device store: the stored measure itself, or a computed measure
        evaluated by one fused kernel over my rows without leaving the device (Cube.evaluateToStore;
        the device half of copyToStoredMeasure, cube.js:205-215)."""
        if measureId in self.storedMeasures:
            return self.storedMeasures[measureId]
        expression = self.computedMeasures[measureId]
        names = expression.variables()
        cell_names = [n for n in names if "__total" not in n]
        totals = {n: self.getTotal(n.replace("__total", "")) for n in names if "__total" in n}
        return self._store_cls.evaluate_to_store(expression, cell_names, [self.storedMeasures[n] for n in cell_names], totals,
                                                 type, defaultValue)

    def setLocalData(self, measureId, values):
        """Cells of MY rows, row-major (length rows_local * inner)."""
        self._set(self.storedMeasures[measureId], values)

    def setData(self, measureId, values):
        """Full-cube data given on every rank: each keeps its own rows (tests, small cubes)."""
        values = np.asarray(values)
        self.setLocalData(measureId, values[self.row0 * self.inner: self.row1 * self.inner])

    def getLocalData(self, measureId):
        if measureId in self.computedMeasures:
            return self._evaluate_local(measureId)
        return self._get(self.storedMeasures[measureId])

    def getData(self, measureId):
        """Whole cube gathered on every rank (verification / small results only)."""
        import torch

        local = torch.from_numpy(np.ascontiguousarray(self.getLocalData(measureId), dtype=np.float64))
        sizes = [(self.row_bounds[r + 1] - self.row_bounds[r]) * self.inner for r in range(self.world)]
        if self.world > 1 and self._store_cls.DEVICE == "cuda":
            local = local.cuda()
        return self.comm.all_gather(local, sizes).cpu().numpy()

    def getTotal(self, measureId):
        store = self.storedMeasures[measureId]
        device = self._store_cls.DEVICE if self.world > 1 else None
        return self.comm.all_reduce_sum(store.total, device)

    # ------------------------------------------------------------ region queries
    def _local_region(self, dimensionsFilter, check_measures):
        """Cube._region on the whole cube (the same validation and errors on every rank, before any collective),
        restricted to my rows: the filter lists of the row dimensions (and the leading multiplicity axis of filter
        keys that are not dimensions) give global rows in product order, repeats kept; those in [row0, row1) are
        the first-axis list of my region.  None when the whole region is empty."""
        region = _cube._region(self.dimensions, dimensionsFilter, check_measures)
        if region is None:
            return None
        lens, keep = region
        lead = len(lens) - len(self.dimensions) + self.prefix  # row axes, the multiplicity axis included
        rows = np.ravel_multi_index(np.ix_(*_cube._region_lists(lens[:lead], keep[:lead])), lens[:lead]).ravel()
        mine = rows[(rows >= self.row0) & (rows < self.row1)] - self.row0
        return [self.rows_local] + self.inner_lens, [mine.astype(np.int32)] + keep[lead:]

    def getTotalForDimensionItems(self, measureId, dimensionsFilter=None):
        """Cube.getTotalForDimensionItems: the region sum of my rows, then one all-reduce that every rank joins."""
        region = self._local_region(dimensionsFilter,
                                    lambda: _cube._check_readable(self.storedMeasures, self.computedMeasures, measureId))
        if region is None:
            return 0
        lens, keep = region
        if measureId in self.storedMeasures:
            local = self.storedMeasures[measureId].regionSum(lens, keep)
        elif (fused := _cube._formula_inputs(self._store_cls, "regionEvalSum", self.computedMeasures, self.storedMeasures,
                                             measureId)) is not None:
            local = self._store_cls.regionEvalSum(*fused, lens, keep)
        else:
            local = _cube._region_sum_f64(np.asarray(self.getLocalData(measureId), dtype=np.float64), lens, keep)
        device = self._store_cls.DEVICE if self.world > 1 else None
        return self.comm.all_reduce_sum(float(local), device)

    def getDistribution(self, measureId, dimensionsFilter=None):
        space = self.getTotalForDimensionItems(measureId, dimensionsFilter)
        total = self.getTotal(measureId)
        return space if total == 0 else space / total

    def copyMeasureData(self, sourceMeasureId, targetMeasureId, dimensionsFilter=None):
        """Cube.copyMeasureData on my rows: both measures have the same row bounds, nothing crosses ranks."""
        def check():
            _cube._check_readable(self.storedMeasures, self.computedMeasures, sourceMeasureId)
            if targetMeasureId not in self.storedMeasures:
                raise ValueError(f"setSingleData: no such stored measure {targetMeasureId}")

        region = self._local_region(dimensionsFilter, check)
        if region is None or region[1][0].size == 0:
            return
        lens, keep = region
        target = self.storedMeasures[targetMeasureId]
        if sourceMeasureId in self.storedMeasures:
            target.regionCopy(self.storedMeasures[sourceMeasureId], lens, keep)
        elif (fused := _cube._formula_inputs(self._store_cls, "regionEvalCopy", self.computedMeasures, self.storedMeasures,
                                             sourceMeasureId)) is not None:
            self._store_cls.regionEvalCopy(target, *fused, lens, keep)
        else:
            _cube._region_set_f64(target, np.asarray(self.getLocalData(sourceMeasureId), dtype=np.float64), lens, keep)

    @staticmethod
    def _set(store, values):
        store.set_data_f32(np.asarray(values, dtype=np.float32))

    @staticmethod
    def _get(store):
        return store.data_f32().astype(np.float64)

    def _derive(self, dimensions, row_bounds=None):
        out = ShardedCube(dimensions, self.prefix, self._store_cls, self.comm.group, row_bounds)
        out.storedMeasuresRules = dict(self.storedMeasuresRules)
        out.computedMeasures = dict(self.computedMeasures)  # formulas follow the cube through every transform (cube.js:1010-1011)
        return out

    # ----------------------------------------------------------- lowered store calls
    def _call(self, name, stores, *args):
        """Batched static form of a lowered transform: one call for all measures."""
        return getattr(self._store_cls, name)(stores, *[list(x) if isinstance(x, _Per) else x for x in args])

    def _local_lens(self):
        return [self.rows_local] + self.inner_lens

    # ------------------------------------------------------------------ transforms
    def drillUp(self, dimensionId, attribute):
        idx = self.getDimensionIndex(dimensionId)
        old_dim = self.dimensions[idx]
        if old_dim.rootAttribute == attribute:
            return self
        new_dim = old_dim.drillUp(attribute)
        if new_dim is old_dim:
            return self
        new_dims = list(self.dimensions)
        new_dims[idx] = new_dim
        ids = list(self.storedMeasures)
        methods = [self.storedMeasuresRules[m].get(dimensionId) or "sum" for m in ids]
        group_map = np.asarray(old_dim.getGroupIndexFromRootIndexMap(new_dim.rootAttribute), dtype=np.int32)
        if idx >= self.prefix:
            return self._drill_up_local(new_dims, idx, group_map, ids, methods)
        new_rows = _prod(d.numItems for d in new_dims[: self.prefix])
        heaviest = -(-new_rows // self.world) * self.world  # rows of the busiest rank x ranks
        deeper = self.prefix < len(self.dimensions)
        uneven = heaviest > MAX_IMBALANCE * new_rows and deeper and self.inner // self.dimensions[self.prefix].numItems >= MIN_DEEP_INNER
        if deeper and (new_rows < self.world or uneven):
            # fewer output rows than ranks, or rows that do not spread evenly (10 rows over 8 ranks:
            # the two ranks with 2 rows would take twice as long as the others; 100 rows over 8
            # ranks: 13 against 12.5, measured 30.8 ms where 29.3 were possible): shard the result
            # on the next dimension as well (SURVEY.md §8e "leaving the result sharded on the next
            # axis").  Nothing moves: the same cells are read as more, shorter rows.
            return self._deepened().drillUp(dimensionId, attribute)
        return self._drill_up_sharded(new_dims, idx, group_map, ids, methods)

    def _deepened(self):
        """The same cells, seen as a cube sharded on one more leading dimension: every row
        becomes numItems rows and the bounds scale with it.  Nothing moves."""
        key = tuple(id(s) for s in self.storedMeasures.values())
        hit = getattr(self, "_deep", None)
        if hit is not None and hit[0] == key:  # the same view again: its peer mappings are still good
            hit[1].storedMeasuresRules = dict(self.storedMeasuresRules)
            hit[1].computedMeasures = dict(self.computedMeasures)
            return hit[1]
        n = self.dimensions[self.prefix].numItems
        out = ShardedCube(self.dimensions, self.prefix + 1, self._store_cls, self.comm.group, [b * n for b in self.row_bounds])
        out.storedMeasures = dict(self.storedMeasures)
        out.storedMeasuresRules = dict(self.storedMeasuresRules)
        out.computedMeasures = dict(self.computedMeasures)
        self._deep = (key, out)
        return out

    def _drill_up_local(self, new_dims, idx, group_map, ids, methods):
        """The drilled dimension lies inside my shard: no communication."""
        out = self._derive(new_dims, self.row_bounds)
        old_len = self._local_lens()
        new_len = [self.rows_local] + [d.numItems for d in new_dims[self.prefix:]]
        maps = [np.arange(n, dtype=np.int32) for n in old_len]
        maps[1 + idx - self.prefix] = group_map
        stores = [self.storedMeasures[m] for m in ids]
        if stores:
            results = self._call("drillUp_lowered", stores, old_len, new_len, maps, _Per(methods))
            out.storedMeasures = dict(zip(ids, results))
        return out

    def _row_map(self, idx, group_map, new_prefix_lens, all_rows=False):
        """my local row (or, with all_rows, every global row) -> global row of the drilled cube"""
        old_prefix_lens = [d.numItems for d in self.dimensions[: self.prefix]]
        rows = np.arange(0 if all_rows else self.row0, self.rows_total if all_rows else self.row1, dtype=np.int64)
        coords = []
        rest = rows
        for n in reversed(old_prefix_lens):
            coords.append(rest % n)
            rest = rest // n
        coords.reverse()
        coords[idx] = group_map[coords[idx]].astype(np.int64)
        new_row = np.zeros_like(rows)
        for c, n in zip(coords, new_prefix_lens):
            new_row = new_row * n + c
        return new_row if all_rows else new_row.astype(np.int32)

    def _drill_up_sharded(self, new_dims, idx, group_map, ids, methods):
        """The drilled dimension is (part of) the sharded row axis."""
        new_prefix_lens = [d.numItems for d in new_dims[: self.prefix]]
        new_rows_total = _prod(new_prefix_lens)
        out_bounds = split_rows(new_rows_total, self.world)
        out = self._derive(new_dims, out_bounds)
        if not ids:
            return out
        W, inner = self.world, self.inner
        if W == 1:
            # a single rank owns every row: the "partial" rollup is the result
            row_map = self._row_map(idx, group_map, new_prefix_lens)
            maps = [row_map] + [np.arange(n, dtype=np.int32) for n in self.inner_lens]
            stores = [self.storedMeasures[m] for m in ids]
            results = self._call("drillUp_lowered", stores, self._local_lens(), [new_rows_total] + self.inner_lens,
                                 maps, _Per(methods))
            out.storedMeasures = dict(zip(ids, results))
            return out
        mode = EXCHANGE
        if mode in ("auto", "pull", "pull2") and self.comm.on and self._store_cls.PEER_MEMORY:
            full_map = self._row_map(idx, group_map, new_prefix_lens, all_rows=True)
            touched = None
            if mode != "pull":
                direct, partial, partial_rows, local_rows, touched = _exchange_costs(full_map, self.row_bounds, out_bounds)
                planes = len(ids) + sum(1 for m in methods if m == "average")
                t_direct = direct * len(ids) / PLAN_NVLINK_GBS
                t_two = (local_rows * len(ids) + 2 * partial_rows * planes) / PLAN_HBM_GBS + partial * planes / PLAN_NVLINK_GBS
                if mode == "auto":
                    mode = "pull" if t_direct <= t_two else "pull2"
            if mode == "pull":
                pulled = self._drill_up_pull(out, full_map, idx, group_map, ids, methods, out_bounds)
            else:
                pulled = self._drill_up_pull2(out, full_map, touched, ids, methods, out_bounds)
            if pulled is not None:
                out.last_exchange = mode
                return pulled
            mode = "push"
        out.last_exchange = mode
        my_out_rows = out_bounds[self.rank + 1] - out_bounds[self.rank]
        row_map = self._row_map(idx, group_map, new_prefix_lens)
        old_len = self._local_lens()
        new_len = [new_rows_total] + self.inner_lens
        maps = [row_map] + [np.arange(n, dtype=np.int32) for n in self.inner_lens]

        # 1. local partial rollup of my rows into the full output row space; `average`
        #    travels as (sum, count)
        plan = []  # (measure, method used for the partial, role)
        for m, method in zip(ids, methods):
            if method == "average":
                plan.append((m, "sum", "avg_sum"))
                plan.append((m, "__count", "avg_cnt"))
            else:
                plan.append((m, method, "plain"))
        stores = [self.storedMeasures[m] for m, _, _ in plan]
        if mode != "nccl" and self.comm.on and self._store_cls.PEER_MEMORY:
            received = self._partials_into_peers(stores, [meth for _, meth, _ in plan], row_map, out_bounds, new_rows_total)
            return self._combine(out, plan, ids, methods, received, my_out_rows)
        partials = self._partials(stores, old_len, new_len, maps, [meth for _, meth, _ in plan])

        # 2. one all-to-all per plane: rank r receives the W partials of ITS output rows
        in_splits = [(out_bounds[r + 1] - out_bounds[r]) * inner for r in range(W)]
        out_splits = [my_out_rows * inner] * W
        received = []
        for src_store in stores:  # every cell is overwritten by the exchange
            received.append(self._store_cls.recv_like(src_store, W * my_out_rows * inner))
        self._exchange_all(partials, received, in_splits, out_splits)
        del partials

        return self._combine(out, plan, ids, methods, received, my_out_rows)

    # ------------------------------------------------------------------ pull exchange
    def _peer_views(self, stores, remember=True):
        """Addresses, in MY address space, of every rank's planes of these stores: two lists
        [K][W] (values, status; None without a plane).  Handles travel once per set of stores (one
        all_gather of ~100 bytes per store) and are remembered on the cube; mappings are cached
        by the library (a recycled block keeps its handle).  None when a store of some rank cannot
        be exported (not created shareable)."""
        key = tuple(s._h for s in stores)
        hit = self._pull_cache.get(key) if remember and hasattr(self, "_pull_cache") else None
        if hit is not None:
            return hit
        import ctypes as C

        from . import _native as N

        try:
            mine = [s.ipc_export() for s in stores]
        except N.OlapError:
            mine = None
        everyone = [None] * self.world
        self.comm.dist.all_gather_object(everyone, mine, group=self.comm.group)
        if any(e is None for e in everyone):
            return None
        lib = N.lib()
        base_v = [[0] * self.world for _ in stores]
        base_s = [[0] * self.world for _ in stores]
        opened = {}
        for r, exported in enumerate(everyone):
            for k, (handle, v_off, s_off) in enumerate(exported):
                if r == self.rank:
                    base_v[k][r] = lib.olap_store_values_cptr(stores[k]._h)
                    base_s[k][r] = lib.olap_store_status_cptr(stores[k]._h) or 0
                    continue
                if handle not in opened:
                    p = C.c_void_p()
                    N.check(lib.olap_peer_map(handle, C.byref(p)))
                    opened[handle] = p.value
                base_v[k][r] = opened[handle] + v_off
                base_s[k][r] = opened[handle] + s_off if s_off >= 0 else 0
        if remember:  # the stores of the cube itself: their handles stay valid as long as the cube holds them
            if not hasattr(self, "_pull_cache"):
                self._pull_cache = {}
            self._pull_cache[key] = (base_v, base_s)
        return base_v, base_s

    def _drill_up_pull(self, out, full_map, idx, group_map, ids, methods, out_bounds):
        """Rollup of a sharded dimension, pull model: I compute MY output rows, reading their child
        rows out of the ranks that hold them (peer-mapped loads over NVLink inside the rollup
        kernel).  Children are walked in ascending global row order, so every method — first /
        last, the double sums, `average` — gives the bits of the unsharded rollup."""
        import ctypes as C

        from . import _native as N
        from .store import _method_code

        stores = [self.storedMeasures[m] for m in ids]
        views = self._peer_views(stores)
        if views is None:
            return None
        base_v, base_s = views
        W, K = self.world, len(stores)
        j0, j1 = out_bounds[self.rank], out_bounds[self.rank + 1]
        key = (idx, group_map.tobytes(), tuple(self.row_bounds), j0, j1)
        tables = self._pull_tables_cache.get(key) if hasattr(self, "_pull_tables_cache") else None
        if tables is None:
            tables = _pull_tables(full_map, self.row_bounds, j0, j1)
            self._pull_tables_cache = {key: tables}
        rank_rows = [self.row_bounds[r + 1] - self.row_bounds[r] for r in range(W)]
        results = self._pull_call(stores, methods, views, tables, rank_rows, j1 - j0)
        out.last_pull_ms, out.last_pull_derived = self.last_pull_ms, self.last_pull_derived
        out.storedMeasures = {m: self._store_cls._wrap(results[k]) for k, m in enumerate(ids)}
        return out

    def _pull_call(self, stores, methods, views, tables, rank_rows, out_rows):
        """olap_drill_up_pull between two barriers: every rank's source stores are complete before
        anyone reads them, and nobody frees or overwrites one while a peer may still be reading."""
        import ctypes as C

        from . import _native as N
        from .store import _method_code

        base_v, base_s = views
        row_start, child_rank, child_row = tables
        W, K = self.world, len(stores)
        lib = N.lib()
        with_status = bool(lib.olap_store_has_status(stores[0]._h))
        flat_v = (C.c_void_p * (K * W))(*[base_v[k][r] or None for k in range(K) for r in range(W)])
        flat_s = (C.c_void_p * (K * W))(*[base_s[k][r] or None for k in range(K) for r in range(W)]) if with_status else None
        rank_rows = N.i64_array(rank_rows)
        results = (C.c_void_p * K)()
        # every rank's stores are complete (their producing kernels have finished) before anyone reads them
        N.check(lib.olap_sync())
        # status planes that follow from the values are not read (4 instead of 5 bytes per cell over NVLink):
        # only if that holds for every store of every rank; the all-reduce doubles as the barrier
        derive = self._all_ranks(with_status and all(s.status_derived for s in stores))
        N.check(lib.olap_drill_up_pull(N.store_array([s._h for s in stores]), K, N.int_array([_method_code(m) for m in methods]),
                                       out_rows, self.inner, row_start.ctypes.data_as(N.p_i32),
                                       child_rank.ctypes.data_as(N.p_i32), child_row.ctypes.data_as(N.p_i64), W, rank_rows,
                                       flat_v, flat_s, int(derive), results))
        self.last_pull_derived = bool(derive)
        # nobody frees or overwrites a store while a peer may still be reading it
        N.check(lib.olap_sync())
        self.last_pull_ms = lib.olap_last_op_ms()  # device time of the pull kernel on this rank (profiling aid)
        self.comm.dist.barrier(group=self.comm.group)
        return results

    def _all_ranks(self, flag):
        """Logical AND of a local flag over the ranks (a MIN all-reduce on the device: also a barrier)."""
        import torch

        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device="cuda")
        self.comm.dist.all_reduce(t, op=self.comm.dist.ReduceOp.MIN, group=self.comm.group)
        return bool(t.item())

    def _drill_up_pull2(self, out, full_map, touched, ids, methods, out_bounds):
        """Two-phase pull: (1) shard-local partial rollup of my rows into ONE compact partial row per
        output row I hold children of (`average` as a sum and a count plane); (2) the pull kernel
        combines, for each of MY output rows, the partial rows of the ranks that have one, in rank
        order — ranks hold contiguous ascending row ranges, so that is ascending row order and
        first / last stay exact; sums of float32 partials (rel 1e-6)."""
        me, W = self.rank, self.world
        if touched is None:
            touched = _exchange_costs(full_map, self.row_bounds, out_bounds)[4]
        plan = []
        for m, method in zip(ids, methods):
            if method == "average":
                plan += [(m, "sum", "sum"), (m, "__count", "sum")]
            else:
                plan.append((m, method, method))
        stores = [self.storedMeasures[m] for m, _, _ in plan]
        mine = touched[me]
        local_map = np.searchsorted(mine, full_map[self.row0:self.row1]).astype(np.int32)
        maps = [local_map] + [None] * len(self.inner_lens)
        partials = self._store_cls.drillUp_lowered(stores, self._local_lens(), [int(mine.size)] + self.inner_lens, maps,
                                                   [meth for _, meth, _ in plan])
        views = self._peer_views(partials, remember=False)
        if views is None:
            return None
        j0, j1 = out_bounds[me], out_bounds[me + 1]
        tables = _pull2_tables(touched, j0, j1)
        results = self._pull_call(partials, [comb for _, _, comb in plan], views, tables, [int(t.size) for t in touched], j1 - j0)
        del partials
        out.last_pull_ms, out.last_pull_derived = self.last_pull_ms, self.last_pull_derived
        combined = [self._store_cls._wrap(h) for h in results]
        k = 0
        for m, method in zip(ids, methods):
            if method == "average":
                out.storedMeasures[m] = self._divide(combined[k], combined[k + 1])
                k += 2
            else:
                out.storedMeasures[m] = combined[k]
                k += 1
        return out

    def _combine(self, out, plan, ids, methods, received, my_out_rows):
        """3. ordered combine of the W partials: a drillUp over the rank axis."""
        W = self.world
        comb_old = [W, my_out_rows] + self.inner_lens
        comb_new = [1, my_out_rows] + self.inner_lens
        comb_maps = [np.zeros(W, dtype=np.int32)] + [np.arange(n, dtype=np.int32) for n in comb_old[1:]]
        comb_methods = ["sum" if role != "plain" else meth for _, meth, role in plan]
        combined = self._call("drillUp_lowered", received, comb_old, comb_new, comb_maps, _Per(comb_methods))
        del received
        k = 0
        for m, method in zip(ids, methods):
            if method == "average":
                out.storedMeasures[m] = self._divide(combined[k], combined[k + 1])
                k += 2
            else:
                out.storedMeasures[m] = combined[k]
                k += 1
        return out

    def _partials_into_peers(self, stores, part_methods, row_map, out_bounds, new_rows_total):
        """1 + 2 fused: the partial rollup of my rows, every output row written by the kernel
        into the receive buffer of its owner (slot = my rank), over NVLink.  Returns my receive
        planes wrapped as stores [W, my_out_rows, inner...]."""
        import ctypes as C

        import torch

        from . import _native as N
        from .store import _method_code

        W, me, inner = self.world, self.rank, self.inner
        K = len(stores)
        rows_of = [out_bounds[r + 1] - out_bounds[r] for r in range(W)]
        with_status = bool(N.lib().olap_store_has_status(stores[0]._h))
        r_max = max(rows_of)
        pad = lambda b: (b + 255) // 256 * 256  # every plane starts on a 256-byte boundary, like a store's own planes
        plane_v, plane_s = pad(W * r_max * inner * 4), pad(W * r_max * inner)
        nbytes = K * plane_v + (K * plane_s if with_status else 0) + 256
        # nobody may still be combining the previous contents of these buffers (the barrier orders
        # host threads only: drain the library's own stream first, whatever the async mode)
        N.check(N.lib().olap_sync())
        self.comm.dist.barrier(group=self.comm.group)
        bases = _PeerBuffers.get(self.comm, nbytes)

        def val_ptr(r, k, src_rank):  # plane k of rank r's buffer, slot of the sending rank
            return bases[r] + k * plane_v + src_rank * rows_of[r] * inner * 4

        def st_ptr(r, k, src_rank):
            return bases[r] + K * plane_v + k * plane_s + src_rank * rows_of[r] * inner

        position, table_v, table_s = _peer_row_tables(bases, out_bounds, me, K, inner, plane_v, plane_s, with_status)
        row_vals = (C.c_void_p * table_v.size)(*table_v.tolist())
        row_sts = (C.c_void_p * table_s.size)(*table_s.tolist()) if with_status else None
        codes = [_method_code(m) for m in part_methods]
        rows_local = self.rows_local
        permuted_map = np.ascontiguousarray(position[np.asarray(row_map, dtype=np.int64)], dtype=np.int32)
        N.check(N.lib().olap_drill_up_rows(N.store_array([s._h for s in stores]), K, N.int_array(codes), rows_local,
                                           new_rows_total, inner, permuted_map.ctypes.data_as(N.p_i32), row_vals, row_sts))
        N.check(N.lib().olap_sync())
        torch.cuda.synchronize()
        # every rank has finished storing into every buffer
        self.comm.dist.barrier(group=self.comm.group)
        received = []
        my_rows = rows_of[me]
        for k, src_store in enumerate(stores):
            h = C.c_void_p()
            N.check(N.lib().olap_store_wrap(C.c_void_p(val_ptr(me, k, 0)), C.c_void_p(st_ptr(me, k, 0)) if with_status else None,
                                            W * my_rows * inner, N.TYPES[src_store._type],
                                            N.DEFAULT_NAN if src_store._defaultValue != src_store._defaultValue else N.DEFAULT_ZERO,
                                            C.byref(h)))
            received.append(self._store_cls._wrap(h.value))
        return received

    def _partials(self, stores, old_len, new_len, maps, methods):
        return self._store_cls.drillUp_lowered(stores, old_len, new_len, maps, methods)

    def _exchange_all(self, parts, recvs, in_splits, out_splits):
        """One all-to-all per plane (values, status) of every partial."""
        cls = self._store_cls
        sent = [cls.exchange_planes(part) for part in parts]
        got = [cls.exchange_planes(recv) for recv in recvs]
        if cls.DEVICE == "cuda":
            import torch

            from . import _native as N

            N.check(N.lib().olap_sync())
            torch.cuda.current_stream().synchronize()
        self.comm.all_to_all_many([(o, i) for outs, ins in zip(got, sent) for o, i in zip(outs, ins)], out_splits, in_splits)
        if cls.DEVICE == "cuda":
            torch.cuda.synchronize()
        for recv, planes in zip(recvs, got):
            cls.exchange_done(recv, planes)

    def _divide(self, sums, counts):
        """average = sum of sums / sum of counts; no contribution -> unset (in-memory.js:323-331)."""
        return self._store_cls.average_of(sums, counts)

    def dice(self, dimensionId, attribute, items, reorder=False):
        """Dice: a shard-local gather, whichever dimension is diced (no communication)."""
        idx = self.getDimensionIndex(dimensionId)
        return self._dice_to(idx, self.dimensions[idx].dice(attribute, items, reorder))

    def diceRange(self, dimensionId, attribute, start, end):  # cube.js:809-832
        idx = self.getDimensionIndex(dimensionId)
        return self._dice_to(idx, self.dimensions[idx].diceRange(attribute, start, end))

    @staticmethod
    def release_peer_buffers():
        """Free the receive buffers of the push exchange (collective; see _PeerBuffers.release)."""
        _PeerBuffers.release()

    def removeDimension(self, dimensionId):
        """cube.js:950-964: roll the dimension up to 'all' with each measure's rule, then forget
        it.  Forgetting a one-item dimension changes no cell and no shard bound."""
        idx = self.getDimensionIndex(dimensionId)
        if len(self.dimensions) == 1:
            raise NotImplementedError("removing the only dimension of a sharded cube leaves one cell: use getTotal")
        rolled = self.drillUp(dimensionId, "all")
        if idx < rolled.prefix and rolled.prefix == 1:
            rolled = rolled._deepened()
        dims = [d for d in rolled.dimensions if d.id != dimensionId]
        out = ShardedCube(dims, rolled.prefix - (1 if idx < rolled.prefix else 0), self._store_cls, self.comm.group,
                          list(rolled.row_bounds))
        out.storedMeasures = dict(rolled.storedMeasures)
        out.computedMeasures = dict(self.computedMeasures)
        out.storedMeasuresRules = {m: {k: v for k, v in rules.items() if k != dimensionId}
                                   for m, rules in self.storedMeasuresRules.items()}
        return out

    def removeDimensions(self, dimensionIds):  # cube.js:899-908
        cube = self
        for dimensionId in dimensionIds:
            cube = cube.removeDimension(dimensionId)
        return cube

    def keepDimensions(self, dimensionIds):  # cube.js:890-897
        return self.removeDimensions([d for d in self.dimensionIds if d not in dimensionIds])

    def slice(self, dimensionId, attribute, value):  # cube.js:799-807
        if self.getDimensionIndex(dimensionId) == -1:
            raise ValueError(f"slice: no such dimension: {dimensionId}")
        return self.dice(dimensionId, attribute, [value]).removeDimension(dimensionId)

    def _dice_to(self, idx, new_dim):
        old_dim = self.dimensions[idx]
        if new_dim is old_dim:
            return self
        new_dims = list(self.dimensions)
        new_dims[idx] = new_dim
        old_idx = old_dim.getItemsToIdx()
        kept = np.asarray([old_idx[i] for i in new_dim.getItems()], dtype=np.int32)
        keep = [np.arange(n, dtype=np.int32) for n in self._local_lens()]
        if idx < self.prefix:
            # Dice of a sharded dimension: whole rows are dropped where they live, nothing moves
            # (SURVEY.md §8e "drop/reassign whole rows; rebalance optional").  Kept rows stay in
            # ascending order, so every rank's survivors are one contiguous range of the new row
            # numbering; the shard sizes may become uneven.
            if kept.size > 1 and np.any(np.diff(kept) <= 0):
                # dice(reorder=True) that permutes a sharded dimension: drop the rows in place first (ascending
                # items, nothing moves), then shuffle whole rows into the requested order (_shuffle_rows)
                order = np.argsort(kept, kind="stable")
                if np.any(np.diff(kept[order]) == 0):
                    raise ValueError("dice: an item is listed twice")
                items = old_dim.getItems()
                ascending = self._dice_to(idx, old_dim.dice(old_dim.rootAttribute, [items[i] for i in kept[order]], False))
                # position of every requested item in the ascending cube
                rank_of = np.empty(kept.size, dtype=np.int64)
                rank_of[order] = np.arange(kept.size)
                new_prefix_lens = [d.numItems for d in new_dims[: self.prefix]]
                below = _prod(new_prefix_lens[idx + 1:])
                new_rows = np.arange(_prod(new_prefix_lens), dtype=np.int64)
                outer, rest = np.divmod(new_rows, new_prefix_lens[idx] * below)
                coord, low = np.divmod(rest, below)
                old_of_new = (outer * new_prefix_lens[idx] + rank_of[coord]) * below + low
                return ascending._shuffle_rows(old_of_new, new_dims)
            old_prefix_lens = [d.numItems for d in self.dimensions[: self.prefix]]
            survives = np.zeros(old_prefix_lens[idx], dtype=bool)
            survives[kept] = True
            coord = (np.arange(self.rows_total, dtype=np.int64) // _prod(old_prefix_lens[idx + 1:])) % old_prefix_lens[idx]
            row_kept = survives[coord]
            before = np.concatenate([[0], np.cumsum(row_kept)])
            out = self._derive(new_dims, [int(before[b]) for b in self.row_bounds])
            keep[0] = np.flatnonzero(row_kept[self.row0:self.row1]).astype(np.int32)
        else:
            out = self._derive(new_dims, self.row_bounds)
            keep[1 + idx - self.prefix] = kept
        ids = list(self.storedMeasures)
        if ids:
            res = self._call("dice_lowered", [self.storedMeasures[m] for m in ids], self._local_lens(), keep)
            out.storedMeasures = dict(zip(ids, res))
        return out

    def _shuffle_rows(self, old_of_new, new_dims):
        """Whole rows into a new global order: new row j is old row old_of_new[j] (a permutation of the rows, or an
        injective selection).  Every rank gathers the rows it has to send in ascending new-row order (so that the
        runs for rank 0, 1, ... follow each other), one all-to-all per plane moves them, and the receiver — whose
        blocks arrive grouped by sending rank — gathers them into ascending new-row order."""
        old_of_new = np.asarray(old_of_new, dtype=np.int64)
        total = int(old_of_new.size)
        W = self.world
        new_bounds = split_rows(total, W)
        out = ShardedCube(new_dims, self.prefix, self._store_cls, self.comm.group, new_bounds)
        out.storedMeasuresRules = dict(self.storedMeasuresRules)
        out.computedMeasures = dict(self.computedMeasures)
        ids = list(self.storedMeasures)
        if not ids:
            return out
        stores = [self.storedMeasures[m] for m in ids]
        src = np.searchsorted(np.asarray(self.row_bounds[1:]), old_of_new, side="right")   # who holds the row now
        dst = np.searchsorted(np.asarray(new_bounds[1:]), np.arange(total), side="right")    # who gets it
        inner_keep = [np.arange(n, dtype=np.int32) for n in self.inner_lens]  # per inner dimension: no table of inner cells
        mine = np.flatnonzero(src == self.rank)  # new rows I hold, ascending: grouped by destination rank
        in_splits = [int(np.count_nonzero(dst[mine] == r)) * self.inner for r in range(W)]
        n0, n1 = new_bounds[self.rank], new_bounds[self.rank + 1]
        src_mine = src[n0:n1]
        out_splits = [int(np.count_nonzero(src_mine == s)) * self.inner for s in range(W)]
        if mine.size and self.inner:
            sent = self._call("dice_lowered", stores, [self.rows_local] + self.inner_lens,
                              [(old_of_new[mine] - self.row0).astype(np.int32)] + inner_keep)
        else:
            sent = [self._empty_like(s, 0) for s in stores]
        received = [self._empty_like(s, (n1 - n0) * self.inner) for s in stores]
        self._exchange_all(sent, received, in_splits, out_splits)
        del sent
        # received: block of rank 0's rows (ascending new row), block of rank 1's rows, ...
        arrival = np.argsort(src_mine, kind="stable")          # arrival position -> local new row
        if (n1 - n0) and self.inner and np.any(arrival != np.arange(n1 - n0)):
            position = np.empty(n1 - n0, dtype=np.int32)
            position[arrival] = np.arange(n1 - n0, dtype=np.int32)  # local new row -> arrival position
            received = self._call("dice_lowered", received, [n1 - n0] + self.inner_lens, [position] + inner_keep)
        out.storedMeasures = dict(zip(ids, received))
        return out

    def rebalance(self):
        """After a dice of a sharded dimension the surviving rows stay where they lived: the shards become uneven,
        some may be empty (SURVEY.md §8e "drop/reassign whole rows; rebalance optional").  Rebalancing gives every
        rank an even share again.  Returns self when the rows are already spread evenly."""
        return self._repartition(split_rows(self.rows_total, self.world))

    def _repartition(self, new_bounds, prefix=None):
        """Move whole rows so that rank r holds rows [new_bounds[r], new_bounds[r + 1]).  The old and the new partition
        are both contiguous in global row order, so rank r sends ONE contiguous run of its rows to every rank whose
        new range overlaps its old one and receives its new rows in ascending order of the sending rank: one
        all-to-all per plane, nothing is reordered on either side.  `prefix`: how many leading dimensions the new
        cube counts as sharded (rows are then rows of THAT prefix; the cells do not move for it)."""
        new_bounds = [int(b) for b in new_bounds]
        prefix = self.prefix if prefix is None else int(prefix)
        if new_bounds == list(self.row_bounds) and prefix == self.prefix:
            return self
        below = _prod(d.numItems for d in self.dimensions[prefix:self.prefix])  # old rows per new row (prefix <= self.prefix)
        if any(b % below for b in new_bounds):
            raise ValueError("new shard bounds must fall on rows of the new prefix")
        out = ShardedCube(self.dimensions, prefix, self._store_cls, self.comm.group, [b // below for b in new_bounds])
        out.storedMeasuresRules = dict(self.storedMeasuresRules)
        out.computedMeasures = dict(self.computedMeasures)
        ids = list(self.storedMeasures)
        if not ids:
            return out
        stores = [self.storedMeasures[m] for m in ids]
        if new_bounds == list(self.row_bounds):  # same cells on every rank, only the bookkeeping changes
            out.storedMeasures = dict(zip(ids, stores))
            return out

        def overlap(a0, a1, b0, b1):
            return max(0, min(a1, b1) - max(a0, b0))

        W = self.world
        n0, n1 = new_bounds[self.rank], new_bounds[self.rank + 1]
        in_splits = [overlap(self.row0, self.row1, new_bounds[r], new_bounds[r + 1]) * self.inner for r in range(W)]
        out_splits = [overlap(self.row_bounds[s], self.row_bounds[s + 1], n0, n1) * self.inner for s in range(W)]
        received = [self._empty_like(s, (n1 - n0) * self.inner) for s in stores]
        self._exchange_all(stores, received, in_splits, out_splits)
        out.storedMeasures = dict(zip(ids, received))
        return out

    def drillDown(self, dimensionId, attribute):
        """drillDown: shard-local whichever dimension is drilled (every child row is produced by
        the rank that holds its parent row; no communication)."""
        idx = self.getDimensionIndex(dimensionId)
        old_dim = self.dimensions[idx]
        if old_dim.rootAttribute == attribute:
            return self
        new_dim = old_dim.drillDown(attribute)
        new_dims = list(self.dimensions)
        new_dims[idx] = new_dim
        child_to_parent = np.asarray(new_dim.getGroupIndexFromRootIndexMap(old_dim.rootAttribute), np.int32)
        old_len = self._local_lens()
        if idx < self.prefix:
            # new global row -> old global row; the rows whose parent I hold must form one
            # contiguous range of the new numbering, rank after rank (true when the drilled
            # dimension is the outermost one, or when the shard bounds fall on its boundaries)
            old_prefix_lens = [d.numItems for d in self.dimensions[: self.prefix]]
            new_prefix_lens = [d.numItems for d in new_dims[: self.prefix]]
            below = _prod(old_prefix_lens[idx + 1:])
            new_rows = np.arange(_prod(new_prefix_lens), dtype=np.int64)
            outer, rest = np.divmod(new_rows, new_prefix_lens[idx] * below)
            coord, low = np.divmod(rest, below)
            old_row = (outer * old_prefix_lens[idx] + child_to_parent[coord]) * below + low
            owner = np.searchsorted(np.asarray(self.row_bounds[1:]), old_row, side="right")
            if owner.size > 1 and np.any(np.diff(owner) < 0):
                # the shard bounds cut through an item of the drilled dimension: move whole rows between
                # neighbouring ranks first, so that every rank holds whole items of it (_repartition), then expand
                aligned = [b * below for b in split_rows(_prod(old_prefix_lens[: idx + 1]), self.world)]
                if aligned == list(self.row_bounds):
                    raise NotImplementedError("drillDown of a sharded dimension whose shard bounds cut through it "
                                              "re-partitions rows; shard on that dimension alone (prefix=1) or align the bounds")
                return self._repartition(aligned).drillDown(dimensionId, attribute)
            new_bounds = [int(b) for b in np.searchsorted(owner, np.arange(self.world + 1), side="left")]
            out = self._derive(new_dims, new_bounds)
            mine = old_row[new_bounds[self.rank]:new_bounds[self.rank + 1]] - self.row0
            new_len = [int(mine.size)] + self.inner_lens
            maps = [np.arange(n, dtype=np.int32) for n in new_len]
            maps[0] = mine.astype(np.int32)
        else:
            out = self._derive(new_dims, self.row_bounds)
            new_len = [self.rows_local] + [d.numItems for d in new_dims[self.prefix:]]
            maps = [np.arange(n, dtype=np.int32) for n in new_len]
            maps[1 + idx - self.prefix] = child_to_parent
        ids = list(self.storedMeasures)
        methods = [self.storedMeasuresRules[m].get(dimensionId) or "sum" for m in ids]
        if ids:
            stores = [self.storedMeasures[m] for m in ids]
            res = self._store_cls.drillDown_lowered(stores, old_len, new_len, maps, methods)
            out.storedMeasures = dict(zip(ids, res))
        return out


    def reorderDimensions(self, dimensionIds):
        """Axis permutation (cube.js:757-783).  Permutations of the dimensions inside the shard
        are shard-local.  With the cube sharded on its outermost dimension alone (prefix = 1),
        a permutation that brings ANOTHER dimension to the front re-partitions the cells on
        that dimension: one local transpose, one all-to-all, a row gather and one more local
        transpose (SURVEY.md §8e)."""
        dimensionIds = list(dimensionIds)
        if dimensionIds == self.dimensionIds:
            return self
        perm = [self.getDimensionIndex(i) for i in dimensionIds]  # new position -> old position
        if sorted(perm) != list(range(len(self.dimensions))):
            raise ValueError("Invalid dimensions provided")
        new_dims = [self.dimensions[j] for j in perm]
        ids = list(self.storedMeasures)
        stores = [self.storedMeasures[m] for m in ids]
        lens = [d.numItems for d in self.dimensions]
        if perm[: self.prefix] == list(range(self.prefix)):
            out = self._derive(new_dims, self.row_bounds)
            if stores:
                order = [0] + [1 + j - self.prefix for j in perm[self.prefix:]]
                out.storedMeasures = dict(zip(ids, self._reorder(stores, self._local_lens(), order)))
            return out
        if self.prefix != 1:
            # shard on the outermost dimension alone first (whole rows of it move between neighbouring ranks: one
            # all-to-all per plane, _repartition), then re-partition on the dimension that comes to the front
            below = _prod(d.numItems for d in self.dimensions[1:self.prefix])
            outer_bounds = [b * below for b in split_rows(lens[0], self.world)]
            return self._repartition(outer_bounds, prefix=1).reorderDimensions(dimensionIds)
        W, k = self.world, perm[0]
        new_bounds = split_rows(lens[k], W)
        out = self._derive(new_dims, new_bounds)
        if not stores:
            return out
        others = [j for j in perm[1:] if j != 0]  # old positions, in their new order, without the two sharded axes
        other_lens = [lens[j] for j in others]
        O = _prod(other_lens)
        my_k = new_bounds[self.rank + 1] - new_bounds[self.rank]
        src_rows = [self.row_bounds[r + 1] - self.row_bounds[r] for r in range(W)]
        # 1. local transpose to [Dk, my rows of D0, others]: the cells for rank r are one contiguous run
        sent = self._reorder(stores, [self.rows_local] + lens[1:], [k, 0] + others)
        # 2. all-to-all: from rank s I receive the block [my Dk items, s's rows of D0, others]
        in_splits = [(new_bounds[r + 1] - new_bounds[r]) * self.rows_local * O for r in range(W)]
        out_splits = [my_k * src_rows[r] * O for r in range(W)]
        if W == 1:
            received = sent
        else:
            received = [self._empty_like(s, sum(out_splits)) for s in stores]
            self._exchange_all(sent, received, in_splits, out_splits)
        del sent
        # 3. rows (k, d0) of the W received blocks -> one block [my Dk items, D0, others]
        d0_total = lens[0]
        block_start = np.concatenate([[0], np.cumsum([my_k * r for r in src_rows])])
        owner = np.searchsorted(np.asarray(self.row_bounds[1:]), np.arange(d0_total), side="right")
        d0_local = np.arange(d0_total) - np.asarray(self.row_bounds)[owner]
        rows = (block_start[owner][None, :] + np.arange(my_k)[:, None] * np.asarray(src_rows)[owner][None, :]
                + d0_local[None, :]).reshape(-1).astype(np.int32)
        if my_k * d0_total * O == 0:
            out.storedMeasures = {m: self._empty_like(s, 0) for m, s in zip(ids, stores)}
            return out
        # (identity lists per remaining dimension, not one list over all O cells of a row: O is 1e8 for a 1e10-cell cube)
        gathered = self._call("dice_lowered", received, [my_k * d0_total] + other_lens,
                              [rows] + [np.arange(n, dtype=np.int32) for n in other_lens])
        del received
        # 4. local transpose to the requested order
        final = [0] + [1 if j == 0 else 2 + others.index(j) for j in perm[1:]]
        if final != list(range(len(final))):
            gathered = self._reorder(gathered, [my_k, d0_total] + other_lens, final)
        out.storedMeasures = dict(zip(ids, gathered))
        return out

    def _reorder(self, stores, old_len, new_to_old):
        if _prod(old_len) == 0:
            return [self._empty_like(s, 0) for s in stores]
        return self._call("reorder_lowered", stores, old_len, new_to_old)

    def _empty_like(self, store, size):
        if getattr(self._store_cls, "SHAREABLE_SHARDS", False):  # a later rollup of the sharded axis may pull from it
            return self._store_cls(size, store._type, store._defaultValue, shareable=True)
        return self._store_cls(size, store._type, store._defaultValue)


class _Per(list):
    """One value per store (methods)."""
