"""GpuStore — device-resident replacement of the reference's per-measure store.

Same members as ``InMemoryStore`` as ``Cube`` uses them
(/root/reference/src/store/in-memory.js:7-431; call sites listed in SURVEY.md
§8b): constructor ``(size, type, defaultValue)``, ``byteLength``, ``size``,
``total``, ``data`` (get/set), ``getValue``, ``setValue``, ``fill``, ``clone``,
``load``, ``reorder``, ``dice``, ``drillUp``, ``drillDown`` and the raw fields
``_type``, ``_defaultValue``, ``_dataMap``.  Dimension objects are lowered here to
dense int32 index maps; everything O(cells) happens in libolapgpu.so (C ABI in
include/olap_gpu.h, hand-written sm_100a kernels).  No CPU fallback exists."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _native as N


def _default_kind(defaultValue):
    if defaultValue != defaultValue:
        return N.DEFAULT_NAN
    if defaultValue == 0:
        return N.DEFAULT_ZERO
    raise N.OlapValueError("Invalid default value, only NaN and 0 are supported")  # in-memory.js:56-57


def _method_code(method):
    name = "sum" if method is None else method
    if name == "__count":  # internal: set children per parent (sharded average)
        return N.COUNT
    code = N.METHODS.get(name)
    if code is None:
        raise N.OlapValueError(f"Unsupported aggregation method: {name}")  # in-memory.js:294-296
    return code


def _lens(dims):
    return [d.numItems for d in dims]


class GpuStore:
    #: allocate a status byte per cell next to the Float32 cells (README.md:698-721)
    WITH_STATUS = True
    FUSED_ROLLUPS = True  # Cube may present a run of removed dimensions as one merged axis (cube.py)
    IMPLIED_MAPS = True   # drillUp_lowered accepts None for unchanged / rolled-to-one dimensions
    SHAREABLE_SHARDS = True  # ShardedCube creates its local shards in memory the peers can map (CUDA IPC)

    def __init__(self, size, type="float32", defaultValue=math.nan, *, _handle=None, with_status=None,
                 uninitialised=False, shareable=False):
        if _handle is not None:
            self._h = _handle
        else:
            kind = _default_kind(defaultValue)
            if type not in N.TYPES:
                raise N.OlapValueError("Invalid type")  # in-memory.js:59-60
            out = C.c_void_p()
            status = self.WITH_STATUS if with_status is None else with_status
            # OLAP_CREATE_UNINITIALISED = 2, OLAP_CREATE_SHAREABLE = 4 (peers of a sharded cube can map it)
            flags = int(bool(status)) | (2 if uninitialised else 0) | (4 if shareable else 0)
            N.check(N.lib().olap_store_create(int(size), N.TYPES[type], kind, flags, C.byref(out)))
            self._h = out.value
        lib = N.lib()
        self._size = lib.olap_store_size(self._h)
        self._type = N.TYPE_NAMES[lib.olap_store_type(self._h)]
        self._defaultValue = math.nan if lib.olap_store_default_kind(self._h) == N.DEFAULT_NAN else 0

    @classmethod
    def _wrap(cls, handle):
        return cls(0, _handle=handle)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and N._lib is not None:
            try:
                N._lib.olap_store_destroy(h)
            except Exception:
                pass

    # ---- in-memory.js:8-46 -------------------------------------------------
    @property
    def byteLength(self):
        return N.lib().olap_store_byte_length(self._h)

    @property
    def size(self):
        return self._size

    @property
    def total(self):
        out = C.c_double()
        N.check(N.lib().olap_store_total(self._h, C.byref(out)))
        return out.value

    @property
    def data(self):
        return self.data_f32().astype(np.float64).tolist()

    @data.setter
    def data(self, values):
        if isinstance(values, np.ndarray) and values.dtype == np.float32:
            return self.set_data_f32(values)
        n = len(values)
        if n != self._size:
            raise N.OlapValueError(f"value length is invalid: {self._size} !== {n}")
        d = float(self._defaultValue)
        arr = np.fromiter((d if v is None else v for v in values), dtype=np.float64, count=n)
        N.check(N.lib().olap_store_upload_f64(self._h, arr.ctypes.data, n))

    def data_f32(self):
        """Cells as a float32 numpy array (the Float32Array fast path of the addon)."""
        out = np.empty(self._size, dtype=np.float32)
        N.check(N.lib().olap_store_download_f32(self._h, out.ctypes.data, self._size))
        return out

    def set_data_f32(self, values):
        values = np.ascontiguousarray(values, dtype=np.float32)
        N.check(N.lib().olap_store_upload_f32(self._h, values.ctypes.data, values.size))

    @property
    def status(self):
        out = np.empty(self._size, dtype=np.uint8)
        N.check(N.lib().olap_store_status(self._h, out.ctypes.data, self._size))
        return out.tolist()

    def presence(self):
        out = np.empty(self._size, dtype=np.uint8)
        N.check(N.lib().olap_store_presence(self._h, out.ctypes.data, self._size))
        return out

    @property
    def _dataMap(self):
        """Set cells as {index: value}, keys ascending (the reference's Map, in-memory.js:63)."""
        keys, values = self.export_sparse()
        return dict(zip(keys.tolist(), values.astype(np.float64).tolist()))

    def export_sparse(self):
        count = C.c_int64()
        N.check(N.lib().olap_store_count_present(self._h, C.byref(count)))
        keys = np.empty(count.value, dtype=np.int64)
        values = np.empty(count.value, dtype=np.float32)
        N.check(N.lib().olap_store_export_sparse(self._h, count.value, keys.ctypes.data, values.ctypes.data, C.byref(count)))
        return keys, values

    def import_sparse(self, keys, values):
        keys = np.ascontiguousarray(keys, dtype=np.int64)
        values = np.ascontiguousarray(values, dtype=np.float32)
        N.check(N.lib().olap_store_import_sparse(self._h, keys.ctypes.data, values.ctypes.data, keys.size))

    def serialize(self):
        """in-memory.js:75-101: {size, type, defaultValue, indexes: Uint32Array, dataBuffer} in the
        reference's wire format; the set cells leave the device through the ordered stream
        compaction (keys ascending: the Map order of a store filled by `set data`)."""
        from .serialization import store_to_buffer

        keys, values = self.export_sparse()
        return store_to_buffer(self._size, self._type, self._defaultValue, keys, values)

    @classmethod
    def deserialize(cls, buffer, size=None):
        """in-memory.js:103-116.  The wire format carries `size` as a Float32
        (serialization.js:71-74); `size`, when given, is the caller's exact cell count and must
        round to the transmitted one."""
        from .serialization import store_from_buffer

        wire_size, type, default, keys, values = store_from_buffer(buffer)
        if size is None:
            size = wire_size
        elif int(np.float32(size)) != wire_size:
            raise N.OlapValueError(f"value length is invalid: {size} !== {wire_size}")
        store = cls(size, type, default)
        if keys.size:
            store.import_sparse(keys, values)
        return store

    @property
    def status_derived(self):
        """True when the status plane holds nothing the values do not say (include/olap_gpu.h,
        olap_store_status_derived): rollups of such a store never read it."""
        return bool(N.lib().olap_store_status_derived(self._h))

    def canonicalise(self):
        """After the planes were written through raw pointers (interop): canonicalise the values and
        re-derive the status plane from them."""
        N.check(N.lib().olap_store_canonicalise(self._h))

    def ipc_export(self):
        """(64-byte CUDA IPC handle, values offset, status offset or -1) of a shareable store."""
        handle = C.create_string_buffer(64)
        v_off, s_off = C.c_int64(), C.c_int64()
        N.check(N.lib().olap_store_ipc_export(self._h, handle, C.byref(v_off), C.byref(s_off)))
        return handle.raw, v_off.value, s_off.value

    def clone(self):  # in-memory.js:66-73
        out = C.c_void_p()
        N.check(N.lib().olap_store_clone(self._h, C.byref(out)))
        return GpuStore._wrap(out.value)

    def __deepcopy__(self, _memo):  # lodash cloneDeep of a store, cube.js:152-154
        return self.clone()

    # ---- in-memory.js:118-137 --------------------------------------------------
    def getValue(self, index):
        out = C.c_double()
        N.check(N.lib().olap_store_get_value(self._h, int(index), C.byref(out)))
        return out.value

    def setValue(self, index, value):
        v = float(self._defaultValue) if value is None else float(value)
        N.check(N.lib().olap_store_set_value(self._h, int(index), v))

    def setValues(self, indexes, values):
        idx = np.ascontiguousarray(indexes, dtype=np.int64)
        val = np.ascontiguousarray(values, dtype=np.float64)
        N.check(N.lib().olap_store_set_values(self._h, idx.ctypes.data, val.ctypes.data, idx.size))

    def fill(self, value):
        N.check(N.lib().olap_store_fill(self._h, float(value)))

    # ---- in-memory.js:139-176 --------------------------------------------------
    def load(self, otherStore, myDimensions, hisDimensions):
        his_to_mine = []
        for i, his in enumerate(hisDimensions):
            mine = myDimensions[i].getItemsToIdx()
            his_to_mine.append([mine.get(item, -1) for item in his.getItems()])
        self.load_lowered(otherStore, _lens(myDimensions), _lens(hisDimensions), his_to_mine)

    def load_lowered(self, otherStore, my_len, his_len, his_to_mine):
        """his_to_mine[d][j] = my item index of his item j; None / -1 when I lack the item."""
        keep, ptrs = N.map_arrays([[-1 if v is None else v for v in m] for m in his_to_mine])
        N.check(
            N.lib().olap_load(self._h, otherStore._h, len(my_len), N.i64_array(my_len), N.i64_array(his_len), ptrs)
        )
        del keep

    # ---- region queries (Cube.getTotalForDimensionItems / copyMeasureData) -------------
    @staticmethod
    def _region_args(lens, keep):
        """keep[d]: item indices of axis d (any order, repeats counted) or None for the whole axis."""
        alive, ptrs = N.map_arrays(keep)
        keep_len = [n if k is None else len(k) for n, k in zip(lens, alive)]
        return alive, len(lens), N.i64_array(lens), N.i64_array(keep_len), ptrs

    def regionSum(self, lens, keep):
        """Double sum of the raw cells (unset cells count as the default) of keep[0] x ... x keep[-1]."""
        alive, nd, len_arr, keep_len, ptrs = self._region_args(lens, keep)
        out = C.c_double()
        N.check(N.lib().olap_region_sum(self._h, nd, len_arr, keep_len, ptrs, C.byref(out)))
        del alive
        return out.value

    def regionCopy(self, src, lens, keep):
        """self.setValue(i, src.getValue(i)) for every cell i of keep[0] x ... x keep[-1], in place."""
        alive, nd, len_arr, keep_len, ptrs = self._region_args(lens, keep)
        N.check(N.lib().olap_region_copy(self._h, src._h, nd, len_arr, keep_len, ptrs))
        del alive

    # ---- computed measures over a region, status of a computed measure (Cube) -----------
    @staticmethod
    def regionEvalSum(expression, cell_names, stores, lens, keep):
        """Sum of a formula of cell variables over keep[0] x ... x keep[-1] (repeats counted): ONE kernel that
        evaluates it only at the region's cells (include/olap_gpu.h, olap_region_eval_sum)."""
        program = GpuStore._program(expression, cell_names, [])
        alive, nd, len_arr, keep_len, ptrs = GpuStore._region_args(lens, keep)
        out = C.c_double()
        N.check(N.lib().olap_region_eval_sum(program.encode(), N.store_array([s._h for s in stores]), len(stores), nd,
                                             len_arr, keep_len, ptrs, C.byref(out)))
        del alive
        return out.value

    @staticmethod
    def regionEvalCopy(target, expression, cell_names, stores, lens, keep):
        """target.setValue(i, formula(i)) for every cell i of the region, in place (olap_region_eval_copy); the
        target may be one of the formula's inputs."""
        program = GpuStore._program(expression, cell_names, [])
        alive, nd, len_arr, keep_len, ptrs = GpuStore._region_args(lens, keep)
        N.check(N.lib().olap_region_eval_copy(target._h, program.encode(), N.store_array([s._h for s in stores]),
                                              len(stores), nd, len_arr, keep_len, ptrs))
        del alive

    @staticmethod
    def statusMerge(stores, size):
        """Status bytes of a computed measure: the OR of its inputs' bytes, one kernel (olap_status_merge)."""
        out = np.empty(size, dtype=np.uint8)
        N.check(N.lib().olap_status_merge(N.store_array([s._h for s in stores]), len(stores), out.ctypes.data, size))
        return out.tolist()

    @staticmethod
    def statusMap_arrays(stores):
        """(keys int64, values float64, is_int uint8) of the status map of a computed measure over `stores`, in
        the order of the dict (olap_status_map_export)."""
        handles = N.store_array([s._h for s in stores])
        count = C.c_int64()
        N.check(N.lib().olap_status_map_export(handles, len(stores), 0, None, None, None, C.byref(count)))
        keys = np.empty(count.value, dtype=np.int64)
        values = np.empty(count.value, dtype=np.float64)
        is_int = np.empty(count.value, dtype=np.uint8)
        if count.value:
            N.check(N.lib().olap_status_map_export(handles, len(stores), count.value, keys.ctypes.data, values.ctypes.data,
                                                   is_int.ctypes.data, C.byref(count)))
        return keys, values, is_int

    @staticmethod
    def statusMap(stores):
        """Cube.getStatusMap of a computed measure: {cell: value} with ints where the fold ORed values."""
        keys, values, is_int = GpuStore.statusMap_arrays(stores)
        vals = values.tolist()
        for j in np.flatnonzero(is_int).tolist():
            vals[j] = int(vals[j])
        return dict(zip(keys.tolist(), vals))

    # ---- single-store forms of the transforms ------------------------------------
    def reorder(self, oldDimensions, newDimensions):
        return GpuStore.reorder_many([self], oldDimensions, newDimensions)[0]

    def dice(self, oldDimensions, newDimensions):
        return GpuStore.dice_many([self], oldDimensions, newDimensions)[0]

    def drillUp(self, oldDimensions, newDimensions, method="sum"):
        return GpuStore.drillUp_many([self], oldDimensions, newDimensions, [method])[0]

    def drillDown(self, oldDimensions, newDimensions, method="sum", distributions=None):
        return GpuStore.drillDown_many([self], oldDimensions, newDimensions, [method], [distributions])[0]

    # ---- batched forms: one call for all stored measures of a cube -----------------
    @staticmethod
    def _finish(out, n):
        return [GpuStore._wrap(out[k]) for k in range(n)]

    @staticmethod
    def reorder_many(stores, oldDimensions, newDimensions):
        """in-memory.js:178-211; the permutation is found by object identity (186-188)."""
        new_to_old = [next(i for i, d in enumerate(oldDimensions) if d is nd) for nd in newDimensions]
        return GpuStore.reorder_lowered(stores, _lens(oldDimensions), new_to_old)

    @staticmethod
    def reorder_lowered(stores, old_len, new_to_old):
        n = len(stores)
        out = (C.c_void_p * n)()
        perm = np.ascontiguousarray(new_to_old, dtype=np.int32)
        N.check(
            N.lib().olap_reorder(
                N.store_array([s._h for s in stores]), n, len(old_len), N.i64_array(old_len),
                perm.ctypes.data_as(N.p_i32), out,
            )
        )
        return GpuStore._finish(out, n)

    @staticmethod
    def dice_many(stores, oldDimensions, newDimensions):
        """in-memory.js:213-263; kept items are matched by name (219-224)."""
        keep = []
        for i, new_dim in enumerate(newDimensions):
            old_idx = oldDimensions[i].getItemsToIdx()
            keep.append([old_idx[item] for item in new_dim.getItems()])
        return GpuStore.dice_lowered(stores, _lens(oldDimensions), keep)

    @staticmethod
    def dice_lowered(stores, old_len, keep):
        n = len(stores)
        out = (C.c_void_p * n)()
        alive, ptrs = N.map_arrays(keep)
        N.check(
            N.lib().olap_dice(
                N.store_array([s._h for s in stores]), n, len(old_len), N.i64_array(old_len),
                N.i64_array([len(k) for k in keep]), ptrs, out,
            )
        )
        del alive
        return GpuStore._finish(out, n)

    @staticmethod
    def drillUp_many(stores, oldDimensions, newDimensions, methods):
        """in-memory.js:265-334; maps come from the OLD dimensions (270-274)."""
        # an untouched dimension needs no map (include/olap_gpu.h: NULL = unchanged): nothing to
        # build, upload or check for it, however many items it has
        maps = [
            None if new_dim is oldDimensions[i] else oldDimensions[i].getGroupIndexFromRootIndexMap(new_dim.rootAttribute)
            for i, new_dim in enumerate(newDimensions)
        ]
        return GpuStore.drillUp_lowered(stores, _lens(oldDimensions), _lens(newDimensions), maps, methods)

    @staticmethod
    def drillUp_lowered(stores, old_len, new_len, maps, methods):
        n = len(stores)
        codes = [_method_code(m) for m in methods]
        out = (C.c_void_p * n)()
        alive, ptrs = N.map_arrays(maps)
        N.check(
            N.lib().olap_drill_up(
                N.store_array([s._h for s in stores]), n, N.int_array(codes), len(old_len),
                N.i64_array(old_len), N.i64_array(new_len), ptrs, out,
            )
        )
        del alive
        return GpuStore._finish(out, n)

    drillUp_lowered_batch = drillUp_lowered  # the name Cube._remove_fused calls (FUSED_ROLLUPS)

    @staticmethod
    def drillDown_many(stores, oldDimensions, newDimensions, methods, distributions=None):
        """in-memory.js:336-430; maps come from the NEW dimensions (349-353)."""
        maps = [
            newDimensions[i].getGroupIndexFromRootIndexMap(old_dim.rootAttribute)
            for i, old_dim in enumerate(oldDimensions)
        ]
        return GpuStore.drillDown_lowered(
            stores, _lens(oldDimensions), _lens(newDimensions), maps, methods, distributions
        )

    @staticmethod
    def drillDown_lowered(stores, old_len, new_len, maps, methods, distributions=None):
        n = len(stores)
        # any method other than 'sum' copies the parent value (in-memory.js:421-423)
        codes = [N.METHODS.get("sum" if m is None else m, N.METHODS["last"]) for m in methods]
        out = (C.c_void_p * n)()
        alive, ptrs = N.map_arrays(maps)
        distributions = distributions or [None] * n
        dist_keep, dist_ptrs, dist_len = [], (N.p_f64 * n)(), (C.c_int64 * n)()
        for k, dist in enumerate(distributions):
            if dist is None:
                dist_ptrs[k] = None
                dist_len[k] = 0
            else:
                arr = np.array([math.nan if v is None else v for v in dist], dtype=np.float64)
                dist_keep.append(arr)
                dist_ptrs[k] = arr.ctypes.data_as(N.p_f64)
                dist_len[k] = arr.size
        N.check(
            N.lib().olap_drill_down(
                N.store_array([s._h for s in stores]), n, N.int_array(codes), len(old_len),
                N.i64_array(old_len), N.i64_array(new_len), ptrs, dist_ptrs, dist_len, out,
            )
        )
        del alive, dist_keep
        return GpuStore._finish(out, n)

    # ---- what ShardedCube needs from a store class beyond the batched transforms -----------
    DEVICE = "cuda"       # where the tensors of the collectives live
    PEER_MEMORY = True    # stores can be mapped by the other processes of the box (pull / push exchange)

    @classmethod
    def recv_like(cls, store, size):
        """A store about to be overwritten cell by cell by an exchange (no default fill)."""
        return cls(size, store._type, store._defaultValue, uninitialised=True, shareable=True)

    @staticmethod
    def exchange_planes(store):
        """The planes of a store as torch tensors an all-to-all can read or write in place."""
        from . import interop

        planes = [interop.values_tensor(store)]
        st = interop.status_tensor(store)
        if st is not None:
            planes.append(st)
        return planes

    @staticmethod
    def exchange_done(store, planes):
        """The tensors of exchange_planes alias the store: nothing to copy back."""

    @classmethod
    def average_of(cls, sums, counts):
        """sum of sums / sum of counts, no contribution -> unset (in-memory.js:323-331): one fused formula
        kernel; the quotient keeps the merged status flags of the sums (the unsharded `average` ORs its
        children's flags exactly like `sum` does; the formula kernel alone would derive SET / UNSET)."""
        default = "#nan" if sums._defaultValue != sums._defaultValue else "#0.0"
        out = cls.eval_program(f"v1 v0 v1 / {default} ?:", [sums, counts], [], sums._type, sums._defaultValue)
        N.check(N.lib().olap_store_copy_status(out._h, sums._h))
        return out

    # ---- computed measures (cube.js:331-363) ------------------------------------------
    @staticmethod
    def _program(expression, cell_names, total_names):
        slots = {name: f"v{k}" for k, name in enumerate(cell_names)}
        slots.update({name: f"t{k}" for k, name in enumerate(total_names)})
        return expression.postfix(slots)

    @staticmethod
    def evaluate(expression, cell_names, stores, totals, size):
        """One fused elementwise kernel over the input planes; returns a list of doubles."""
        return GpuStore.evaluate_f64(expression, cell_names, stores, totals, size).tolist()

    @staticmethod
    def evaluate_f64(expression, cell_names, stores, totals, size):
        if not stores:
            # a formula of constants/totals only: nothing per-cell to read
            value = expression.evaluate(dict(totals))
            return np.full(size, value, dtype=np.float64)
        total_names = list(totals.keys())
        program = GpuStore._program(expression, cell_names, total_names)
        out = np.empty(size, dtype=np.float64)
        tot = (C.c_double * max(1, len(total_names)))(*[totals[t] for t in total_names])
        N.check(
            N.lib().olap_eval(
                program.encode(), N.store_array([s._h for s in stores]), len(stores), tot, len(total_names),
                out.ctypes.data, 0, 0, None,
            )
        )
        return out

    @staticmethod
    def evaluate_to_store(expression, cell_names, stores, totals, type="float32", defaultValue=0):
        """copyToStoredMeasure without leaving the device (cube.js:205-215)."""
        total_names = list(totals.keys())
        program = GpuStore._program(expression, cell_names, total_names)
        return GpuStore.eval_program(program, stores, [totals[t] for t in total_names], type, defaultValue)

    @staticmethod
    def eval_program(program, stores, totals, type="float32", defaultValue=0):
        """Run a postfix formula program (include/olap_gpu.h, olap_eval) into a new store."""
        tot = (C.c_double * max(1, len(totals)))(*totals)
        out = C.c_void_p()
        N.check(
            N.lib().olap_eval(
                program.encode(), N.store_array([s._h for s in stores]), len(stores), tot, len(totals),
                None, N.TYPES[type], _default_kind(defaultValue), C.byref(out),
            )
        )
        return GpuStore._wrap(out.value)
