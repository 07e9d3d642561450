/*
 * olap_gpu.h — C ABI of the B200-native cell store for olap-in-memory.
 *
 * This is the drop-in boundary for ONE path of the reference: the per-measure
 * store `InMemoryStore` (/root/reference/src/store/in-memory.js:7-431) as it is
 * driven by `Cube` (/root/reference/src/cube.js).  Every entry point names the
 * reference member it replaces.  The JavaScript facade / N-API shim that binds
 * these symbols is shown in INTEGRATION.md (js/, addon/); in this repository
 * the same symbols are bound from Python with ctypes
 * (olap_in_memory_b200/_native.py).
 *
 * Conventions
 *  - plain C types only; all functions return 0 on success, a negative
 *    OLAP_E_* code otherwise; olap_last_error() gives the message of the last
 *    failure on the calling thread.  Messages of argument errors are the
 *    reference's own Error texts (in-memory.js:40-43, 56-60, 294-296, 397-398).
 *  - a store handle owns device memory: `float values[size]` and, optionally,
 *    `uint8_t status[size]` (README.md:698-721 flags).  Cells that are not set
 *    hold the canonical default (+0.0f or the quiet NaN 0x7fc00000), so
 *    presence is `default==NaN ? v==v : v!=0` exactly as in-memory.js:122-133.
 *  - transforms never mutate their inputs and return NEW handles (the
 *    reference's query methods are immutable, README.md:419-423); all stores
 *    returned by one call live in ONE contiguous device allocation.
 *  - batched entry points take `n` stores (all stored measures of a cube) so
 *    one launch sequence serves every measure and index maps cross PCIe once.
 *  - index maps are dense int32 arrays, one per dimension, exactly what
 *    `dimension.getGroupIndexFromRootIndexMap()` yields
 *    (src/dimension/generic.js:243-247, src/dimension/time.js:182-197).
 *    Linear cell indices are int64 (cubes exceed 2^32 cells).
 *  - calls are synchronous (the stream is drained before returning) unless
 *    olap_set_async(1); the library is driven from one host thread per device.
 *  - there is NO CPU fallback: without a CUDA device every call fails with
 *    OLAP_E_CUDA.
 */
#ifndef OLAP_GPU_H
#define OLAP_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OLAP_ABI_VERSION 1
#define OLAP_MAX_DIMS 16
#define OLAP_MAX_MEASURES 64

/* error codes */
#define OLAP_OK 0
#define OLAP_E_INVALID (-1)  /* bad argument; message = the reference's Error text */
#define OLAP_E_CUDA (-2)     /* CUDA runtime / driver / NVRTC failure, or no device */
#define OLAP_E_NOMEM (-3)    /* device allocation failed */
#define OLAP_E_UNSUPPORTED (-4)

/* `type` of a store (in-memory.js:59-60).  Cells are Float32 on the device for
 * every type; the tag drives byteLength (in-memory.js:8-16) and the integer
 * rounding of drillDown (in-memory.js:343, 403-417). */
#define OLAP_INT32 0
#define OLAP_UINT32 1
#define OLAP_FLOAT32 2
#define OLAP_FLOAT64 3

/* default value (in-memory.js:56-57: only 0 and NaN are legal) */
#define OLAP_DEFAULT_ZERO 0
#define OLAP_DEFAULT_NAN 1

/* aggregation methods (in-memory.js:282-290) */
#define OLAP_SUM 0
#define OLAP_AVERAGE 1
#define OLAP_HIGHEST 2
#define OLAP_LOWEST 3
#define OLAP_FIRST 4
#define OLAP_LAST 5
#define OLAP_PRODUCT 6
/* extension (not a reference method): number of set children per parent, as a float.
 * Used to finish `average` when the drilled dimension is sharded across GPUs. */
#define OLAP_COUNT 7

/* status flags (README.md:698-721) */
#define OLAP_STATUS_UNSET 0x1
#define OLAP_STATUS_SET 0x2
#define OLAP_STATUS_INTERPOLATED 0x4

typedef struct olap_store olap_store;

/* ---- library ------------------------------------------------------------ */
int olap_abi_version(void);
/* Bind the calling thread's library state to CUDA device `device`. */
int olap_init(int device);
/* Run all work on `cuda_stream` (a cudaStream_t); NULL restores the library's own stream. */
int olap_set_stream(void* cuda_stream);
/* 1: calls return without draining the stream (caller uses olap_sync). */
int olap_set_async(int enabled);
int olap_sync(void);
/* 1: every store created from now on (results of transforms included) is shareable with the other
 * processes of the box (OLAP_CREATE_SHAREABLE) — what a process holding one shard of a sharded cube
 * wants: any of its stores may be the source of a peer's pull. */
int olap_set_shareable(int enabled);
const char* olap_last_error(void);
/* Translate a method name ("sum", "average", ...) — in-memory.js:282-296.
 * Unknown names fail with "Unsupported aggregation method: <name>". */
int olap_method_from_name(const char* name, int* method);
/* Number of kernels this library launched since process start (bench evidence). */
int64_t olap_kernel_launches(void);
/* Device time in ms of the kernels of the most recent transform/eval call. */
double olap_last_op_ms(void);
/* Name of the kernel path the most recent transform took (for tests/profiles). */
const char* olap_last_op_path(void);

/* Debug aid: with OLAP_GUARD=1 in the environment every plane is followed by a guard region
 * that is checked when the store is destroyed; returns the number of overwritten guard bytes. */
int64_t olap_guard_violations(void);

/* Page-locked host buffers for the data boundary: uploads/downloads from these run at
 * PCIe speed (the N-API shim backs Float32Array results with them). */
int olap_host_alloc(size_t bytes, void** out);
int olap_host_free(void* p);

/* ---- store life cycle: `new InMemoryStore(size, type, defaultValue)` in-memory.js:48-64 */
/* with_status: bit 0 = allocate the status plane; bit 1 (OLAP_CREATE_UNINITIALISED) = do not
 * fill the planes with the default — only for a store whose every cell is about to be
 * overwritten (receive buffers of the multi-GPU exchange). */
#define OLAP_CREATE_UNINITIALISED 2
/* bit 2 (OLAP_CREATE_SHAREABLE): the store lives in memory that the other processes of the box can
 * map (cudaMalloc + CUDA IPC instead of the stream-ordered pool): the local shard of a sharded
 * cube.  Results of transforms of a shareable store are shareable too. */
#define OLAP_CREATE_SHAREABLE 4
int olap_store_create(int64_t size, int type, int default_kind, int with_status, olap_store** out);
/* n stores of equal size (a cube's stored measures), carved from one allocation while they are
 * small (< 32 MiB each) or share a status plane; larger stores own their allocation, so that
 * destroying some of them frees their memory.
 * shared_status != 0: one status plane shared by all n stores. */
int olap_store_create_batch(int n, int64_t size, const int* types, const int* default_kinds,
                            int with_status, int shared_status, olap_store** out);
int olap_store_destroy(olap_store* s);
/* `.clone()` in-memory.js:66-73 */
int olap_store_clone(const olap_store* s, olap_store** out);

/* ---- peer memory (sharded cubes, SURVEY.md §8e: "each rank pulls/pushes its slice through
 * peer-mapped pointers") -------------------------------------------------------------------
 * olap_peer_alloc: device memory that another process of the box can map; `handle64` receives
 * the 64-byte CUDA IPC handle to send to the peers.  olap_peer_open maps a peer's buffer.
 * olap_store_wrap: a store over memory the library does not own (destroy leaves it alone). */
int olap_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int olap_peer_open(const unsigned char* handle64, void** ptr);
int olap_peer_close(void* ptr);
int olap_peer_free(void* ptr);
int olap_store_wrap(void* values, void* status, int64_t size, int type, int default_kind, olap_store** out);
/* drillUp (in-memory.js:265-334) of the OUTERMOST axis, [c_rows, inner] -> [p_rows, inner], where
 * output row r of store k is written to row_values[k * p_rows + r] (and its status bytes to
 * row_status[k * p_rows + r]; NULL when the stores carry no status plane) instead of a new
 * store: with peer pointers, the partial rollup of a sharded dimension lands directly in the
 * owning rank's receive buffer — rollup and exchange in ONE kernel over NVLink. */
int olap_drill_up_rows(olap_store* const* src, int n, const int* methods, int64_t c_rows, int64_t p_rows,
                       int64_t inner, const int32_t* row_map, float* const* row_values,
                       uint8_t* const* row_status);
/* Pull model of the same rollup (the default on GPUs).  olap_store_ipc_export: the 64-byte CUDA IPC
 * handle of the block a SHAREABLE store lives in, and the byte offsets of its values / status plane
 * (-1: none) inside that block, to be sent to the peers.  olap_peer_map: map a peer's block (cached
 * by handle; a block recycled by its owner keeps its handle).  olap_peer_unmap_all closes them.
 * olap_drill_up_pull: drillUp (in-memory.js:265-334) of the sharded row axis where the rank that
 * OWNS output rows reads their child rows out of the ranks that hold them: output row j (of
 * out_rows, `inner` cells each) aggregates child rows row_start[j] .. row_start[j+1]-1 of the child
 * tables, in that order (ascending global row = the reference's iteration order); child c is row
 * child_row[c] of rank child_rank[c], whose store k starts at base_values[k * n_ranks + rank] (an
 * address valid in THIS process: local, or peer-mapped) and holds rank_rows[rank] rows.  `like`
 * gives type / default / status layout of the n results.  One kernel; cells cross NVLink once;
 * bit-equal to the unsharded olap_drill_up for every method.  derive_status != 0: the status planes of
 * ALL source stores on ALL ranks are derived (olap_store_status_derived): they are not read (base_status
 * may be NULL), the children's status bytes are recomputed from their values — 4 instead of 5 bytes per
 * cell over NVLink. */
int olap_store_ipc_export(const olap_store* s, unsigned char* handle64, int64_t* values_offset, int64_t* status_offset);
int olap_peer_map(const unsigned char* handle64, void** ptr);
int olap_peer_unmap_all(void);
int olap_drill_up_pull(olap_store* const* like, int n, const int* methods, int64_t out_rows, int64_t inner,
                       const int32_t* row_start, const int32_t* child_rank, const int64_t* child_row, int n_ranks,
                       const int64_t* rank_rows, const void* const* base_values, const void* const* base_status,
                       int derive_status, olap_store** out);
/* dst's status plane := src's (same size; a no-op when either store has none).  Finishes the
 * `average` of a sharded rollup: the quotient sum / count keeps the merged flags of the sums. */
int olap_store_copy_status(olap_store* dst, const olap_store* src);
int64_t olap_store_size(const olap_store* s);        /* `.size` in-memory.js:18-20 */
int64_t olap_store_byte_length(const olap_store* s); /* `.byteLength` in-memory.js:8-16 */
int olap_store_type(const olap_store* s);
int olap_store_default_kind(const olap_store* s);
int olap_store_has_status(const olap_store* s);
/* Raw device pointers (for NCCL / torch interop on the host side).  The _ptr forms give MUTABLE access and
 * make the library forget that the status plane follows from the values (see olap_store_status_derived);
 * the _cptr forms are for reading only.  olap_store_canonicalise re-derives the status plane from the
 * values (and canonicalises them: -0 -> +0 under a zero default, any NaN -> the canonical NaN) after the
 * planes were written through raw pointers. */
void* olap_store_values_ptr(olap_store* s);
void* olap_store_status_ptr(olap_store* s);
const void* olap_store_values_cptr(const olap_store* s);
const void* olap_store_status_cptr(const olap_store* s);
int olap_store_canonicalise(olap_store* s);
/* 1 when every status byte of the store equals  set ? OLAP_STATUS_SET : OLAP_STATUS_UNSET  by construction
 * (after create / upload / fill / sparse import / eval, and through dice, reorder, clone; not after
 * drillUp, drillDown, load from a store that is not, for planes shared by several stores, wrapped memory
 * or once a mutable raw pointer was handed out).  drillUp of such a store never reads its status plane. */
int olap_store_status_derived(const olap_store* s);

/* ---- data boundary -------------------------------------------------------- */
/* `set data` in-memory.js:39-46.  n != size fails with
 * "value length is invalid: <size> !== <n>".  Values equal to the default are unset.
 * Host buffers of every call of this section are borrowed for the call.  They may be pinned
 * (olap_host_alloc: one copy at PCIe speed) or plain pageable memory (a typed array of the Node
 * addon): transfers of 8 MiB and more then travel in chunks through the library's ring of pinned
 * buffers, the host-side copies on worker threads (csrc/host_pipe.cuh). */
int olap_store_upload_f32(olap_store* s, const float* host, int64_t n);
int olap_store_upload_f64(olap_store* s, const double* host, int64_t n);
/* `get data` in-memory.js:30-37 (unset cells read as the default) */
int olap_store_download_f32(const olap_store* s, float* host, int64_t n);
int olap_store_download_f64(const olap_store* s, double* host, int64_t n);
/* `getValue` / `setValue` in-memory.js:118-133 */
int olap_store_get_value(const olap_store* s, int64_t index, double* out);
int olap_store_set_value(olap_store* s, int64_t index, double value);
/* batched setValue: hydrateFromSparseNestedObject (cube.js:472-491) */
int olap_store_set_values(olap_store* s, const int64_t* indexes, const double* values, int64_t n);
/* `fill` in-memory.js:135-137 */
int olap_store_fill(olap_store* s, double value);
/* `get total` in-memory.js:22-28 (double sum of the set cells) */
int olap_store_total(const olap_store* s, double* out);
/* set-ness of every cell, one byte each (1 = key in `_dataMap`) — cube.js:368-371 */
int olap_store_presence(const olap_store* s, uint8_t* host, int64_t n);
int olap_store_count_present(const olap_store* s, int64_t* out);
/* status plane (README.md:698-721); stores without a plane derive SET/UNSET from presence */
int olap_store_status(const olap_store* s, uint8_t* host, int64_t n);
/* `_dataMap` / `serialize()` as COO, keys ascending (in-memory.js:75-101).
 * capacity < count fails; *count always receives the number of set cells. */
int olap_store_export_sparse(const olap_store* s, int64_t capacity, int64_t* keys, float* values,
                             int64_t* count);
/* `deserialize()` in-memory.js:103-116: unset everything, then set the given cells */
int olap_store_import_sparse(olap_store* s, const int64_t* keys, const float* values, int64_t count);

/* ---- transforms (each returns n NEW stores in out[0..n)) -------------------- */
/* `drillUp(oldDims, newDims, method)` in-memory.js:265-334, called per measure by
 * Cube.drillUp (cube.js:1012-1020).  maps[d][i] = new item index of old item i of
 * dimension d, length old_len[d] (in-memory.js:270-274).  methods[k] per store.
 * maps[d] may be NULL for a dimension that does not change (old_len == new_len) or that
 * rolls up to ONE item (new_len == 1): no table has to be built or checked for it. */
int olap_drill_up(olap_store* const* src, int n, const int* methods, int ndim, const int64_t* old_len,
                  const int64_t* new_len, const int32_t* const* maps, olap_store** out);
/* `drillDown(oldDims, newDims, method, distributions)` in-memory.js:336-430
 * (Cube.drillDown cube.js:978-986, Cube.addDimension cube.js:937-945).
 * maps[d][j] = OLD item index of NEW item j, length new_len[d] (in-memory.js:349-353).
 * dist[k] may be NULL; a NaN entry means "missing" and fails with
 * "distribution missing for index <i>" when a set parent needs it. */
int olap_drill_down(olap_store* const* src, int n, const int* methods, int ndim, const int64_t* old_len,
                    const int64_t* new_len, const int32_t* const* maps, const double* const* dist,
                    const int64_t* dist_len, olap_store** out);
/* `dice(oldDims, newDims)` in-memory.js:213-263 (Cube.dice/diceRange/diceByDimensionItems).
 * keep[d][j] = old item index of new item j, length new_len[d]; any order, several
 * dimensions at once. */
int olap_dice(olap_store* const* src, int n, int ndim, const int64_t* old_len, const int64_t* new_len,
              const int32_t* const* keep, olap_store** out);
/* `reorder(oldDims, newDims)` in-memory.js:178-211: new axis i is old axis new_to_old[i]. */
int olap_reorder(olap_store* const* src, int n, int ndim, const int64_t* old_len, const int32_t* new_to_old,
                 olap_store** out);
/* `load(otherStore, myDims, hisDims)` in-memory.js:139-176: dst[mine(his)] = src[his] for every
 * cell of src, defaults included.  his_to_mine[d][j] = my item index of his item j, or -1 when
 * I do not have the item (the cell is dropped). */
int olap_load(olap_store* dst, const olap_store* src, int ndim, const int64_t* my_len, const int64_t* his_len,
              const int32_t* const* his_to_mine);

/* ---- region queries (Cube.getTotalForDimensionItems / getDistribution / copyMeasureData, cube.js,
 * which loop over the cartesian product of the filter's items with getSingleData / setSingleData).
 * The region of a store of len[0] x ... x len[ndim-1] cells is keep[0] x ... x keep[ndim-1]:
 * keep[d] = item indices of axis d (keep_len[d] of them), any order, repeats counted; keep[d] == NULL
 * (or keep == NULL) = the whole axis in order.  One kernel (region/sum, region/copy); olap_last_op_ms()
 * gives its time.  An empty region launches nothing. */
/* getTotalForDimensionItems: double sum of the raw cells (unset = default) of the region
 * keep[0] x ... x keep[ndim-1]; keep[d] = item indices of axis d, any order, repeats counted, NULL = whole axis.
 * NaN cells (a NaN default's unset cells included) make the sum NaN.  Summation order is fixed for a
 * given region: repeated calls give the same bits. */
int olap_region_sum(const olap_store* s, int ndim, const int64_t* len, const int64_t* keep_len,
                    const int32_t* const* keep, double* out);
/* copyMeasureData: dst.setValue(i, src.getValue(i)) for every cell i of the region (dst, src same size):
 * the source's raw value, canonicalised for dst's default, status byte SET / UNSET by dst's presence rule.
 * dst may be src.  Cells outside the region are not touched. */
int olap_region_copy(olap_store* dst, const olap_store* src, int ndim, const int64_t* len,
                     const int64_t* keep_len, const int32_t* const* keep);

/* ---- computed measures: Cube.getData(computedId) cube.js:331-363 --------------- */
/* `program` is the formula in postfix text, space separated:
 *   v<k>  cell of input store k      t<k>  totals[k] (an `x__total` variable)
 *   #<number>                        + - * / % ^ || neg  ?:
 *   call:<name>:<argc>               (abs sqrt min max isNaN ... — src/parser.js:3-26)
 * It is lowered to ONE fused elementwise sm_100a kernel (NVRTC) evaluating in double.
 * Exactly one of out_host_f64 / out_store is used: a host array of `size` doubles, or a
 * new float32 store with the given type/default (copyToStoredMeasure, cube.js:205-215). */
int olap_eval(const char* program, olap_store* const* inputs, int n_inputs, const double* totals, int n_totals,
              double* out_host_f64, int out_type, int out_default_kind, olap_store** out_store);

/* ---- computed measures over a region (Cube.getTotalForDimensionItems / getDistribution / copyMeasureData
 * of a computed measure).  `program` is a formula as for olap_eval, without totals (t<k>); inputs[k] is the
 * store of v<k>.  The region is that of olap_region_sum.  The formula is evaluated only at the region's cells,
 * in double, by the same function olap_eval uses (so a cell gets the bits getData returns for it), in ONE
 * NVRTC kernel that walks the region like region_kernel.  An empty region launches nothing. */
/* Sum over the region's cells of the formula's value, repeats counted (region/eval-sum, one launch).
 * NaN and +-inf propagate as in a double sum; summation order is fixed for a given region: repeated calls
 * give the same bits. */
int olap_region_eval_sum(const char* program, olap_store* const* inputs, int n_inputs, int ndim, const int64_t* len,
                         const int64_t* keep_len, const int32_t* const* keep, double* out);
/* dst.setValue(i, formula(i)) for every cell i of the region (region/eval-copy): the value rounded to
 * Float32, canonicalised for dst's default, status byte SET / UNSET.  dst may be one of the inputs: every
 * value is computed before its cell is written (each item list is de-duplicated first; a repeat would write
 * the same value again).  Cells outside the region are not touched.  An int32 / uint32 target refuses the
 * whole call, before anything is written, when a value does not survive its Float32 cell (as
 * olap_store_set_values does), naming the first such cell in product order: a check launch, then the write. */
int olap_region_eval_copy(olap_store* dst, const char* program, olap_store* const* inputs, int n_inputs, int ndim,
                          const int64_t* len, const int64_t* keep_len, const int32_t* const* keep);

/* ---- the status accessors of a computed measure (Cube.getStatus / getStatusMap, cube.js:368-389) ---- */
/* getStatus: host[i] = OR over the inputs of their status byte of cell i: the plane's byte, or SET / UNSET
 * from the values for an input without a plane (what olap_store_status reports for it).  n_cells = the
 * stores' size.  One launch (status/merge), then the download. */
int olap_status_merge(olap_store* const* inputs, int n, uint8_t* host, int64_t n_cells);
/* getStatusMap: the union of the stores' set cells (by value, as olap_store_export_sparse), keys grouped by
 * the first store in which the cell is set and ascending within a group (the insertion order of cube.js's
 * Map).  values[j] folds the key's set values over the stores in order: the first one; then, for each later
 * one, ToInt32(prev) | ToInt32(v) when prev is truthy (not NaN, not 0; is_int[j] = 1), else v itself
 * (is_int[j] = 0).  Two calls, as olap_store_export_sparse: keys / values / is_int all NULL -> *count only; then
 * all three arrays, of `capacity` >= *count entries (status/map).  A mix of NULL and non-NULL arrays is an error. */
int olap_status_map_export(olap_store* const* stores, int n, int64_t capacity, int64_t* keys, double* values,
                           uint8_t* is_int, int64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* OLAP_GPU_H */
