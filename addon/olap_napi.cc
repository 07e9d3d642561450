// N-API shim: the JavaScript binding of include/olap_gpu.h.
//
// UNEXECUTED in this repository: the build image has no Node.js and no node_api.h
// (SURVEY.md F4).  It is shipped so a maintainer with Node 20 can `node-gyp rebuild` it
// (addon/binding.gyp) next to a built libolapgpu.so.  By design it holds no logic: it
// unpacks arguments, extracts TypedArray pointers, calls the C ABI and turns an error
// code into a thrown JS Error carrying olap_last_error() — the texts are the reference's
// own (`value length is invalid: a !== b`, `Unsupported aggregation method: x`, ...).
#include <node_api.h>

#include <vector>

#include "../include/olap_gpu.h"

#define NAPI_OK(call)                                                      \
    do {                                                                   \
        if ((call) != napi_ok) {                                           \
            napi_throw_error(env, nullptr, "N-API call failed: " #call);   \
            return nullptr;                                                \
        }                                                                  \
    } while (0)

static napi_value throw_last(napi_env env) {
    napi_throw_error(env, nullptr, olap_last_error());
    return nullptr;
}
#define OLAP_CALL(expr)                                \
    do {                                               \
        if ((expr) != OLAP_OK) return throw_last(env); \
    } while (0)

static void finalize_store(napi_env env, void* data, void*) {
    olap_store* s = static_cast<olap_store*>(data);
    int64_t freed = -(olap_store_size(s) * (olap_store_has_status(s) ? 5 : 4));
    int64_t adjusted;
    napi_adjust_external_memory(env, freed, &adjusted);  // let V8's GC see HBM pressure
    olap_store_destroy(s);
}

static napi_value wrap_store(napi_env env, olap_store* s) {
    napi_value ext;
    NAPI_OK(napi_create_external(env, s, finalize_store, nullptr, &ext));
    int64_t adjusted;
    napi_adjust_external_memory(env, olap_store_size(s) * (olap_store_has_status(s) ? 5 : 4), &adjusted);
    return ext;
}

static olap_store* unwrap(napi_env env, napi_value v) {
    void* p = nullptr;
    napi_get_value_external(env, v, &p);
    return static_cast<olap_store*>(p);
}

struct Args {
    napi_value v[10];
    size_t n = 10;
};
#define GET_ARGS() \
    Args a;        \
    NAPI_OK(napi_get_cb_info(env, info, &a.n, a.v, nullptr, nullptr))

static std::vector<olap_store*> store_list(napi_env env, napi_value arr) {
    uint32_t n = 0;
    napi_get_array_length(env, arr, &n);
    std::vector<olap_store*> out(n);
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, arr, i, &e);
        out[i] = unwrap(env, e);
    }
    return out;
}

static std::vector<int64_t> int64_list(napi_env env, napi_value arr) {
    uint32_t n = 0;
    napi_get_array_length(env, arr, &n);
    std::vector<int64_t> out(n);
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, arr, i, &e);
        napi_get_value_int64(env, e, &out[i]);
    }
    return out;
}

// Array of Int32Array -> const int32_t* const*
static std::vector<const int32_t*> map_list(napi_env env, napi_value arr) {
    uint32_t n = 0;
    napi_get_array_length(env, arr, &n);
    std::vector<const int32_t*> out(n);
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, arr, i, &e);
        napi_typedarray_type t;
        size_t len;
        void* data;
        napi_get_typedarray_info(env, e, &t, &len, &data, nullptr, nullptr);
        out[i] = static_cast<const int32_t*>(data);
    }
    return out;
}

static napi_value store_array_out(napi_env env, std::vector<olap_store*>& out) {
    napi_value arr;
    NAPI_OK(napi_create_array_with_length(env, out.size(), &arr));
    for (size_t i = 0; i < out.size(); ++i) napi_set_element(env, arr, i, wrap_store(env, out[i]));
    return arr;
}

// create(size, type, defaultKind, withStatus) -> external
static napi_value Create(napi_env env, napi_callback_info info) {
    GET_ARGS();
    int64_t size;
    int32_t type, kind;
    bool status;
    napi_get_value_int64(env, a.v[0], &size);
    napi_get_value_int32(env, a.v[1], &type);
    napi_get_value_int32(env, a.v[2], &kind);
    napi_get_value_bool(env, a.v[3], &status);
    olap_store* s = nullptr;
    OLAP_CALL(olap_store_create(size, type, kind, status, &s));
    return wrap_store(env, s);
}

// upload(store, Float32Array | Float64Array)
static napi_value Upload(napi_env env, napi_callback_info info) {
    GET_ARGS();
    napi_typedarray_type t;
    size_t len;
    void* data;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &data, nullptr, nullptr));
    if (t == napi_float32_array) {
        OLAP_CALL(olap_store_upload_f32(unwrap(env, a.v[0]), static_cast<float*>(data), (int64_t)len));
    } else {
        OLAP_CALL(olap_store_upload_f64(unwrap(env, a.v[0]), static_cast<double*>(data), (int64_t)len));
    }
    return nullptr;
}

// download(store, Float32Array | Float64Array)
static napi_value Download(napi_env env, napi_callback_info info) {
    GET_ARGS();
    napi_typedarray_type t;
    size_t len;
    void* data;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &data, nullptr, nullptr));
    if (t == napi_float32_array) {
        OLAP_CALL(olap_store_download_f32(unwrap(env, a.v[0]), static_cast<float*>(data), (int64_t)len));
    } else {
        OLAP_CALL(olap_store_download_f64(unwrap(env, a.v[0]), static_cast<double*>(data), (int64_t)len));
    }
    return nullptr;
}

// drillUp(stores[], methods Int32Array, oldLen[], newLen[], maps Int32Array[]) -> stores[]
static napi_value DrillUp(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto src = store_list(env, a.v[0]);
    napi_typedarray_type t;
    size_t len;
    void* mdata;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &mdata, nullptr, nullptr));
    auto old_len = int64_list(env, a.v[2]), new_len = int64_list(env, a.v[3]);
    auto maps = map_list(env, a.v[4]);
    std::vector<olap_store*> out(src.size());
    OLAP_CALL(olap_drill_up(src.data(), (int)src.size(), static_cast<const int*>(mdata), (int)old_len.size(),
                            old_len.data(), new_len.data(), maps.data(), out.data()));
    return store_array_out(env, out);
}

// dice(stores[], oldLen[], newLen[], keep Int32Array[]) -> stores[]
static napi_value Dice(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto src = store_list(env, a.v[0]);
    auto old_len = int64_list(env, a.v[1]), new_len = int64_list(env, a.v[2]);
    auto keep = map_list(env, a.v[3]);
    std::vector<olap_store*> out(src.size());
    OLAP_CALL(olap_dice(src.data(), (int)src.size(), (int)old_len.size(), old_len.data(), new_len.data(), keep.data(), out.data()));
    return store_array_out(env, out);
}

// reorder(stores[], oldLen[], newToOld Int32Array) -> stores[]
static napi_value Reorder(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto src = store_list(env, a.v[0]);
    auto old_len = int64_list(env, a.v[1]);
    napi_typedarray_type t;
    size_t len;
    void* perm;
    NAPI_OK(napi_get_typedarray_info(env, a.v[2], &t, &len, &perm, nullptr, nullptr));
    std::vector<olap_store*> out(src.size());
    OLAP_CALL(olap_reorder(src.data(), (int)src.size(), (int)old_len.size(), old_len.data(), static_cast<const int32_t*>(perm), out.data()));
    return store_array_out(env, out);
}

// total(store) -> number
static napi_value Total(napi_env env, napi_callback_info info) {
    GET_ARGS();
    double v;
    OLAP_CALL(olap_store_total(unwrap(env, a.v[0]), &v));
    napi_value out;
    NAPI_OK(napi_create_double(env, v, &out));
    return out;
}

// Float64Array[] (entries may be null) -> const double* const*, with the lengths
static void f64_list(napi_env env, napi_value arr, std::vector<const double*>& ptrs, std::vector<int64_t>& lens) {
    uint32_t n = 0;
    napi_get_array_length(env, arr, &n);
    ptrs.assign(n, nullptr);
    lens.assign(n, 0);
    for (uint32_t i = 0; i < n; ++i) {
        napi_value e;
        napi_get_element(env, arr, i, &e);
        bool typed = false;
        napi_is_typedarray(env, e, &typed);
        if (!typed) continue;  // null: no distribution for this store
        napi_typedarray_type t;
        size_t len;
        void* data;
        napi_get_typedarray_info(env, e, &t, &len, &data, nullptr, nullptr);
        ptrs[i] = static_cast<const double*>(data);
        lens[i] = (int64_t)len;
    }
}

// drillDown(stores[], methods Int32Array, oldLen[], newLen[], maps Int32Array[], dist (Float64Array|null)[]) -> stores[]
static napi_value DrillDown(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto src = store_list(env, a.v[0]);
    napi_typedarray_type t;
    size_t len;
    void* mdata;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &mdata, nullptr, nullptr));
    auto old_len = int64_list(env, a.v[2]), new_len = int64_list(env, a.v[3]);
    auto maps = map_list(env, a.v[4]);
    std::vector<const double*> dist;
    std::vector<int64_t> dist_len;
    f64_list(env, a.v[5], dist, dist_len);
    dist.resize(src.size(), nullptr);
    dist_len.resize(src.size(), 0);
    std::vector<olap_store*> out(src.size());
    OLAP_CALL(olap_drill_down(src.data(), (int)src.size(), static_cast<const int*>(mdata), (int)old_len.size(),
                              old_len.data(), new_len.data(), maps.data(), dist.data(), dist_len.data(), out.data()));
    return store_array_out(env, out);
}

// load(dst, src, myLen[], hisLen[], hisToMine Int32Array[])
static napi_value Load(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto my_len = int64_list(env, a.v[2]), his_len = int64_list(env, a.v[3]);
    auto maps = map_list(env, a.v[4]);
    OLAP_CALL(olap_load(unwrap(env, a.v[0]), unwrap(env, a.v[1]), (int)my_len.size(), my_len.data(), his_len.data(), maps.data()));
    return nullptr;
}

// (Int32Array | null)[] -> item lists and their lengths; null = the whole axis
static void region_lists(napi_env env, napi_value arr, const std::vector<int64_t>& lens,
                         std::vector<const int32_t*>& ptrs, std::vector<int64_t>& keep_len) {
    ptrs.assign(lens.size(), nullptr);
    keep_len = lens;
    for (uint32_t i = 0; i < (uint32_t)lens.size(); ++i) {
        napi_value e;
        napi_get_element(env, arr, i, &e);
        bool typed = false;
        napi_is_typedarray(env, e, &typed);
        if (!typed) continue;
        napi_typedarray_type t;
        size_t len;
        void* data;
        napi_get_typedarray_info(env, e, &t, &len, &data, nullptr, nullptr);
        ptrs[i] = static_cast<const int32_t*>(data);
        keep_len[i] = (int64_t)len;
    }
}

// regionSum(store, len[], keep (Int32Array|null)[]) -> number   (cube.js getTotalForDimensionItems)
static napi_value RegionSum(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto len = int64_list(env, a.v[1]);
    std::vector<const int32_t*> keep;
    std::vector<int64_t> keep_len;
    region_lists(env, a.v[2], len, keep, keep_len);
    double v;
    OLAP_CALL(olap_region_sum(unwrap(env, a.v[0]), (int)len.size(), len.data(), keep_len.data(), keep.data(), &v));
    napi_value out;
    NAPI_OK(napi_create_double(env, v, &out));
    return out;
}

// regionCopy(dst, src, len[], keep (Int32Array|null)[])   (cube.js copyMeasureData)
static napi_value RegionCopy(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto len = int64_list(env, a.v[2]);
    std::vector<const int32_t*> keep;
    std::vector<int64_t> keep_len;
    region_lists(env, a.v[3], len, keep, keep_len);
    OLAP_CALL(olap_region_copy(unwrap(env, a.v[0]), unwrap(env, a.v[1]), (int)len.size(), len.data(), keep_len.data(), keep.data()));
    return nullptr;
}

// clone(store) -> external
static napi_value Clone(napi_env env, napi_callback_info info) {
    GET_ARGS();
    olap_store* s = nullptr;
    OLAP_CALL(olap_store_clone(unwrap(env, a.v[0]), &s));
    return wrap_store(env, s);
}

// getValue(store, index) -> number
static napi_value GetValue(napi_env env, napi_callback_info info) {
    GET_ARGS();
    int64_t index;
    napi_get_value_int64(env, a.v[1], &index);
    double v;
    OLAP_CALL(olap_store_get_value(unwrap(env, a.v[0]), index, &v));
    napi_value out;
    NAPI_OK(napi_create_double(env, v, &out));
    return out;
}

// setValue(store, index, value)
static napi_value SetValue(napi_env env, napi_callback_info info) {
    GET_ARGS();
    int64_t index;
    double v;
    napi_get_value_int64(env, a.v[1], &index);
    napi_get_value_double(env, a.v[2], &v);
    OLAP_CALL(olap_store_set_value(unwrap(env, a.v[0]), index, v));
    return nullptr;
}

// setValues(store, indexes BigInt64Array, values Float64Array): batched point updates
static napi_value SetValues(napi_env env, napi_callback_info info) {
    GET_ARGS();
    napi_typedarray_type t;
    size_t n, nv;
    void *idx, *val;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &n, &idx, nullptr, nullptr));
    NAPI_OK(napi_get_typedarray_info(env, a.v[2], &t, &nv, &val, nullptr, nullptr));
    OLAP_CALL(olap_store_set_values(unwrap(env, a.v[0]), static_cast<const int64_t*>(idx), static_cast<const double*>(val),
                                    (int64_t)(n < nv ? n : nv)));
    return nullptr;
}

// fill(store, value)
static napi_value Fill(napi_env env, napi_callback_info info) {
    GET_ARGS();
    double v;
    napi_get_value_double(env, a.v[1], &v);
    OLAP_CALL(olap_store_fill(unwrap(env, a.v[0]), v));
    return nullptr;
}

// presence(store, Uint8Array) / status(store, Uint8Array)
static napi_value Presence(napi_env env, napi_callback_info info) {
    GET_ARGS();
    napi_typedarray_type t;
    size_t len;
    void* data;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &data, nullptr, nullptr));
    OLAP_CALL(olap_store_presence(unwrap(env, a.v[0]), static_cast<uint8_t*>(data), (int64_t)len));
    return nullptr;
}
static napi_value Status(napi_env env, napi_callback_info info) {
    GET_ARGS();
    napi_typedarray_type t;
    size_t len;
    void* data;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &data, nullptr, nullptr));
    OLAP_CALL(olap_store_status(unwrap(env, a.v[0]), static_cast<uint8_t*>(data), (int64_t)len));
    return nullptr;
}

// exportSparse(store) -> { keys: BigInt64Array, values: Float32Array }   (keys ascending)
static napi_value ExportSparse(napi_env env, napi_callback_info info) {
    GET_ARGS();
    olap_store* s = unwrap(env, a.v[0]);
    int64_t count = 0;
    OLAP_CALL(olap_store_count_present(s, &count));
    napi_value kbuf, vbuf, keys, values, out;
    void *kdata, *vdata;
    NAPI_OK(napi_create_arraybuffer(env, (size_t)count * 8, &kdata, &kbuf));
    NAPI_OK(napi_create_arraybuffer(env, (size_t)count * 4, &vdata, &vbuf));
    OLAP_CALL(olap_store_export_sparse(s, count, static_cast<int64_t*>(kdata), static_cast<float*>(vdata), &count));
    NAPI_OK(napi_create_typedarray(env, napi_bigint64_array, (size_t)count, kbuf, 0, &keys));
    NAPI_OK(napi_create_typedarray(env, napi_float32_array, (size_t)count, vbuf, 0, &values));
    NAPI_OK(napi_create_object(env, &out));
    NAPI_OK(napi_set_named_property(env, out, "keys", keys));
    NAPI_OK(napi_set_named_property(env, out, "values", values));
    return out;
}

// importSparse(store, keys BigInt64Array, values Float32Array)
static napi_value ImportSparse(napi_env env, napi_callback_info info) {
    GET_ARGS();
    napi_typedarray_type t;
    size_t n, nv;
    void *keys, *values;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &n, &keys, nullptr, nullptr));
    NAPI_OK(napi_get_typedarray_info(env, a.v[2], &t, &nv, &values, nullptr, nullptr));
    OLAP_CALL(olap_store_import_sparse(unwrap(env, a.v[0]), static_cast<const int64_t*>(keys), static_cast<const float*>(values),
                                       (int64_t)(n < nv ? n : nv)));
    return nullptr;
}

// evaluate(program string, stores[], totals Float64Array, out Float64Array)  — Cube.getData(computedId)
static napi_value Evaluate(napi_env env, napi_callback_info info) {
    GET_ARGS();
    size_t plen = 0;
    NAPI_OK(napi_get_value_string_utf8(env, a.v[0], nullptr, 0, &plen));
    std::vector<char> program(plen + 1);
    NAPI_OK(napi_get_value_string_utf8(env, a.v[0], program.data(), program.size(), &plen));
    auto src = store_list(env, a.v[1]);
    napi_typedarray_type t;
    size_t nt, n;
    void *totals, *out;
    NAPI_OK(napi_get_typedarray_info(env, a.v[2], &t, &nt, &totals, nullptr, nullptr));
    NAPI_OK(napi_get_typedarray_info(env, a.v[3], &t, &n, &out, nullptr, nullptr));
    OLAP_CALL(olap_eval(program.data(), src.data(), (int)src.size(), static_cast<const double*>(totals), (int)nt,
                        static_cast<double*>(out), 0, 0, nullptr));
    return nullptr;
}

// evaluateToStore(program string, stores[], totals Float64Array, type, defaultKind) -> external  — copyToStoredMeasure
static napi_value EvaluateToStore(napi_env env, napi_callback_info info) {
    GET_ARGS();
    size_t plen = 0;
    NAPI_OK(napi_get_value_string_utf8(env, a.v[0], nullptr, 0, &plen));
    std::vector<char> program(plen + 1);
    NAPI_OK(napi_get_value_string_utf8(env, a.v[0], program.data(), program.size(), &plen));
    auto src = store_list(env, a.v[1]);
    napi_typedarray_type t;
    size_t nt;
    void* totals;
    NAPI_OK(napi_get_typedarray_info(env, a.v[2], &t, &nt, &totals, nullptr, nullptr));
    int32_t type, kind;
    napi_get_value_int32(env, a.v[3], &type);
    napi_get_value_int32(env, a.v[4], &kind);
    olap_store* s = nullptr;
    OLAP_CALL(olap_eval(program.data(), src.data(), (int)src.size(), static_cast<const double*>(totals), (int)nt, nullptr, type,
                        kind, &s));
    return wrap_store(env, s);
}

// program string argument -> NUL-terminated buffer
static napi_status utf8_arg(napi_env env, napi_value v, std::vector<char>& out) {
    size_t plen = 0;
    const napi_status st = napi_get_value_string_utf8(env, v, nullptr, 0, &plen);
    if (st != napi_ok) return st;
    out.assign(plen + 1, '\0');
    return napi_get_value_string_utf8(env, v, out.data(), out.size(), &plen);
}

// regionEvalSum(program string, stores[], len[], keep (Int32Array|null)[]) -> number
//   (getTotalForDimensionItems of a computed measure)
static napi_value RegionEvalSum(napi_env env, napi_callback_info info) {
    GET_ARGS();
    std::vector<char> program;
    NAPI_OK(utf8_arg(env, a.v[0], program));
    auto src = store_list(env, a.v[1]);
    auto len = int64_list(env, a.v[2]);
    std::vector<const int32_t*> keep;
    std::vector<int64_t> keep_len;
    region_lists(env, a.v[3], len, keep, keep_len);
    double v;
    OLAP_CALL(olap_region_eval_sum(program.data(), src.data(), (int)src.size(), (int)len.size(), len.data(), keep_len.data(),
                                   keep.data(), &v));
    napi_value out;
    NAPI_OK(napi_create_double(env, v, &out));
    return out;
}

// regionEvalCopy(dst, program string, stores[], len[], keep (Int32Array|null)[])   (copyMeasureData, computed source)
static napi_value RegionEvalCopy(napi_env env, napi_callback_info info) {
    GET_ARGS();
    std::vector<char> program;
    NAPI_OK(utf8_arg(env, a.v[1], program));
    auto src = store_list(env, a.v[2]);
    auto len = int64_list(env, a.v[3]);
    std::vector<const int32_t*> keep;
    std::vector<int64_t> keep_len;
    region_lists(env, a.v[4], len, keep, keep_len);
    OLAP_CALL(olap_region_eval_copy(unwrap(env, a.v[0]), program.data(), src.data(), (int)src.size(), (int)len.size(), len.data(),
                                    keep_len.data(), keep.data()));
    return nullptr;
}

// statusMerge(stores[], Uint8Array)   (getStatus of a computed measure)
static napi_value StatusMerge(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto src = store_list(env, a.v[0]);
    napi_typedarray_type t;
    size_t len;
    void* data;
    NAPI_OK(napi_get_typedarray_info(env, a.v[1], &t, &len, &data, nullptr, nullptr));
    OLAP_CALL(olap_status_merge(src.data(), (int)src.size(), static_cast<uint8_t*>(data), (int64_t)len));
    return nullptr;
}

// statusMap(stores[]) -> { keys: BigInt64Array, values: Float64Array, isInt: Uint8Array }   (getStatusMap of a computed measure)
static napi_value StatusMap(napi_env env, napi_callback_info info) {
    GET_ARGS();
    auto src = store_list(env, a.v[0]);
    int64_t count = 0;
    OLAP_CALL(olap_status_map_export(src.data(), (int)src.size(), 0, nullptr, nullptr, nullptr, &count));
    napi_value kbuf, vbuf, ibuf, keys, values, is_int, out;
    void *kdata, *vdata, *idata;
    NAPI_OK(napi_create_arraybuffer(env, (size_t)count * 8, &kdata, &kbuf));
    NAPI_OK(napi_create_arraybuffer(env, (size_t)count * 8, &vdata, &vbuf));
    NAPI_OK(napi_create_arraybuffer(env, (size_t)count, &idata, &ibuf));
    OLAP_CALL(olap_status_map_export(src.data(), (int)src.size(), count, static_cast<int64_t*>(kdata), static_cast<double*>(vdata),
                                     static_cast<uint8_t*>(idata), &count));
    NAPI_OK(napi_create_typedarray(env, napi_bigint64_array, (size_t)count, kbuf, 0, &keys));
    NAPI_OK(napi_create_typedarray(env, napi_float64_array, (size_t)count, vbuf, 0, &values));
    NAPI_OK(napi_create_typedarray(env, napi_uint8_array, (size_t)count, ibuf, 0, &is_int));
    NAPI_OK(napi_create_object(env, &out));
    NAPI_OK(napi_set_named_property(env, out, "keys", keys));
    NAPI_OK(napi_set_named_property(env, out, "values", values));
    NAPI_OK(napi_set_named_property(env, out, "isInt", is_int));
    return out;
}

static napi_value Init(napi_env env, napi_value exports) {
    const napi_property_descriptor props[] = {
        {"create", nullptr, Create, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"upload", nullptr, Upload, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"download", nullptr, Download, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"drillUp", nullptr, DrillUp, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"dice", nullptr, Dice, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"reorder", nullptr, Reorder, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"total", nullptr, Total, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"drillDown", nullptr, DrillDown, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"load", nullptr, Load, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"regionSum", nullptr, RegionSum, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"regionCopy", nullptr, RegionCopy, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"clone", nullptr, Clone, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"getValue", nullptr, GetValue, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"setValue", nullptr, SetValue, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"setValues", nullptr, SetValues, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"fill", nullptr, Fill, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"presence", nullptr, Presence, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"status", nullptr, Status, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"exportSparse", nullptr, ExportSparse, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"importSparse", nullptr, ImportSparse, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"evaluate", nullptr, Evaluate, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"evaluateToStore", nullptr, EvaluateToStore, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"regionEvalSum", nullptr, RegionEvalSum, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"regionEvalCopy", nullptr, RegionEvalCopy, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"statusMerge", nullptr, StatusMerge, nullptr, nullptr, nullptr, napi_default, nullptr},
        {"statusMap", nullptr, StatusMap, nullptr, nullptr, nullptr, napi_default, nullptr},
    };
    napi_define_properties(env, exports, sizeof props / sizeof props[0], props);
    if (olap_init(0) != OLAP_OK) return throw_last(env);  // no CPU fallback: fail at require() time
    return exports;
}
NAPI_MODULE(olap_gpu, Init)
