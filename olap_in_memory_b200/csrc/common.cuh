// Shared declarations of the native store: context, handles, error plumbing,
// device helpers.  sm_100a only.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/olap_gpu.h"
#include "region_walk.cuh"  // FastDiv

namespace olap {

// ---------------------------------------------------------------- errors
extern thread_local std::string g_error;
int fail(int code, const char* fmt, ...);

#define OLAP_CUDA(expr)                                                                     \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return ::olap::fail(_e == cudaErrorMemoryAllocation ? OLAP_E_NOMEM : OLAP_E_CUDA, \
                                "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, \
                                __LINE__, cudaGetErrorString(_e));                          \
    } while (0)

#define OLAP_TRY(expr)          \
    do {                        \
        int _rc = (expr);       \
        if (_rc != OLAP_OK) return _rc; \
    } while (0)

// ---------------------------------------------------------------- context
struct Ctx {
    bool ready = false;
    int device = -1;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    bool async = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing_pending = false;
    double last_ms = 0.0;
    const char* last_path = "";
    // pinned staging for small per-query tables (index maps, CSR, descriptors): a ring of
    // slots so that the host can prepare several calls ahead of the device in async mode
    static constexpr int kPinSlots = 8;
    struct PinSlot {
        char* ptr = nullptr;
        size_t cap = 0;
        cudaEvent_t free_ev = nullptr;  // recorded after the copy out of this slot
        bool busy = false;
    } pin[kPinSlots];
    int pin_next = 0;
};
extern Ctx g;
extern std::atomic<int64_t> g_launches;

int ensure_ctx();
void mark_kernels_begin();       // records the op's start event before its first kernel
int finish_op();                       // sync unless async; surfaces launch errors
int dev_alloc(void** p, size_t bytes); // stream-ordered
int dev_free(void* p);

// One device allocation shared by the stores of one batched call.
struct Arena {
    void* base = nullptr;
    size_t bytes = 0;
    std::atomic<int> refs{0};
    // shareable: the block comes from cudaMalloc (CUDA IPC cannot export the stream-ordered pool), so
    // that the other ranks of a sharded cube can map it and read its cells over NVLink
    // (olap_store_ipc_export / olap_drill_up_pull).  Freed blocks are recycled by size.
    bool shareable = false;
};

}  // namespace olap

struct olap_store {
    int64_t size = 0;
    int type = OLAP_FLOAT32;
    int default_kind = OLAP_DEFAULT_ZERO;
    float* values = nullptr;
    uint8_t* status = nullptr;  // optional plane (may be shared with sibling stores)
    olap::Arena* arena = nullptr;
    // The status plane says nothing the values do not: every cell holds  set ? SET : UNSET.  True after
    // create / upload / fill / sparse import / eval and through dice, reorder and clone; false after
    // drillUp (OR-merged flags), drillDown (INTERPOLATED), for planes shared by several stores, wrapped
    // memory, and as soon as a raw plane pointer is handed out.  Kernels that load the values anyway
    // (drillUp) then never read the plane: 4 instead of 5 bytes per input cell.
    bool derived = false;
    bool shared_plane = false;
};

namespace olap {

// Allocate `n` stores of `size` cells in one arena.  Layout (contiguous):
//   values[0][size] ... values[n-1][size]  |  status planes (n, 1 or 0), each padded to 256 B.
int alloc_batch(int n, int64_t size, const int* types, const int* default_kinds, bool with_status,
                bool shared_status, olap_store** out, bool shareable = false);

// Small host->device table upload through pinned staging (async on the stream).
// Tables of one call are packed into a single device buffer.
struct TablePack {
    std::vector<char> host;
    void* dev = nullptr;
    size_t add(const void* data, size_t bytes, size_t align = 16);  // returns the offset (aligned; the device base is 256-byte aligned)
    int upload();
    int release();
    TablePack() = default;
    TablePack(const TablePack&) = delete;
    TablePack& operator=(const TablePack&) = delete;
    ~TablePack() { if (dev) dev_free(dev); }  // error returns between upload() and release() (stream-ordered free)
    template <typename T>
    T* ptr(size_t off) const { return reinterpret_cast<T*>(static_cast<char*>(dev) + off); }
};

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

#define CANON_NAN_BITS 0x7fc00000u

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ float canon_nan() { return __int_as_float(CANON_NAN_BITS); }
__device__ __forceinline__ float default_of(int nan_default) { return nan_default ? canon_nan() : 0.0f; }
// in-memory.js:122-133: a cell is set iff its value differs from the default
// (-0 === 0 in JS, so -0 is "default" under a zero default; NaN is set under it).
__device__ __forceinline__ bool present_f(float v, int nan_default) { return nan_default ? (v == v) : (v != 0.0f); }
__device__ __forceinline__ bool present_d(double v, int nan_default) { return nan_default ? (v == v) : (v != 0.0); }
// canonical cell content for a value about to be stored
__device__ __forceinline__ float canon_store(float v, int nan_default) {
    if (v != v) return canon_nan();  // NaN: the default under NaN, a set NaN under zero
    if (!nan_default && v == 0.0f) return 0.0f;  // -0 -> +0
    return v;
}

// 128-bit streaming accesses: inputs are read once, outputs written once.
__device__ __forceinline__ float4 ld_stream4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float ld_stream1(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ float2 ld_stream2(const float* p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ld_stream_u16(const void* p) {
    uint16_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(r) : "l"(p));
    return (uint32_t)r;
}
__device__ __forceinline__ uint32_t ld_stream_u32(const void* p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// JS Math.max / Math.min on floats: NaN-propagating, max(-0,+0) = +0, min(+0,-0) = -0
// (in-memory.js:285-286).
__device__ __forceinline__ float js_max(float a, float b) {
    float r = a > b ? a : b;
    if (a == b) r = __int_as_float(__float_as_int(a) & __float_as_int(b));
    if (a != a || b != b) r = canon_nan();
    return r;
}
__device__ __forceinline__ float js_min(float a, float b) {
    float r = a < b ? a : b;
    if (a == b) r = __int_as_float(__float_as_int(a) | __float_as_int(b));
    if (a != a || b != b) r = canon_nan();
    return r;
}

}  // namespace olap
