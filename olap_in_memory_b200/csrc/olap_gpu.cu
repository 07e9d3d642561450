// libolapgpu.so — C ABI (include/olap_gpu.h) over the sm_100a kernels.
// Host logic here: argument validation with the reference's error texts, lowering of
// the per-dimension int32 maps to CSR / offset tables, shape canonicalisation
// ([O, C, I] view, merging of untouched axes), launch configuration.
#include <math.h>
#include <stdarg.h>

#include <algorithm>
#include <array>
#include <map>
#include <numeric>
#include <unordered_set>

#include "common.cuh"
#include "jit_eval.cuh"
#include "kernels_drillup.cuh"
#include "kernels_gather.cuh"
#include "kernels_store.cuh"
#include "kernels_pair.cuh"
#include "kernels_pair_async.cuh"
#include "kernels_tile.cuh"
#include "kernels_long.cuh"
#include "kernels_lanes.cuh"
#include "kernels_pull.cuh"
#include "kernels_region.cuh"
#include "kernels_tma.cuh"
#include "host_pipe.cuh"

namespace olap {

thread_local std::string g_error;
Ctx g;
std::atomic<int64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
    char buf[2048];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define LAUNCHED() (++::olap::g_launches)
#define KERNELS_BEGIN() ::olap::mark_kernels_begin()

int ensure_ctx() {
    if (g.ready) {
        // the calling thread may not have the device current yet
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess || cur != g.device) OLAP_CUDA(cudaSetDevice(g.device));
        return OLAP_OK;
    }
    return olap_init(0);
}

// ev0 is recorded right before the FIRST kernel of an op (after the small table upload),
// ev1 after the last one: olap_last_op_ms() is kernel time, not host-side preparation.
static bool g_op_started = false;
static void begin_op() { g_op_started = false; }
void mark_kernels_begin() {
    if (!g_op_started && g.ev0) cudaEventRecord(g.ev0, g.stream);
    g_op_started = true;
}
static void end_op(const char* path) {
    mark_kernels_begin();  // an op without kernels still gets a (zero-length) bracket
    if (g.ev1) cudaEventRecord(g.ev1, g.stream);
    g.timing_pending = true;
    g.last_path = path;
}

int finish_op() {
    OLAP_CUDA(cudaGetLastError());
    if (!g.async) OLAP_CUDA(cudaStreamSynchronize(g.stream));
    return OLAP_OK;
}

int dev_alloc(void** p, size_t bytes) {
    *p = nullptr;
    if (bytes == 0) bytes = 256;
    cudaError_t e = cudaMallocAsync(p, bytes, g.stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? OLAP_E_NOMEM : OLAP_E_CUDA,
                    "device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    }
    return OLAP_OK;
}
int dev_free(void* p) {
    if (p) OLAP_CUDA(cudaFreeAsync(p, g.stream));
    return OLAP_OK;
}

static size_t pad256(size_t b) { return (b + 255) & ~(size_t)255; }

// OLAP_GUARD=1 (debug aid; compute-sanitizer is not available on every pool): every plane is
// followed by a 256-byte guard filled with 0xA5; destroying a store checks its guards and
// olap_guard_violations() reports how many bytes were overwritten.
static const bool g_guard = [] { const char* e = getenv("OLAP_GUARD"); return e && atoi(e) != 0; }();
static std::atomic<int64_t> g_guard_violations{0};
constexpr size_t kGuardBytes = 256;

// Shareable blocks (cudaMalloc, exportable through CUDA IPC) are recycled by exact size: a sharded
// cube re-creates result stores of the same sizes query after query, and a recycled block keeps its
// IPC handle, so the mappings the peers hold stay valid.  All library work runs on one stream, so
// handing a freed block to a later call is stream-ordered by construction.
static std::multimap<size_t, void*> g_share_free;
static bool g_share_all = false;  // olap_set_shareable(1): every new store of this process is shareable
// cudaMalloc carves small requests out of shared 2 MiB slabs, and an IPC handle names the slab:
// every exported block gets whole slabs of its own, so that handle <-> block is one to one
static size_t share_round(size_t bytes) { return std::max<size_t>(1, (bytes + (2u << 20) - 1) >> 21) << 21; }
static int share_alloc(void** p, size_t bytes) {
    bytes = share_round(bytes);
    auto it = g_share_free.find(bytes);
    if (it != g_share_free.end()) {
        *p = it->second;
        g_share_free.erase(it);
        return OLAP_OK;
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation) {  // give the cached blocks back and try again
        cudaGetLastError();
        for (auto& kv : g_share_free) cudaFree(kv.second);
        g_share_free.clear();
        e = cudaMalloc(p, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        *p = nullptr;
        return fail(e == cudaErrorMemoryAllocation ? OLAP_E_NOMEM : OLAP_E_CUDA,
                    "device allocation of %zu shareable bytes failed: %s", bytes, cudaGetErrorString(e));
    }
    return OLAP_OK;
}
static void share_free(void* p, size_t bytes) {
    if (p) g_share_free.emplace(share_round(bytes), p);
}

int alloc_batch(int n, int64_t size, const int* types, const int* default_kinds, bool with_status,
                bool shared_status, olap_store** out, bool shareable) {
    const size_t guard = g_guard ? kGuardBytes : 0;
    const size_t vplane = pad256((size_t)size * sizeof(float)) + guard;
    const size_t splane = with_status ? pad256((size_t)size) + guard : 0;
    const int n_status = with_status ? (shared_status ? 1 : n) : 0;
    const size_t bytes = vplane * n + splane * n_status;
    shareable |= g_share_all;
    // Large stores with planes of their own get an allocation EACH: a cube that keeps 1 of 64 measures
    // (dropMeasure, keepMeasures, dice by measures) must not pin the planes of the other 63.  Small ones share one
    // block (one pool call per query); shared status planes and peer-mapped blocks need the single block.
    const char* own_env = getenv("OLAP_OWN_ARENA_MB");  // read per call: a test lowers it
    const size_t own_arena_bytes = (size_t)(own_env ? atoi(own_env) : 32) << 20;
    if (n > 1 && !shareable && !(with_status && shared_status) && vplane + splane >= own_arena_bytes) {
        for (int k = 0; k < n; ++k) {
            const int rc = alloc_batch(1, size, types + k, default_kinds + k, with_status, false, out + k, false);
            if (rc != OLAP_OK) {
                for (int q = 0; q < k; ++q) { olap_store_destroy(out[q]); out[q] = nullptr; }
                return rc;
            }
        }
        return OLAP_OK;
    }
    Arena* arena = new Arena();
    int rc = shareable ? share_alloc(&arena->base, bytes) : dev_alloc(&arena->base, bytes);
    if (rc != OLAP_OK) { delete arena; return rc; }
    arena->bytes = bytes;
    arena->shareable = shareable;
    arena->refs = n;
    char* base = static_cast<char*>(arena->base);
    if (g_guard && bytes) cudaMemsetAsync(base, 0xA5, bytes, g.stream);
    for (int k = 0; k < n; ++k) {
        olap_store* s = new olap_store();
        s->size = size;
        s->type = types[k];
        s->default_kind = default_kinds[k];
        s->values = reinterpret_cast<float*>(base + vplane * k);
        s->status = with_status ? reinterpret_cast<uint8_t*>(base + vplane * n + splane * (shared_status ? 0 : k)) : nullptr;
        s->arena = arena;
        s->shared_plane = with_status && shared_status && n > 1;
        out[k] = s;
    }
    return OLAP_OK;
}

// see olap_store::derived
static bool is_derived(const olap_store* s) { return !s->status || (s->derived && !s->shared_plane); }
static void set_derived(olap_store* s, bool yes) { s->derived = yes && !s->shared_plane; }

// bytes of the guard (and of the alignment padding before it) that no longer hold 0xA5
static void check_guards(const olap_store* s) {
    if (!g_guard || !g.ready || !s->arena) return;  // wrapped stores (olap_store_wrap) carry no guard regions
    auto check = [&](const char* plane, size_t used) {
        const size_t span = pad256(used) + kGuardBytes - used;
        std::vector<unsigned char> host(span);
        if (cudaMemcpyAsync(host.data(), plane + used, span, cudaMemcpyDeviceToHost, g.stream) != cudaSuccess) return;
        if (cudaStreamSynchronize(g.stream) != cudaSuccess) return;
        for (unsigned char c : host) g_guard_violations += c != 0xA5;
    };
    check(reinterpret_cast<const char*>(s->values), (size_t)s->size * 4);
    if (s->status) check(reinterpret_cast<const char*>(s->status), (size_t)s->size);
}

size_t TablePack::add(const void* data, size_t bytes, size_t align) {
    const size_t off = (host.size() + align - 1) & ~(align - 1);
    host.resize(off + bytes);
    if (bytes) memcpy(host.data() + off, data, bytes);
    return off;
}

int TablePack::upload() {
    const size_t bytes = host.size();
    OLAP_TRY(dev_alloc(&dev, bytes));
    if (!bytes) return OLAP_OK;
    Ctx::PinSlot& slot = g.pin[g.pin_next];
    g.pin_next = (g.pin_next + 1) % Ctx::kPinSlots;
    if (slot.busy) {
        OLAP_CUDA(cudaEventSynchronize(slot.free_ev));
        slot.busy = false;
    }
    if (slot.cap < bytes) {
        if (slot.ptr) cudaFreeHost(slot.ptr);
        slot.ptr = nullptr;
        slot.cap = 0;
        const size_t cap = std::max(bytes * 2, (size_t)256 << 10);
        OLAP_CUDA(cudaHostAlloc((void**)&slot.ptr, cap, cudaHostAllocDefault));
        slot.cap = cap;
    }
    if (!slot.free_ev) OLAP_CUDA(cudaEventCreateWithFlags(&slot.free_ev, cudaEventDisableTiming));
    memcpy(slot.ptr, host.data(), bytes);
    OLAP_CUDA(cudaMemcpyAsync(dev, slot.ptr, bytes, cudaMemcpyHostToDevice, g.stream));
    OLAP_CUDA(cudaEventRecord(slot.free_ev, g.stream));
    slot.busy = true;
    return OLAP_OK;
}

int TablePack::release() {
    int rc = dev_free(dev);
    dev = nullptr;
    return rc;
}

// Device copies of map-derived tables, keyed by content (a few recent ones are kept).
struct CachedTable {
    std::vector<char> host;
    void* dev = nullptr;
    uint64_t stamp = 0;
};
static int cached_tables(const TablePack& pack, const char** dev_out) {
    static CachedTable cache[8];
    static uint64_t clock = 0;
    ++clock;
    CachedTable* victim = &cache[0];
    for (auto& e : cache) {
        if (e.dev && e.host.size() == pack.host.size() && !memcmp(e.host.data(), pack.host.data(), pack.host.size())) {
            e.stamp = clock;
            *dev_out = static_cast<const char*>(e.dev);
            return OLAP_OK;
        }
        if (e.stamp < victim->stamp) victim = &e;
    }
    if (victim->dev) OLAP_TRY(dev_free(victim->dev));  // stream-ordered: earlier kernels finish first
    victim->dev = nullptr;
    TablePack up;
    up.host = pack.host;
    OLAP_TRY(up.upload());
    victim->dev = up.dev;
    victim->host = pack.host;
    victim->stamp = clock;
    *dev_out = static_cast<const char*>(up.dev);
    up.dev = nullptr;  // the cache owns it now
    return OLAP_OK;
}

static int grid_for(int64_t n, int per_block) {
    const int64_t want = ceil_div(n, per_block);
    const int64_t cap = (int64_t)g.sm_count * 32;
    return (int)std::max<int64_t>(1, std::min(want, cap));
}

static bool mul_overflow(int64_t a, int64_t b, int64_t* out) { return __builtin_mul_overflow(a, b, out); }

static int product(const int64_t* len, int nd, int64_t* out, const char* what) {
    int64_t p = 1;
    for (int d = 0; d < nd; ++d) {
        if (len[d] < 0) return fail(OLAP_E_INVALID, "%s: negative dimension length", what);
        if (mul_overflow(p, len[d], &p)) return fail(OLAP_E_INVALID, "%s: cube size overflows int64", what);
    }
    *out = p;
    return OLAP_OK;
}

static int check_batch(olap_store* const* src, int n, const char* what, int64_t* size) {
    if (!src || n < 1 || n > OLAP_MAX_MEASURES) return fail(OLAP_E_INVALID, "%s: 1..%d stores expected", what, OLAP_MAX_MEASURES);
    for (int k = 0; k < n; ++k) {
        if (!src[k]) return fail(OLAP_E_INVALID, "%s: null store", what);
        if (src[k]->size != src[0]->size) return fail(OLAP_E_INVALID, "%s: stores of one call must have the same size", what);
    }
    *size = src[0]->size;
    return OLAP_OK;
}

// Result stores of a transform: same type/default as their source, one arena.
static int alloc_like(olap_store* const* src, int n, int64_t new_size, olap_store** out) {
    int types[OLAP_MAX_MEASURES], defaults[OLAP_MAX_MEASURES];
    bool with_status = true, shared = n > 1;
    for (int k = 0; k < n; ++k) {
        types[k] = src[k]->type;
        defaults[k] = src[k]->default_kind;
        with_status &= src[k]->status != nullptr;
        shared &= src[k]->status == src[0]->status;
    }
    // results of a shareable store stay shareable: the next query may be a rollup of the sharded axis
    const bool shareable = src[0]->arena && src[0]->arena->shareable;
    return alloc_batch(n, new_size, types, defaults, with_status, with_status && shared, out, shareable);
}

// Result stores of a call in flight: destroyed (and the caller's out[] cleared) on every early
// return; `done()` hands them over on success.
struct OutGuard {
    olap_store** out;
    int n;
    OutGuard(olap_store** o, int count) : out(o), n(count) {}
    ~OutGuard() {
        if (!out) return;
        for (int k = 0; k < n; ++k) { olap_store_destroy(out[k]); out[k] = nullptr; }
    }
    int done(int rc) {
        if (rc == OLAP_OK) out = nullptr;
        return rc;
    }
};

static int fill_default(olap_store* s) {
    if (s->size == 0) return OLAP_OK;
    fill_kernel<<<grid_for(s->size, kStoreThreads), kStoreThreads, 0, g.stream>>>(
        s->values, s->status, s->size, s->default_kind ? __builtin_nanf("") : 0.0f, OLAP_STATUS_UNSET);
    LAUNCHED();
    return OLAP_OK;
}

// status planes that several stores share must be written by one of them only
static uint8_t* st_out_of(olap_store** out, int k) {
    for (int q = 0; q < k; ++q)
        if (out[q]->status == out[k]->status) return nullptr;
    return out[k]->status;
}

// ---------------------------------------------------------------- drillUp
struct Csr {
    std::vector<int32_t> pstart, children;
    bool contiguous = true;
};

static Csr build_csr(const int32_t* map, int64_t C, int64_t P, bool lean = false) {
    Csr c;
    if (P == 1 && lean) {  // everything rolls up to one parent: the child list is 0..C-1, never materialised
        c.pstart = {0, (int32_t)C};
        return c;
    }
    c.pstart.assign(P + 1, 0);
    for (int64_t i = 0; i < C; ++i) c.pstart[map[i] + 1]++;
    for (int64_t p = 0; p < P; ++p) c.pstart[p + 1] += c.pstart[p];
    c.children.resize(C);
    std::vector<int32_t> fill(c.pstart.begin(), c.pstart.end() - 1);
    for (int64_t i = 0; i < C; ++i) c.children[fill[map[i]]++] = (int32_t)i;
    for (int64_t i = 0; i < C; ++i)
        if (c.children[i] != i) { c.contiguous = false; break; }
    return c;
}

static uint32_t next_pow2(uint32_t v) {
    uint32_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

static int launch_up_mid(const UpMeasure* d_meas, const UpMeasure* h_meas, int n, const Csr& csr,
                         const int32_t* d_pstart, const int32_t* d_children, int64_t O, int64_t C, int64_t P, int64_t I,
                         float* const* d_row_out = nullptr, uint8_t* const* d_row_st = nullptr) {
    const int VEC = (I % 4 == 0) ? 4 : (I % 2 == 0 ? 2 : 1);
    const int64_t IV_total = I / VEC;
    // chunk the inner run so that one row of output vectors fits 32-bit math
    const int64_t max_row = ((int64_t)1 << 30);
    int64_t chunk_iv = IV_total;
    if (P * IV_total > max_row) chunk_iv = std::max<int64_t>(1, max_row / P);
    for (int64_t iv0 = 0; iv0 < IV_total; iv0 += chunk_iv) {
        const int64_t iv_n = std::min(chunk_iv, IV_total - iv0);
        UpMidParams p{};
        p.meas = d_meas;
        if (!d_meas) for (int k = 0; k < n; ++k) p.meas_inline[k] = h_meas[k];
        p.pstart = d_pstart;
        p.children = d_children;
        p.O = O; p.C = (int32_t)C; p.P = (int32_t)P;
        p.I = iv_n * VEC;
        p.I_total = I;
        p.in_row = C * I;
        p.out_row = P * I;
        p.i_base = iv0 * VEC;
        p.IV = (uint32_t)iv_n;
        p.div_iv = FastDiv((uint32_t)iv_n);
        p.row_vecs = (uint32_t)(P * iv_n);
        p.n_measures = n;
        p.row_out = d_row_out;
        p.row_st = d_row_st;
        // too few output vectors to fill the chip and long child lists: split each parent's
        // children over G thread rows (drillup_split_kernel)
        static const int split_knob = [] { const char* e = getenv("OLAP_SPLIT"); return e ? atoi(e) : -1; }();
        const int64_t threads = O * (int64_t)p.row_vecs;
        const int64_t want_threads = (int64_t)g.sm_count * 2048;
        const int64_t avg_children = std::max<int64_t>(1, C / std::max<int64_t>(P, 1));
        int G = 1;
        while (G < 32 && threads * G * 4 <= want_threads && avg_children >= 8 * G) G *= 2;
        if (split_knob >= 0) G = split_knob;
        if (d_row_out) G = 1;  // row pointer tables: plain mid kernel only
        if (G >= 2 && O * ceil_div(p.row_vecs, 32) <= 0x7fffffffLL) {
            p.blocks_per_row = (uint32_t)ceil_div(p.row_vecs, 32);
            const size_t smem = (size_t)G * 32 * VEC * 16 + (size_t)G * 32 * 4;
            dim3 grid((unsigned)(O * p.blocks_per_row), (unsigned)n), block(32, G);
            KERNELS_BEGIN();
#define OLAP_SPLIT_LAUNCH(V, R)                                                                            \
    do {                                                                                                   \
        static bool attr = false;                                                                          \
        if (!attr) {                                                                                       \
            OLAP_CUDA(cudaFuncSetAttribute(drillup_split_kernel<V, R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           32 * 32 * 4 * 16 + 32 * 32 * 4));                               \
            attr = true;                                                                                   \
        }                                                                                                  \
        if (wide) drillup_split_kernel<V, R, true><<<grid, block, smem, g.stream>>>(p);                    \
        else drillup_split_kernel<V, R, false><<<grid, block, smem, g.stream>>>(p);                        \
    } while (0)
            static const int wide_knob = [] { const char* e = getenv("OLAP_SPLIT_WIDE"); return e ? atoi(e) : 1; }();
            const bool wide = wide_knob && G <= 8;
            if (VEC == 4) { if (csr.contiguous) OLAP_SPLIT_LAUNCH(4, true); else OLAP_SPLIT_LAUNCH(4, false); }
            else if (VEC == 2) { if (csr.contiguous) OLAP_SPLIT_LAUNCH(2, true); else OLAP_SPLIT_LAUNCH(2, false); }
            else { if (csr.contiguous) OLAP_SPLIT_LAUNCH(1, true); else OLAP_SPLIT_LAUNCH(1, false); }
#undef OLAP_SPLIT_LAUNCH
            LAUNCHED();
            continue;
        }
        const uint32_t bx = std::min<uint32_t>(256, next_pow2(p.row_vecs));
        const uint32_t by = 256 / bx;
        p.blocks_per_row = (uint32_t)ceil_div(p.row_vecs, bx);
        const int64_t gx = ceil_div(O, by) * p.blocks_per_row;
        if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "drillUp: grid too large (%lld blocks)", (long long)gx);
        dim3 grid((unsigned)gx, (unsigned)n), block(bx, by);
        KERNELS_BEGIN();
        // 8 children in flight per thread (80 registers) for long child lists, 4 (60 registers,
        // one more resident CTA per SM) when a parent has only a handful of children
        static const int U_knob = [] { const char* e = getenv("OLAP_UP_U"); return e ? atoi(e) : 0; }();
        const int U = U_knob ? U_knob : (C / std::max<int64_t>(P, 1) < 8 ? 4 : 8);
#define OLAP_UP_LAUNCH(V, R)                                                                         \
    do {                                                                                             \
        if (U == 4) drillup_mid_kernel<V, R, 4><<<grid, block, 0, g.stream>>>(p);                    \
        else drillup_mid_kernel<V, R, 8><<<grid, block, 0, g.stream>>>(p);                           \
    } while (0)
        if (VEC == 4) {
            if (csr.contiguous) OLAP_UP_LAUNCH(4, true); else OLAP_UP_LAUNCH(4, false);
        } else if (VEC == 2) {
            if (csr.contiguous) OLAP_UP_LAUNCH(2, true); else OLAP_UP_LAUNCH(2, false);
        } else {
            if (csr.contiguous) OLAP_UP_LAUNCH(1, true); else OLAP_UP_LAUNCH(1, false);
        }
#undef OLAP_UP_LAUNCH
        LAUNCHED();
    }
    return OLAP_OK;
}

static int launch_down_mid(const DownMeasure* d_meas, int n, const Csr& csr, const int32_t* d_pstart,
                           const int32_t* d_children, int64_t O, int64_t P, int64_t C, int64_t I, int kind) {
    const int VEC = (I % 4 == 0) ? 4 : (I % 2 == 0 ? 2 : 1);
    const int64_t IV_total = I / VEC;
    const int64_t max_row = ((int64_t)1 << 30);
    int64_t chunk_iv = IV_total;
    if (P * IV_total > max_row) chunk_iv = std::max<int64_t>(1, max_row / P);
    for (int64_t iv0 = 0; iv0 < IV_total; iv0 += chunk_iv) {
        const int64_t iv_n = std::min(chunk_iv, IV_total - iv0);
        DownMidParams p{};
        p.meas = d_meas;
        p.pstart = d_pstart;
        p.children = d_children;
        p.O = O; p.C = (int32_t)C; p.P = (int32_t)P;
        p.I_total = I;
        p.in_row = P * I;
        p.out_row = C * I;
        p.i_base = iv0 * VEC;
        p.IV = (uint32_t)iv_n;
        p.div_iv = FastDiv((uint32_t)iv_n);
        p.row_vecs = (uint32_t)(P * iv_n);
        const uint32_t bx = std::min<uint32_t>(256, next_pow2(p.row_vecs));
        const uint32_t by = 256 / bx;
        p.blocks_per_row = (uint32_t)ceil_div(p.row_vecs, bx);
        const int64_t gx = ceil_div(O, by) * p.blocks_per_row;
        if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "drillDown: grid too large (%lld blocks)", (long long)gx);
        dim3 grid((unsigned)gx, (unsigned)n), block(bx, by);
        KERNELS_BEGIN();
#define OLAP_DOWN_K(V, R)                                                                              \
    do {                                                                                               \
        if (kind == 0) drilldown_mid_kernel<V, R, 0><<<grid, block, 0, g.stream>>>(p);                 \
        else if (kind == 1) drilldown_mid_kernel<V, R, 1><<<grid, block, 0, g.stream>>>(p);            \
        else if (kind == 2) drilldown_mid_kernel<V, R, 2><<<grid, block, 0, g.stream>>>(p);            \
        else drilldown_mid_kernel<V, R, -1><<<grid, block, 0, g.stream>>>(p);                          \
    } while (0)
        if (VEC == 4) { if (csr.contiguous) OLAP_DOWN_K(4, true); else OLAP_DOWN_K(4, false); }
        else if (VEC == 2) { if (csr.contiguous) OLAP_DOWN_K(2, true); else OLAP_DOWN_K(2, false); }
        else { if (csr.contiguous) OLAP_DOWN_K(1, true); else OLAP_DOWN_K(1, false); }
#undef OLAP_DOWN_K
        LAUNCHED();
    }
    return OLAP_OK;
}

// The block kernel's dynamic shared memory: RB rows of P * I staged parent cells (step, result, status, truthy:
// 14 bytes each), the [C] parent and rank tables, and 16 bytes of alignment.  It opts in to kDownBlockSmem bytes.
constexpr size_t kDownBlockSmem = 160 * 1024;
static int64_t down_block_rows(int64_t O, int64_t C, int64_t I) { return std::max<int64_t>(1, std::min<int64_t>(O, 8192 / (C * I))); }
static size_t down_block_smem(int64_t O, int64_t P, int64_t C, int64_t I) {
    return (size_t)down_block_rows(O, C, I) * P * I * (8 + 4 + 1 + 1) + (size_t)C * 8 + 16;
}

// The block kernel stages P * I parent cells (14 bytes each) of at least one outer index in shared memory.
// With an inner run behind the drilled axis the integer-spreading measures stay on the parent-driven
// kernel, which carries floor((k - 1) * step) from child to child (the block kernel would redo both
// floors per cell: 0.38 against 0.64 of peak).  Shapes whose staging exceeds kDownBlockSmem (long rows, or
// many parents without children) take the mid or gather kernels.
static bool down_block_fits(int64_t O, int64_t P, int64_t C, int64_t I, bool any_int = false) {
    static const int knob = [] { const char* e = getenv("OLAP_DOWN_BLOCK"); return e ? atoi(e) : 1; }();
    bool fits = I == 1 ? C <= 8192 && P <= 8192 : knob && !any_int && P * I <= 8192 && C <= 8192 && C * I < (1 << 28) && I <= 2048;
    return fits && down_block_smem(O, P, C, I) <= kDownBlockSmem;
}

static int launch_down_inner(const DownMeasure* d_meas, int n, const int32_t* d_parent, const int32_t* d_rank,
                             const int32_t* d_cnt, int64_t O, int64_t P, int64_t C, int64_t I) {
    DownInnerParams p{};
    p.meas = d_meas;
    p.parent_of = d_parent;
    p.rank_of = d_rank;
    p.cnt_of = d_cnt;
    p.O = O; p.P = (int32_t)P; p.C = (int32_t)C; p.I = (uint32_t)I;
    p.RB = (uint32_t)down_block_rows(O, C, I);
    p.vec4 = I == 1 ? (C % 4 == 0 && ((int64_t)p.RB * C) % 4 == 0) : (I % 4 == 0);
    p.div_i = FastDiv((uint32_t)I);
    p.div_pi = FastDiv((uint32_t)(P * I));
    p.div_ci = FastDiv((uint32_t)(C * I));
    const size_t smem = down_block_smem(O, P, C, I);
    const int64_t gx = ceil_div(O, p.RB);
    if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "drillDown: grid too large");
    static bool attr = false;
    if (!attr) {
        OLAP_CUDA(cudaFuncSetAttribute(drilldown_inner_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDownBlockSmem));
        attr = true;
    }
    KERNELS_BEGIN();
    drilldown_inner_kernel<<<dim3((unsigned)gx, (unsigned)n), 256, smem, g.stream>>>(p);
    LAUNCHED();
    return OLAP_OK;
}

}  // namespace olap

using namespace olap;

// =====================================================================================
extern "C" {

int olap_abi_version(void) { return OLAP_ABI_VERSION; }

const char* olap_last_error(void) { return g_error.c_str(); }

int olap_init(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(OLAP_E_CUDA, "no CUDA device available (%s); this store has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= count) return fail(OLAP_E_INVALID, "olap_init: device %d out of range [0, %d)", device, count);
    if (g.ready && g.device == device) return OLAP_OK;
    if (g.ready) return fail(OLAP_E_UNSUPPORTED, "olap_init: already bound to device %d (one device per process)", g.device);
    OLAP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    OLAP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(OLAP_E_UNSUPPORTED, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
    g.device = device;
    g.sm_count = prop.multiProcessorCount;
    OLAP_CUDA(cudaStreamCreateWithFlags(&g.own_stream, cudaStreamNonBlocking));
    g.stream = g.own_stream;
    OLAP_CUDA(cudaEventCreate(&g.ev0));
    OLAP_CUDA(cudaEventCreate(&g.ev1));
    cudaMemPool_t pool;
    OLAP_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = UINT64_MAX;  // keep freed blocks cached: transforms allocate every call
    OLAP_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    g.ready = true;
    return OLAP_OK;
}

int olap_set_stream(void* cuda_stream) {
    OLAP_TRY(ensure_ctx());
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    g.stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : g.own_stream;
    return OLAP_OK;
}

int olap_set_async(int enabled) {
    g.async = enabled != 0;
    return OLAP_OK;
}

int olap_set_shareable(int enabled) {
    g_share_all = enabled != 0;
    return OLAP_OK;
}

int olap_sync(void) {
    OLAP_TRY(ensure_ctx());
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    OLAP_CUDA(cudaGetLastError());
    return OLAP_OK;
}

int olap_method_from_name(const char* name, int* method) {
    static const char* names[] = {"sum", "average", "highest", "lowest", "first", "last", "product"};
    if (name)
        for (int k = 0; k < 7; ++k)
            if (!strcmp(name, names[k])) { *method = k; return OLAP_OK; }
    return fail(OLAP_E_INVALID, "Unsupported aggregation method: %s", name ? name : "undefined");
}

int64_t olap_kernel_launches(void) { return g_launches.load(); }

double olap_last_op_ms(void) {
    if (!g.ready) return 0.0;
    if (g.timing_pending) {
        float ms = 0.f;
        if (cudaEventSynchronize(g.ev1) == cudaSuccess && cudaEventElapsedTime(&ms, g.ev0, g.ev1) == cudaSuccess) g.last_ms = ms;
        g.timing_pending = false;
    }
    return g.last_ms;
}

const char* olap_last_op_path(void) { return g.last_path; }

// ---- pinned host buffers for the data boundary (so H2D/D2H run at PCIe speed) ----
int olap_host_alloc(size_t bytes, void** out) {
    OLAP_TRY(ensure_ctx());
    static const bool wc = [] { const char* e = getenv("OLAP_PIN_WC"); return e && atoi(e) != 0; }();  // experiment knob
    OLAP_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, wc ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
    return OLAP_OK;
}
int olap_host_free(void* p) {
    if (p) OLAP_CUDA(cudaFreeHost(p));
    return OLAP_OK;
}

// ---- life cycle -------------------------------------------------------------------
static int check_type_default(int type, int default_kind) {
    if (default_kind != OLAP_DEFAULT_ZERO && default_kind != OLAP_DEFAULT_NAN)
        return fail(OLAP_E_INVALID, "Invalid default value, only NaN and 0 are supported");
    if (type < OLAP_INT32 || type > OLAP_FLOAT64) return fail(OLAP_E_INVALID, "Invalid type");
    return OLAP_OK;
}

int olap_store_create_batch(int n, int64_t size, const int* types, const int* default_kinds, int with_status,
                            int shared_status, olap_store** out) {
    if (n < 1 || n > OLAP_MAX_MEASURES || !out) return fail(OLAP_E_INVALID, "olap_store_create_batch: 1..%d stores expected", OLAP_MAX_MEASURES);
    if (size < 0) return fail(OLAP_E_INVALID, "olap_store_create_batch: negative size");
    for (int k = 0; k < n; ++k) OLAP_TRY(check_type_default(types[k], default_kinds[k]));
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_batch(n, size, types, default_kinds, (with_status & 1) != 0, shared_status != 0, out,
                         (with_status & OLAP_CREATE_SHAREABLE) != 0));
    OutGuard guard(out, n);
    if (with_status & OLAP_CREATE_UNINITIALISED) return guard.done(finish_op());  // the caller overwrites every cell
    for (int k = 0; k < n; ++k) {
        olap_store tmp = *out[k];
        tmp.status = st_out_of(out, k);
        OLAP_TRY(fill_default(&tmp));
        set_derived(out[k], true);
    }
    return guard.done(finish_op());
}

int olap_store_create(int64_t size, int type, int default_kind, int with_status, olap_store** out) {
    return olap_store_create_batch(1, size, &type, &default_kind, with_status, 0, out);
}

int64_t olap_guard_violations(void) { return g_guard_violations.load(); }

int olap_store_destroy(olap_store* s) {
    if (!s) return OLAP_OK;
    check_guards(s);
    Arena* a = s->arena;
    delete s;
    if (a && --a->refs == 0) {
        if (a->shareable) share_free(a->base, a->bytes);
        else if (g.ready) cudaFreeAsync(a->base, g.stream);
        delete a;
    }
    return OLAP_OK;
}

int olap_store_clone(const olap_store* s, olap_store** out) {
    if (!s || !out) return fail(OLAP_E_INVALID, "olap_store_clone: null argument");
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_batch(1, s->size, &s->type, &s->default_kind, s->status != nullptr, false, out,
                         s->arena && s->arena->shareable));
    OutGuard guard(out, 1);
    (*out)->derived = s->derived && !s->shared_plane;
    if (s->size) {
        OLAP_CUDA(cudaMemcpyAsync((*out)->values, s->values, (size_t)s->size * 4, cudaMemcpyDeviceToDevice, g.stream));
        if (s->status) OLAP_CUDA(cudaMemcpyAsync((*out)->status, s->status, (size_t)s->size, cudaMemcpyDeviceToDevice, g.stream));
    }
    return guard.done(finish_op());
}

int olap_store_copy_status(olap_store* dst, const olap_store* src) {
    if (!dst || !src) return fail(OLAP_E_INVALID, "olap_store_copy_status: null store");
    if (dst->size != src->size) return fail(OLAP_E_INVALID, "value length is invalid: %lld !== %lld", (long long)dst->size, (long long)src->size);
    OLAP_TRY(ensure_ctx());
    dst->derived = false;
    if (dst->status && src->status && dst->size)
        OLAP_CUDA(cudaMemcpyAsync(dst->status, src->status, (size_t)dst->size, cudaMemcpyDeviceToDevice, g.stream));
    return finish_op();
}

int64_t olap_store_size(const olap_store* s) { return s ? s->size : -1; }
int64_t olap_store_byte_length(const olap_store* s) {
    if (!s) return -1;
    return s->size * (s->type == OLAP_FLOAT64 ? 8 : 4);
}
int olap_store_type(const olap_store* s) { return s ? s->type : -1; }
int olap_store_default_kind(const olap_store* s) { return s ? s->default_kind : -1; }
int olap_store_has_status(const olap_store* s) { return s && s->status ? 1 : 0; }
// mutable access: whatever is written through these pointers, the library no longer knows that the status
// plane follows from the values (olap_store_canonicalise re-establishes it)
void* olap_store_values_ptr(olap_store* s) { if (s) s->derived = false; return s ? s->values : nullptr; }
void* olap_store_status_ptr(olap_store* s) { if (s) s->derived = false; return s ? s->status : nullptr; }
const void* olap_store_values_cptr(const olap_store* s) { return s ? s->values : nullptr; }
const void* olap_store_status_cptr(const olap_store* s) { return s ? s->status : nullptr; }
int olap_store_status_derived(const olap_store* s) { return s && is_derived(s) ? 1 : 0; }

int olap_store_canonicalise(olap_store* s) {
    if (!s) return fail(OLAP_E_INVALID, "olap_store_canonicalise: null store");
    OLAP_TRY(ensure_ctx());
    if (s->size) {
        canon_f32_kernel<<<grid_for(ceil_div(s->size, 4), kStoreThreads), kStoreThreads, 0, g.stream>>>(s->values, s->status, s->size, s->default_kind);
        LAUNCHED();
    }
    set_derived(s, true);
    return finish_op();
}

// ---- data boundary ------------------------------------------------------------------
static int check_len(const olap_store* s, int64_t n) {
    if (!s) return fail(OLAP_E_INVALID, "null store");
    if (s->size != n) return fail(OLAP_E_INVALID, "value length is invalid: %lld !== %lld", (long long)s->size, (long long)n);
    return OLAP_OK;
}

// Cells are Float32 for every store type.  The reference keeps JS doubles, so an int32 / uint32 store
// there holds counts above 2^24 exactly; here such a value would silently become a neighbour.  Uploads
// and setValue(s) of integer stores therefore refuse values that do not survive Math.fround
// (OLAP_LOSSY_INTS=1 restores the silent rounding).  float64 stores round by declared contract.
static bool strict_ints(const olap_store* s) {
    static const bool relaxed = [] { const char* e = getenv("OLAP_LOSSY_INTS"); return e && atoi(e) != 0; }();
    return !relaxed && (s->type == OLAP_INT32 || s->type == OLAP_UINT32);
}
static int lossy_error(const olap_store* s, int64_t index, double value) {
    return fail(OLAP_E_UNSUPPORTED, "value %.17g at index %lld of an %s store is not representable in its Float32 cell "
                "(the reference would keep it exact; use a float32 store or set OLAP_LOSSY_INTS=1 to round)", value,
                (long long)index, s->type == OLAP_INT32 ? "int32" : "uint32");
}

int olap_store_upload_f32(olap_store* s, const float* host, int64_t n) {
    OLAP_TRY(check_len(s, n));
    OLAP_TRY(ensure_ctx());
    if (n == 0) return OLAP_OK;
    OLAP_TRY(copy_h2d(s->values, host, (size_t)n * 4));
    canon_f32_kernel<<<grid_for(ceil_div(n, 4), kStoreThreads), kStoreThreads, 0, g.stream>>>(s->values, s->status, n, s->default_kind);
    LAUNCHED();
    set_derived(s, true);
    return finish_op();
}

int olap_store_upload_f64(olap_store* s, const double* host, int64_t n) {
    OLAP_TRY(check_len(s, n));
    OLAP_TRY(ensure_ctx());
    if (n == 0) return OLAP_OK;
    void* tmp;
    OLAP_TRY(dev_alloc(&tmp, (size_t)n * 8 + 8));
    OLAP_TRY(copy_h2d(tmp, host, (size_t)n * 8));
    // integer stores hold exact integers in the reference (JS doubles): refuse what a Float32 cell would change
    unsigned long long* lossy = strict_ints(s) ? reinterpret_cast<unsigned long long*>(static_cast<char*>(tmp) + (size_t)n * 8) : nullptr;
    if (lossy) OLAP_CUDA(cudaMemsetAsync(lossy, 0xff, 8, g.stream));
    from_f64_kernel<<<grid_for(n, kStoreThreads), kStoreThreads, 0, g.stream>>>((const double*)tmp, s->values, s->status, n, s->default_kind, lossy);
    LAUNCHED();
    unsigned long long first = ~0ull;
    if (lossy) OLAP_CUDA(cudaMemcpyAsync(&first, lossy, 8, cudaMemcpyDeviceToHost, g.stream));
    OLAP_TRY(dev_free(tmp));
    // the host buffer is borrowed for the call only
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    set_derived(s, true);
    if (first != ~0ull) return lossy_error(s, (int64_t)first - 1, host[first - 1]);
    return finish_op();
}

int olap_store_download_f32(const olap_store* s, float* host, int64_t n) {
    OLAP_TRY(check_len(s, n));
    OLAP_TRY(ensure_ctx());
    if (n == 0) return OLAP_OK;
    return copy_d2h(host, s->values, (size_t)n * 4);
}

int olap_store_download_f64(const olap_store* s, double* host, int64_t n) {
    OLAP_TRY(check_len(s, n));
    OLAP_TRY(ensure_ctx());
    if (n == 0) return OLAP_OK;
    void* tmp;
    OLAP_TRY(dev_alloc(&tmp, (size_t)n * 8));
    to_f64_kernel<<<grid_for(n, kStoreThreads), kStoreThreads, 0, g.stream>>>(s->values, (double*)tmp, n);
    LAUNCHED();
    OLAP_TRY(copy_d2h(host, tmp, (size_t)n * 8));
    return dev_free(tmp);
}

int olap_store_get_value(const olap_store* s, int64_t index, double* out) {
    if (!s || !out) return fail(OLAP_E_INVALID, "olap_store_get_value: null argument");
    OLAP_TRY(ensure_ctx());
    if (index < 0 || index >= s->size) {  // Map.get(missing) ?? default
        *out = s->default_kind ? NAN : 0.0;
        return OLAP_OK;
    }
    float v;
    OLAP_CUDA(cudaMemcpyAsync(&v, s->values + index, 4, cudaMemcpyDeviceToHost, g.stream));
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    *out = (double)v;
    return OLAP_OK;
}

int olap_store_set_values(olap_store* s, const int64_t* indexes, const double* values, int64_t n) {
    if (!s || (n && (!indexes || !values))) return fail(OLAP_E_INVALID, "olap_store_set_values: null argument");
    OLAP_TRY(ensure_ctx());
    if (n == 0) return OLAP_OK;
    if (strict_ints(s))  // the values are on the host: check before anything is written
        for (int64_t i = 0; i < n; ++i)
            if (values[i] == values[i] && (double)(float)values[i] != values[i] && indexes[i] >= 0 && indexes[i] < s->size)
                return lossy_error(s, indexes[i], values[i]);
    TablePack t;
    const size_t oi = t.add(indexes, (size_t)n * 8);
    const size_t ov = t.add(values, (size_t)n * 8);
    OLAP_TRY(t.upload());
    set_values_kernel<<<(unsigned)ceil_div(n, kStoreThreads), kStoreThreads, 0, g.stream>>>(
        s->values, s->status, t.ptr<int64_t>(oi), t.ptr<double>(ov), n, s->size, s->default_kind, nullptr);
    LAUNCHED();
    OLAP_TRY(t.release());
    return finish_op();
}

int olap_store_set_value(olap_store* s, int64_t index, double value) { return olap_store_set_values(s, &index, &value, 1); }

int olap_store_fill(olap_store* s, double value) {
    if (!s) return fail(OLAP_E_INVALID, "olap_store_fill: null store");
    OLAP_TRY(ensure_ctx());
    if (s->size == 0) return OLAP_OK;
    float v = (float)value;
    const bool nan_default = s->default_kind != 0;
    if (v != v) v = __builtin_nanf("");
    if (!nan_default && v == 0.0f) v = 0.0f;
    const bool set = nan_default ? (v == v) : (v != 0.0f);
    fill_kernel<<<grid_for(s->size, kStoreThreads), kStoreThreads, 0, g.stream>>>(
        s->values, s->status, s->size, v, set ? OLAP_STATUS_SET : OLAP_STATUS_UNSET);
    LAUNCHED();
    set_derived(s, true);
    return finish_op();
}

static int total_and_count(const olap_store* s, double* sum, int64_t* count) {
    OLAP_TRY(ensure_ctx());
    *sum = 0.0;
    *count = 0;
    if (s->size == 0) return OLAP_OK;
    const int blocks = grid_for(ceil_div(s->size, 4), kStoreThreads);
    void* scratch;
    const size_t bytes = (size_t)blocks * 16 + 64;
    OLAP_TRY(dev_alloc(&scratch, bytes));
    char* b = (char*)scratch;
    double* psum = (double*)b;
    unsigned long long* pcnt = (unsigned long long*)(b + (size_t)blocks * 8);
    double* osum = (double*)(b + (size_t)blocks * 16);
    unsigned long long* ocnt = (unsigned long long*)(b + (size_t)blocks * 16 + 8);
    unsigned int* ticket = (unsigned int*)(b + (size_t)blocks * 16 + 16);
    OLAP_CUDA(cudaMemsetAsync(ticket, 0, 4, g.stream));
    begin_op();
    KERNELS_BEGIN();
    total_kernel<<<blocks, kStoreThreads, 0, g.stream>>>(s->values, s->size, s->default_kind, psum, pcnt, ticket, osum, ocnt);
    LAUNCHED();
    end_op("total");
    struct { double s; unsigned long long c; } host;
    OLAP_CUDA(cudaMemcpyAsync(&host, osum, 16, cudaMemcpyDeviceToHost, g.stream));
    OLAP_TRY(dev_free(scratch));
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    *sum = host.s;
    *count = (int64_t)host.c;
    return OLAP_OK;
}

int olap_store_total(const olap_store* s, double* out) {
    if (!s || !out) return fail(OLAP_E_INVALID, "olap_store_total: null argument");
    int64_t c;
    return total_and_count(s, out, &c);
}

int olap_store_count_present(const olap_store* s, int64_t* out) {
    if (!s || !out) return fail(OLAP_E_INVALID, "olap_store_count_present: null argument");
    double t;
    return total_and_count(s, &t, out);
}

static int bytes_out(const olap_store* s, uint8_t* host, int64_t n, bool status) {
    OLAP_TRY(check_len(s, n));
    OLAP_TRY(ensure_ctx());
    if (n == 0) return OLAP_OK;
    if (status && s->status) {
        return copy_d2h(host, s->status, (size_t)n);
    }
    void* tmp;
    OLAP_TRY(dev_alloc(&tmp, (size_t)n));
    presence_kernel<<<grid_for(n, kStoreThreads), kStoreThreads, 0, g.stream>>>(
        s->values, (uint8_t*)tmp, n, s->default_kind, status ? OLAP_STATUS_SET : 1, status ? OLAP_STATUS_UNSET : 0);
    LAUNCHED();
    OLAP_TRY(copy_d2h(host, tmp, (size_t)n));
    return dev_free(tmp);
}

int olap_store_presence(const olap_store* s, uint8_t* host, int64_t n) { return bytes_out(s, host, n, false); }
int olap_store_status(const olap_store* s, uint8_t* host, int64_t n) { return bytes_out(s, host, n, true); }

int olap_store_export_sparse(const olap_store* s, int64_t capacity, int64_t* keys, float* values, int64_t* count) {
    if (!s || !count) return fail(OLAP_E_INVALID, "olap_store_export_sparse: null argument");
    OLAP_TRY(ensure_ctx());
    *count = 0;
    if (s->size == 0) return OLAP_OK;
    const int64_t nb = ceil_div(s->size, kCompactTile);
    void* cnt;
    OLAP_TRY(dev_alloc(&cnt, (size_t)(nb + 1) * 8));
    unsigned long long* d_cnt = (unsigned long long*)cnt;
    compact_count_kernel<<<(unsigned)nb, 256, 0, g.stream>>>(s->values, s->size, s->default_kind, d_cnt);
    LAUNCHED();
    compact_scan_kernel<<<1, 1024, 0, g.stream>>>(d_cnt, nb, d_cnt + nb);
    LAUNCHED();
    unsigned long long total = 0;
    OLAP_CUDA(cudaMemcpyAsync(&total, d_cnt + nb, 8, cudaMemcpyDeviceToHost, g.stream));
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    *count = (int64_t)total;
    int rc = OLAP_OK;
    if (keys && values && total) {
        if ((int64_t)total > capacity) {
            rc = fail(OLAP_E_INVALID, "olap_store_export_sparse: capacity %lld < %llu set cells", (long long)capacity, total);
        } else {
            void *dk, *dv;
            OLAP_TRY(dev_alloc(&dk, (size_t)total * 8));
            OLAP_TRY(dev_alloc(&dv, (size_t)total * 4));
            compact_write_kernel<<<(unsigned)nb, 256, 0, g.stream>>>(s->values, s->size, s->default_kind, d_cnt, (int64_t*)dk, (float*)dv);
            LAUNCHED();
            OLAP_TRY(copy_d2h(keys, dk, (size_t)total * 8));
            OLAP_TRY(copy_d2h(values, dv, (size_t)total * 4));
            OLAP_TRY(dev_free(dk));
            OLAP_TRY(dev_free(dv));
        }
    }
    OLAP_TRY(dev_free(cnt));
    return rc;
}

int olap_store_import_sparse(olap_store* s, const int64_t* keys, const float* values, int64_t count) {
    if (!s || (count && (!keys || !values))) return fail(OLAP_E_INVALID, "olap_store_import_sparse: null argument");
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(fill_default(s));
    set_derived(s, true);
    if (count >= ((int64_t)1 << 20)) {  // large lists go straight to the device (pageable memory: through the pinned ring)
        void *dk, *dv;
        OLAP_TRY(dev_alloc(&dk, (size_t)count * 8));
        OLAP_TRY(dev_alloc(&dv, (size_t)count * 4));
        OLAP_TRY(copy_h2d(dk, keys, (size_t)count * 8));
        OLAP_TRY(copy_h2d(dv, values, (size_t)count * 4));
        import_sparse_kernel<<<(unsigned)ceil_div(count, kStoreThreads), kStoreThreads, 0, g.stream>>>(
            s->values, s->status, (const int64_t*)dk, (const float*)dv, count, s->size, s->default_kind);
        LAUNCHED();
        OLAP_TRY(dev_free(dk));
        OLAP_TRY(dev_free(dv));
        OLAP_CUDA(cudaStreamSynchronize(g.stream));  // the host lists are borrowed for the call only
    } else if (count) {
        TablePack t;
        const size_t ok = t.add(keys, (size_t)count * 8);
        const size_t ov = t.add(values, (size_t)count * 4);
        OLAP_TRY(t.upload());
        import_sparse_kernel<<<(unsigned)ceil_div(count, kStoreThreads), kStoreThreads, 0, g.stream>>>(
            s->values, s->status, t.ptr<int64_t>(ok), t.ptr<float>(ov), count, s->size, s->default_kind);
        LAUNCHED();
        OLAP_TRY(t.release());
    }
    return finish_op();
}

// ---- drillUp --------------------------------------------------------------------------
int olap_drill_up(olap_store* const* src, int n, const int* methods, int ndim, const int64_t* old_len,
                  const int64_t* new_len, const int32_t* const* maps, olap_store** out) {
    int64_t size = 0, old_size = 0, new_size = 0;
    OLAP_TRY(check_batch(src, n, "olap_drill_up", &size));
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "olap_drill_up: at most %d dimensions", OLAP_MAX_DIMS);
    if (!out || (ndim && (!old_len || !new_len || !maps))) return fail(OLAP_E_INVALID, "olap_drill_up: null argument");
    OLAP_TRY(product(old_len, ndim, &old_size, "olap_drill_up"));
    OLAP_TRY(product(new_len, ndim, &new_size, "olap_drill_up"));
    if (old_size != size) return fail(OLAP_E_INVALID, "olap_drill_up: dimensions describe %lld cells, store has %lld", (long long)old_size, (long long)size);
    for (int k = 0; k < n; ++k)
        if (methods[k] < OLAP_SUM || methods[k] > OLAP_COUNT) return fail(OLAP_E_INVALID, "Unsupported aggregation method: %d", methods[k]);
    std::vector<int> changed;
    for (int d = 0; d < ndim; ++d) {
        if (old_len[d] > 0x7fffffffLL || new_len[d] > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "olap_drill_up: dimension %d longer than 2^31-1", d);
        bool identity = old_len[d] == new_len[d];
        if (!maps[d]) {
            // no map: the dimension is untouched, or every item rolls up to the single new item
            if (!identity && new_len[d] != 1) return fail(OLAP_E_INVALID, "olap_drill_up: dimension %d changes length without a map", d);
            if (!identity) changed.push_back(d);
            continue;
        }
        for (int64_t i = 0; i < old_len[d]; ++i) {
            const int32_t m = maps[d][i];
            if (m < 0 || m >= new_len[d]) return fail(OLAP_E_INVALID, "olap_drill_up: map of dimension %d sends item %lld to %d, outside [0, %lld)", d, (long long)i, m, (long long)new_len[d]);
            identity &= m == i;
        }
        if (!identity) changed.push_back(d);
    }
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_like(src, n, new_size, out));
    OutGuard guard(out, n);
    begin_op();
    const char* path = "drillup/empty";
    if (new_size == 0) {
        // nothing to compute
    } else if (old_size == 0) {
        for (int k = 0; k < n; ++k) { olap_store t = *out[k]; t.status = st_out_of(out, k); OLAP_TRY(fill_default(&t)); }
    } else {
        std::vector<UpMeasure> meas(n);
        for (int k = 0; k < n; ++k) {
            // a status plane shared by the RESULTS is written by the first of them only; results with
            // planes of their own each merge their source's plane, even when one source store is
            // passed twice (sum and count of a sharded `average`)
            uint8_t* so = out[k]->status && src[k]->status ? st_out_of(out, k) : nullptr;
            meas[k] = UpMeasure{src[k]->values, out[k]->values, so ? src[k]->status : nullptr, so, methods[k], src[k]->default_kind};
        }
        TablePack t;
        const size_t o_meas = t.add(meas.data(), sizeof(UpMeasure) * n);
        if (changed.size() <= 1) {
            // view the cube as [O, C, I] around the changed dimension (or the last one for a plain copy)
            const int d = changed.empty() ? std::max(0, ndim - 1) : changed[0];
            int64_t O = 1, I = 1;
            for (int q = 0; q < d; ++q) O *= old_len[q];
            for (int q = d + 1; q < ndim; ++q) I *= old_len[q];
            const int64_t C = ndim ? old_len[d] : 1, P = ndim ? new_len[d] : 1;
            static const int32_t zero = 0;
            std::vector<int32_t> implied;
            if (ndim && !maps[d] && P != 1) { implied.resize(C); std::iota(implied.begin(), implied.end(), 0); }  // plain copy
            const Csr csr = build_csr(!ndim ? &zero : (maps[d] ? maps[d] : implied.data()), C, P, true);
            // the CSR depends only on the map: keep it on the device across calls (a cube is
            // usually drilled the same way many times); measure descriptors change every call
            // (new output planes) and travel in the kernel parameters when they fit
            bool any_status = false;
            for (int k = 0; k < n; ++k) any_status |= meas[k].st_in != nullptr;
            const TileDecision tile = tile_plan(O, C, P, I, any_status);
            LongDecision lng;
            LanesDecision lanes;
            static const int derive_knob = [] { const char* e = getenv("OLAP_DERIVE_STATUS"); return e ? atoi(e) : 1; }();
            if (!tile.use) {
                // planes that will really be read (the others follow from the values; read in words of 4 status bytes)
                bool loaded = false, aligned = true;
                for (int k = 0; k < n; ++k) {
                    loaded |= meas[k].st_in && !(derive_knob && src[k]->derived && !src[k]->shared_plane);
                    aligned &= (reinterpret_cast<uintptr_t>(meas[k].st_in) & 3) == 0;
                }
                if (aligned) lanes = lanes_plan(O, C, P, I, n, g.sm_count, loaded);
            }
            if (!tile.use && !lanes.use) lng = long_plan(O, C, P, I, any_status, n, g.sm_count, csr.contiguous);
            TablePack stat;
            const size_t o_ps = stat.add(csr.pstart.data(), csr.pstart.size() * 4);
            // a contiguous map needs no child list on the device (children[k] == k)
            const size_t o_ch = csr.contiguous ? 0 : stat.add(csr.children.data(), csr.children.size() * 4);
            size_t o_seg = 0, o_perm = 0;
            if (lng.use) {
                const LongTables lt = long_seg_table(csr.pstart, csr.children, csr.contiguous, C, P, lng);
                o_seg = stat.add(lt.seg_ptr.data(), lt.seg_ptr.size() * 4);
                if (!lt.perm16.empty()) o_perm = stat.add(lt.perm16.data(), lt.perm16.size() * 2);
            }
            size_t o_map8 = 0;
            if (lanes.use) {
                const std::vector<uint8_t> lists = lanes_lists(maps[d], C, lanes.tile);
                o_map8 = stat.add(lists.data(), lists.size());
            }
            const char* d_stat = nullptr;
            OLAP_TRY(cached_tables(stat, &d_stat));
            const bool inline_meas = n <= kInlineMeasures;
            if (!inline_meas) OLAP_TRY(t.upload());
            const UpMeasure* d_meas = inline_meas ? nullptr : t.ptr<UpMeasure>(o_meas);
            const int32_t* d_ps = reinterpret_cast<const int32_t*>(d_stat + o_ps);
            const int32_t* d_ch = csr.contiguous ? nullptr : reinterpret_cast<const int32_t*>(d_stat + o_ch);
            // sources whose status plane follows from their values: the mid / split / tile kernels recompute the
            // bytes from the cells they load anyway and never read the plane (4 instead of 5 bytes per input cell)
            const UpMeasure* d_meas_drv = d_meas;
            TablePack t2;
            if (derive_knob && (tile.use || lanes.use || !lng.use)) {
                bool changed_desc = false;
                for (int k = 0; k < n; ++k)
                    if (meas[k].st_in && src[k]->derived && !src[k]->shared_plane) {
                        meas[k].st_in = nullptr;
                        meas[k].derive = 1;
                        changed_desc = true;
                    }
                if (changed_desc && !inline_meas) {  // descriptors travel through a device table: upload the edited ones
                    const size_t o2 = t2.add(meas.data(), sizeof(UpMeasure) * n);
                    OLAP_TRY(t2.upload());
                    d_meas_drv = t2.ptr<UpMeasure>(o2);
                }
            }
            if (tile.use) {
                path = "drillup/tile";
                OLAP_TRY(launch_up_tile(d_meas_drv, meas.data(), n, csr.contiguous, d_ps, d_ch, O, C, P, I, tile));
            } else if (lanes.use) {
                path = "drillup/lanes";
                void* scratch = nullptr;
                if (lanes.SS > 1) OLAP_TRY(dev_alloc(&scratch, (size_t)lanes.scratch_stride * n));
                OLAP_TRY(launch_up_lanes(d_meas_drv, meas.data(), n, csr.contiguous, d_ps, d_ch,
                                         reinterpret_cast<const uint8_t*>(d_stat + o_map8), O, C, P, lanes,
                                         static_cast<unsigned char*>(scratch)));
                if (scratch) OLAP_TRY(dev_free(scratch));
            } else if (lng.use) {
                path = "drillup/long";
                void* scratch = nullptr;
                if (lng.SS > 1) OLAP_TRY(dev_alloc(&scratch, (size_t)lng.scratch_stride * n));
                OLAP_TRY(launch_up_long(d_meas, meas.data(), n, csr.contiguous, d_ps, d_ch,
                                        reinterpret_cast<const int32_t*>(d_stat + o_seg),
                                        csr.contiguous ? nullptr : reinterpret_cast<const uint16_t*>(d_stat + o_perm), O, C, P, I, lng,
                                        static_cast<unsigned char*>(scratch)));
                if (scratch) OLAP_TRY(dev_free(scratch));
            } else {
                path = (I % 4 == 0) ? "drillup/mid-vec4" : (I % 2 == 0 ? "drillup/mid-vec2" : "drillup/mid-scalar");
                OLAP_TRY(launch_up_mid(d_meas_drv, meas.data(), n, csr, d_ps, d_ch, O, C, P, I));
            }
        } else {
            path = "drillup/generic";
            UpGenParams p{};
            p.nd = ndim;
            p.n_out = new_size;
            std::vector<size_t> o_ps(ndim), o_ch(ndim);
            int64_t stride = 1;
            for (int d = ndim - 1; d >= 0; --d) {
                p.new_len[d] = new_len[d];
                p.old_stride[d] = stride;
                stride *= old_len[d];
                std::vector<int32_t> implied;
                if (!maps[d]) {  // untouched (identity) or rolled up to one item (zeros)
                    implied.assign(old_len[d], 0);
                    if (old_len[d] == new_len[d]) std::iota(implied.begin(), implied.end(), 0);
                }
                const Csr csr = build_csr(maps[d] ? maps[d] : implied.data(), old_len[d], new_len[d]);
                o_ps[d] = t.add(csr.pstart.data(), csr.pstart.size() * 4);
                o_ch[d] = t.add(csr.children.data(), csr.children.size() * 4);
            }
            OLAP_TRY(t.upload());
            p.meas = t.ptr<UpMeasure>(o_meas);
            for (int d = 0; d < ndim; ++d) { p.pstart[d] = t.ptr<int32_t>(o_ps[d]); p.children[d] = t.ptr<int32_t>(o_ch[d]); }
            const int64_t gx = ceil_div(new_size, 256);
            if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "olap_drill_up: grid too large");
            KERNELS_BEGIN();
            drillup_generic_kernel<<<dim3((unsigned)gx, (unsigned)n), 256, 0, g.stream>>>(p);
            LAUNCHED();
        }
        OLAP_TRY(t.release());
    }
    end_op(path);
    return guard.done(finish_op());
}

// ---- gather family ----------------------------------------------------------------------
namespace {

// COPY gathers of a store whose status plane follows from its values (olap_store::derived): the kernels that
// support it (vector gather, pair transpose) write the bytes from the cells they move and never read the plane
static void gather_derive(std::vector<GatherMeasure>& meas, olap_store* const* src, int n) {
    static const int knob = [] { const char* e = getenv("OLAP_DERIVE_STATUS"); return e ? atoi(e) : 1; }();
    if (!knob) return;
    for (int k = 0; k < n; ++k)
        if (meas[k].st_in && meas[k].st_out && src[k]->derived && !src[k]->shared_plane) {
            meas[k].st_in = nullptr;
            meas[k].derive = 1;
        }
}

// COPY gathers that only rearrange cells INSIDE contiguous blocks of the source (gather_inner_flat_kernel): the
// leading axes are untouched and merge into one linear "row" axis whose stride D is the block length, and every
// source offset of the trailing axes stays inside the block — dice / slice of the innermost axes, reorders that
// swap trailing axes (the 10 x 10 inner swap of config 3).  `dims` is in output order.  *done says whether the
// kernel was launched.
static int try_gather_flat(olap_store* const* src, int n, std::vector<GDim> dims, const std::vector<GatherMeasure>& meas_in,
                           bool* done, const char** path) {
    *done = false;
    static const int flat_knob = [] { const char* e = getenv("OLAP_FLAT"); return e ? atoi(e) : 1; }();
    if (!flat_knob) return OLAP_OK;
    const FlatPlan fp = flat_plan(std::move(dims), src[0]->size);
    if (!fp.use) return OLAP_OK;
    const bool front = fp.front;
    const int64_t const_off = fp.const_off, rows = fp.rows, D = fp.D, K = fp.K, RB = fp.RB;
    const std::vector<int32_t>& keep = fp.keep;
    for (int k = 0; k < n; ++k)  // wrapped memory may sit anywhere
        if ((reinterpret_cast<uintptr_t>(meas_in[k].in) & 15) || (reinterpret_cast<uintptr_t>(meas_in[k].st_in) & 15) ||
            (reinterpret_cast<uintptr_t>(meas_in[k].out) & 3) || (reinterpret_cast<uintptr_t>(meas_in[k].st_out) & 3))
            return OLAP_OK;
    FlatParams p{};
    TablePack t;
    std::vector<GatherMeasure> meas = meas_in;
    gather_derive(meas, src, n);
    bool any_plane = false;
    for (auto& m : meas) { m.in += const_off; if (m.st_in) m.st_in += const_off; any_plane |= m.st_in != nullptr; }
    const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
    const size_t o_keep = t.add(keep.data(), keep.size() * 4);
    OLAP_TRY(t.upload());
    p.meas = t.ptr<GatherMeasure>(o_meas);
    p.keep = t.ptr<int32_t>(o_keep);
    p.rows = rows;
    p.D = (uint32_t)D; p.K = (uint32_t)K; p.RB = (uint32_t)RB;
    p.div_k = FastDiv((uint32_t)K);
    p.div_rb = FastDiv((uint32_t)RB);
    const int64_t n_tiles = ceil_div(rows, RB);
    p.n_tiles = (uint32_t)n_tiles;
    const int64_t per_thread = ceil_div(RB * K, 256);
    const int per_sm = per_thread <= 16 ? 4 : 3;
    const int64_t gx = std::min<int64_t>(n_tiles, std::max<int64_t>(1, (int64_t)g.sm_count * per_sm / n));  // persistent CTAs
    const size_t smem = (size_t)RB * D * (any_plane ? 5 : 4);
    const dim3 grid((unsigned)gx, (unsigned)n);
    KERNELS_BEGIN();
    if (front) {
        if (per_thread <= 16) gather_inner_flat_kernel<16, 4, true><<<grid, 256, smem, g.stream>>>(p);
        else gather_inner_flat_kernel<32, 3, true><<<grid, 256, smem, g.stream>>>(p);
    } else if (per_thread <= 8) gather_inner_flat_kernel<8, 4, false><<<grid, 256, smem, g.stream>>>(p);
    else if (per_thread <= 16) gather_inner_flat_kernel<16, 4, false><<<grid, 256, smem, g.stream>>>(p);
    else gather_inner_flat_kernel<32, 3, false><<<grid, 256, smem, g.stream>>>(p);
    LAUNCHED();
    *path = front ? "gather/flat-to-front" : "gather/inner-flat";
    OLAP_TRY(t.release());
    *done = true;
    return OLAP_OK;
}

// [K, R] -> [R, K]: short outer axes of the source become the innermost axes of the output (gather_planes_flat_kernel).
// `dims` is in output order: the row axis comes first and is contiguous in the source.
static int try_gather_planes(olap_store* const* src, int n, std::vector<GDim> dims, const std::vector<GatherMeasure>& meas_in,
                             bool* done, const char** path) {
    *done = false;
    static const int knob = [] { const char* e = getenv("OLAP_FLAT"); return e ? atoi(e) : 1; }();
    if (!knob) return OLAP_OK;
    const PlanesPlan pl = planes_plan(std::move(dims), src[0]->size);
    if (!pl.use) return OLAP_OK;
    const int64_t rows = pl.rows, K = pl.K, RB = pl.RB;
    const std::vector<int64_t>& plane = pl.plane;
    for (int k = 0; k < n; ++k)  // wrapped memory may sit anywhere
        if ((reinterpret_cast<uintptr_t>(meas_in[k].in) & 15) || (reinterpret_cast<uintptr_t>(meas_in[k].st_in) & 3) ||
            (reinterpret_cast<uintptr_t>(meas_in[k].out) & 3))
            return OLAP_OK;
    PlanesParams p{};
    TablePack t;
    std::vector<GatherMeasure> meas = meas_in;
    gather_derive(meas, src, n);
    bool any_plane = false;
    for (auto& m : meas) any_plane |= m.st_in != nullptr;
    const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
    const size_t o_off = t.add(plane.data(), plane.size() * 8);
    OLAP_TRY(t.upload());
    p.meas = t.ptr<GatherMeasure>(o_meas);
    p.plane_off = t.ptr<int64_t>(o_off);
    p.rows = rows;
    p.K = (uint32_t)K; p.RB = (uint32_t)RB;
    p.div_k = FastDiv((uint32_t)K);
    p.div_rb4 = FastDiv((uint32_t)(RB / 4));
    const int64_t n_tiles = ceil_div(rows, RB);
    p.n_tiles = (uint32_t)n_tiles;
    const int64_t per_thread = RB * K / 256;
    const int per_sm = per_thread <= 16 ? 4 : 3;
    const int64_t gx = std::min<int64_t>(n_tiles, std::max<int64_t>(1, (int64_t)g.sm_count * per_sm / n));  // persistent CTAs
    const size_t smem = (size_t)K * (RB + 4) * (any_plane ? 5 : 4);
    const dim3 grid((unsigned)gx, (unsigned)n);
    KERNELS_BEGIN();
    if (per_thread <= 16) gather_planes_flat_kernel<16, 4><<<grid, 256, smem, g.stream>>>(p);
    else gather_planes_flat_kernel<32, 3><<<grid, 256, smem, g.stream>>>(p);
    LAUNCHED();
    *path = "gather/planes-to-inner";
    OLAP_TRY(t.release());
    *done = true;
    return OLAP_OK;
}

static int run_gather(int mode, olap_store* const* src, int n, std::vector<GDim>& dims, int64_t new_size, int64_t old_size,
                      const std::vector<GatherMeasure>& meas_in, int* d_error, const char** path) {
    if (mode == G_COPY) {
        bool done = false;
        OLAP_TRY(try_gather_flat(src, n, dims, meas_in, &done, path));
        if (done) return OLAP_OK;
    }
    int64_t const_off = 0;
    merge_dims(dims, &const_off);
    int64_t I = 1;
    if (!dims.empty() && dims.back().linear && dims.back().stride == 1 && dims.back().aux.empty()) {
        I = dims.back().len;
        dims.pop_back();
    }
    if ((int)dims.size() > OLAP_MAX_DIMS) return fail(OLAP_E_UNSUPPORTED, "too many dimensions");
    int VEC = (I % 4 == 0) ? 4 : 1;
    // scalar case: the amortised row kernel (innermost axis = short run or a table axis)
    static const int rows_knob = [] { const char* e = getenv("OLAP_ROWS"); return e ? atoi(e) : 1; }();
    if (VEC == 1 && rows_knob && (I > 1 || !dims.empty())) {
        GDim last;
        std::vector<GDim> outer = dims;
        if (I > 1) { last.len = I; last.linear = true; last.stride = 1; }
        else { last = outer.back(); outer.pop_back(); }
        int64_t rows = 1;
        bool fits = last.len <= kRowsMaxL && last.len >= 1;
        for (auto& d : outer) { rows *= d.len; fits &= d.len <= 0x7fffffffLL; }
        if (fits && rows < ((int64_t)1 << 31)) {
            GatherParams p{};
            RowsTail tail{};
            TablePack t;
            std::vector<GatherMeasure> meas = meas_in;
            for (auto& m : meas) { m.in += const_off; if (m.st_in) m.st_in += const_off; }
            const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
            std::vector<size_t> o_tbl(outer.size(), 0), o_aux(outer.size(), 0);
            for (size_t d = 0; d < outer.size(); ++d) {
                if (!outer[d].linear) o_tbl[d] = t.add(outer[d].tbl.data(), outer[d].tbl.size() * 8);
                if (!outer[d].aux.empty()) o_aux[d] = t.add(outer[d].aux.data(), outer[d].aux.size() * sizeof(DownAux));
            }
            const size_t o_ltbl = last.linear ? 0 : t.add(last.tbl.data(), last.tbl.size() * 8);
            const size_t o_laux = last.aux.empty() ? 0 : t.add(last.aux.data(), last.aux.size() * sizeof(DownAux));
            OLAP_TRY(t.upload());
            p.meas = t.ptr<GatherMeasure>(o_meas);
            p.nd = (int)outer.size();
            for (size_t d = 0; d < outer.size(); ++d) {
                p.len[d] = (uint32_t)outer[d].len;
                p.div[d] = FastDiv((uint32_t)outer[d].len);
                p.tbl[d] = outer[d].linear ? nullptr : t.ptr<int64_t>(o_tbl[d]);
                p.lin[d] = outer[d].stride;
                p.aux[d] = outer[d].aux.empty() ? nullptr : t.ptr<DownAux>(o_aux[d]);
            }
            p.new_size = new_size;
            p.old_size = old_size;
            p.error_flag = d_error;
            tail.L = (uint32_t)last.len;
            tail.div_l = FastDiv((uint32_t)last.len);
            tail.tbl = last.linear ? nullptr : t.ptr<int64_t>(o_ltbl);
            tail.lin = last.stride;
            tail.aux = last.aux.empty() ? nullptr : t.ptr<DownAux>(o_laux);
            tail.RB = (uint32_t)std::max<int64_t>(1, std::min<int64_t>(kRowsPerBlock, 4096 / last.len));
            tail.rows = rows;
            const int64_t gx = ceil_div(rows, tail.RB);
            if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "grid too large");
            dim3 grid((unsigned)gx, (unsigned)n);
            KERNELS_BEGIN();
            if (mode == G_COPY) gather_rows_kernel<G_COPY><<<grid, 256, 0, g.stream>>>(p, tail);
            else if (mode == G_DOWN_FLOAT) gather_rows_kernel<G_DOWN_FLOAT><<<grid, 256, 0, g.stream>>>(p, tail);
            else gather_rows_kernel<G_DOWN><<<grid, 256, 0, g.stream>>>(p, tail);
            LAUNCHED();
            *path = "gather/rows";
            OLAP_TRY(t.release());
            return OLAP_OK;
        }
    }
    // every offset must keep 16-byte alignment for the 128-bit path
    if (VEC == 4) {
        if (const_off % 4) VEC = 1;
        for (auto& d : dims) {
            if (d.linear) { if (d.stride % 4) VEC = 1; }
            else for (int64_t v : d.tbl) if (v % 4) { VEC = 1; break; }
        }
    }
    GatherParams p{};
    TablePack t;
    std::vector<GatherMeasure> meas = meas_in;
    if (mode == G_COPY) gather_derive(meas, src, n);
    for (auto& m : meas) { m.in += const_off; if (m.st_in) m.st_in += const_off; }
    const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
    std::vector<size_t> o_tbl(dims.size(), 0), o_aux(dims.size(), 0);
    int64_t rows = 1;
    bool big = false;
    for (size_t d = 0; d < dims.size(); ++d) {
        if (dims[d].len > 0x7fffffffLL) {
            if (!dims[d].linear) return fail(OLAP_E_UNSUPPORTED, "dimension longer than 2^31-1");
            big = true;
        }
        if (!dims[d].linear) o_tbl[d] = t.add(dims[d].tbl.data(), dims[d].tbl.size() * 8);
        if (!dims[d].aux.empty()) o_aux[d] = t.add(dims[d].aux.data(), dims[d].aux.size() * sizeof(DownAux));
        rows *= dims[d].len;
    }
    OLAP_TRY(t.upload());
    p.meas = t.ptr<GatherMeasure>(o_meas);
    p.nd = (int)dims.size();
    for (size_t d = 0; d < dims.size(); ++d) {
        p.len[d] = (uint32_t)dims[d].len;
        p.div[d] = FastDiv((uint32_t)dims[d].len);
        p.tbl[d] = dims[d].linear ? nullptr : t.ptr<int64_t>(o_tbl[d]);
        p.lin[d] = dims[d].stride;
        p.aux[d] = dims[d].aux.empty() ? nullptr : t.ptr<DownAux>(o_aux[d]);
        p.n_aux += dims[d].aux.empty() ? 0 : 1;
    }
    p.I = I;
    const int64_t IV = I / VEC;
    if (IV > 0x7fffffffLL) big = true;
    p.IV = (uint32_t)IV;
    p.div_iv = FastDiv((uint32_t)IV);
    p.rows = rows;
    p.n_vec = rows * IV;
    if (p.n_vec >= ((int64_t)1 << 31) || rows >= ((int64_t)1 << 31)) big = true;
    if (big && (IV > 0xffffffffLL)) return fail(OLAP_E_UNSUPPORTED, "inner run too long");
    if (big) {
        for (size_t d = 0; d < dims.size(); ++d)
            if (dims[d].len > 0xffffffffLL) return fail(OLAP_E_UNSUPPORTED, "merged dimension longer than 2^32-1");
        p.IV = (uint32_t)IV;
    }
    p.new_size = new_size;
    p.old_size = old_size;
    p.error_flag = d_error;
    const int64_t gx = ceil_div(p.n_vec, 512);
    if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "grid too large");
    dim3 grid((unsigned)gx, (unsigned)n);
    KERNELS_BEGIN();
#define OLAP_GATHER(M, V, B) gather_kernel<M, V, B><<<grid, 256, 0, g.stream>>>(p)
#define OLAP_GATHER_VB(M)                                                                      \
    do {                                                                                       \
        if (VEC == 4) { if (big) OLAP_GATHER(M, 4, true); else OLAP_GATHER(M, 4, false); }     \
        else { if (big) OLAP_GATHER(M, 1, true); else OLAP_GATHER(M, 1, false); }              \
    } while (0)
    if (mode == G_COPY) OLAP_GATHER_VB(G_COPY);
    else if (mode == G_DOWN_FLOAT) OLAP_GATHER_VB(G_DOWN_FLOAT);
    else OLAP_GATHER_VB(G_DOWN);
#undef OLAP_GATHER_VB
#undef OLAP_GATHER
    LAUNCHED();
    *path = VEC == 4 ? (big ? "gather/vec4-big" : "gather/vec4") : (big ? "gather/scalar-big" : "gather/scalar");
    OLAP_TRY(t.release());
    return OLAP_OK;
}

static std::vector<GatherMeasure> gather_measures(olap_store* const* src, olap_store** out, int n) {
    std::vector<GatherMeasure> meas(n);
    for (int k = 0; k < n; ++k) {
        GatherMeasure m{};
        m.in = src[k]->values;
        m.out = out[k]->values;
        m.st_out = out[k]->status && src[k]->status ? st_out_of(out, k) : nullptr;
        m.st_in = m.st_out ? src[k]->status : nullptr;
        m.nan_default = src[k]->default_kind;
        m.int_rounding = src[k]->type == OLAP_INT32 || src[k]->type == OLAP_UINT32;
        m.method_is_sum = 1;
        meas[k] = m;
    }
    return meas;
}

}  // namespace

int olap_dice(olap_store* const* src, int n, int ndim, const int64_t* old_len, const int64_t* new_len,
              const int32_t* const* keep, olap_store** out) {
    int64_t size = 0, old_size = 0, new_size = 0;
    OLAP_TRY(check_batch(src, n, "olap_dice", &size));
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "olap_dice: at most %d dimensions", OLAP_MAX_DIMS);
    if (!out || (ndim && (!old_len || !new_len || !keep))) return fail(OLAP_E_INVALID, "olap_dice: null argument");
    OLAP_TRY(product(old_len, ndim, &old_size, "olap_dice"));
    OLAP_TRY(product(new_len, ndim, &new_size, "olap_dice"));
    if (old_size != size) return fail(OLAP_E_INVALID, "olap_dice: dimensions describe %lld cells, store has %lld", (long long)old_size, (long long)size);
    std::vector<GDim> dims(ndim);
    int64_t stride = 1;
    for (int d = ndim - 1; d >= 0; --d) {
        GDim& g_ = dims[d];
        g_.len = new_len[d];
        bool identity = new_len[d] == old_len[d];
        for (int64_t j = 0; j < new_len[d]; ++j) {
            const int32_t o = keep[d][j];
            if (o < 0 || o >= old_len[d]) return fail(OLAP_E_INVALID, "olap_dice: dimension %d keeps item %d, outside [0, %lld)", d, o, (long long)old_len[d]);
            identity &= o == j;
        }
        if (identity) { g_.linear = true; g_.stride = stride; }
        else {
            g_.linear = false;
            g_.tbl.resize(new_len[d]);
            for (int64_t j = 0; j < new_len[d]; ++j) g_.tbl[j] = (int64_t)keep[d][j] * stride;
        }
        stride *= old_len[d];
    }
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_like(src, n, new_size, out));
    OutGuard guard(out, n);
    begin_op();
    const char* path = "dice/empty";
    for (int k = 0; k < n; ++k) set_derived(out[k], is_derived(src[k]));  // a gather copies value and status together
    if (new_size) {
        auto meas = gather_measures(src, out, n);
        OLAP_TRY(run_gather(G_COPY, src, n, dims, new_size, old_size, meas, nullptr, &path));
    }
    end_op(path);
    return guard.done(finish_op());
}

int olap_reorder(olap_store* const* src, int n, int ndim, const int64_t* old_len, const int32_t* new_to_old,
                 olap_store** out) {
    int64_t size = 0, old_size = 0;
    OLAP_TRY(check_batch(src, n, "olap_reorder", &size));
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "olap_reorder: at most %d dimensions", OLAP_MAX_DIMS);
    if (!out || (ndim && (!old_len || !new_to_old))) return fail(OLAP_E_INVALID, "olap_reorder: null argument");
    OLAP_TRY(product(old_len, ndim, &old_size, "olap_reorder"));
    if (old_size != size) return fail(OLAP_E_INVALID, "olap_reorder: dimensions describe %lld cells, store has %lld", (long long)old_size, (long long)size);
    std::vector<int64_t> old_stride(ndim);
    int64_t stride = 1;
    for (int d = ndim - 1; d >= 0; --d) { old_stride[d] = stride; stride *= old_len[d]; }
    std::vector<bool> seen(ndim, false);
    std::vector<GDim> dims(ndim);
    for (int i = 0; i < ndim; ++i) {
        const int o = new_to_old[i];
        if (o < 0 || o >= ndim || seen[o]) return fail(OLAP_E_INVALID, "olap_reorder: new_to_old is not a permutation");
        seen[o] = true;
        dims[i].len = old_len[o];
        dims[i].linear = true;
        dims[i].stride = old_stride[o];
    }
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_like(src, n, size, out));
    OutGuard guard(out, n);
    begin_op();
    const char* path = "reorder/empty";
    for (int k = 0; k < n; ++k) set_derived(out[k], is_derived(src[k]));
    if (size) {
        auto meas = gather_measures(src, out, n);
        TmaPlan tm = transpose_tma_plan(dims);
        if (tm.use && !tma_encode_fn()) tm.use = false;  // a driver without cuTensorMapEncodeTiled
        PairPlan pp;
        if (!tm.use) pp = transpose_pair_plan(dims);
        bool flat_done = false;
        if (!tm.use && !pp.use) OLAP_TRY(try_gather_flat(src, n, dims, meas, &flat_done, &path));  // trailing axes swapped inside short blocks
        if (!tm.use && !pp.use && !flat_done) OLAP_TRY(try_gather_planes(src, n, dims, meas, &flat_done, &path));  // short outer axes rotated to innermost
        TransposePlan tp;
        if (!tm.use && !pp.use && !flat_done) tp = transpose_plan(dims);
        if (flat_done) {
        } else if (tm.use) {
            path = "reorder/tma-transpose";
            std::vector<CUtensorMap> maps;
            OLAP_TRY(tma_encode_maps(tm, meas, maps));
            TablePack t;
            const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
            const size_t o_src = t.add(tm.pair.src_row.data(), tm.pair.src_row.size() * sizeof(uint32_t));
            const size_t o_dst = t.add(tm.pair.dst_row.data(), tm.pair.dst_row.size() * sizeof(uint32_t));
            const size_t o_maps = t.add(maps.data(), maps.size() * sizeof(CUtensorMap), 64);
            OLAP_TRY(t.upload());
            OLAP_TRY(launch_transpose_tma(t.ptr<GatherMeasure>(o_meas), t.ptr<uint32_t>(o_src), t.ptr<uint32_t>(o_dst),
                                          t.ptr<CUtensorMap>(o_maps), n, tm));
            OLAP_TRY(t.release());
        } else if (pp.use) {
            path = "reorder/pair-transpose";
            if (pp.p.split == 1) gather_derive(meas, src, n);  // the 2-CTA cluster variant always stages the status bytes
            bool loaded = false;
            for (int k = 0; k < n; ++k) loaded |= meas[k].st_in != nullptr;
            const bool async = transpose_async_fits(pp, loaded);
            if (async) path = "reorder/pair-async";
            TablePack t;
            const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
            const size_t o_src = t.add(pp.src_row.data(), pp.src_row.size() * sizeof(uint32_t));
            const size_t o_dst = t.add(pp.dst_row.data(), pp.dst_row.size() * sizeof(uint32_t));
            OLAP_TRY(t.upload());
            if (async) OLAP_TRY(launch_transpose_async(t.ptr<GatherMeasure>(o_meas), t.ptr<uint32_t>(o_src), t.ptr<uint32_t>(o_dst), n, pp, loaded));
            else OLAP_TRY(launch_transpose_pair(t.ptr<GatherMeasure>(o_meas), t.ptr<uint32_t>(o_src), t.ptr<uint32_t>(o_dst), n, pp));
            OLAP_TRY(t.release());
        } else if (tp.use) {
            path = "reorder/box-transpose";
            gather_derive(meas, src, n);
            TablePack t;
            const size_t o_meas = t.add(meas.data(), sizeof(GatherMeasure) * n);
            const size_t o_rd = t.add(tp.rd_tab.data(), tp.rd_tab.size() * sizeof(uint2));
            const size_t o_wr = t.add(tp.wr_tab.data(), tp.wr_tab.size() * sizeof(uint2));
            OLAP_TRY(t.upload());
            bool derive_all = true;  // no measure moves a loaded status plane
            for (int k = 0; k < n; ++k) derive_all &= meas[k].st_in == nullptr;
            OLAP_TRY(launch_transpose(derive_all, t.ptr<GatherMeasure>(o_meas), t.ptr<uint2>(o_rd), t.ptr<uint2>(o_wr), n, tp));
            OLAP_TRY(t.release());
        } else {
            OLAP_TRY(run_gather(G_COPY, src, n, dims, size, size, meas, nullptr, &path));
        }
    }
    end_op(path);
    return guard.done(finish_op());
}

int olap_drill_down(olap_store* const* src, int n, const int* methods, int ndim, const int64_t* old_len,
                    const int64_t* new_len, const int32_t* const* maps, const double* const* dist,
                    const int64_t* dist_len, olap_store** out) {
    int64_t size = 0, old_size = 0, new_size = 0;
    OLAP_TRY(check_batch(src, n, "olap_drill_down", &size));
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "olap_drill_down: at most %d dimensions", OLAP_MAX_DIMS);
    if (!out || (ndim && (!old_len || !new_len || !maps))) return fail(OLAP_E_INVALID, "olap_drill_down: null argument");
    OLAP_TRY(product(old_len, ndim, &old_size, "olap_drill_down"));
    OLAP_TRY(product(new_len, ndim, &new_size, "olap_drill_down"));
    if (old_size != size) return fail(OLAP_E_INVALID, "olap_drill_down: dimensions describe %lld cells, store has %lld", (long long)old_size, (long long)size);
    std::vector<GDim> dims(ndim);
    std::vector<int> changed;
    int64_t inner_of_changed = 1;
    int64_t stride = 1;
    for (int d = ndim - 1; d >= 0; --d) {
        GDim& g_ = dims[d];
        g_.len = new_len[d];
        bool identity = new_len[d] == old_len[d];
        for (int64_t j = 0; j < new_len[d]; ++j) {
            const int32_t o = maps[d][j];
            if (o < 0 || o >= old_len[d]) return fail(OLAP_E_INVALID, "olap_drill_down: map of dimension %d sends item %lld to %d, outside [0, %lld)", d, (long long)j, o, (long long)old_len[d]);
            identity &= o == j;
        }
        if (identity) { g_.linear = true; g_.stride = stride; }
        else {
            changed.push_back(d);
            inner_of_changed = stride;  // product of the (old == new) lengths after d when d is the only change
            g_.linear = false;
            g_.tbl.resize(new_len[d]);
            g_.aux.resize(new_len[d]);
            std::vector<int32_t> count(old_len[d], 0);
            for (int64_t j = 0; j < new_len[d]; ++j) {
                g_.tbl[j] = (int64_t)maps[d][j] * stride;
                g_.aux[j].rank = count[maps[d][j]]++;  // rank among siblings, ascending new index
            }
            for (int64_t j = 0; j < new_len[d]; ++j) {
                g_.aux[j].cnt = count[maps[d][j]];
                g_.aux[j].inv = 1.0 / (double)g_.aux[j].cnt;
            }
        }
        stride *= old_len[d];
    }
    bool any_dist = false;
    for (int k = 0; k < n; ++k) any_dist |= dist && dist[k];
    if (any_dist && (old_size == 0 || new_size % old_size != 0)) return fail(OLAP_E_INVALID, "olap_drill_down: distributions need newSize to be a multiple of oldSize");
    bool any_int_sum = false;
    for (int k = 0; k < n; ++k)
        any_int_sum |= (src[k]->type == OLAP_INT32 || src[k]->type == OLAP_UINT32) && (methods ? methods[k] == OLAP_SUM : true);
    int64_t O_changed = 1;  // cells in front of the changed dimension when there is one
    for (int q = 0; changed.size() == 1 && q < changed[0]; ++q) O_changed *= old_len[q];
    const bool block = new_size && !any_dist && changed.size() == 1 &&
                       down_block_fits(O_changed, old_len[changed[0]], new_len[changed[0]], inner_of_changed, any_int_sum);
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_like(src, n, new_size, out));
    OutGuard guard(out, n);
    begin_op();
    const char* path = "drilldown/empty";
    int rc = OLAP_OK;
    if (new_size && old_size == 0) {
        for (int k = 0; k < n; ++k) { olap_store t = *out[k]; t.status = st_out_of(out, k); OLAP_TRY(fill_default(&t)); }
    } else if (new_size && !any_dist && changed.size() == 1 && !block &&
               ((inner_of_changed % 4 == 0 && inner_of_changed >= 32) || (inner_of_changed % 2 == 0 && inner_of_changed >= 64) ||
                inner_of_changed >= 128)) {
        // one changed dimension with a long inner run: parent-driven kernel
        const int d = changed[0];
        int64_t O = 1;
        for (int q = 0; q < d; ++q) O *= old_len[q];
        // CSR parent -> new items: build from the new->old map
        const Csr csr = build_csr(maps[d], new_len[d], old_len[d]);
        std::vector<DownMeasure> dm(n);
        for (int k = 0; k < n; ++k) {
            const bool is_int = src[k]->type == OLAP_INT32 || src[k]->type == OLAP_UINT32;
            const bool is_sum = methods ? methods[k] == OLAP_SUM : true;
            uint8_t* so = out[k]->status && src[k]->status ? st_out_of(out, k) : nullptr;
            dm[k] = DownMeasure{src[k]->values, out[k]->values, so ? src[k]->status : nullptr, so,
                                src[k]->default_kind, !is_sum ? 1 : (is_int ? 2 : 0)};
        }
        TablePack t;
        const size_t o_meas = t.add(dm.data(), sizeof(DownMeasure) * n);
        const size_t o_ps = t.add(csr.pstart.data(), csr.pstart.size() * 4);
        const size_t o_ch = t.add(csr.children.data(), csr.children.size() * 4);
        OLAP_TRY(t.upload());
        path = inner_of_changed % 4 == 0 ? "drilldown/mid-vec4" : (inner_of_changed % 2 == 0 ? "drilldown/mid-vec2" : "drilldown/mid-scalar");
        int kind = dm[0].kind;  // the kind all measures share, or -1
        for (int k = 1; k < n; ++k) if (dm[k].kind != kind) kind = -1;
        OLAP_TRY(launch_down_mid(t.ptr<DownMeasure>(o_meas), n, csr, t.ptr<int32_t>(o_ps), t.ptr<int32_t>(o_ch), O,
                                 old_len[d], new_len[d], inner_of_changed, kind));
        OLAP_TRY(t.release());
    } else if (block) {
        // the drilled dimension is the innermost one, or the run behind it is short: block kernel,
        // parents staged in shared memory, output written front to back with 128-bit stores
        const int d = changed[0];
        int64_t O = 1;
        for (int q = 0; q < d; ++q) O *= old_len[q];
        const int64_t P = old_len[d], C = new_len[d];
        std::vector<int32_t> rank(C), cnt(P, 0);
        for (int64_t j = 0; j < C; ++j) rank[j] = cnt[maps[d][j]]++;
        std::vector<DownMeasure> dm(n);
        for (int k = 0; k < n; ++k) {
            const bool is_int = src[k]->type == OLAP_INT32 || src[k]->type == OLAP_UINT32;
            const bool is_sum = methods ? methods[k] == OLAP_SUM : true;
            uint8_t* so = out[k]->status && src[k]->status ? st_out_of(out, k) : nullptr;
            dm[k] = DownMeasure{src[k]->values, out[k]->values, so ? src[k]->status : nullptr, so,
                                src[k]->default_kind, !is_sum ? 1 : (is_int ? 2 : 0)};
        }
        TablePack t;
        const size_t o_meas = t.add(dm.data(), sizeof(DownMeasure) * n);
        const size_t o_par = t.add(maps[d], (size_t)C * 4);
        const size_t o_rank = t.add(rank.data(), (size_t)C * 4);
        const size_t o_cnt = t.add(cnt.data(), (size_t)P * 4);
        OLAP_TRY(t.upload());
        path = inner_of_changed == 1 ? "drilldown/inner-rows" : "drilldown/block-rows";
        OLAP_TRY(launch_down_inner(t.ptr<DownMeasure>(o_meas), n, t.ptr<int32_t>(o_par), t.ptr<int32_t>(o_rank),
                                   t.ptr<int32_t>(o_cnt), O, P, C, inner_of_changed));
        OLAP_TRY(t.release());
    } else if (new_size) {
        auto meas = gather_measures(src, out, n);
        TablePack dpack;
        std::vector<size_t> o_dist(n, 0);
        if (any_dist) {
            int zero = 0;
            dpack.add(&zero, 4);  // error flag at offset 0
            for (int k = 0; k < n; ++k)
                if (dist[k]) o_dist[k] = dpack.add(dist[k], (size_t)dist_len[k] * 8);
            OLAP_TRY(dpack.upload());
        }
        for (int k = 0; k < n; ++k) {
            meas[k].method_is_sum = methods ? (methods[k] == OLAP_SUM) : 1;
            if (any_dist && dist[k]) { meas[k].dist = dpack.ptr<double>(o_dist[k]); meas[k].dist_len = dist_len[k]; }
        }
        bool fast = !any_dist;
        for (int k = 0; k < n; ++k) fast &= meas[k].method_is_sum && !meas[k].int_rounding;
        rc = run_gather(fast ? G_DOWN_FLOAT : G_DOWN, src, n, dims, new_size, old_size, meas,
                        any_dist ? dpack.ptr<int>(0) : nullptr, &path);
        if (rc == OLAP_OK && any_dist) {
            int flag = 0;
            OLAP_CUDA(cudaMemcpyAsync(&flag, dpack.ptr<int>(0), 4, cudaMemcpyDeviceToHost, g.stream));
            OLAP_CUDA(cudaStreamSynchronize(g.stream));
            if (flag) rc = fail(OLAP_E_INVALID, "distribution missing for index %d", flag - 1);
        }
        if (any_dist) OLAP_TRY(dpack.release());
    }
    end_op(path);
    if (rc != OLAP_OK) return rc;  // the guard destroys the results
    return guard.done(finish_op());
}

int olap_load(olap_store* dst, const olap_store* src, int ndim, const int64_t* my_len, const int64_t* his_len,
              const int32_t* const* his_to_mine) {
    if (!dst || !src) return fail(OLAP_E_INVALID, "olap_load: null store");
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "olap_load: at most %d dimensions", OLAP_MAX_DIMS);
    int64_t my_size = 0, his_size = 0;
    OLAP_TRY(product(my_len, ndim, &my_size, "olap_load"));
    OLAP_TRY(product(his_len, ndim, &his_size, "olap_load"));
    if (my_size != dst->size || his_size != src->size) return fail(OLAP_E_INVALID, "olap_load: dimensions do not match the stores");
    OLAP_TRY(ensure_ctx());
    begin_op();
    dst->derived = dst->derived && is_derived(src);  // set cells take the other store's flags (README.md:704)
    // Trailing axes that both stores have in full and in the same order (his item j -> my item j) are ONE contiguous
    // run on both sides: fold them into a single innermost axis (identity, no table) so that the vectorised scatter
    // moves the run with 128-bit accesses (hydrateFromCube of cubes that differ in their outer dimensions only)
    std::vector<int64_t> my_len_m(my_len, my_len + ndim), his_len_m(his_len, his_len + ndim);
    std::vector<const int32_t*> maps_m(his_to_mine, his_to_mine + ndim);
    int64_t id_run = 0;  // > 0: the (folded) innermost axis is the identity over id_run cells
    if (his_size && my_size && his_size < ((int64_t)1 << 31)) {  // the vectorised scatter below takes these
        int64_t run = 1;
        int k = 0;
        while (ndim - k >= 1) {
            const int L = ndim - 1 - k;
            bool identity = my_len_m[L] == his_len_m[L] && his_len_m[L] > 0 && run * his_len_m[L] < ((int64_t)1 << 31);
            for (int64_t j = 0; j < his_len_m[L] && identity; ++j) identity = maps_m[L][j] == (int32_t)j;
            if (!identity) break;
            run *= his_len_m[L];
            ++k;
        }
        if (k >= 2) {
            ndim -= k - 1;
            my_len_m[ndim - 1] = his_len_m[ndim - 1] = run;
            maps_m[ndim - 1] = nullptr;
            id_run = run;
        }
    }
    my_len = my_len_m.data();
    his_len = his_len_m.data();
    his_to_mine = maps_m.data();
    bool fast = false;
    if (his_size && my_size && ndim >= 1 && his_size < ((int64_t)1 << 31)) {
        // innermost axis: his item j -> my item m0 + j ?  then runs stay contiguous
        const int L = ndim - 1;
        bool linear = his_len[L] > 0;
        const int32_t first = id_run ? 0 : (his_len[L] > 0 ? his_to_mine[L][0] : 0);
        if (!id_run)
            for (int64_t j = 0; j < his_len[L] && linear; ++j) linear = his_to_mine[L][j] >= 0 && his_to_mine[L][j] == first + (int32_t)j;
        if (linear && first + his_len[L] > my_len[L]) return fail(OLAP_E_INVALID, "olap_load: item index outside [0, %lld)", (long long)my_len[L]);
        const int64_t I = linear ? his_len[L] : 1;
        const int nd = linear ? ndim - 1 : ndim;
        const int VEC = (linear && I % 4 == 0 && first % 4 == 0 && my_len[L] % 4 == 0) ? 4 : 1;
        bool ok = true;
        for (int d = 0; d < nd; ++d) ok &= his_len[d] <= 0x7fffffffLL;
        if (ok) {
            ScatterVecParams p{};
            TablePack t;
            std::vector<size_t> offs(nd);
            int64_t stride = linear ? my_len[L] : 1;
            for (int d = nd - 1; d >= 0; --d) {
                std::vector<int64_t> tbl(his_len[d]);
                for (int64_t j = 0; j < his_len[d]; ++j) {
                    const int32_t m = his_to_mine[d][j];
                    if (m >= my_len[d]) return fail(OLAP_E_INVALID, "olap_load: item index %d outside [0, %lld)", m, (long long)my_len[d]);
                    tbl[j] = m < 0 ? INT64_MIN / 32 : (int64_t)m * stride;
                }
                offs[d] = t.add(tbl.data(), tbl.size() * 8);
                p.len[d] = (uint32_t)his_len[d];
                p.div[d] = FastDiv((uint32_t)his_len[d]);
                stride *= my_len[d];
            }
            OLAP_TRY(t.upload());
            for (int d = 0; d < nd; ++d) p.tbl[d] = t.ptr<int64_t>(offs[d]);
            p.src = src->values; p.dst = dst->values;
            p.st_src = src->status; p.st_dst = dst->status;
            p.dst_nan_default = dst->default_kind;
            p.nd = nd;
            p.IV = (uint32_t)(I / VEC);
            p.div_iv = FastDiv(p.IV);
            p.inner_off = linear ? first : 0;
            p.n_vec = (uint32_t)(his_size / VEC);
            const int64_t gx = ceil_div((int64_t)p.n_vec, 256);
            KERNELS_BEGIN();
            if (VEC == 4) load_scatter_vec_kernel<4><<<(unsigned)gx, 256, 0, g.stream>>>(p);
            else load_scatter_vec_kernel<1><<<(unsigned)gx, 256, 0, g.stream>>>(p);
            LAUNCHED();
            OLAP_TRY(t.release());
            fast = true;
            end_op(VEC == 4 ? "load/scatter-vec4" : "load/scatter-rows");
        }
    }
    if (fast) return finish_op();
    if (his_size && my_size) {
        ScatterParams p{};
        TablePack t;
        std::vector<size_t> offs(ndim);
        int64_t stride = 1;
        for (int d = ndim - 1; d >= 0; --d) {
            std::vector<int64_t> tbl(his_len[d]);
            for (int64_t j = 0; j < his_len[d]; ++j) {
                const int32_t m = his_to_mine[d][j];
                if (m >= my_len[d]) return fail(OLAP_E_INVALID, "olap_load: item index %d outside [0, %lld)", m, (long long)my_len[d]);
                tbl[j] = m < 0 ? INT64_MIN / 32 : (int64_t)m * stride;
            }
            offs[d] = t.add(tbl.data(), tbl.size() * 8);
            p.len[d] = his_len[d];
            stride *= my_len[d];
        }
        OLAP_TRY(t.upload());
        for (int d = 0; d < ndim; ++d) p.tbl[d] = t.ptr<int64_t>(offs[d]);
        p.src = src->values; p.dst = dst->values;
        p.st_src = src->status; p.st_dst = dst->status;
        p.dst_nan_default = dst->default_kind; p.src_nan_default = src->default_kind;
        p.nd = ndim; p.n = his_size;
        const int64_t gx = ceil_div(his_size, 256);
        if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "olap_load: grid too large");
        KERNELS_BEGIN();
        load_scatter_kernel<<<(unsigned)gx, 256, 0, g.stream>>>(p);
        LAUNCHED();
        OLAP_TRY(t.release());
    }
    end_op("load/scatter");
    return finish_op();
}

// ---- region queries: getTotalForDimensionItems / copyMeasureData -------------------------
namespace {

// The region keep[0] x ... x keep[ndim-1] of a store of len[0] x ... x len[ndim-1] cells, lowered like a
// dice (olap_dice): an identity list becomes a stride, any other list an int64 offset table; one-item axes
// fold into a constant offset, whole neighbours merge, and the trailing whole axes form the inner run.
struct RegionPlan {
    std::vector<GDim> dims;   // outer axes (tables or strides)
    int64_t const_off = 0, I = 1, cells = 0;
};

static int plan_region(const char* what, int64_t size, int ndim, const int64_t* len, const int64_t* keep_len,
                       const int32_t* const* keep, RegionPlan* plan) {
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "%s: at most %d dimensions", what, OLAP_MAX_DIMS);
    if (ndim && !len) return fail(OLAP_E_INVALID, "%s: null argument", what);
    int64_t total = 0;
    OLAP_TRY(product(len, ndim, &total, what));
    if (total != size) return fail(OLAP_E_INVALID, "%s: dimensions describe %lld cells, store has %lld", what, (long long)total, (long long)size);
    std::vector<int64_t> n(ndim);
    for (int d = 0; d < ndim; ++d) {
        const bool whole = !keep || !keep[d];
        if (!whole && (!keep_len || keep_len[d] < 0)) return fail(OLAP_E_INVALID, "%s: dimension %d has no list length", what, d);
        n[d] = whole ? len[d] : keep_len[d];
    }
    OLAP_TRY(product(n.data(), ndim, &plan->cells, what));
    plan->dims.assign(ndim, GDim{});
    int64_t stride = 1;
    for (int d = ndim - 1; d >= 0; --d) {
        GDim& g_ = plan->dims[d];
        g_.len = n[d];
        bool identity = n[d] == len[d];
        if (keep && keep[d])
            for (int64_t j = 0; j < n[d]; ++j) {
                const int32_t o = keep[d][j];
                if (o < 0 || o >= len[d]) return fail(OLAP_E_INVALID, "%s: dimension %d lists item %d, outside [0, %lld)", what, d, o, (long long)len[d]);
                identity &= o == j;
            }
        if (identity) { g_.linear = true; g_.stride = stride; }
        else {
            g_.linear = false;
            g_.tbl.resize(n[d]);
            for (int64_t j = 0; j < n[d]; ++j) g_.tbl[j] = (int64_t)keep[d][j] * stride;
        }
        stride *= len[d];
    }
    if (plan->cells == 0) return OLAP_OK;
    merge_dims(plan->dims, &plan->const_off);
    if (!plan->dims.empty() && plan->dims.back().linear && plan->dims.back().stride == 1) {
        plan->I = plan->dims.back().len;
        plan->dims.pop_back();
    }
    if ((int)plan->dims.size() > OLAP_MAX_DIMS) return fail(OLAP_E_UNSUPPORTED, "%s: too many dimensions", what);
    for (auto& d : plan->dims)
        if (d.len > 0xffffffffLL) return fail(OLAP_E_UNSUPPORTED, "%s: merged dimension longer than 2^32-1", what);
    return OLAP_OK;
}

// 128-bit accesses when the inner run, every offset and the planes allow them
static int region_vec(const RegionPlan& plan, const void* a, const void* b, const void* st) {
    if (plan.I % 4 || plan.const_off % 4) return 1;
    if ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) return 1;
    if (reinterpret_cast<uintptr_t>(st) & 3) return 1;
    for (auto& d : plan.dims) {
        if (d.linear) { if (d.stride % 4) return 1; }
        else for (int64_t v : d.tbl) if (v % 4) return 1;
    }
    return 4;
}

// Tables to the device, index fields of p.ix; returns the grid
static int region_params(const RegionPlan& plan, int VEC, TablePack& t, RegionParams& p) {
    std::vector<size_t> o_tbl(plan.dims.size(), 0);
    int64_t rows = 1;
    for (size_t d = 0; d < plan.dims.size(); ++d) {
        if (!plan.dims[d].linear) o_tbl[d] = t.add(plan.dims[d].tbl.data(), plan.dims[d].tbl.size() * 8);
        rows *= plan.dims[d].len;
    }
    OLAP_TRY(t.upload());
    GatherParams& q = p.ix;
    q.nd = (int)plan.dims.size();
    for (size_t d = 0; d < plan.dims.size(); ++d) {
        q.len[d] = (uint32_t)plan.dims[d].len;
        q.div[d] = FastDiv((uint32_t)plan.dims[d].len);
        q.tbl[d] = plan.dims[d].linear ? nullptr : t.ptr<int64_t>(o_tbl[d]);
        q.lin[d] = plan.dims[d].stride;
    }
    const int64_t IV = plan.I / VEC;
    q.I = plan.I;
    q.rows = rows;
    q.n_vec = rows * IV;
    p.big = q.n_vec >= ((int64_t)1 << 31) || IV > 0xffffffffLL;
    for (auto& d : plan.dims) p.big |= d.len >= ((int64_t)1 << 31);
    if (IV > 0xffffffffLL) return fail(OLAP_E_UNSUPPORTED, "region: inner run too long");
    q.IV = (uint32_t)IV;
    q.div_iv = FastDiv(p.big ? 1u : (uint32_t)IV);
    return OLAP_OK;
}

}  // namespace

int olap_region_sum(const olap_store* s, int ndim, const int64_t* len, const int64_t* keep_len,
                    const int32_t* const* keep, double* out) {
    if (!s || !out) return fail(OLAP_E_INVALID, "olap_region_sum: null argument");
    RegionPlan plan;
    OLAP_TRY(plan_region("olap_region_sum", s->size, ndim, len, keep_len, keep, &plan));
    OLAP_TRY(ensure_ctx());
    *out = 0.0;
    begin_op();
    if (plan.cells == 0) {
        end_op("region/sum");
        return finish_op();
    }
    const int VEC = region_vec(plan, s->values + plan.const_off, s->values + plan.const_off, nullptr);
    RegionParams p{};
    TablePack t;
    OLAP_TRY(region_params(plan, VEC, t, p));
    const int blocks = grid_for(p.ix.n_vec, 256);
    void* scratch;
    OLAP_TRY(dev_alloc(&scratch, (size_t)blocks * 8 + 16));
    p.src = s->values + plan.const_off;
    p.partial = static_cast<double*>(scratch);
    p.out = p.partial + blocks;
    p.ticket = reinterpret_cast<unsigned int*>(p.out + 1);
    OLAP_CUDA(cudaMemsetAsync(p.ticket, 0, 4, g.stream));
    KERNELS_BEGIN();
    if (VEC == 4) region_kernel<REGION_SUM, 4><<<blocks, 256, 0, g.stream>>>(p);
    else region_kernel<REGION_SUM, 1><<<blocks, 256, 0, g.stream>>>(p);
    LAUNCHED();
    end_op("region/sum");
    double host = 0.0;
    OLAP_CUDA(cudaMemcpyAsync(&host, p.out, 8, cudaMemcpyDeviceToHost, g.stream));
    OLAP_TRY(t.release());
    OLAP_TRY(dev_free(scratch));
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    *out = host;
    return finish_op();
}

int olap_region_copy(olap_store* dst, const olap_store* src, int ndim, const int64_t* len, const int64_t* keep_len,
                     const int32_t* const* keep) {
    if (!dst || !src) return fail(OLAP_E_INVALID, "olap_region_copy: null store");
    if (dst->size != src->size) return fail(OLAP_E_INVALID, "olap_region_copy: stores of %lld and %lld cells", (long long)dst->size, (long long)src->size);
    RegionPlan plan;
    OLAP_TRY(plan_region("olap_region_copy", src->size, ndim, len, keep_len, keep, &plan));
    OLAP_TRY(ensure_ctx());
    begin_op();
    // the derived flag stays as it is, as for olap_store_set_values: every byte written is  set ? SET : UNSET
    if (plan.cells) {
        const int VEC = region_vec(plan, src->values + plan.const_off, dst->values + plan.const_off,
                                   dst->status ? dst->status + plan.const_off : nullptr);
        RegionParams p{};
        TablePack t;
        OLAP_TRY(region_params(plan, VEC, t, p));
        p.src = src->values + plan.const_off;
        p.dst = dst->values + plan.const_off;
        p.st_dst = dst->status ? dst->status + plan.const_off : nullptr;
        p.dst_nan_default = dst->default_kind;
        const int blocks = grid_for(p.ix.n_vec, 256);
        KERNELS_BEGIN();
        if (VEC == 4) region_kernel<REGION_COPY, 4><<<blocks, 256, 0, g.stream>>>(p);
        else region_kernel<REGION_COPY, 1><<<blocks, 256, 0, g.stream>>>(p);
        LAUNCHED();
        OLAP_TRY(t.release());
    }
    end_op("region/copy");
    return finish_op();
}

// ---- peer memory and the fused rollup + exchange (sharded cubes) --------------------------
// Buffers that other processes of the box can map (cudaMalloc + CUDA IPC; the stream-ordered
// pool cannot be exported), stores that wrap such memory, and a drillUp of the OUTERMOST axis
// that writes every output row to a caller-given pointer: with peer-mapped pointers each rank
// stores its partial rollup of a sharded dimension STRAIGHT into the receive buffer of the
// rank that owns the row, over NVLink, from inside the rollup kernel — no partial plane in
// local HBM, no separate all-to-all.
int olap_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64) {
    if (!ptr || !handle64) return fail(OLAP_E_INVALID, "olap_peer_alloc: null argument");
    OLAP_TRY(ensure_ctx());
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    OLAP_CUDA(cudaMalloc(ptr, share_round(bytes)));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, *ptr);
    if (e != cudaSuccess) {
        cudaFree(*ptr);
        *ptr = nullptr;
        return fail(OLAP_E_CUDA, "olap_peer_alloc: cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    }
    memcpy(handle64, &h, 64);
    return OLAP_OK;
}

int olap_peer_open(const unsigned char* handle64, void** ptr) {
    if (!ptr || !handle64) return fail(OLAP_E_INVALID, "olap_peer_open: null argument");
    OLAP_TRY(ensure_ctx());
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    OLAP_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return OLAP_OK;
}

int olap_peer_close(void* ptr) {
    if (!ptr) return OLAP_OK;
    OLAP_CUDA(cudaIpcCloseMemHandle(ptr));
    return OLAP_OK;
}

int olap_peer_free(void* ptr) {
    if (!ptr) return OLAP_OK;
    OLAP_CUDA(cudaFree(ptr));
    return OLAP_OK;
}

int olap_store_wrap(void* values, void* status, int64_t size, int type, int default_kind, olap_store** out) {
    if (!values || !out || size < 0) return fail(OLAP_E_INVALID, "olap_store_wrap: invalid argument");
    OLAP_TRY(check_type_default(type, default_kind));
    olap_store* s = new olap_store();
    s->size = size;
    s->type = type;
    s->default_kind = default_kind;
    s->values = static_cast<float*>(values);
    s->status = static_cast<uint8_t*>(status);
    s->arena = nullptr;  // not owned: olap_store_destroy leaves the memory alone
    *out = s;
    return OLAP_OK;
}

int olap_drill_up_rows(olap_store* const* src, int n, const int* methods, int64_t c_rows, int64_t p_rows, int64_t inner,
                       const int32_t* row_map, float* const* row_values, uint8_t* const* row_status) {
    int64_t size = 0;
    OLAP_TRY(check_batch(src, n, "olap_drill_up_rows", &size));
    if (!methods || !row_map || !row_values) return fail(OLAP_E_INVALID, "olap_drill_up_rows: null argument");
    // c_rows == 0 is legal: a rank that holds no row of the sharded axis still fills its slot of
    // every receive buffer with "unset" (the combine step reads all W slots)
    if (c_rows < 0 || p_rows <= 0 || inner <= 0 || c_rows > 0x7fffffffLL || p_rows > 0x7fffffffLL)
        return fail(OLAP_E_INVALID, "olap_drill_up_rows: invalid shape");
    if (c_rows * inner != size) return fail(OLAP_E_INVALID, "olap_drill_up_rows: shape describes %lld cells, store has %lld", (long long)(c_rows * inner), (long long)size);
    for (int k = 0; k < n; ++k)
        if (methods[k] < OLAP_SUM || methods[k] > OLAP_COUNT) return fail(OLAP_E_INVALID, "Unsupported aggregation method: %d", methods[k]);
    for (int64_t i = 0; i < c_rows; ++i)
        if (row_map[i] < 0 || row_map[i] >= p_rows) return fail(OLAP_E_INVALID, "olap_drill_up_rows: row %lld maps to %d, outside [0, %lld)", (long long)i, row_map[i], (long long)p_rows);
    bool any_status = false;
    for (int k = 0; k < n; ++k) any_status |= src[k]->status != nullptr;
    if (any_status && !row_status) return fail(OLAP_E_INVALID, "olap_drill_up_rows: stores carry a status plane but no status rows were given");
    OLAP_TRY(ensure_ctx());
    begin_op();
    std::vector<UpMeasure> meas(n);
    for (int k = 0; k < n; ++k) {
        const uint8_t* si = row_status ? src[k]->status : nullptr;  // every row buffer is written, shared source plane or not
        // out / st_out are placeholders (non-null where a plane exists): the kernel rebases them per row
        meas[k] = UpMeasure{src[k]->values, const_cast<float*>(src[k]->values), si, si ? const_cast<uint8_t*>(si) : nullptr,
                            methods[k], src[k]->default_kind};
    }
    const Csr csr = build_csr(row_map, c_rows, p_rows);
    TablePack t;
    const size_t o_meas = t.add(meas.data(), sizeof(UpMeasure) * n);
    const size_t o_ps = t.add(csr.pstart.data(), csr.pstart.size() * 4);
    const size_t o_ch = t.add(csr.children.data(), csr.children.size() * 4);
    const size_t o_rv = t.add(row_values, sizeof(float*) * (size_t)n * p_rows);
    std::vector<uint8_t*> no_status((size_t)n * p_rows, nullptr);
    const size_t o_rs = t.add(row_status ? (const void*)row_status : (const void*)no_status.data(), sizeof(uint8_t*) * (size_t)n * p_rows);
    OLAP_TRY(t.upload());
    OLAP_TRY(launch_up_mid(t.ptr<UpMeasure>(o_meas), meas.data(), n, csr, t.ptr<int32_t>(o_ps), t.ptr<int32_t>(o_ch), 1, c_rows,
                           p_rows, inner, t.ptr<float*>(o_rv), t.ptr<uint8_t*>(o_rs)));
    OLAP_TRY(t.release());
    end_op("drillup/mid-rows-p2p");
    return finish_op();
}

// ---- pull model: stores that peers can map, and the rollup that reads them ------------------
int olap_store_ipc_export(const olap_store* s, unsigned char* handle64, int64_t* values_offset, int64_t* status_offset) {
    if (!s || !handle64 || !values_offset || !status_offset) return fail(OLAP_E_INVALID, "olap_store_ipc_export: null argument");
    if (!s->arena || !s->arena->shareable)
        return fail(OLAP_E_UNSUPPORTED, "olap_store_ipc_export: the store was not created with OLAP_CREATE_SHAREABLE");
    OLAP_TRY(ensure_ctx());
    cudaIpcMemHandle_t h;
    OLAP_CUDA(cudaIpcGetMemHandle(&h, s->arena->base));
    memcpy(handle64, &h, 64);
    *values_offset = reinterpret_cast<const char*>(s->values) - static_cast<const char*>(s->arena->base);
    *status_offset = s->status ? reinterpret_cast<const char*>(s->status) - static_cast<const char*>(s->arena->base) : -1;
    return OLAP_OK;
}

// Mappings of peers' blocks, by IPC handle.  A recycled block keeps its handle, so a sharded cube
// that is queried repeatedly opens each peer block once.  Least recently used mappings are closed
// beyond kPeerMapCap entries (their blocks may have been freed by the owner since).
namespace {
struct PeerMapping { void* ptr; uint64_t stamp; };
std::map<std::array<unsigned char, 64>, PeerMapping> g_peer_maps;
uint64_t g_peer_clock = 0;
constexpr size_t kPeerMapCap = 512;
}  // namespace

int olap_peer_map(const unsigned char* handle64, void** ptr) {
    if (!ptr || !handle64) return fail(OLAP_E_INVALID, "olap_peer_map: null argument");
    OLAP_TRY(ensure_ctx());
    std::array<unsigned char, 64> key;
    memcpy(key.data(), handle64, 64);
    auto it = g_peer_maps.find(key);
    if (it != g_peer_maps.end()) {
        it->second.stamp = ++g_peer_clock;
        *ptr = it->second.ptr;
        return OLAP_OK;
    }
    if (g_peer_maps.size() >= kPeerMapCap) {
        auto victim = g_peer_maps.begin();
        for (auto q = g_peer_maps.begin(); q != g_peer_maps.end(); ++q)
            if (q->second.stamp < victim->second.stamp) victim = q;
        OLAP_CUDA(cudaStreamSynchronize(g.stream));  // no kernel may still be reading it
        cudaIpcCloseMemHandle(victim->second.ptr);
        g_peer_maps.erase(victim);
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    OLAP_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    g_peer_maps[key] = PeerMapping{*ptr, ++g_peer_clock};
    return OLAP_OK;
}

int olap_peer_unmap_all(void) {
    if (!g.ready) return OLAP_OK;
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    for (auto& kv : g_peer_maps) cudaIpcCloseMemHandle(kv.second.ptr);
    g_peer_maps.clear();
    return OLAP_OK;
}

int olap_drill_up_pull(olap_store* const* like, int n, const int* methods, int64_t out_rows, int64_t inner,
                       const int32_t* row_start, const int32_t* child_rank, const int64_t* child_row, int n_ranks,
                       const int64_t* rank_rows, const void* const* base_values, const void* const* base_status,
                       int derive_status, olap_store** out) {
    int64_t like_size = 0;
    OLAP_TRY(check_batch(like, n, "olap_drill_up_pull", &like_size));
    if (!methods || !row_start || !rank_rows || !base_values || !out) return fail(OLAP_E_INVALID, "olap_drill_up_pull: null argument");
    if (out_rows < 0 || inner <= 0 || n_ranks < 1) return fail(OLAP_E_INVALID, "olap_drill_up_pull: invalid shape");
    for (int k = 0; k < n; ++k)
        if (methods[k] < OLAP_SUM || methods[k] > OLAP_COUNT) return fail(OLAP_E_INVALID, "Unsupported aggregation method: %d", methods[k]);
    int64_t new_size = 0;
    if (mul_overflow(out_rows, inner, &new_size)) return fail(OLAP_E_INVALID, "olap_drill_up_pull: cube size overflows int64");
    if (out_rows > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "olap_drill_up_pull: more than 2^31-1 output rows");
    if (row_start[0] != 0) return fail(OLAP_E_INVALID, "olap_drill_up_pull: row_start[0] must be 0");
    for (int64_t j = 0; j < out_rows; ++j)
        if (row_start[j + 1] < row_start[j]) return fail(OLAP_E_INVALID, "olap_drill_up_pull: row_start is not ascending");
    const int64_t nc = row_start[out_rows];
    if (nc && (!child_rank || !child_row)) return fail(OLAP_E_INVALID, "olap_drill_up_pull: null child tables");
    std::vector<int64_t> child_off((size_t)nc);
    for (int64_t c = 0; c < nc; ++c) {
        const int32_t r = child_rank[c];
        if (r < 0 || r >= n_ranks) return fail(OLAP_E_INVALID, "olap_drill_up_pull: child %lld lives on rank %d, outside [0, %d)", (long long)c, r, n_ranks);
        if (child_row[c] < 0 || child_row[c] >= rank_rows[r])
            return fail(OLAP_E_INVALID, "olap_drill_up_pull: child %lld is row %lld of rank %d, which holds %lld rows", (long long)c, (long long)child_row[c], r, (long long)rank_rows[r]);
        child_off[c] = child_row[c] * inner;
    }
    bool any_status = false;
    for (int k = 0; k < n; ++k) any_status |= like[k]->status != nullptr;
    if (any_status && !base_status && !derive_status) return fail(OLAP_E_INVALID, "olap_drill_up_pull: stores carry a status plane but no status bases were given");
    for (int k = 0; k < n; ++k)
        for (int r = 0; r < n_ranks; ++r) {
            // a rank without rows is never dereferenced; every other base must be a real address
            if (rank_rows[r] && !base_values[(size_t)k * n_ranks + r]) return fail(OLAP_E_INVALID, "olap_drill_up_pull: null base of store %d on rank %d", k, r);
        }
    OLAP_TRY(ensure_ctx());
    OLAP_TRY(alloc_like(like, n, new_size, out));
    OutGuard guard(out, n);
    begin_op();
    if (new_size) {
        std::vector<PullMeasure> meas(n);
        std::vector<const void*> bs((size_t)n * n_ranks, nullptr);
        for (int k = 0; k < n; ++k) {
            // a status plane shared by several measures is read and written by the first of them only
            const bool own_status = out[k]->status && like[k]->status && st_out_of(out, k);
            meas[k] = PullMeasure{out[k]->values, own_status ? out[k]->status : nullptr, methods[k], like[k]->default_kind,
                                  derive_status ? 1 : 0};
            if (own_status && !derive_status)
                for (int r = 0; r < n_ranks; ++r) bs[(size_t)k * n_ranks + r] = base_status[(size_t)k * n_ranks + r];
        }
        TablePack t;
        const size_t o_meas = t.add(meas.data(), sizeof(PullMeasure) * n);
        const size_t o_rs = t.add(row_start, sizeof(int32_t) * (size_t)(out_rows + 1));
        const size_t o_cr = t.add(child_rank, sizeof(int32_t) * (size_t)nc);
        const size_t o_co = t.add(child_off.data(), sizeof(int64_t) * (size_t)nc);
        const size_t o_bv = t.add(base_values, sizeof(void*) * (size_t)n * n_ranks);
        const size_t o_bs = t.add(bs.data(), sizeof(void*) * (size_t)n * n_ranks);
        OLAP_TRY(t.upload());
        // 128-bit path: every row of every rank must start on a 16-byte boundary
        bool vec4 = inner % 4 == 0;
        for (size_t q = 0; q < (size_t)n * n_ranks && vec4; ++q) {
            vec4 &= (reinterpret_cast<uintptr_t>(base_values[q]) & 15) == 0;
            vec4 &= (reinterpret_cast<uintptr_t>(bs[q]) & 3) == 0;
        }
        UpPullParams p{};
        p.meas = t.ptr<PullMeasure>(o_meas);
        p.row_start = t.ptr<int32_t>(o_rs);
        p.child_rank = t.ptr<int32_t>(o_cr);
        p.child_off = t.ptr<int64_t>(o_co);
        p.base_v = t.ptr<const float*>(o_bv);
        p.base_s = t.ptr<const uint8_t*>(o_bs);
        p.n_ranks = n_ranks;
        p.rows = out_rows;
        p.inner = inner;
        p.IV = vec4 ? inner / 4 : inner;
        const uint32_t bx = (uint32_t)std::min<int64_t>(256, next_pow2((uint32_t)std::min<int64_t>(p.IV, 256)));
        const uint32_t by = 256 / bx;
        const int64_t gx = ceil_div(p.IV, bx);
        if (gx > 0x7fffffffLL) return fail(OLAP_E_UNSUPPORTED, "olap_drill_up_pull: inner run too long");
        const int64_t rows_per_launch = (int64_t)65535 * by;
        // staged variant (cp.async into the thread's own shared-memory slots): all children of a row in flight at once
        static const int staged_knob = [] { const char* e = getenv("OLAP_PULL_STAGED"); return e ? atoi(e) : 1; }();
        int32_t max_children = 1;
        for (int64_t j = 0; j < out_rows; ++j) max_children = std::max(max_children, row_start[j + 1] - row_start[j]);
        const int chunk = std::min(16, (int)max_children);
        const bool staged = staged_knob != 0 && vec4;
        bool st_loaded = false;
        for (int k = 0; k < n; ++k) st_loaded |= meas[k].st_out && !meas[k].derive;
        const size_t staged_smem = (size_t)chunk * 256 * (16 + (st_loaded ? 4 : 0));
        if (staged) {
            static size_t attr = 0;
            if (staged_smem > attr) {
                OLAP_CUDA(cudaFuncSetAttribute(drillup_pull_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 256 * 20));
                attr = 16 * 256 * 20;
            }
        }
        KERNELS_BEGIN();
        for (int64_t r0 = 0; r0 < out_rows; r0 += rows_per_launch) {
            p.row0 = r0;
            const int64_t gy = ceil_div(std::min(rows_per_launch, out_rows - r0), by);
            dim3 grid((unsigned)gx, (unsigned)gy, (unsigned)n), block(bx, by);
            if (vec4 && staged) drillup_pull_staged_kernel<<<grid, block, staged_smem, g.stream>>>(p, chunk);
            else if (vec4) drillup_pull_kernel<4><<<grid, block, 0, g.stream>>>(p);
            else drillup_pull_kernel<1><<<grid, block, 0, g.stream>>>(p);
            LAUNCHED();
        }
        OLAP_TRY(t.release());
    }
    end_op("drillup/pull-peers");
    return guard.done(finish_op());
}

// ---- computed measures --------------------------------------------------------------------
int olap_eval(const char* program, olap_store* const* inputs, int n_inputs, const double* totals, int n_totals,
              double* out_host_f64, int out_type, int out_default_kind, olap_store** out_store) {
    if (!program) return fail(OLAP_E_INVALID, "olap_eval: null program");
    if (n_inputs < 0 || n_inputs > OLAP_MAX_MEASURES || n_totals < 0 || n_totals > OLAP_MAX_MEASURES) return fail(OLAP_E_INVALID, "olap_eval: too many inputs");
    if ((out_host_f64 != nullptr) == (out_store != nullptr)) return fail(OLAP_E_INVALID, "olap_eval: exactly one of out_host_f64 / out_store");
    if (n_inputs == 0) return fail(OLAP_E_INVALID, "olap_eval: a formula needs at least one stored measure to give the cube size");
    int64_t size = 0;
    OLAP_TRY(check_batch(inputs, n_inputs, "olap_eval", &size));
    OLAP_TRY(ensure_ctx());
    JitKernel* k = nullptr;
    OLAP_TRY(jit_get(program, n_inputs, n_totals, JIT_EVAL, &k));

    float* out32 = nullptr;
    uint8_t* st_out = nullptr;
    double* out64 = nullptr;
    olap_store* result = nullptr;
    if (out_store) {
        OLAP_TRY(check_type_default(out_type, out_default_kind));
        bool with_status = true;
        for (int q = 0; q < n_inputs; ++q) with_status &= inputs[q]->status != nullptr;
        OLAP_TRY(alloc_batch(1, size, &out_type, &out_default_kind, with_status, false, &result,
                             inputs[0]->arena && inputs[0]->arena->shareable));
        out32 = result->values;
        st_out = result->status;
        set_derived(result, true);  // the formula kernel writes SET / UNSET from the result it stores
    } else if (size) {
        void* tmp;
        OLAP_TRY(dev_alloc(&tmp, (size_t)size * 8));
        out64 = (double*)tmp;
    }
    begin_op();
    if (size) {
        std::vector<void*> args;
        std::vector<const float*> ptrs(n_inputs);
        std::vector<double> tot(n_totals);
        for (int q = 0; q < n_inputs; ++q) { ptrs[q] = inputs[q]->values; args.push_back(&ptrs[q]); }
        for (int q = 0; q < n_totals; ++q) { tot[q] = totals[q]; args.push_back(&tot[q]); }
        long long n = size;
        int nan_default = out_default_kind;
        args.push_back(&out32); args.push_back(&st_out); args.push_back(&out64); args.push_back(&n); args.push_back(&nan_default);
        const int blocks = (int)std::min<int64_t>(ceil_div(ceil_div(size, 4), 256), (int64_t)g.sm_count * 16);
        KERNELS_BEGIN();
        CUresult cr = jit_api().LaunchKernel(k->fn, blocks, 1, 1, 256, 1, 1, 0, (CUstream)g.stream, args.data(), nullptr);
        if (cr != CUDA_SUCCESS) {
            const char* msg = "?";
            jit_api().GetErrorString(cr, &msg);
            olap_store_destroy(result);
            dev_free(out64);
            return fail(OLAP_E_CUDA, "launching the formula kernel failed: %s", msg);
        }
        LAUNCHED();
    }
    end_op("eval/jit");
    if (out_store) {
        *out_store = result;
        return finish_op();
    }
    if (size) {
        OLAP_CUDA(cudaMemcpyAsync(out_host_f64, out64, (size_t)size * 8, cudaMemcpyDeviceToHost, g.stream));
        OLAP_TRY(dev_free(out64));
        OLAP_CUDA(cudaStreamSynchronize(g.stream));
    }
    return OLAP_OK;
}

// ---- computed measures over a region: getTotalForDimensionItems / copyMeasureData ------------------
namespace {

static int formula_inputs(const char* what, const char* program, olap_store* const* inputs, int n, int64_t* size) {
    if (!program) return fail(OLAP_E_INVALID, "%s: null program", what);
    return check_batch(inputs, n, what, size);
}

// VEC 4 when the plan and the planes of every input (and of the target) allow it
static int region_vec_all(const RegionPlan& plan, olap_store* const* in, int n, const olap_store* dst) {
    int vec = 4;
    const int64_t c = plan.const_off;
    for (int k = 0; k < n; ++k) vec = std::min(vec, region_vec(plan, in[k]->values + c, in[k]->values + c, nullptr));
    if (dst) vec = std::min(vec, region_vec(plan, dst->values + c, dst->values + c, dst->status ? dst->status + c : nullptr));
    return vec;
}

// the index fields of region_params as the RegionWalk the NVRTC kernels take
static int region_walk_of(const RegionPlan& plan, int VEC, TablePack& t, RegionWalk& w) {
    RegionParams p{};
    OLAP_TRY(region_params(plan, VEC, t, p));
    w = RegionWalk{};
    w.nd = p.ix.nd;
    for (int d = 0; d < p.ix.nd; ++d) {
        w.len[d] = p.ix.len[d];
        w.div[d] = p.ix.div[d];
        w.tbl[d] = p.ix.tbl[d];
        w.lin[d] = p.ix.lin[d];
    }
    w.IV = p.ix.IV;
    w.div_iv = p.ix.div_iv;
    w.n_vec = p.ix.n_vec;
    w.big = p.big;
    return OLAP_OK;
}

static int jit_launch(CUfunction fn, int blocks, std::vector<void*>& args) {
    const CUresult cr = jit_api().LaunchKernel(fn, blocks, 1, 1, 256, 1, 1, 0, (CUstream)g.stream, args.data(), nullptr);
    if (cr != CUDA_SUCCESS) {
        const char* msg = "?";
        jit_api().GetErrorString(cr, &msg);
        return fail(OLAP_E_CUDA, "launching the formula region kernel failed: %s", msg);
    }
    LAUNCHED();
    return OLAP_OK;
}

}  // namespace

int olap_region_eval_sum(const char* program, olap_store* const* inputs, int n_inputs, int ndim, const int64_t* len,
                         const int64_t* keep_len, const int32_t* const* keep, double* out) {
    if (!out) return fail(OLAP_E_INVALID, "olap_region_eval_sum: null argument");
    int64_t size = 0;
    OLAP_TRY(formula_inputs("olap_region_eval_sum", program, inputs, n_inputs, &size));
    RegionPlan plan;
    OLAP_TRY(plan_region("olap_region_eval_sum", size, ndim, len, keep_len, keep, &plan));
    OLAP_TRY(ensure_ctx());
    *out = 0.0;
    if (plan.cells == 0) {
        begin_op();
        end_op("region/eval-sum");
        return finish_op();
    }
    JitKernel* k = nullptr;
    OLAP_TRY(jit_get(program, n_inputs, 0, JIT_REGION_SUM, &k));
    begin_op();
    const int VEC = region_vec_all(plan, inputs, n_inputs, nullptr);
    RegionWalk w;
    TablePack t;
    OLAP_TRY(region_walk_of(plan, VEC, t, w));
    const int blocks = grid_for(w.n_vec, 256);
    void* scratch;
    OLAP_TRY(dev_alloc(&scratch, (size_t)blocks * 8 + 16));
    double* partial = static_cast<double*>(scratch);
    double* dout = partial + blocks;
    unsigned int* ticket = reinterpret_cast<unsigned int*>(dout + 1);
    OLAP_CUDA(cudaMemsetAsync(ticket, 0, 4, g.stream));
    std::vector<const float*> ptrs(n_inputs);
    std::vector<void*> args{&w};
    for (int q = 0; q < n_inputs; ++q) { ptrs[q] = inputs[q]->values + plan.const_off; args.push_back(&ptrs[q]); }
    args.push_back(&partial); args.push_back(&ticket); args.push_back(&dout);
    KERNELS_BEGIN();
    OLAP_TRY(jit_launch(VEC == 4 ? k->vec4 : k->vec1, blocks, args));
    end_op("region/eval-sum");
    double host = 0.0;
    OLAP_CUDA(cudaMemcpyAsync(&host, dout, 8, cudaMemcpyDeviceToHost, g.stream));
    OLAP_TRY(t.release());
    OLAP_TRY(dev_free(scratch));
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    *out = host;
    return finish_op();
}

int olap_region_eval_copy(olap_store* dst, const char* program, olap_store* const* inputs, int n_inputs, int ndim,
                          const int64_t* len, const int64_t* keep_len, const int32_t* const* keep) {
    if (!dst) return fail(OLAP_E_INVALID, "olap_region_eval_copy: null store");
    int64_t size = 0;
    OLAP_TRY(formula_inputs("olap_region_eval_copy", program, inputs, n_inputs, &size));
    if (dst->size != size) return fail(OLAP_E_INVALID, "olap_region_eval_copy: stores of %lld and %lld cells", (long long)dst->size, (long long)size);
    if (ndim < 0 || ndim > OLAP_MAX_DIMS) return fail(OLAP_E_INVALID, "olap_region_eval_copy: at most %d dimensions", OLAP_MAX_DIMS);
    // Each list de-duplicated, first occurrences in order (the multiplicity axis becomes one item): every cell is
    // then read and written by one thread, once, so the target may be an input.  A repeat writes the value it
    // wrote before, so the planes end as those of the setValue per combination.
    std::vector<std::vector<int32_t>> uniq(ndim);
    std::vector<const int32_t*> kp(ndim, nullptr);
    std::vector<int64_t> kl(ndim, 0);
    for (int d = 0; d < ndim; ++d) {
        if (!keep || !keep[d]) continue;
        if (!keep_len || keep_len[d] < 0) return fail(OLAP_E_INVALID, "olap_region_eval_copy: dimension %d has no list length", d);
        std::unordered_set<int32_t> seen;
        for (int64_t j = 0; j < keep_len[d]; ++j)
            if (seen.insert(keep[d][j]).second) uniq[d].push_back(keep[d][j]);
        // an empty list stays a list (of no items): data() of an empty vector may be NULL, which means "whole axis"
        static const int32_t no_items = 0;
        kp[d] = uniq[d].empty() ? &no_items : uniq[d].data();
        kl[d] = (int64_t)uniq[d].size();
    }
    RegionPlan plan;
    OLAP_TRY(plan_region("olap_region_eval_copy", size, ndim, len, kl.data(), kp.data(), &plan));
    OLAP_TRY(ensure_ctx());
    // the derived flag stays as it is, as for olap_region_copy: every byte written is  set ? SET : UNSET
    if (plan.cells == 0) {
        begin_op();
        end_op("region/eval-copy");
        return finish_op();
    }
    JitKernel* k = nullptr;
    OLAP_TRY(jit_get(program, n_inputs, 0, JIT_REGION_COPY, &k));
    begin_op();
    const int VEC = region_vec_all(plan, inputs, n_inputs, dst);
    RegionWalk w;
    TablePack t;
    OLAP_TRY(region_walk_of(plan, VEC, t, w));
    const int blocks = grid_for(w.n_vec, 256);
    std::vector<const float*> ptrs(n_inputs);
    std::vector<void*> args{&w};
    for (int q = 0; q < n_inputs; ++q) { ptrs[q] = inputs[q]->values + plan.const_off; args.push_back(&ptrs[q]); }
    KERNELS_BEGIN();
    if (strict_ints(dst)) {
        // olap_store_set_values refuses the whole call when a value would not survive its Float32 cell: a check
        // pass finds the first such cell in product order (and its value) before anything is written
        struct { unsigned long long first; int64_t off; double val; unsigned int ticket; } host;
        void* scratch;
        OLAP_TRY(dev_alloc(&scratch, sizeof host));
        char* b = static_cast<char*>(scratch);
        unsigned long long* first = reinterpret_cast<unsigned long long*>(b);
        int64_t* bad_off = reinterpret_cast<int64_t*>(b + 8);
        double* bad_val = reinterpret_cast<double*>(b + 16);
        unsigned int* ticket = reinterpret_cast<unsigned int*>(b + 24);
        OLAP_CUDA(cudaMemsetAsync(first, 0xff, 8, g.stream));
        OLAP_CUDA(cudaMemsetAsync(ticket, 0, 4, g.stream));
        std::vector<void*> cargs = args;
        cargs.push_back(&first); cargs.push_back(&ticket); cargs.push_back(&bad_off); cargs.push_back(&bad_val);
        OLAP_TRY(jit_launch(VEC == 4 ? k->check4 : k->check1, blocks, cargs));
        OLAP_CUDA(cudaMemcpyAsync(&host, scratch, sizeof host, cudaMemcpyDeviceToHost, g.stream));
        OLAP_TRY(dev_free(scratch));
        OLAP_CUDA(cudaStreamSynchronize(g.stream));
        if (host.first != ~0ull) {
            end_op("region/eval-copy");
            OLAP_TRY(t.release());
            return lossy_error(dst, plan.const_off + host.off, host.val);
        }
    }
    float* dv = dst->values + plan.const_off;
    uint8_t* ds = dst->status ? dst->status + plan.const_off : nullptr;
    int nan_default = dst->default_kind;
    args.push_back(&dv); args.push_back(&ds); args.push_back(&nan_default);
    OLAP_TRY(jit_launch(VEC == 4 ? k->vec4 : k->vec1, blocks, args));
    end_op("region/eval-copy");
    OLAP_TRY(t.release());
    return finish_op();
}

// ---- the status accessors of a computed measure: Cube.getStatus / getStatusMap --------------------
namespace {
static int status_inputs(const char* what, olap_store* const* s, int n, int64_t* size, TablePack& t, size_t* o_in) {
    if (!s || n < 1) return fail(OLAP_E_INVALID, "%s: at least one store expected", what);
    std::vector<StatusIn> in(n);
    for (int k = 0; k < n; ++k) {
        if (!s[k]) return fail(OLAP_E_INVALID, "%s: null store", what);
        if (s[k]->size != s[0]->size) return fail(OLAP_E_INVALID, "%s: stores of one call must have the same size", what);
        in[k] = StatusIn{s[k]->values, s[k]->status, s[k]->default_kind};
    }
    *size = s[0]->size;
    *o_in = t.add(in.data(), sizeof(StatusIn) * n);
    return OLAP_OK;
}
}  // namespace

int olap_status_merge(olap_store* const* inputs, int n, uint8_t* host, int64_t n_cells) {
    TablePack t;
    size_t o_in = 0;
    int64_t size = 0;
    OLAP_TRY(status_inputs("olap_status_merge", inputs, n, &size, t, &o_in));
    if (size != n_cells) return fail(OLAP_E_INVALID, "value length is invalid: %lld !== %lld", (long long)size, (long long)n_cells);
    if (n_cells && !host) return fail(OLAP_E_INVALID, "olap_status_merge: null argument");
    OLAP_TRY(ensure_ctx());
    begin_op();
    if (n_cells == 0) {
        end_op("status/merge");
        return finish_op();
    }
    bool vec4 = n_cells % 4 == 0;
    for (int k = 0; k < n; ++k)
        vec4 &= ((reinterpret_cast<uintptr_t>(inputs[k]->values) & 15) | (reinterpret_cast<uintptr_t>(inputs[k]->status) & 3)) == 0;
    OLAP_TRY(t.upload());
    void* tmp;
    OLAP_TRY(dev_alloc(&tmp, (size_t)n_cells));
    KERNELS_BEGIN();
    if (vec4) status_merge_kernel<4><<<grid_for(n_cells / 4, kStoreThreads), kStoreThreads, 0, g.stream>>>(t.ptr<StatusIn>(o_in), n, (uint8_t*)tmp, n_cells);
    else status_merge_kernel<1><<<grid_for(n_cells, kStoreThreads), kStoreThreads, 0, g.stream>>>(t.ptr<StatusIn>(o_in), n, (uint8_t*)tmp, n_cells);
    LAUNCHED();
    end_op("status/merge");
    OLAP_TRY(copy_d2h(host, tmp, (size_t)n_cells));
    OLAP_TRY(t.release());
    OLAP_TRY(dev_free(tmp));
    return finish_op();
}

int olap_status_map_export(olap_store* const* stores, int n, int64_t capacity, int64_t* keys, double* values,
                           uint8_t* is_int, int64_t* count) {
    if (!count) return fail(OLAP_E_INVALID, "olap_status_map_export: null argument");
    const bool fill = keys != nullptr;
    if ((values != nullptr) != fill || (is_int != nullptr) != fill)
        return fail(OLAP_E_INVALID, "olap_status_map_export: keys, values and is_int must be all NULL (count) or all given (fill)");
    *count = 0;
    TablePack t;
    size_t o_in = 0;
    int64_t size = 0;
    OLAP_TRY(status_inputs("olap_status_map_export", stores, n, &size, t, &o_in));
    OLAP_TRY(ensure_ctx());
    if (size == 0) {
        begin_op();
        end_op("status/map");
        return finish_op();
    }
    OLAP_TRY(t.upload());
    const int64_t nb = ceil_div(size, kCompactTile);
    const int64_t nc = (int64_t)n * nb;
    void* cnt;
    OLAP_TRY(dev_alloc(&cnt, (size_t)(nc + 1) * 8));
    unsigned long long* d_cnt = (unsigned long long*)cnt;
    const StatusIn* in = t.ptr<StatusIn>(o_in);
    begin_op();
    KERNELS_BEGIN();
    map_count_kernel<<<(unsigned)nb, 256, (size_t)n * 4, g.stream>>>(in, n, size, d_cnt, nb);
    LAUNCHED();
    compact_scan_kernel<<<1, 1024, 0, g.stream>>>(d_cnt, nc, d_cnt + nc);
    LAUNCHED();
    unsigned long long total = 0;
    OLAP_CUDA(cudaMemcpyAsync(&total, d_cnt + nc, 8, cudaMemcpyDeviceToHost, g.stream));
    OLAP_CUDA(cudaStreamSynchronize(g.stream));
    *count = (int64_t)total;
    const bool write = fill && total && (int64_t)total <= capacity;
    void *dk = nullptr, *dv = nullptr, *di = nullptr;
    if (write) {
        OLAP_TRY(dev_alloc(&dk, (size_t)total * 8));
        OLAP_TRY(dev_alloc(&dv, (size_t)total * 8));
        OLAP_TRY(dev_alloc(&di, (size_t)total));
        map_write_kernel<<<(unsigned)nb, 256, (size_t)n * 9 * 4, g.stream>>>(in, n, size, d_cnt, nb, (int64_t*)dk, (double*)dv, (uint8_t*)di);
        LAUNCHED();
    }
    end_op("status/map");  // every path that launched closes the op here
    int rc = OLAP_OK;
    if (fill && (int64_t)total > capacity)
        rc = fail(OLAP_E_INVALID, "olap_status_map_export: capacity %lld < %llu keys", (long long)capacity, total);
    if (write) {
        OLAP_TRY(copy_d2h(keys, dk, (size_t)total * 8));
        OLAP_TRY(copy_d2h(values, dv, (size_t)total * 8));
        OLAP_TRY(copy_d2h(is_int, di, (size_t)total));
        OLAP_TRY(dev_free(dk));
        OLAP_TRY(dev_free(dv));
        OLAP_TRY(dev_free(di));
    }
    OLAP_TRY(t.release());
    OLAP_TRY(dev_free(cnt));
    return rc == OLAP_OK ? finish_op() : rc;
}

}  // extern "C"
