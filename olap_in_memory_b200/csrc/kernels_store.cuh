// Elementwise / reduction kernels of the store itself: the data boundary
// (in-memory.js:30-46), fill (135-137), total (22-28), presence and status planes,
// and the COO export/import used by `_dataMap` / serialize (75-116).
#pragma once
#include "common.cuh"

namespace olap {

constexpr int kStoreThreads = 256;

// `set data`: canonicalise freshly copied float cells in place and (re)build status.
__global__ void __launch_bounds__(kStoreThreads) canon_f32_kernel(float* __restrict__ v, uint8_t* __restrict__ st,
                                                                  int64_t n, int nan_default) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
        if (i + 4 <= n) {
            float4 t = *reinterpret_cast<float4*>(v + i);
            t.x = canon_store(t.x, nan_default); t.y = canon_store(t.y, nan_default);
            t.z = canon_store(t.z, nan_default); t.w = canon_store(t.w, nan_default);
            *reinterpret_cast<float4*>(v + i) = t;
            if (st) {
                uchar4 s;
                s.x = present_f(t.x, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
                s.y = present_f(t.y, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
                s.z = present_f(t.z, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
                s.w = present_f(t.w, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
                *reinterpret_cast<uchar4*>(st + i) = s;
            }
        } else {
            for (int64_t k = i; k < n; ++k) {
                const float t = canon_store(v[k], nan_default);
                v[k] = t;
                if (st) st[k] = present_f(t, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
            }
        }
    }
}

// `set data` from doubles: Math.fround then canonicalise.
// `lossy` (nullable): first index (+1) whose double does not survive the Float32 cell — integer stores
// are expected to hold exact integers (counts above 2^24 would silently change, ADVICE r01).
__global__ void __launch_bounds__(kStoreThreads) from_f64_kernel(const double* __restrict__ src, float* __restrict__ v,
                                                                 uint8_t* __restrict__ st, int64_t n, int nan_default,
                                                                 unsigned long long* __restrict__ lossy) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (lossy && src[i] == src[i] && (double)(float)src[i] != src[i]) atomicMin(lossy, (unsigned long long)i + 1);
        const float t = canon_store((float)src[i], nan_default);
        v[i] = t;
        if (st) st[i] = present_f(t, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
    }
}

__global__ void __launch_bounds__(kStoreThreads) to_f64_kernel(const float* __restrict__ v, double* __restrict__ dst,
                                                               int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = (double)v[i];
}

__global__ void __launch_bounds__(kStoreThreads) fill_kernel(float* __restrict__ v, uint8_t* __restrict__ st, int64_t n,
                                                             float value, uint8_t status) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        v[i] = value;
        if (st) st[i] = status;
    }
}

// setValue of one cell (in-memory.js:122-133): the canonical content of `x` and its status byte
__device__ __forceinline__ float set_cell(float x, int nan_default, uint8_t& status) {
    const float t = canon_store(x, nan_default);
    status = present_f(t, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
    return t;
}

// batched setValue (hydrateFromSparseNestedObject, setSingleData)
__global__ void __launch_bounds__(kStoreThreads) set_values_kernel(float* __restrict__ v, uint8_t* __restrict__ st,
                                                                   const int64_t* __restrict__ idx,
                                                                   const double* __restrict__ val, int64_t n,
                                                                   int64_t size, int nan_default,
                                                                   unsigned long long* __restrict__ lossy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = idx[i];
    if (k < 0 || k >= size) return;
    if (lossy && val[i] == val[i] && (double)(float)val[i] != val[i]) atomicMin(lossy, (unsigned long long)i + 1);
    uint8_t s;
    v[k] = set_cell((float)val[i], nan_default, s);
    if (st) st[k] = s;
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// `get total`: double sum of the set cells, plus their count.  Per-block partials are
// written to scratch and folded by the last block (threadfence + ticket), which keeps
// the result deterministic for a given grid.
__global__ void __launch_bounds__(kStoreThreads, 4) total_kernel(const float* __restrict__ v, int64_t n, int nan_default,
                                                              double* __restrict__ partial_sum,
                                                              unsigned long long* __restrict__ partial_cnt,
                                                              unsigned int* __restrict__ ticket,
                                                              double* __restrict__ out_sum,
                                                              unsigned long long* __restrict__ out_cnt) {
    __shared__ double s_sum[kStoreThreads / 32];
    __shared__ unsigned long long s_cnt[kStoreThreads / 32];
    __shared__ bool s_last;
    // U vectors in flight per thread, one accumulator per vector slot (independent add chains),
    // presence folded into the arithmetic (an unset cell adds 0.0 and counts 0)
    constexpr int U = 4;
    double accs[U] = {0.0, 0.0, 0.0, 0.0};
    uint32_t cnts[U] = {0u, 0u, 0u, 0u};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    for (; i + (U - 1) * stride + 4 <= n; i += U * stride) {
        float4 t[U];
#pragma unroll
        for (int u = 0; u < U; ++u) t[u] = ld_stream4(v + i + u * stride);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float e[4] = {t[u].x, t[u].y, t[u].z, t[u].w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool set = present_f(e[k], nan_default);
                accs[u] += set ? (double)e[k] : 0.0;
                cnts[u] += set ? 1u : 0u;
            }
        }
    }
    double acc = (accs[0] + accs[1]) + (accs[2] + accs[3]);
    unsigned long long cnt = (unsigned long long)cnts[0] + cnts[1] + cnts[2] + cnts[3];
    for (; i < n; i += stride) {
        float e[4];
        int m = 4;
        if (i + 4 <= n) {
            const float4 t = ld_stream4(v + i);
            e[0] = t.x; e[1] = t.y; e[2] = t.z; e[3] = t.w;
        } else {
            m = (int)(n - i);
            for (int k = 0; k < m; ++k) e[k] = v[i + k];
        }
        for (int k = 0; k < m; ++k)
            if (present_f(e[k], nan_default)) { acc += (double)e[k]; ++cnt; }
    }
    acc = warp_sum(acc);
    cnt = warp_sum_u64(cnt);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { s_sum[w] = acc; s_cnt[w] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0;
        unsigned long long c = 0;
        for (int k = 0; k < kStoreThreads / 32; ++k) { a += s_sum[k]; c += s_cnt[k]; }
        partial_sum[blockIdx.x] = a;
        partial_cnt[blockIdx.x] = c;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last) {
        // the last block folds the per-block partials cooperatively (fixed order for a given grid)
        double a = 0.0;
        unsigned long long c = 0;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
            a += ((volatile double*)partial_sum)[b];
            c += ((volatile unsigned long long*)partial_cnt)[b];
        }
        a = warp_sum(a);
        c = warp_sum_u64(c);
        __syncthreads();
        if (l == 0) { s_sum[w] = a; s_cnt[w] = c; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double ta = 0.0;
            unsigned long long tc = 0;
            for (int k = 0; k < kStoreThreads / 32; ++k) { ta += s_sum[k]; tc += s_cnt[k]; }
            *out_sum = ta;
            *out_cnt = tc;
            *ticket = 0;
        }
    }
}

// presence (1 = set) or status bytes for stores without a status plane
__global__ void __launch_bounds__(kStoreThreads) presence_kernel(const float* __restrict__ v, uint8_t* __restrict__ out,
                                                                 int64_t n, int nan_default, uint8_t yes, uint8_t no) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = present_f(v[i], nan_default) ? yes : no;
}

// ---- ordered stream compaction (keys ascending), three passes --------------------
constexpr int kCompactTile = 2048;  // cells per block

__global__ void __launch_bounds__(256) compact_count_kernel(const float* __restrict__ v, int64_t n, int nan_default,
                                                            unsigned long long* __restrict__ block_cnt) {
    __shared__ unsigned int s[8];
    const int64_t base = (int64_t)blockIdx.x * kCompactTile;
    unsigned int c = 0;
    for (int k = threadIdx.x; k < kCompactTile; k += 256) {
        const int64_t i = base + k;
        if (i < n && present_f(v[i], nan_default)) ++c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
        for (int k = 0; k < 8; ++k) t += s[k];
        block_cnt[blockIdx.x] = t;
    }
}

// single block exclusive scan over the per-block counts (in place); total to out
__global__ void __launch_bounds__(1024) compact_scan_kernel(unsigned long long* __restrict__ block_cnt, int64_t nb,
                                                            unsigned long long* __restrict__ total) {
    __shared__ unsigned long long s[1024];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nb; base += 1024) {
        const int64_t i = base + threadIdx.x;
        const unsigned long long x = i < nb ? block_cnt[i] : 0ull;
        s[threadIdx.x] = x;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            const unsigned long long y = threadIdx.x >= o ? s[threadIdx.x - o] : 0ull;
            __syncthreads();
            s[threadIdx.x] += y;
            __syncthreads();
        }
        if (i < nb) block_cnt[i] = carry + s[threadIdx.x] - x;
        __syncthreads();
        if (threadIdx.x == 1023) carry += s[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(256) compact_write_kernel(const float* __restrict__ v, int64_t n, int nan_default,
                                                            const unsigned long long* __restrict__ block_off,
                                                            int64_t* __restrict__ keys, float* __restrict__ vals) {
    __shared__ unsigned int s_warp[8];
    __shared__ unsigned int s_run;
    const int64_t base = (int64_t)blockIdx.x * kCompactTile;
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    const unsigned long long off = block_off[blockIdx.x];
    for (int k0 = 0; k0 < kCompactTile; k0 += 256) {
        const int64_t i = base + k0 + threadIdx.x;
        const float x = i < n ? v[i] : 0.0f;
        const bool pres = i < n && present_f(x, nan_default);
        const unsigned int ballot = __ballot_sync(0xffffffffu, pres);
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane == 0) s_warp[w] = __popc(ballot);
        __syncthreads();
        unsigned int before = s_run;
        for (int q = 0; q < w; ++q) before += s_warp[q];
        if (pres) {
            const unsigned long long pos = off + before + __popc(ballot & ((1u << lane) - 1u));
            keys[pos] = i;
            vals[pos] = x;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int t = 0;
            for (int q = 0; q < 8; ++q) t += s_warp[q];
            s_run += t;
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kStoreThreads) import_sparse_kernel(float* __restrict__ v, uint8_t* __restrict__ st,
                                                                      const int64_t* __restrict__ keys,
                                                                      const float* __restrict__ vals, int64_t count,
                                                                      int64_t size, int nan_default) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int64_t k = keys[i];
    if (k < 0 || k >= size) return;
    const float t = canon_store(vals[i], nan_default);
    v[k] = t;
    if (st) st[k] = present_f(t, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET;
}

// ---- the status accessors of a computed measure (Cube.getStatus / getStatusMap) ---------------
// One input store: its status plane, or (nullptr) SET / UNSET from its values.
struct StatusIn {
    const float* v;
    const uint8_t* st;
    int nan_default;
};

// getStatus: the OR over the inputs of each cell's status byte (the bytes olap_store_status reports per input)
template <int VEC>
__global__ void __launch_bounds__(kStoreThreads) status_merge_kernel(const StatusIn* __restrict__ in, int n,
                                                                     uint8_t* __restrict__ out, int64_t cells) {
    const int64_t nv = cells / VEC;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
        uint32_t acc = 0;
        for (int k = 0; k < n; ++k) {
            const StatusIn m = in[k];
            if (VEC == 4) {
                if (m.st) {
                    acc |= ld_stream_u32(m.st + i * 4);
                } else {
                    const float4 x = ld_stream4(m.v + i * 4);
                    acc |= (uint32_t)(present_f(x.x, m.nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET) |
                           (uint32_t)(present_f(x.y, m.nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET) << 8 |
                           (uint32_t)(present_f(x.z, m.nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET) << 16 |
                           (uint32_t)(present_f(x.w, m.nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET) << 24;
                }
            } else {
                acc |= m.st ? m.st[i] : (present_f(m.v[i], m.nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET);
            }
        }
        if (VEC == 4) *reinterpret_cast<uint32_t*>(out + i * 4) = acc;
        else out[i] = (uint8_t)acc;
    }
}

// JS ToInt32 of a float32 value held in a double: NaN and +-inf give 0, then truncation and the wrap modulo 2^32.
// A float32 of magnitude >= 2^55 is a multiple of 2^32, so ToInt32 is 0 for every one of them beyond 2^63.
__device__ __forceinline__ int js_to_int32(double x) {
    if (!(fabs(x) < 9223372036854775808.0)) return 0;
    return (int)(uint32_t)(unsigned long long)(long long)x;
}

// getStatusMap of a computed measure (cube.js:374-386) for one cell: `g` = the first input in which the cell is
// set (-1: none), `val` / `is_int` = the fold over the inputs in order: the first set value; then for each later
// set value, ToInt32(prev) | ToInt32(v) (an int) when the previous value is truthy, else the value itself.
__device__ __forceinline__ int status_map_cell(const StatusIn* __restrict__ in, int n, int64_t i, double& val,
                                               uint8_t& is_int) {
    int g = -1;
    val = 0.0;
    is_int = 0;
    for (int k = 0; k < n; ++k) {
        const float x = in[k].v[i];
        if (!present_f(x, in[k].nan_default)) continue;
        if (g < 0) {
            g = k;
            val = x;
        } else if (val == val && val != 0.0) {
            val = (double)(js_to_int32(val) | js_to_int32(x));
            is_int = 1;
        } else {
            val = x;
            is_int = 0;
        }
    }
    return g;
}

__device__ __forceinline__ int first_set(const StatusIn* __restrict__ in, int n, int64_t i) {
    for (int k = 0; k < n; ++k)
        if (present_f(in[k].v[i], in[k].nan_default)) return k;
    return -1;
}

// Ordered compaction with one bucket per input (compact_* with keys grouped by their first input): tile b's
// count of group g goes to cnt[g * nb + b], so that one exclusive scan of cnt gives every (group, tile) its
// first output slot.  Dynamic shared memory: n counters.
__global__ void __launch_bounds__(256) map_count_kernel(const StatusIn* __restrict__ in, int n, int64_t cells,
                                                        unsigned long long* __restrict__ cnt, int64_t nb) {
    extern __shared__ unsigned int s_cnt[];
    for (int g = threadIdx.x; g < n; g += 256) s_cnt[g] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kCompactTile;
    for (int k = threadIdx.x; k < kCompactTile; k += 256) {
        const int64_t i = base + k;
        const int g = i < cells ? first_set(in, n, i) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, g);
        if (g >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_cnt[g], (unsigned)__popc(peers));
    }
    __syncthreads();
    for (int g = threadIdx.x; g < n; g += 256) cnt[(int64_t)g * nb + blockIdx.x] = s_cnt[g];
}

// Dynamic shared memory: n running counts, then 8 per-warp counts per group.
__global__ void __launch_bounds__(256) map_write_kernel(const StatusIn* __restrict__ in, int n, int64_t cells,
                                                        const unsigned long long* __restrict__ off, int64_t nb,
                                                        int64_t* __restrict__ keys, double* __restrict__ vals,
                                                        uint8_t* __restrict__ is_int) {
    extern __shared__ unsigned int s_map[];
    unsigned int* s_run = s_map;
    unsigned int* s_warp = s_map + n;
    for (int g = threadIdx.x; g < n; g += 256) s_run[g] = 0;
    const int64_t base = (int64_t)blockIdx.x * kCompactTile;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int k0 = 0; k0 < kCompactTile; k0 += 256) {
        for (int q = threadIdx.x; q < n * 8; q += 256) s_warp[q] = 0;
        __syncthreads();
        const int64_t i = base + k0 + threadIdx.x;
        double val = 0.0;
        uint8_t as_int = 0;
        const int g = i < cells ? status_map_cell(in, n, i, val, as_int) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, g);
        if (g >= 0 && lane == __ffs(peers) - 1) s_warp[g * 8 + w] = __popc(peers);
        __syncthreads();
        if (g >= 0) {
            unsigned long long pos = off[(int64_t)g * nb + blockIdx.x] + s_run[g] + __popc(peers & ((1u << lane) - 1u));
            for (int q = 0; q < w; ++q) pos += s_warp[g * 8 + q];
            keys[pos] = i;
            vals[pos] = val;
            is_int[pos] = as_int;
        }
        __syncthreads();
        for (int q = threadIdx.x; q < n; q += 256) {
            unsigned int t = 0;
            for (int x = 0; x < 8; ++x) t += s_warp[q * 8 + x];
            s_run[q] += t;
        }
        __syncthreads();
    }
}

}  // namespace olap
