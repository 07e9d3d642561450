// Region queries over ONE store: getTotalForDimensionItems (cube.js) as a double sum of the raw cells of
// the cartesian product keep[0] x ... x keep[ndim-1] of per-axis item lists, and copyMeasureData as
// dst.setValue(i, src.getValue(i)) for every cell i of that product.
//
// The region is lowered exactly like a dice (kernels_gather.cuh): one int64 offset table per filtered axis
// (or a stride for an axis taken whole and in order), neighbouring whole axes merged, and the trailing whole
// axes merged into one contiguous inner run of I cells.  Work item t is vector `t % IV` of row `t / IV`; the
// row decodes into one table read per outer axis with 32-bit magic division (GatherParams).  Repeated items
// are table entries like any other, and the multiplicity of filter keys that are not dimensions is a leading
// axis whose table is all zeros.
#pragma once
#include "common.cuh"
#include "kernels_gather.cuh"
#include "kernels_store.cuh"
#include "region_walk.cuh"

namespace olap {

static_assert(kWalkMaxDims == OLAP_MAX_DIMS, "region_walk.cuh sizes its tables for OLAP_MAX_DIMS");

enum RegionOp { REGION_SUM = 0, REGION_COPY = 1 };

struct RegionParams {
    GatherParams ix;          // nd / len / div / tbl / lin, I / IV / div_iv, n_vec (meas, aux unused)
    int big;                  // n_vec or a row index >= 2^31: 64-bit division instead of FastDiv
    const float* src;         // values of the source, advanced by the constant offset of dropped one-item axes
    float* dst;               // REGION_COPY: values of the target (same offsets)
    uint8_t* st_dst;          // REGION_COPY: status plane of the target (nullable)
    int dst_nan_default;
    double* partial;          // REGION_SUM: one partial per CTA
    unsigned int* ticket;     // REGION_SUM: CTAs done (the last one folds the partials)
    double* out;
};

// source offset (in cells, relative to src) of work item t: the walk of region_walk.cuh, which the NVRTC
// formula region kernels (jit_eval.cuh) share
__device__ __forceinline__ int64_t region_offset(const RegionParams& p, int64_t t, int vec) { return walk_offset(p.ix, p.big, t, vec); }

// One grid-stride loop, U vectors of VEC cells in flight per thread.
// REGION_SUM adds the raw floats in double (the status plane is never read: an unset cell holds the
// default, which is what getSingleData returns for it); per-CTA partials are folded by the last CTA in
// a fixed order, so a given region on a given grid always gives the same bits (as total_kernel).
// REGION_COPY applies setValue's element body (set_cell, shared with set_values_kernel) to the source's
// raw value at the same offset of the target.  Source and target may be the same store: the loads are
// plain (not .nc) and a repeated item writes the same value to the same cell again.
// Min-blocks bound: 4 CTAs of 256 (64 registers) for both: U int64 offsets and U float4 in flight, plus U
// double accumulators for the sum; the copy spills at 8 CTAs (32 registers).
template <int OP, int VEC>
__global__ void __launch_bounds__(256, 4) region_kernel(const __grid_constant__ RegionParams p) {
    constexpr int U = 4;
    const int64_t n = p.ix.n_vec;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    double accs[U] = {0.0, 0.0, 0.0, 0.0};
    for (int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t0 < n; t0 += U * stride) {
        int64_t off[U];
        float v[U][VEC];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t t = t0 + u * stride;
            off[u] = t < n ? region_offset(p, t, VEC) : -1;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (off[u] < 0) continue;
            if (VEC == 4) {
                const float4 x = OP == REGION_SUM ? ld_stream4(p.src + off[u]) : *reinterpret_cast<const float4*>(p.src + off[u]);
                v[u][0] = x.x; v[u][1 % VEC] = x.y; v[u][2 % VEC] = x.z; v[u][3 % VEC] = x.w;
            } else {
                v[u][0] = OP == REGION_SUM ? ld_stream1(p.src + off[u]) : p.src[off[u]];
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (off[u] < 0) continue;
            if (OP == REGION_SUM) {
#pragma unroll
                for (int e = 0; e < VEC; ++e) accs[u] += (double)v[u][e];
            } else {
                uint32_t so = 0;
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    uint8_t s;
                    v[u][e] = set_cell(v[u][e], p.dst_nan_default, s);
                    so |= (uint32_t)s << (8 * e);
                }
                if (VEC == 4) {
                    *reinterpret_cast<float4*>(p.dst + off[u]) = make_float4(v[u][0], v[u][1 % VEC], v[u][2 % VEC], v[u][3 % VEC]);
                    if (p.st_dst) *reinterpret_cast<uint32_t*>(p.st_dst + off[u]) = so;
                } else {
                    p.dst[off[u]] = v[u][0];
                    if (p.st_dst) p.st_dst[off[u]] = (uint8_t)so;
                }
            }
        }
    }
    if (OP != REGION_SUM) return;

    __shared__ double s_sum[256 / 32];
    __shared__ bool s_last;
    double acc = warp_sum((accs[0] + accs[1]) + (accs[2] + accs[3]));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) s_sum[w] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0;
        for (int k = 0; k < 256 / 32; ++k) a += s_sum[k];
        p.partial[blockIdx.x] = a;
        __threadfence();
        s_last = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    double a = 0.0;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) a += ((volatile double*)p.partial)[b];
    a = warp_sum(a);
    __syncthreads();
    if (l == 0) s_sum[w] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        double ta = 0.0;
        for (int k = 0; k < 256 / 32; ++k) ta += s_sum[k];
        *p.out = ta;
        *p.ticket = 0;
    }
}

}  // namespace olap
