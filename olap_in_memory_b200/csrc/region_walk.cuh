// The region walk, shared by region_kernel (kernels_region.cuh, nvcc) and the fused formula region kernels
// (jit_eval.cuh, NVRTC): 32-bit magic division, the index fields of a lowered region, and the source offset
// of one work item.  The library embeds this file as a string (Makefile) and hands it to NVRTC as an
// in-memory header, so both compilers walk a region with the same code.  It must stay dependency-free.
#pragma once
#ifdef __CUDACC_RTC__
typedef unsigned int uint32_t;
typedef long long int64_t;
#else
#include <stdint.h>
#endif

namespace olap {

constexpr int kWalkMaxDims = 16;  // OLAP_MAX_DIMS (include/olap_gpu.h)

// Division by a runtime constant without the 64-bit divide unit.
struct FastDiv {
    uint32_t d = 1, mul = 0, shift = 0;
#ifndef __CUDACC_RTC__
    FastDiv() {}
    explicit FastDiv(uint32_t div) : d(div) {
        // round-up method valid for n < 2^31
        if (div <= 1) { mul = 0; shift = 0; return; }
        uint32_t l = 0;
        while ((1ull << l) < div) ++l;
        shift = l;
        mul = (uint32_t)(((1ull << 32) * ((1ull << l) - div)) / div + 1);
    }
#endif
    __host__ __device__ __forceinline__ uint32_t div(uint32_t n) const {
        if (d == 1) return n;
#ifdef __CUDA_ARCH__
        uint32_t t = __umulhi(mul, n);
#else
        uint32_t t = (uint32_t)(((uint64_t)mul * n) >> 32);
#endif
        return (t + ((n - t) >> 1)) >> (shift - 1);
    }
};

// The index fields of a region lowered like a dice (plan_region, olap_gpu.cu); same meaning as the fields of
// GatherParams that the walk reads.  Work item t is vector `t % IV` (of VEC cells) of row `t / IV`; the row
// decodes into one table read (or coordinate * lin) per outer axis, innermost last.
struct RegionWalk {
    int nd;                              // outer axes
    uint32_t len[kWalkMaxDims];          // items of each outer axis
    FastDiv div[kWalkMaxDims];
    const int64_t* tbl[kWalkMaxDims];    // source offset per item, or
    int64_t lin[kWalkMaxDims];           // nullptr: the offset is item * lin[d]
    uint32_t IV;                         // inner run / VEC
    FastDiv div_iv;
    int64_t n_vec;                       // rows * IV work items
    int big;                             // n_vec or an axis >= 2^31: 64-bit division instead of FastDiv
};

// source offset (in cells) of work item t; `q` is a RegionWalk or a GatherParams
template <class Ix>
__device__ __forceinline__ int64_t walk_offset(const Ix& q, int big, int64_t t, int vec) {
    int64_t row, off;
    if (big) {
        row = t / q.IV;
        off = (t - row * q.IV) * vec;
        for (int d = q.nd - 1; d >= 0; --d) {
            const int64_t r = row / q.len[d];
            const uint32_t c = (uint32_t)(row - r * q.len[d]);
            row = r;
            off += q.tbl[d] ? q.tbl[d][c] : (int64_t)c * q.lin[d];
        }
        return off;
    }
    uint32_t rest = q.div_iv.div((uint32_t)t);
    off = (int64_t)((uint32_t)t - rest * q.IV) * vec;
    for (int d = q.nd - 1; d >= 0; --d) {
        const uint32_t r = q.div[d].div(rest);
        const uint32_t c = rest - r * q.len[d];
        rest = r;
        off += q.tbl[d] ? q.tbl[d][c] : (int64_t)c * q.lin[d];
    }
    return off;
}

__device__ __forceinline__ int64_t region_offset(const RegionWalk& w, int64_t t, int vec) { return walk_offset(w, w.big, t, vec); }

}  // namespace olap
