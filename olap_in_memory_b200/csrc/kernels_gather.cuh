// Output-driven gather kernels: dice (in-memory.js:213-263), reorder (178-211),
// drillDown (336-430) and the scatter of load (139-176).
//
// All four are "re-index every cell through one small table per dimension".  The host
// folds each dimension's map and the source stride into an int64 offset table
//     tbl_d[new coordinate] = old coordinate * old stride
// so the source offset of an output cell is a sum of D table reads.  Trailing
// dimensions that are untouched and contiguous on both sides are merged into an inner
// run of length I that is moved with 128-bit accesses.
#pragma once
#include <algorithm>
#include <numeric>

#include "common.cuh"

namespace olap {

struct GatherMeasure {
    const float* in;
    float* out;
    const uint8_t* st_in;
    uint8_t* st_out;
    const double* dist;  // drillDown distributions (nullable)
    int64_t dist_len;
    int nan_default;
    int int_rounding;  // store type is int32/uint32 (in-memory.js:343)
    int method_is_sum;
    // st_in == nullptr, st_out != nullptr: the source's status plane follows from its values (olap_store::derived);
    // a COPY gather then writes  set ? SET : UNSET  from the cells it moves and never reads the plane
    int derive = 0;
};

// drillDown bookkeeping of one new item: siblings under its parent, rank among them
// (ascending new index), and 1.0 / siblings.
struct DownAux {
    int32_t cnt, rank;
    double inv;
};

// one new-side dimension of a gather: either linear (offset = coord * stride) or a table
struct GDim {
    int64_t len = 1;
    bool linear = true;
    int64_t stride = 0;
    std::vector<int64_t> tbl;
    std::vector<DownAux> aux;  // drillDown only
};

enum GatherMode { G_COPY = 0, G_DOWN = 1, G_DOWN_FLOAT = 2 };  // G_DOWN_FLOAT: float cells, method sum, no distributions

struct GatherParams {
    const GatherMeasure* meas;
    int nd;                              // outer dimensions (tables)
    uint32_t len[OLAP_MAX_DIMS];         // new length of each outer dimension
    FastDiv div[OLAP_MAX_DIMS];
    const int64_t* tbl[OLAP_MAX_DIMS];   // source offset contribution per new coordinate, or
    int64_t lin[OLAP_MAX_DIMS];          // nullptr: the contribution is coordinate * lin[d]
    const DownAux* aux[OLAP_MAX_DIMS];   // drillDown: siblings / rank / 1/siblings per new item; nullable
    int n_aux;                           // how many dimensions carry aux
    int64_t I;                           // inner run (elements), contiguous on both sides
    uint32_t IV;                         // I / VEC
    FastDiv div_iv;
    int64_t n_vec;                       // rows * IV
    int64_t rows;
    int64_t new_size, old_size;          // for the distributions index formula
    int* error_flag;                     // set to 1 + dist index when a distribution is missing
};

// in-memory.js:383-427 for one cell: `v` parent value, `n` siblings, `k` rank.
// `inv` = 1.0 / n, computed once per thread.  For the float path the reference computes
// fround(v / n) in double; v * (1/n) differs from v / n by < 2^-52 relative, and v / n
// (v float32, n < 2^20) is never that close to a float32 rounding boundary, so the float32
// result is identical; larger n take the exact division.
__device__ __forceinline__ float down_value(const GatherMeasure& m, const GatherParams& p, float v, uint32_t n,
                                            double inv, uint32_t k, int64_t new_idx, bool& ok) {
    ok = false;
    if (v == 0.0f || v != v) return default_of(m.nan_default);  // `if (!oldValue) continue`
    double r;
    if (m.dist) {
        const int64_t added = p.new_size / p.old_size;
        const int64_t shared = m.dist_len / added;
        const int64_t di = (new_idx / (p.new_size / (shared > 0 ? shared : 1))) * added + (new_idx % added);
        const double w = (di >= 0 && di < m.dist_len) ? m.dist[di] : __longlong_as_double(0x7ff8000000000000ll);
        if (w != w) {
            atomicCAS(p.error_flag, 0, (int)(di < 0x7ffffffe ? di + 1 : 0x7fffffff));
            return default_of(m.nan_default);
        }
        r = (double)v * w;
    } else if (m.method_is_sum) {
        if (m.int_rounding) {
            // floor(v/n), v % n (sign of the dividend), then the reference's spreading rule
            const double dv = (double)v, dn = (double)n;
            const double quot = dv / dn;
            const double base = floor(quot);
            const double rem = fma(-trunc(quot), dn, dv);  // == fmod(v, n): exact in double
            const double step = rem / dn;
            const bool last_is_same = floor((double)k * step) == floor(((double)k - 1.0) * step);
            r = last_is_same ? base : base + 1.0;
        } else {
            r = n < (1u << 20) ? (double)v * inv : (double)v / (double)n;
        }
    } else {
        r = (double)v;
    }
    const float f = canon_store((float)r, m.nan_default);
    ok = present_f(f, m.nan_default);
    return f;
}

template <int MODE, int VEC, bool BIG>
__global__ void __launch_bounds__(256, MODE == G_COPY ? 8 : 4) gather_kernel(const __grid_constant__ GatherParams p) {
    constexpr int U = 2;  // independent vectors per thread
    const GatherMeasure m = p.meas[blockIdx.y];
    const int64_t base = (int64_t)blockIdx.x * (256 * U) + threadIdx.x;

    int64_t src_off[U], dst_off[U];
    uint32_t sib[U], rank[U];
    double inv_of[U];
    bool live[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int64_t t = base + u * 256;
        live[u] = t < p.n_vec;
        int64_t row;
        uint32_t colv;
        if (BIG) {
            row = t / p.IV;
            colv = (uint32_t)(t - row * p.IV);
        } else {
            const uint32_t r32 = p.div_iv.div((uint32_t)t);
            colv = (uint32_t)t - r32 * p.IV;
            row = r32;
        }
        int64_t off = (int64_t)colv * VEC;
        dst_off[u] = row * p.I + off;
        uint32_t n = 1, k = 0;
        double inv1 = 1.0;
        if (live[u]) {
            if (BIG) {
                int64_t rest = row;
                for (int d = p.nd - 1; d >= 0; --d) {
                    const int64_t q = rest / p.len[d];
                    const uint32_t c = (uint32_t)(rest - q * p.len[d]);
                    rest = q;
                    off += p.tbl[d] ? p.tbl[d][c] : (int64_t)c * p.lin[d];
                    if (MODE != G_COPY && p.aux[d]) {
                        const DownAux a = p.aux[d][c];
                        k += (uint32_t)a.rank * n;  // ranks compose last-dimension-fastest
                        n *= (uint32_t)a.cnt;
                        inv1 = a.inv;
                    }
                }
            } else {
                uint32_t rest = (uint32_t)row;
                for (int d = p.nd - 1; d >= 0; --d) {
                    const uint32_t q = p.div[d].div(rest);
                    const uint32_t c = rest - q * p.len[d];
                    rest = q;
                    off += p.tbl[d] ? p.tbl[d][c] : (int64_t)c * p.lin[d];
                    if (MODE != G_COPY && p.aux[d]) {
                        const DownAux a = p.aux[d][c];
                        k += (uint32_t)a.rank * n;
                        n *= (uint32_t)a.cnt;
                        inv1 = a.inv;
                    }
                }
            }
        }
        src_off[u] = off;
        sib[u] = n;
        rank[u] = k;
        inv_of[u] = inv1;
    }

    float v[U][VEC];
    uint32_t s[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        s[u] = 0;
        if (!live[u]) continue;
        if (VEC == 4) {
            const float4 t = ld_stream4(m.in + src_off[u]);
            v[u][0] = t.x; v[u][1 % VEC] = t.y; v[u][2 % VEC] = t.z; v[u][3 % VEC] = t.w;
            if (m.st_in) s[u] = ld_stream_u32(m.st_in + src_off[u]);
        } else {
            v[u][0] = ld_stream1(m.in + src_off[u]);
            if (m.st_in) s[u] = m.st_in[src_off[u]];
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!live[u]) continue;
        if (MODE != G_COPY) {
            uint32_t so = 0;
            const double inv = p.n_aux == 1 ? inv_of[u] : 1.0 / (double)sib[u];
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                bool ok;
                if (MODE == G_DOWN_FLOAT) {
                    // fround(v / n) for a truthy parent, else unset (in-memory.js:386-387, 419)
                    const float x = v[u][e];
                    const float r = canon_store((float)(sib[u] < (1u << 20) ? (double)x * inv : (double)x / (double)sib[u]),
                                                m.nan_default);
                    const bool truthy = x != 0.0f && x == x;
                    v[u][e] = truthy ? r : default_of(m.nan_default);
                    ok = truthy && present_f(r, m.nan_default);
                } else {
                    v[u][e] = down_value(m, p, v[u][e], sib[u], inv, rank[u], dst_off[u] + e, ok);
                }
                const uint32_t sb = (s[u] >> (8 * e)) & 0xffu;
                so |= (ok ? ((sb | OLAP_STATUS_INTERPOLATED) & 0xffu) : (uint32_t)OLAP_STATUS_UNSET) << (8 * e);
            }
            s[u] = so;
        }
        if (MODE == G_COPY && m.derive) {
            s[u] = 0;
#pragma unroll
            for (int e = 0; e < VEC; ++e)
                s[u] |= (present_f(v[u][e], m.nan_default) ? (uint32_t)OLAP_STATUS_SET : (uint32_t)OLAP_STATUS_UNSET) << (8 * e);
        }
        if (VEC == 4) {
            st_stream4(m.out + dst_off[u], make_float4(v[u][0], v[u][1 % VEC], v[u][2 % VEC], v[u][3 % VEC]));
            if (m.st_out) *reinterpret_cast<uint32_t*>(m.st_out + dst_off[u]) = s[u];
        } else {
            m.out[dst_off[u]] = v[u][0];
            if (m.st_out) m.st_out[dst_off[u]] = (uint8_t)s[u];
        }
    }
}

// ---- scalar gathers, amortised: gather_rows_kernel ------------------------------------
// When the innermost output axis cannot be moved with 128-bit accesses (it is diced /
// drilled itself, or shorter than 4), the per-element cost of gather_kernel is the full
// index decode.  Here a CTA owns RB consecutive output rows (a row = the innermost axis, L
// cells): RB threads decode one row each (source offset, drillDown sibling count / rank)
// into shared memory, the innermost axis' table sits in shared memory too, and every
// element then costs one division by L, two shared-memory reads, one load, one store.
// Output is written as one contiguous span.
constexpr int kRowsMaxL = 1024;
constexpr int kRowsPerBlock = 256;

struct RowsTail {
    uint32_t L;
    FastDiv div_l;
    const int64_t* tbl;   // source offset per innermost coordinate (nullptr: coordinate * lin)
    int64_t lin;
    const DownAux* aux;   // drillDown aux of the innermost axis (nullable)
    uint32_t RB;          // rows per CTA
    int64_t rows;
};

template <int MODE>
__global__ void __launch_bounds__(256) gather_rows_kernel(const __grid_constant__ GatherParams p,
                                                          const __grid_constant__ RowsTail tail) {
    __shared__ int64_t s_off[kRowsPerBlock];
    __shared__ uint32_t s_n[kRowsPerBlock], s_k[kRowsPerBlock];
    __shared__ int64_t s_tbl[kRowsMaxL];
    __shared__ DownAux s_aux[MODE == G_COPY ? 1 : kRowsMaxL];
    const GatherMeasure m = p.meas[blockIdx.y];
    const int64_t row0 = (int64_t)blockIdx.x * tail.RB;
    const uint32_t rows = (uint32_t)min((int64_t)tail.RB, tail.rows - row0);
    for (uint32_t c = threadIdx.x; c < tail.L; c += 256) {
        s_tbl[c] = tail.tbl ? tail.tbl[c] : (int64_t)c * tail.lin;
        if (MODE != G_COPY) s_aux[c] = tail.aux ? tail.aux[c] : DownAux{1, 0, 1.0};
    }
    if (threadIdx.x < rows) {
        uint32_t rest = (uint32_t)(row0 + threadIdx.x);
        int64_t off = 0;
        uint32_t n = 1, k = 0;
        for (int d = p.nd - 1; d >= 0; --d) {
            const uint32_t q = p.div[d].div(rest);
            const uint32_t c = rest - q * p.len[d];
            rest = q;
            off += p.tbl[d] ? p.tbl[d][c] : (int64_t)c * p.lin[d];
            if (MODE != G_COPY && p.aux[d]) {
                const DownAux a = p.aux[d][c];
                k += (uint32_t)a.rank * n;
                n *= (uint32_t)a.cnt;
            }
        }
        s_off[threadIdx.x] = off;
        s_n[threadIdx.x] = n;
        s_k[threadIdx.x] = k;
    }
    __syncthreads();
    const uint32_t cells = rows * tail.L;
    const int64_t base = row0 * tail.L;
    constexpr int U = 4;
    for (uint32_t t0 = threadIdx.x; t0 < cells; t0 += 256 * U) {
        float v[U];
        uint32_t sb[U], rr[U], cc[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t t = t0 + u * 256;
            if (t < cells) {
                rr[u] = tail.div_l.div(t);
                cc[u] = t - rr[u] * tail.L;
                const int64_t off = s_off[rr[u]] + s_tbl[cc[u]];
                v[u] = ld_stream1(m.in + off);
                sb[u] = m.st_in ? (uint32_t)m.st_in[off] : 0u;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t t = t0 + u * 256;
            if (t >= cells) continue;
            float r = v[u];
            uint32_t so = sb[u];
            if (MODE != G_COPY) {
                const DownAux a = s_aux[cc[u]];
                const uint32_t n = s_n[rr[u]] * (uint32_t)a.cnt;
                const uint32_t k = s_k[rr[u]] * (uint32_t)a.cnt + (uint32_t)a.rank;
                const double inv = s_n[rr[u]] == 1 ? a.inv : 1.0 / (double)n;
                bool ok;
                if (MODE == G_DOWN_FLOAT) {
                    const float x = v[u];
                    const float q = canon_store((float)(n < (1u << 20) ? (double)x * inv : (double)x / (double)n), m.nan_default);
                    const bool truthy = x != 0.0f && x == x;
                    r = truthy ? q : default_of(m.nan_default);
                    ok = truthy && present_f(q, m.nan_default);
                } else {
                    r = down_value(m, p, v[u], n, inv, k, base + t, ok);
                }
                so = ok ? ((sb[u] | OLAP_STATUS_INTERPOLATED) & 0xffu) : (uint32_t)OLAP_STATUS_UNSET;
            }
            m.out[base + t] = r;
            if (m.st_out) m.st_out[base + t] = (uint8_t)so;
        }
    }
}

// Drop single-item dimensions (their constant offset goes to `const_off`) and merge
// neighbours that stay adjacent and contiguous in the source.
inline void merge_dims(std::vector<GDim>& dims, int64_t* const_off) {
    std::vector<GDim> out;
    for (auto& d : dims) {
        if (d.len == 1) {
            if (!d.linear) *const_off += d.tbl[0];
            continue;  // aux of a single item is {1 sibling, rank 0}: neutral
        }
        if (!out.empty() && out.back().linear && d.linear && out.back().stride == d.len * d.stride) {
            out.back().len *= d.len;
            out.back().stride = d.stride;
        } else {
            out.push_back(std::move(d));
        }
    }
    dims.swap(out);
}

// ---- rearrangements inside short contiguous blocks: gather_inner_flat_kernel -------------
// [R, D] -> [R, K] with the leading axes untouched: dice / slice of the innermost axes (in-memory.js:213-263) and
// reorders that only swap trailing axes (in-memory.js:178-211; keep[] is then a permutation of the block):
// the source rows are ONE contiguous span, so nothing has to be decoded per row, and a tile of RB rows looks the
// same wherever it starts: output j of a tile always comes from cell (j / K) * D + keep[j % K] of the tile.
// A persistent CTA computes that offset ONCE for each of the <= 32 outputs a thread owns per tile (consecutive
// lanes, consecutive outputs), then for every tile: stages the RB rows with 16-byte cp.async copies, all in
// flight at once (every sector of the span is touched anyway: kept and dropped cells share sectors) and per output issues one shared load and one
// coalesced store (values: 128 bytes per warp, status: one full 32-byte sector per warp).
// gather_rows_kernel spends a row decode (one division per outer axis) per row of K outputs and a division per
// cell: 1.1e9 warp instructions on every-other of a 10-item axis of 1e9 cells (ncu: issue-bound, 0.48 of peak).
constexpr int kFlatCells = 8192;

struct FlatParams {
    const GatherMeasure* meas;
    const int32_t* keep;   // [K] source offset of every kept item inside a row
    int64_t rows;
    uint32_t D, K, RB, n_tiles;
    FastDiv div_k;
    FastDiv div_rb;        // FRONT: the block's axes move to the FRONT of the output ([R, D] -> [K, R]); RB % 256 == 0
};

// Output j of a tile (consecutive lanes, consecutive j) is row r of the tile and position k of the block; it comes
// from cell r * D + keep[k] of the staged span.  Shared by the kernel and the CPU emulation (tests/host/plan_check.cu).
struct FlatIdx { uint32_t r, k; };
__host__ __device__ __forceinline__ FlatIdx flat_split(const FlatParams& p, bool front, uint32_t j) {
    FlatIdx ix;
    if (front) { ix.k = p.div_rb.div(j); ix.r = j - ix.k * p.RB; }
    else { ix.r = p.div_k.div(j); ix.k = j - ix.r * p.K; }
    return ix;
}

// Host side of gather_inner_flat_kernel.  `dims` is the gather in output order (GDim: length and source stride or
// offset table per output axis).  The untouched leading axes of the source merge into one linear "row" axis whose
// stride D is the block length; they are either still the leading axes of the output (rows first: the block stays
// innermost) or its trailing axes (rows last: the block's axes moved to the FRONT).
struct FlatPlan {
    bool use = false, front = false;
    int64_t rows = 0, D = 0, K = 0, RB = 0, const_off = 0;
    std::vector<int32_t> keep;  // [K] source offset inside a block of every output position of the block (row-major)
};

inline FlatPlan flat_plan(std::vector<GDim> dims, int64_t src_size) {
    FlatPlan plan;
    int64_t const_off = 0;
    merge_dims(dims, &const_off);
    if (dims.size() < 2 || const_off % 16) return plan;
    const GDim& lead = dims[0];
    const GDim& tail = dims.back();
    bool front = false;
    auto block_inside = [&](size_t first, size_t last, int64_t D) {  // every offset of axes [first, last] stays in [0, D)
        int64_t hi = 0;
        for (size_t d = first; d <= last; ++d) {
            if (!dims[d].aux.empty()) return false;
            int64_t lo_d = 0, hi_d = 0;
            if (dims[d].linear) { hi_d = (dims[d].len - 1) * dims[d].stride; if (dims[d].stride < 0) return false; }
            else for (int64_t v : dims[d].tbl) { lo_d = std::min(lo_d, v); hi_d = std::max(hi_d, v); }
            if (lo_d < 0) return false;
            hi += hi_d;
        }
        return hi < D;
    };
    if (lead.linear && lead.aux.empty() && lead.stride >= 2 && lead.stride <= kFlatCells && block_inside(1, dims.size() - 1, lead.stride)) front = false;
    else if (tail.linear && tail.aux.empty() && tail.stride >= 2 && tail.stride <= 32 && block_inside(0, dims.size() - 2, tail.stride)) front = true;
    else return plan;
    const GDim& row_axis = front ? tail : lead;
    const size_t b0 = front ? 0 : 1, b1 = front ? dims.size() - 2 : dims.size() - 1;  // the block's axes, in output order
    const int64_t rows = row_axis.len, D = row_axis.stride;
    if (rows < 64 || rows >= ((int64_t)1 << 31) || const_off + rows * D > src_size) return plan;  // whole blocks are staged
    // long 128-bit inner runs are the vector gather's (0.87-0.94 of peak)
    if (!front && tail.linear && tail.stride == 1 && tail.len % 4 == 0 && tail.len >= 16) return plan;
    int64_t K = 1;
    for (size_t d = b0; d <= b1; ++d) {
        K *= dims[d].len;
        if (K > D || K < 1) return plan;
    }
    plan.keep.resize((size_t)K);
    for (int64_t k = 0; k < K; ++k) {  // row-major over the block's output axes
        int64_t rest = k, off = 0;
        for (size_t d = b1 + 1; d-- > b0;) {
            const int64_t c = rest % dims[d].len;
            rest /= dims[d].len;
            off += dims[d].linear ? c * dims[d].stride : dims[d].tbl[(size_t)c];
        }
        plan.keep[(size_t)k] = (int32_t)off;
    }
    // rows per tile: spans start on 16 cells (16-byte copies of values and of status bytes); FRONT: whole groups of
    // 256 rows, so that the plane a thread writes to depends on the loop index only
    const int64_t step = front ? 256 : 16 / std::gcd<int64_t, int64_t>(D, 16);
    const int64_t RB = (kFlatCells / D) / step * step;
    if (RB < 1) return plan;
    // consecutive lanes read neighbouring outputs: decline patterns that pile onto few shared-memory banks
    {
        const int64_t tile_out = RB * K;
        int64_t conflicts = 0, warps = 0;
        for (int64_t j0 = 0; j0 < tile_out; j0 += 32, ++warps) {
            int bank[32] = {0};
            int worst = 0;
            for (int64_t j = j0; j < std::min(tile_out, j0 + 32); ++j) {
                const int64_t cell = front ? (j % RB) * D + plan.keep[(size_t)(j / RB)] : (j / K) * D + plan.keep[(size_t)(j % K)];
                worst = std::max(worst, ++bank[cell & 31]);
            }
            conflicts += worst;
        }
        if (conflicts > 4 * warps) return plan;
    }
    plan.use = true;
    plan.front = front;
    plan.rows = rows; plan.D = D; plan.K = K; plan.RB = RB; plan.const_off = const_off;
    return plan;
}

__device__ __forceinline__ void flat_cp_async16(void* smem_dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(src) : "memory");
}

// E: outputs per thread and tile (the smallest of 8 / 16 / 32 that covers RB * K / 256); MINB: CTAs per SM the
// register allocation aims at (32 offsets per thread do not fit the 64 registers of 4 CTAs)
// FRONT: the rearranged block does not stay innermost but becomes the OUTERMOST part of the output ([R, D] -> [K, R]:
// a short innermost axis rotated to the front): output k of row r goes to plane k, cell r — a tile writes K runs
// of RB consecutive cells instead of one span.  Thread t owns rows t, t + 256, ... of every plane.
template <int E, int MINB, bool FRONT>
static __global__ void __launch_bounds__(256, MINB) gather_inner_flat_kernel(const __grid_constant__ FlatParams p) {
    extern __shared__ __align__(16) unsigned char smem_flat[];
    float* s_val = reinterpret_cast<float*>(smem_flat);           // [RB * D]
    uint8_t* s_st = smem_flat + (size_t)p.RB * p.D * 4;            // [RB * D]
    const GatherMeasure m = p.meas[blockIdx.y];
    // where my outputs of a tile come from (the same for every tile)
    uint32_t off[E];
    const uint32_t tile_out = p.RB * p.K;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const uint32_t j = threadIdx.x + 256u * e;
        off[e] = 0;
        if (j < tile_out) {
            const FlatIdx ix = flat_split(p, FRONT, j);
            off[e] = ix.r * p.D + (uint32_t)p.keep[ix.k];
        }
    }
    const bool load_plane = m.st_in != nullptr, write_plane = m.st_out != nullptr, nan_default = m.nan_default != 0;
    for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * p.RB;
        const uint32_t rows = (uint32_t)min((int64_t)p.RB, p.rows - row0);
        const uint32_t n_in = rows * p.D, n_out = rows * p.K;
        const float* g_in = m.in + row0 * p.D;
        const uint8_t* g_st = load_plane ? m.st_in + row0 * p.D : nullptr;
        // the span starts on 16 bytes (RB * D is a multiple of 16 cells): asynchronous 16-byte copies, all in flight
        for (uint32_t i = threadIdx.x * 4; i + 4 <= n_in; i += 1024) flat_cp_async16(s_val + i, g_in + i);
        if (load_plane)
            for (uint32_t i = threadIdx.x * 16; i + 16 <= n_in; i += 4096) flat_cp_async16(s_st + i, g_st + i);
        asm volatile("cp.async.commit_group;" ::: "memory");
        for (uint32_t i = (n_in & ~3u) + threadIdx.x; i < n_in; i += 256) s_val[i] = g_in[i];
        if (load_plane)
            for (uint32_t i = (n_in & ~15u) + threadIdx.x; i < n_in; i += 256) s_st[i] = g_st[i];
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        if (FRONT) {
            float* g_out = m.out + row0;
            uint8_t* g_so = write_plane ? m.st_out + row0 : nullptr;
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const uint32_t j = threadIdx.x + 256u * e;
                const FlatIdx ix = flat_split(p, true, j);  // the plane k is warp-uniform (RB % 256 == 0)
                const uint32_t k = ix.k, r = ix.r;
                if (k < p.K && r < rows) {
                    const int64_t g = (int64_t)k * p.rows + r;
                    const float v = s_val[off[e]];
                    g_out[g] = v;
                    if (write_plane)
                        g_so[g] = load_plane ? s_st[off[e]] : (uint8_t)(present_f(v, nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET);
                }
            }
        } else {
        float* g_out = m.out + row0 * p.K + threadIdx.x;
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (threadIdx.x + 256u * e < n_out) g_out[256 * e] = s_val[off[e]];
        if (write_plane) {
            uint8_t* g_so = m.st_out + row0 * p.K + threadIdx.x;
            if (load_plane) {
#pragma unroll
                for (int e = 0; e < E; ++e)
                    if (threadIdx.x + 256u * e < n_out) g_so[256 * e] = s_st[off[e]];
            } else if (nan_default) {  // derived plane
#pragma unroll
                for (int e = 0; e < E; ++e)
                    if (threadIdx.x + 256u * e < n_out) g_so[256 * e] = (uint8_t)(present_f(s_val[off[e]], 1) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET);
            } else {
#pragma unroll
                for (int e = 0; e < E; ++e)
                    if (threadIdx.x + 256u * e < n_out) g_so[256 * e] = (uint8_t)(present_f(s_val[off[e]], 0) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET);
            }
        }
        }
        __syncthreads();  // the next tile overwrites the staged rows
    }
}

// ---- the mirror image of FRONT: gather_planes_flat_kernel --------------------------------
// [K, R] -> [R, K]: short OUTER axes (K <= 32 planes of the source, anywhere in it) become the innermost axes of
// the output.  A tile is RB consecutive rows: K runs of RB cells are staged (16-byte cp.async for the values,
// 4-byte for the status bytes; plane pitch RB + 4: the fold reads at 4 k + r, conflict-free up to 8 planes, 2-way
// beyond), then the RB * K outputs leave as ONE contiguous span, consecutive lanes consecutive cells.
struct PlanesParams {
    const GatherMeasure* meas;
    const int64_t* plane_off;  // [K] source offset of plane k (cells, multiples of 4)
    int64_t rows;
    uint32_t K, RB, n_tiles;
    FastDiv div_k, div_rb4;
};

// Host side: `dims` in output order — the row axis comes first and is contiguous in the source, the trailing
// output axes select one of K <= 32 planes (any offsets that are multiples of 4 cells).
struct PlanesPlan {
    bool use = false;
    int64_t rows = 0, K = 0, RB = 0;
    std::vector<int64_t> plane;  // [K] source offset of every plane (row-major over the trailing output axes)
};

inline PlanesPlan planes_plan(std::vector<GDim> dims, int64_t src_size) {
    PlanesPlan plan;
    int64_t const_off = 0;
    merge_dims(dims, &const_off);
    if (dims.size() < 2 || const_off % 4 || !dims[0].linear || dims[0].stride != 1 || !dims[0].aux.empty()) return plan;
    const int64_t rows = dims[0].len;
    if (rows < 4096 || rows >= ((int64_t)1 << 31)) return plan;
    int64_t K = 1;
    for (size_t d = 1; d < dims.size(); ++d) {
        if (!dims[d].aux.empty()) return plan;
        K *= dims[d].len;
        if (K > 32 || K < 1) return plan;
    }
    if (K < 2) return plan;
    plan.plane.resize((size_t)K);
    for (int64_t k = 0; k < K; ++k) {  // row-major over the trailing output axes
        int64_t rest = k, off = const_off;
        for (size_t d = dims.size(); d-- > 1;) {
            const int64_t c = rest % dims[d].len;
            rest /= dims[d].len;
            off += dims[d].linear ? c * dims[d].stride : dims[d].tbl[(size_t)c];
        }
        if (off < 0 || off % 4 || off + rows > src_size) return plan;
        plan.plane[(size_t)k] = off;
    }
    const int64_t RB = (kFlatCells / K) / 256 * 256;
    if (RB < 256) return plan;
    plan.use = true;
    plan.rows = rows; plan.K = K; plan.RB = RB;
    return plan;
}

template <int E, int MINB>
static __global__ void __launch_bounds__(256, MINB) gather_planes_flat_kernel(const __grid_constant__ PlanesParams p) {
    extern __shared__ __align__(16) unsigned char smem_planes[];
    const uint32_t pitch = p.RB + 4;
    float* s_val = reinterpret_cast<float*>(smem_planes);          // [K][pitch]
    uint8_t* s_st = smem_planes + (size_t)p.K * pitch * 4;         // [K][pitch]
    __shared__ int64_t s_off[32];
    const GatherMeasure m = p.meas[blockIdx.y];
    if (threadIdx.x < p.K) s_off[threadIdx.x] = p.plane_off[threadIdx.x];
    uint32_t off[E];
    const uint32_t tile_out = p.RB * p.K;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const uint32_t j = threadIdx.x + 256u * e;
        off[e] = 0;
        if (j < tile_out) {
            const uint32_t r = p.div_k.div(j), k = j - r * p.K;
            off[e] = k * pitch + r;
        }
    }
    __syncthreads();
    const bool load_plane = m.st_in != nullptr, write_plane = m.st_out != nullptr, nan_default = m.nan_default != 0;
    const uint32_t rb4 = p.RB >> 2;
    for (uint32_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * p.RB;
        const uint32_t rows = (uint32_t)min((int64_t)p.RB, p.rows - row0);
        for (uint32_t c = threadIdx.x; c < p.K * rb4; c += 256) {
            const uint32_t k = p.div_rb4.div(c), i = (c - k * rb4) << 2;
            const int64_t g = s_off[k] + row0 + i;
            if (i + 4 <= rows) {
                flat_cp_async16(s_val + k * pitch + i, m.in + g);
                if (load_plane) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(s_st + k * pitch + i)), "l"(m.st_in + g) : "memory");
            } else {
                for (uint32_t q = i; q < rows; ++q) {  // the ragged end of the last tile
                    s_val[k * pitch + q] = m.in[g + (q - i)];
                    if (load_plane) s_st[k * pitch + q] = m.st_in[g + (q - i)];
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        const uint32_t n_out = rows * p.K;
        float* g_out = m.out + row0 * p.K + threadIdx.x;
#pragma unroll
        for (int e = 0; e < E; ++e)
            if (threadIdx.x + 256u * e < n_out) g_out[256 * e] = s_val[off[e]];
        if (write_plane) {
            uint8_t* g_so = m.st_out + row0 * p.K + threadIdx.x;
            if (load_plane) {
#pragma unroll
                for (int e = 0; e < E; ++e)
                    if (threadIdx.x + 256u * e < n_out) g_so[256 * e] = s_st[off[e]];
            } else {
#pragma unroll
                for (int e = 0; e < E; ++e)
                    if (threadIdx.x + 256u * e < n_out)
                        g_so[256 * e] = (uint8_t)(present_f(s_val[off[e]], nan_default) ? OLAP_STATUS_SET : OLAP_STATUS_UNSET);  // derived plane
            }
        }
        __syncthreads();  // the next tile overwrites the staged runs
    }
}

// ---- load: input-driven scatter  dst[mine(his)] = src[his]  (in-memory.js:159-175).
// Tables hold my offset contribution per his coordinate, or -1 when I lack the item
// (then the cell is dropped).  His items are distinct, so the scatter is injective.
struct ScatterParams {
    const float* src;
    float* dst;
    const uint8_t* st_src;
    uint8_t* st_dst;
    int dst_nan_default;
    int src_nan_default;
    int nd;
    int64_t len[OLAP_MAX_DIMS];
    const int64_t* tbl[OLAP_MAX_DIMS];
    int64_t n;
};

// Status byte of a cell load writes: "status flags are copied between cubes" (README.md:704), but whether the cell
// is set follows MY default.  A set cell takes the source's byte when that byte says set, else SET: a zero-default
// source's unset 0 (0x1) is a set cell of a NaN-default target, and a plane that says UNSET there would no longer
// follow from the values (olap_store::derived).
__device__ __forceinline__ uint32_t load_status(bool set, uint32_t src_byte) {
    if (!set) return OLAP_STATUS_UNSET;
    return (src_byte & OLAP_STATUS_SET) ? src_byte : (uint32_t)OLAP_STATUS_SET;
}

static __global__ void __launch_bounds__(256) load_scatter_kernel(const __grid_constant__ ScatterParams p) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.n) return;
    int64_t rest = t, off = 0;
    bool drop = false;
    for (int d = p.nd - 1; d >= 0; --d) {
        const int64_t q = rest / p.len[d];
        const int64_t c = rest - q * p.len[d];
        rest = q;
        const int64_t o = p.tbl[d][c];
        drop |= o < 0;
        off += o;
    }
    if (drop) return;
    // otherStore.getValue(): unset cells read as HIS default; setValue() applies MY presence rule
    const float v = p.src[t];
    p.dst[off] = canon_store(v, p.dst_nan_default);
    if (p.st_dst) {
        const bool set = present_f(canon_store(v, p.dst_nan_default), p.dst_nan_default);
        p.st_dst[off] = load_status(set, p.st_src ? p.st_src[t] : (uint32_t)OLAP_STATUS_SET);
    }
}

// Same scatter with 32-bit index math and, when the innermost axis of the other store lands
// as one contiguous run in mine (his item j -> my item m0 + j), VEC cells per thread: one
// decode per vector, 128-bit loads and stores.
struct ScatterVecParams {
    const float* src;
    float* dst;
    const uint8_t* st_src;
    uint8_t* st_dst;
    int dst_nan_default;
    int nd;                         // outer axes (tables)
    uint32_t len[OLAP_MAX_DIMS];
    FastDiv div[OLAP_MAX_DIMS];
    const int64_t* tbl[OLAP_MAX_DIMS];
    uint32_t IV;                    // vectors per inner run
    FastDiv div_iv;
    int64_t inner_off;              // my offset of his first inner item
    uint32_t n_vec;
};

template <int VEC>
__global__ void __launch_bounds__(256) load_scatter_vec_kernel(const __grid_constant__ ScatterVecParams p) {
    const uint32_t t = blockIdx.x * 256u + threadIdx.x;
    if (t >= p.n_vec) return;
    uint32_t rest = p.div_iv.div(t);
    int64_t off = p.inner_off + (int64_t)(t - rest * p.IV) * VEC;
    bool drop = false;
    for (int d = p.nd - 1; d >= 0; --d) {
        const uint32_t q = p.div[d].div(rest);
        const int64_t o = p.tbl[d][rest - q * p.len[d]];
        rest = q;
        drop |= o < 0;
        off += o;
    }
    if (drop) return;
    const int64_t s0 = (int64_t)t * VEC;
    float v[VEC];
    if (VEC == 4) {
        const float4 x = ld_stream4(p.src + s0);
        v[0] = x.x; v[1 % VEC] = x.y; v[2 % VEC] = x.z; v[3 % VEC] = x.w;
    } else {
        v[0] = ld_stream1(p.src + s0);
    }
    uint32_t sb = 0;
    if (p.st_dst && p.st_src) {
        if (VEC == 4) sb = ld_stream_u32(p.st_src + s0);
        else sb = p.st_src[s0];
    }
    uint32_t so = 0;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        v[e] = canon_store(v[e], p.dst_nan_default);
        const bool set = present_f(v[e], p.dst_nan_default);
        so |= load_status(set, p.st_src ? (sb >> (8 * e)) & 0xffu : (uint32_t)OLAP_STATUS_SET) << (8 * e);
    }
    if (VEC == 4) {
        st_stream4(p.dst + off, make_float4(v[0], v[1 % VEC], v[2 % VEC], v[3 % VEC]));
        if (p.st_dst) *reinterpret_cast<uint32_t*>(p.st_dst + off) = so;
    } else {
        p.dst[off] = v[0];
        if (p.st_dst) p.st_dst[off] = (uint8_t)so;
    }
}

}  // namespace olap
