// Computed measures (cube.js:331-363, parser.js:3-26): the formula arrives in postfix
// text, is lowered to ONE fused elementwise CUDA kernel evaluating in double on the
// float32 cells of its inputs, compiled for sm_100a with NVRTC and cached per
// (program, input count, total count).  libnvrtc and libcuda are resolved with dlopen
// so the library loads on machines without a driver (where every call then fails).
#pragma once
#include <cuda.h>
#include <dlfcn.h>
#include <nvrtc.h>

#include <map>
#include <sstream>

#include "common.cuh"

namespace olap {

struct JitApi {
    bool tried = false, ok = false;
    std::string why;
    // nvrtc
    nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
    nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*);
    nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*);
    nvrtcResult (*GetCUBIN)(nvrtcProgram, char*);
    nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*);
    nvrtcResult (*GetProgramLog)(nvrtcProgram, char*);
    nvrtcResult (*DestroyProgram)(nvrtcProgram*);
    // driver
    CUresult (*ModuleLoadData)(CUmodule*, const void*);
    CUresult (*ModuleGetFunction)(CUfunction*, CUmodule, const char*);
    CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream,
                             void**, void**);
    CUresult (*GetErrorString)(CUresult, const char**);
};

inline JitApi& jit_api() {
    static JitApi api;
    if (api.tried) return api;
    api.tried = true;
    void* rtc = nullptr;
    for (const char* name : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12"}) {
        rtc = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        if (rtc) break;
    }
    if (!rtc) { api.why = "libnvrtc.so.12 not found"; return api; }
    void* drv = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!drv) { api.why = "libcuda.so.1 not found (no NVIDIA driver)"; return api; }
#define OLAP_SYM(lib, field, sym)                                         \
    *(void**)(&api.field) = dlsym(lib, sym);                              \
    if (!api.field) { api.why = std::string("missing symbol ") + sym; return api; }
    OLAP_SYM(rtc, CreateProgram, "nvrtcCreateProgram")
    OLAP_SYM(rtc, CompileProgram, "nvrtcCompileProgram")
    OLAP_SYM(rtc, GetCUBINSize, "nvrtcGetCUBINSize")
    OLAP_SYM(rtc, GetCUBIN, "nvrtcGetCUBIN")
    OLAP_SYM(rtc, GetProgramLogSize, "nvrtcGetProgramLogSize")
    OLAP_SYM(rtc, GetProgramLog, "nvrtcGetProgramLog")
    OLAP_SYM(rtc, DestroyProgram, "nvrtcDestroyProgram")
    OLAP_SYM(drv, ModuleLoadData, "cuModuleLoadData")
    OLAP_SYM(drv, ModuleGetFunction, "cuModuleGetFunction")
    OLAP_SYM(drv, LaunchKernel, "cuLaunchKernel")
    OLAP_SYM(drv, GetErrorString, "cuGetErrorString")
#undef OLAP_SYM
    api.ok = true;
    return api;
}

// ---- postfix -> C expression ----------------------------------------------------
struct Lowered {
    std::string expr;
    int max_input = -1, max_total = -1;
};

inline bool lower_program(const char* program, Lowered& out, std::string& err) {
    std::vector<std::string> st;
    std::istringstream in(program ? program : "");
    std::string tok;
    auto pop = [&](std::string& s) {
        if (st.empty()) return false;
        s = st.back();
        st.pop_back();
        return true;
    };
    static const std::map<std::string, std::string> unary = {
        {"abs", "fabs"}, {"ceil", "ceil"}, {"floor", "floor"}, {"trunc", "trunc"}, {"sqrt", "sqrt"}, {"cbrt", "cbrt"},
        {"exp", "exp"}, {"expm1", "expm1"}, {"ln", "log"}, {"log", "log"}, {"log1p", "log1p"}, {"log2", "log2"},
        {"log10", "log10"}, {"lg", "log10"}, {"sin", "sin"}, {"cos", "cos"}, {"tan", "tan"}, {"asin", "asin"},
        {"acos", "acos"}, {"atan", "atan"}, {"sinh", "sinh"}, {"cosh", "cosh"}, {"tanh", "tanh"}, {"asinh", "asinh"},
        {"acosh", "acosh"}, {"atanh", "atanh"}, {"sign", "olap_sign"}, {"round", "olap_round"}, {"isNaN", "olap_isnan"}};
    while (in >> tok) {
        if (tok[0] == 'v' && tok.size() > 1 && isdigit((unsigned char)tok[1])) {
            int k = atoi(tok.c_str() + 1);
            if (k > out.max_input) out.max_input = k;
            st.push_back("x" + std::to_string(k));
        } else if (tok[0] == 't' && tok.size() > 1 && isdigit((unsigned char)tok[1])) {
            int k = atoi(tok.c_str() + 1);
            if (k > out.max_total) out.max_total = k;
            st.push_back("t" + std::to_string(k));
        } else if (tok[0] == '#') {
            const std::string num = tok.substr(1);
            if (num == "nan") st.push_back("olap_nan()");
            else if (num == "inf") st.push_back("olap_inf()");
            else if (num == "-inf") st.push_back("(-olap_inf())");
            else {
                char* end = nullptr;
                const double v = strtod(num.c_str(), &end);
                if (!end || *end) { err = "bad number token: " + tok; return false; }
                char buf[64];
                snprintf(buf, sizeof buf, "%.17g", v);
                std::string lit = buf;
                if (lit.find_first_of(".eEn") == std::string::npos) lit += ".0";
                st.push_back("(" + lit + ")");
            }
        } else if (tok == "neg") {
            std::string a;
            if (!pop(a)) { err = "stack underflow at neg"; return false; }
            st.push_back("(-" + a + ")");
        } else if (tok == "+" || tok == "-" || tok == "*" || tok == "/" || tok == "%" || tok == "^" || tok == "||") {
            std::string a, b;
            if (!pop(b) || !pop(a)) { err = "stack underflow at " + tok; return false; }
            if (tok == "%") st.push_back("fmod(" + a + ", " + b + ")");
            else if (tok == "^") st.push_back("olap_pow(" + a + ", " + b + ")");
            else if (tok == "||") st.push_back("olap_coalesce_add(" + a + ", " + b + ")");
            else st.push_back("(" + a + " " + tok + " " + b + ")");
        } else if (tok == "?:") {
            std::string c, a, b;
            if (!pop(b) || !pop(a) || !pop(c)) { err = "stack underflow at ?:"; return false; }
            st.push_back("(olap_truthy(" + c + ") ? " + a + " : " + b + ")");
        } else if (tok.rfind("call:", 0) == 0) {
            const size_t c2 = tok.rfind(':');
            if (c2 <= 5) { err = "bad call token: " + tok; return false; }
            const std::string name = tok.substr(5, c2 - 5);
            const int argc = atoi(tok.c_str() + c2 + 1);
            if (argc < 1 || (int)st.size() < argc) { err = "stack underflow at " + tok; return false; }
            std::vector<std::string> args(st.end() - argc, st.end());
            st.resize(st.size() - argc);
            auto u = unary.find(name);
            if (u != unary.end() && argc == 1) st.push_back(u->second + "(" + args[0] + ")");
            else if (name == "min" || name == "max") {
                // a single argument still goes through the helper so NaN stays NaN
                std::string e = argc == 1 ? "olap_" + name + "(" + args[0] + ", " + args[0] + ")" : args[0];
                for (int k = 1; k < argc; ++k) e = "olap_" + name + "(" + e + ", " + args[k] + ")";
                st.push_back(e);
            } else if (name == "hypot") {
                std::string e = "sqrt(";
                for (int k = 0; k < argc; ++k) e += (k ? " + " : "") + ("(" + args[k] + ")*(" + args[k] + ")");
                st.push_back(e + ")");
            } else if (name == "pow" && argc == 2) st.push_back("olap_pow(" + args[0] + ", " + args[1] + ")");
            else if (name == "atan2" && argc == 2) st.push_back("atan2(" + args[0] + ", " + args[1] + ")");
            else if (name == "roundTo" && argc == 2)
                st.push_back("(olap_round(" + args[0] + " * pow(10.0, " + args[1] + ")) / pow(10.0, " + args[1] + "))");
            else if (name == "if" && argc == 3)
                st.push_back("(olap_truthy(" + args[0] + ") ? " + args[1] + " : " + args[2] + ")");
            else { err = "unsupported function in formula: " + name; return false; }
        } else {
            err = "unknown token in formula program: " + tok;
            return false;
        }
    }
    if (st.size() != 1) { err = "formula program does not reduce to one value"; return false; }
    out.expr = st[0];
    return true;
}

// Helpers and `olap_formula`: the same text in every kernel kind, so a cell gets the same bits in each.
inline void formula_prelude(std::ostringstream& s, const Lowered& lw, int n_inputs, int n_totals) {
    s << "typedef long long i64;\n"
         "__device__ __forceinline__ double olap_nan() { return __longlong_as_double(0x7ff8000000000000LL); }\n"
         "__device__ __forceinline__ double olap_inf() { return __longlong_as_double(0x7ff0000000000000LL); }\n"
         "__device__ __forceinline__ bool olap_truthy(double c) { return c == c && c != 0.0; }\n"
         "__device__ __forceinline__ double olap_isnan(double a) { return a != a ? 1.0 : 0.0; }\n"
         "__device__ __forceinline__ double olap_round(double a) { return floor(a + 0.5); }\n"
         "__device__ __forceinline__ double olap_sign(double a) { return a != a ? a : (a > 0.0 ? 1.0 : (a < 0.0 ? -1.0 : a)); }\n"
         // parser.js:18-23
         "__device__ __forceinline__ double olap_coalesce_add(double a, double b) {\n"
         "  if (a != a && b == b) return b; if (a == a && b != b) return a; return a + b; }\n"
         // Math.max / Math.min / Math.pow semantics
         "__device__ __forceinline__ double olap_max(double a, double b) {\n"
         "  if (a != a || b != b) return olap_nan();\n"
         "  if (a == b) return __longlong_as_double(__double_as_longlong(a) & __double_as_longlong(b));\n"
         "  return a > b ? a : b; }\n"
         "__device__ __forceinline__ double olap_min(double a, double b) {\n"
         "  if (a != a || b != b) return olap_nan();\n"
         "  if (a == b) return __longlong_as_double(__double_as_longlong(a) | __double_as_longlong(b));\n"
         "  return a < b ? a : b; }\n"
         "__device__ __forceinline__ double olap_pow(double a, double b) {\n"
         "  if (b != b) return olap_nan(); if (b == 0.0) return 1.0;\n"
         "  if (fabs(a) == 1.0 && isinf(b)) return olap_nan();\n"
         // integer exponents by squaring: exact whenever the result is representable
         // (CUDA pow() is only 2-ulp accurate, which breaks e.g. (7 ^ 2) % 7)
         "  if (b == trunc(b) && fabs(b) <= 1024.0) { double r = 1.0, x = a; long long e = (long long)fabs(b);\n"
         "    while (e) { if (e & 1) r *= x; x *= x; e >>= 1; } return b < 0.0 ? 1.0 / r : r; }\n"
         "  return pow(a, b); }\n"
         "__device__ __forceinline__ float olap_canon(float v, int nan_default) {\n"
         "  if (v != v) return __int_as_float(0x7fc00000); if (!nan_default && v == 0.0f) return 0.0f; return v; }\n";
    s << "__device__ __forceinline__ double olap_formula(";
    bool first = true;
    for (int k = 0; k < n_inputs; ++k) { s << (first ? "" : ", ") << "double x" << k; first = false; }
    for (int k = 0; k < n_totals; ++k) { s << (first ? "" : ", ") << "double t" << k; first = false; }
    s << ") { return " << lw.expr << "; }\n";
}

inline std::string eval_source(const Lowered& lw, int n_inputs, int n_totals) {
    std::ostringstream s;
    bool first = true;
    formula_prelude(s, lw, n_inputs, n_totals);
    s << "extern \"C\" __global__ void __launch_bounds__(256) olap_eval_kernel(";
    for (int k = 0; k < n_inputs; ++k) s << "const float* __restrict__ v" << k << ", ";
    for (int k = 0; k < n_totals; ++k) s << "double t" << k << ", ";
    s << "float* __restrict__ out32, unsigned char* __restrict__ st_out, double* __restrict__ out64, i64 n, "
         "int nan_default) {\n"
         "  const i64 stride = (i64)gridDim.x * blockDim.x * 4;\n"
         "  for (i64 i = ((i64)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {\n"
         "    if (i + 4 <= n) {\n";
    for (int k = 0; k < n_inputs; ++k)
        s << "      const float4 a" << k << " = __ldcs(reinterpret_cast<const float4*>(v" << k << " + i));\n";
    const char* comp[4] = {"x", "y", "z", "w"};
    for (int e = 0; e < 4; ++e) {
        s << "      const double r" << e << " = olap_formula(";
        first = true;
        for (int k = 0; k < n_inputs; ++k) { s << (first ? "" : ", ") << "(double)a" << k << "." << comp[e]; first = false; }
        for (int k = 0; k < n_totals; ++k) { s << (first ? "" : ", ") << "t" << k; first = false; }
        s << ");\n";
    }
    s << "      if (out64) { double2 lo = make_double2(r0, r1), hi = make_double2(r2, r3);\n"
         "        __stcs(reinterpret_cast<double2*>(out64 + i), lo); __stcs(reinterpret_cast<double2*>(out64 + i + 2), hi); }\n"
         "      if (out32) { float4 o = make_float4(olap_canon((float)r0, nan_default), olap_canon((float)r1, nan_default),\n"
         "                                          olap_canon((float)r2, nan_default), olap_canon((float)r3, nan_default));\n"
         "        __stcs(reinterpret_cast<float4*>(out32 + i), o);\n"
         "        if (st_out) { uchar4 q;\n"
         "          q.x = (nan_default ? o.x == o.x : o.x != 0.0f) ? 2 : 1; q.y = (nan_default ? o.y == o.y : o.y != 0.0f) ? 2 : 1;\n"
         "          q.z = (nan_default ? o.z == o.z : o.z != 0.0f) ? 2 : 1; q.w = (nan_default ? o.w == o.w : o.w != 0.0f) ? 2 : 1;\n"
         "          *reinterpret_cast<uchar4*>(st_out + i) = q; } }\n"
         "    } else {\n"
         "      for (i64 j = i; j < n; ++j) {\n"
         "        const double r = olap_formula(";
    first = true;
    for (int k = 0; k < n_inputs; ++k) { s << (first ? "" : ", ") << "(double)v" << k << "[j]"; first = false; }
    for (int k = 0; k < n_totals; ++k) { s << (first ? "" : ", ") << "t" << k; first = false; }
    s << ");\n"
         "        if (out64) out64[j] = r;\n"
         "        if (out32) { const float o = olap_canon((float)r, nan_default); out32[j] = o;\n"
         "          if (st_out) st_out[j] = (nan_default ? o == o : o != 0.0f) ? 2 : 1; }\n"
         "      }\n"
         "    }\n"
         "  }\n"
         "}\n";
    return s.str();
}

// ---- the formula over a region (olap_region_eval_sum / olap_region_eval_copy) -------------------------
// The region is walked by region_walk.cuh exactly as region_kernel walks it; each input is read at the same
// offset, the formula is evaluated in double, and the value is summed (kind JIT_REGION_SUM, epilogue of
// region_kernel's SUM) or stored into the target with setValue's element body (kind JIT_REGION_COPY).
// A module holds each kernel for VEC 4 (128-bit accesses) and VEC 1.
enum JitKind { JIT_EVAL = 0, JIT_REGION_SUM = 1, JIT_REGION_COPY = 2 };

inline std::string region_source(const Lowered& lw, int n_inputs, int kind) {
    std::ostringstream s;
    s << "#include \"region_walk.cuh\"\n";
    formula_prelude(s, lw, n_inputs, 0);
    // vectors in flight per thread: U x n_inputs loads of VEC floats
    const int U = n_inputs >= 4 ? 1 : (n_inputs >= 2 ? 2 : 4);
    s << "constexpr int U = " << U << ";\n"
         "template <int VEC, bool NC> __device__ __forceinline__ void olap_ld(const float* p, float (&x)[VEC]) {\n"
         "  if (VEC == 4) { const float4 a = NC ? __ldcs(reinterpret_cast<const float4*>(p)) : *reinterpret_cast<const float4*>(p);\n"
         "    x[0] = a.x; x[1 % VEC] = a.y; x[2 % VEC] = a.z; x[3 % VEC] = a.w; }\n"
         "  else x[0] = NC ? __ldcs(p) : *p; }\n";
    auto params = [&](std::ostringstream& o) {
        for (int k = 0; k < n_inputs; ++k) o << ", const float* v" << k;
    };
    auto formula_at = [&](const char* u, const char* e) {
        std::ostringstream o;
        o << "olap_formula(";
        for (int k = 0; k < n_inputs; ++k) o << (k ? ", " : "") << "(double)x" << k << "[" << u << "][" << e << "]";
        o << ")";
        return o.str();
    };
    auto loads = [&](bool nc) {
        std::ostringstream o;
        for (int k = 0; k < n_inputs; ++k) o << "float x" << k << "[U][VEC];\n";
        o << "#pragma unroll\n  for (int u = 0; u < U; ++u) { if (off[u] < 0) continue;\n";
        for (int k = 0; k < n_inputs; ++k) o << "    olap_ld<VEC, " << (nc ? "true" : "false") << ">(v" << k << " + off[u], x" << k << "[u]);\n";
        o << "  }\n";
        return o.str();
    };
    const char* walk_head =
        "  const i64 n = w.n_vec;\n"
        "  const i64 stride = (i64)gridDim.x * blockDim.x;\n"
        "  for (i64 t0 = (i64)blockIdx.x * blockDim.x + threadIdx.x; t0 < n; t0 += U * stride) {\n"
        "    i64 off[U];\n"
        "#pragma unroll\n"
        "    for (int u = 0; u < U; ++u) { const i64 t = t0 + u * stride; off[u] = t < n ? olap::region_offset(w, t, VEC) : -1; }\n";
    // the last CTA of a ticketed grid: s_last in shared memory
    const char* ticket =
        "  __shared__ bool s_last;\n"
        "  __threadfence();\n"
        "  __syncthreads();\n"
        "  if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;\n"
        "  __syncthreads();\n";
    if (kind == JIT_REGION_SUM) {
        s << "__device__ __forceinline__ double olap_warp_sum(double x) {\n"
             "#pragma unroll\n  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);\n  return x; }\n";
        s << "template <int VEC> __device__ __forceinline__ void region_eval_sum(const olap::RegionWalk& w";
        params(s);
        s << ", double* partial, unsigned* ticket, double* out) {\n"
             "  double accs[U];\n"
             "#pragma unroll\n  for (int u = 0; u < U; ++u) accs[u] = 0.0;\n"
          << walk_head << loads(true)
          << "#pragma unroll\n    for (int u = 0; u < U; ++u) { if (off[u] < 0) continue;\n"
             "#pragma unroll\n      for (int e = 0; e < VEC; ++e) accs[u] += " << formula_at("u", "e") << "; }\n"
             "  }\n"
             // region_kernel's epilogue: per-CTA partials folded in a fixed order by the last CTA
             "  __shared__ double s_sum[256 / 32];\n"
             "  double a0 = accs[0];\n"
             "#pragma unroll\n  for (int u = 1; u < U; ++u) a0 += accs[u];\n"
             "  const double acc = olap_warp_sum(a0);\n"
             "  const int wi = threadIdx.x >> 5, l = threadIdx.x & 31;\n"
             "  if (l == 0) s_sum[wi] = acc;\n"
             "  __shared__ bool s_last;\n"
             "  __syncthreads();\n"
             "  if (threadIdx.x == 0) {\n"
             "    double a = 0.0;\n"
             "    for (int k = 0; k < 256 / 32; ++k) a += s_sum[k];\n"
             "    partial[blockIdx.x] = a;\n"
             "    __threadfence();\n"
             "    s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;\n"
             "  }\n"
             "  __syncthreads();\n"
             "  if (!s_last) return;\n"
             "  double a = 0.0;\n"
             "  for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) a += ((volatile double*)partial)[b];\n"
             "  a = olap_warp_sum(a);\n"
             "  __syncthreads();\n"
             "  if (l == 0) s_sum[wi] = a;\n"
             "  __syncthreads();\n"
             "  if (threadIdx.x == 0) {\n"
             "    double ta = 0.0;\n"
             "    for (int k = 0; k < 256 / 32; ++k) ta += s_sum[k];\n"
             "    *out = ta;\n"
             "    *ticket = 0;\n"
             "  }\n"
             "}\n";
        for (int vec : {4, 1}) {
            s << "extern \"C\" __global__ void __launch_bounds__(256, 4) olap_region_eval_sum_v" << vec
              << "(const __grid_constant__ olap::RegionWalk w";
            params(s);
            s << ", double* partial, unsigned* ticket, double* out) { region_eval_sum<" << vec << ">(w";
            for (int k = 0; k < n_inputs; ++k) s << ", v" << k;
            s << ", partial, ticket, out); }\n";
        }
        return s.str();
    }
    // JIT_REGION_COPY.  Every cell of the (de-duplicated) region is read and written by one thread, once, so
    // the target may be an input: the loads are plain (not .nc) and each value is computed before its cell
    // is written.  The check kernel (integer targets) writes nothing: it finds the first cell, in product
    // order, whose value does not survive the Float32 cell; its last CTA evaluates that cell once more and
    // reports its offset and value.
    s << "template <int VEC> __device__ __forceinline__ void region_eval_copy(const olap::RegionWalk& w";
    params(s);
    s << ", float* dst, unsigned char* st_dst, int nan_default) {\n"
      << walk_head << loads(false)
      << "#pragma unroll\n    for (int u = 0; u < U; ++u) { if (off[u] < 0) continue;\n"
         "      float o[VEC]; unsigned so = 0;\n"
         "#pragma unroll\n      for (int e = 0; e < VEC; ++e) {\n"
         "        o[e] = olap_canon((float)" << formula_at("u", "e") << ", nan_default);\n"
         "        so |= (unsigned)((nan_default ? o[e] == o[e] : o[e] != 0.0f) ? 2 : 1) << (8 * e); }\n"
         "      if (VEC == 4) {\n"
         "        *reinterpret_cast<float4*>(dst + off[u]) = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);\n"
         "        if (st_dst) *reinterpret_cast<unsigned*>(st_dst + off[u]) = so;\n"
         "      } else {\n"
         "        dst[off[u]] = o[0];\n"
         "        if (st_dst) st_dst[off[u]] = (unsigned char)so;\n"
         "      }\n"
         "    }\n"
         "  }\n"
         "}\n";
    s << "template <int VEC> __device__ __forceinline__ void region_eval_check(const olap::RegionWalk& w";
    params(s);
    s << ", unsigned long long* first, unsigned* ticket, i64* bad_off, double* bad_val) {\n"
      << walk_head << loads(false)
      << "#pragma unroll\n    for (int u = 0; u < U; ++u) { if (off[u] < 0) continue;\n"
         "#pragma unroll\n      for (int e = 0; e < VEC; ++e) {\n"
         "        const double r = " << formula_at("u", "e") << ";\n"
         "        if (r == r && (double)(float)r != r) atomicMin(first, (unsigned long long)((t0 + u * stride) * VEC + e)); } }\n"
         "  }\n"
      << ticket
      << "  if (!s_last || threadIdx.x != 0) return;\n"
         "  *ticket = 0;\n"
         "  const unsigned long long pos = atomicAdd(first, 0ull);\n"
         "  if (pos == ~0ull) return;\n"
         "  const i64 o = olap::region_offset(w, (i64)(pos / VEC), VEC) + (i64)(pos % VEC);\n"
         "  *bad_off = o;\n"
         "  *bad_val = olap_formula(";
    for (int k = 0; k < n_inputs; ++k) s << (k ? ", " : "") << "(double)v" << k << "[o]";
    s << ");\n}\n";
    for (int vec : {4, 1}) {
        s << "extern \"C\" __global__ void __launch_bounds__(256, 4) olap_region_eval_copy_v" << vec
          << "(const __grid_constant__ olap::RegionWalk w";
        params(s);
        s << ", float* dst, unsigned char* st_dst, int nan_default) { region_eval_copy<" << vec << ">(w";
        for (int k = 0; k < n_inputs; ++k) s << ", v" << k;
        s << ", dst, st_dst, nan_default); }\n";
        s << "extern \"C\" __global__ void __launch_bounds__(256, 4) olap_region_eval_check_v" << vec
          << "(const __grid_constant__ olap::RegionWalk w";
        params(s);
        s << ", unsigned long long* first, unsigned* ticket, i64* bad_off, double* bad_val) { region_eval_check<" << vec << ">(w";
        for (int k = 0; k < n_inputs; ++k) s << ", v" << k;
        s << ", first, ticket, bad_off, bad_val); }\n";
    }
    return s.str();
}

// region_walk.cuh as text (generated by the Makefile): the in-memory header of the region kinds
static const char kRegionWalkHeader[] =
#include "region_walk.inc"
    ;

struct JitKernel {
    CUmodule mod = nullptr;
    CUfunction fn = nullptr;             // JIT_EVAL: olap_eval_kernel
    CUfunction vec4 = nullptr, vec1 = nullptr;      // region kinds: the sum or copy kernel
    CUfunction check4 = nullptr, check1 = nullptr;  // JIT_REGION_COPY: the check pass of integer targets
};

// CUDA source of a formula program for one kernel kind; on error `code` is set and `err` says why
inline std::string jit_source(const char* program, int n_inputs, int n_totals, int kind, std::string& err, int* code) {
    Lowered lw;
    *code = OLAP_OK;
    if (!lower_program(program, lw, err)) { *code = OLAP_E_INVALID; return ""; }
    char buf[128];
    if (lw.max_input >= n_inputs) {
        snprintf(buf, sizeof buf, "formula reads input %d but only %d given", lw.max_input, n_inputs);
        err = buf; *code = OLAP_E_INVALID; return "";
    }
    if (lw.max_total >= n_totals) {
        snprintf(buf, sizeof buf, "formula reads total %d but only %d given", lw.max_total, n_totals);
        err = buf; *code = OLAP_E_INVALID; return "";
    }
    return kind == JIT_EVAL ? eval_source(lw, n_inputs, n_totals) : region_source(lw, n_inputs, kind);
}

inline int jit_get(const char* program, int n_inputs, int n_totals, int kind, JitKernel** out) {
    static std::map<std::string, JitKernel> cache;
    const std::string key = std::to_string(kind) + "|" + std::to_string(n_inputs) + "|" + std::to_string(n_totals) + "|" +
                            (program ? program : "");
    auto it = cache.find(key);
    if (it != cache.end()) { *out = &it->second; return OLAP_OK; }

    std::string err;
    int code;
    const std::string src = jit_source(program, n_inputs, n_totals, kind, err, &code);
    if (code != OLAP_OK) return fail(code, "%s", err.c_str());

    JitApi& api = jit_api();
    if (!api.ok) return fail(OLAP_E_CUDA, "computed-measure JIT unavailable: %s", api.why.c_str());

    nvrtcProgram prog;
    const char* hdr_src[] = {kRegionWalkHeader};
    const char* hdr_name[] = {"region_walk.cuh"};
    const int n_hdr = kind == JIT_EVAL ? 0 : 1;
    if (api.CreateProgram(&prog, src.c_str(), "olap_eval.cu", n_hdr, n_hdr ? hdr_src : nullptr, n_hdr ? hdr_name : nullptr) != NVRTC_SUCCESS)
        return fail(OLAP_E_CUDA, "nvrtcCreateProgram failed");
    const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", "--fmad=false"};
    const nvrtcResult rc = api.CompileProgram(prog, 4, opts);
    if (rc != NVRTC_SUCCESS) {
        size_t n = 0;
        api.GetProgramLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) api.GetProgramLog(prog, &log[0]);
        api.DestroyProgram(&prog);
        return fail(OLAP_E_CUDA, "NVRTC failed to compile formula kernel: %s", log.c_str());
    }
    size_t sz = 0;
    api.GetCUBINSize(prog, &sz);
    std::vector<char> cubin(sz);
    api.GetCUBIN(prog, cubin.data());
    api.DestroyProgram(&prog);

    JitKernel k;
    CUresult cr = api.ModuleLoadData(&k.mod, cubin.data());
    if (cr == CUDA_SUCCESS && kind == JIT_EVAL) cr = api.ModuleGetFunction(&k.fn, k.mod, "olap_eval_kernel");
    const char* base = kind == JIT_REGION_SUM ? "olap_region_eval_sum_v" : "olap_region_eval_copy_v";
    if (cr == CUDA_SUCCESS && kind != JIT_EVAL) cr = api.ModuleGetFunction(&k.vec4, k.mod, (std::string(base) + "4").c_str());
    if (cr == CUDA_SUCCESS && kind != JIT_EVAL) cr = api.ModuleGetFunction(&k.vec1, k.mod, (std::string(base) + "1").c_str());
    if (cr == CUDA_SUCCESS && kind == JIT_REGION_COPY) cr = api.ModuleGetFunction(&k.check4, k.mod, "olap_region_eval_check_v4");
    if (cr == CUDA_SUCCESS && kind == JIT_REGION_COPY) cr = api.ModuleGetFunction(&k.check1, k.mod, "olap_region_eval_check_v1");
    if (cr != CUDA_SUCCESS) {
        const char* msg = "?";
        api.GetErrorString(cr, &msg);
        return fail(OLAP_E_CUDA, "loading the formula kernel failed: %s", msg);
    }
    auto ins = cache.emplace(key, k);
    *out = &ins.first->second;
    return OLAP_OK;
}

}  // namespace olap
