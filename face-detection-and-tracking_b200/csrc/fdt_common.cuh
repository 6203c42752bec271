// Shared helpers for libfdt_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "fdt_b200.h"

#define FDT_API extern "C" __attribute__((visibility("default")))

void fdt_set_error(const char *fmt, ...);

// library-internal form of fdt_detect (hostctx.cu): `loc` may be a device view of pinned HOST memory that k_sort_nms gathers in place
constexpr unsigned FDT_FLAG_LOC_HOST_MAPPED = 1u;
int fdt_detect_flags(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                     float conf_thresh, float nms_thresh, float var0, float var1, float *out, int32_t *counts, int64_t *kept_prior,
                     void *ws, size_t ws_bytes, void *stream, unsigned flags);

constexpr int FDT_DETECT_MAX_DEPTH = 4;     // slots of the stateful Detect workspace (calls of one stream in flight)
int fdt_option_host_chunk();     // images per copy/compute chunk of the host-buffer pipeline (hostctx.cu); option "host_chunk"

// greedy NMS for any n and for float64 (nms_generic.cu): sort + pairwise bit mask + serial reduce
constexpr int FDT_MAX_NMS_GENERIC = 131072;
size_t fdt_nms_generic_workspace_bytes(int64_t n);
template <typename T>
int fdt_nms_generic(const T *boxes, const T *scores, int64_t n, T thresh, int64_t top_k, int variant,
                    int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, cudaStream_t st);

#define FDT_CUDA(expr)                                                                            \
    do {                                                                                          \
        cudaError_t e_ = (expr);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            fdt_set_error("%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__);   \
            return FDT_E_CUDA;                                                                    \
        }                                                                                         \
    } while (0)

#define FDT_REQUIRE(cond, code, ...)                                                              \
    do {                                                                                          \
        if (!(cond)) { fdt_set_error(__VA_ARGS__); return (code); }                               \
    } while (0)

#define FDT_LAUNCH_CHECK() FDT_CUDA(cudaGetLastError())

static inline size_t fdt_align256(size_t x) { return (x + 255) & ~(size_t)255; }
static inline bool fdt_aligned(const void *p, size_t a) { return ((uintptr_t)p & (a - 1)) == 0; }

constexpr int FDT_NUM_SMS = 148;            // B200
constexpr int FDT_SMEM_MAX = 232448;        // 227 KB opt-in dynamic shared memory per CTA

// ---- device helpers -------------------------------------------------------------------------
// sign of (r + h)^4 - x, with (r + h)^2 and its square carried in double-double (error ~2^-100 relative; h = half an ulp of r)
__device__ __forceinline__ int fdt_qroot_side(double r, double h, double x)
{
    const double p = __dmul_rn(r, r), pe = fma(r, r, -p);
    const double b = __dmul_rn(2.0 * r, h), c = __dmul_rn(h, h);                     // exact: h is a power of two
    const double s = __dadd_rn(p, b), bb = __dsub_rn(s, p);
    const double e1 = __dadd_rn(__dsub_rn(p, __dsub_rn(s, bb)), __dsub_rn(b, bb));   // two-sum error of p + b
    const double lo0 = __dadd_rn(__dadd_rn(pe, e1), c);
    const double hi = __dadd_rn(s, lo0), lo = __dsub_rn(lo0, __dsub_rn(hi, s));
    const double q = __dmul_rn(hi, hi), qe = fma(hi, hi, -q);
    const double d = __dadd_rn(__dsub_rn(q, x), __dadd_rn(qe, __dmul_rn(2.0 * hi, lo)));
    return (d > 0.0) - (d < 0.0);
}
// x ** 0.25 correctly rounded (utils/calc_performance.py:49 `dis ** 0.25`).  CUDA's pow is off by an ulp for about a quarter of all
// inputs, exact fourth powers included (pow(k^4, 0.25) != k for 491 integers k < 8192), which moves ties and the `< sigma_dis`
// edge of the tracker.  sqrt(sqrt(x)) is within one ulp; the neighbour across the nearer rounding midpoint is taken when
// the midpoint's fourth power says so.  0, +inf, NaN and negative x give what pow gives.
__device__ __forceinline__ double fdt_qroot_cr(double x)
{
    if (!(x > 0.0) || x == INFINITY) return sqrt(sqrt(x)) + 0.0;
    double sc = 1.0;                                                                 // keep r^4 and its error terms in range
    if (x < 0x1p-900) { x *= 0x1p800; sc = 0x1p-200; }
    else if (x > 0x1p900) { x *= 0x1p-800; sc = 0x1p200; }
    double r = sqrt(sqrt(x));
    const long long rb = __double_as_longlong(r);                                   // r > 0 and normal here
    const double up = __longlong_as_double(rb + 1), dn = __longlong_as_double(rb - 1);
    if (fdt_qroot_side(r, 0.5 * (up - r), x) < 0) r = up;
    else if (fdt_qroot_side(r, 0.5 * (dn - r), x) > 0) r = dn;
    return r * sc;
}

// Order-preserving float -> uint32 map (larger float -> larger uint; +NaN above +inf like torch.sort).
__device__ __forceinline__ uint32_t fdt_float_key(float f)
{
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fdt_key_float(uint32_t k)
{
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
// exp/log evaluated in fp64, rounded once to fp32 (see include/fdt_b200.h conventions): (float)exp((double)x), (float)log((double)x).
// The library routines spend more instructions on materialising their 64-bit constants and on special cases than on arithmetic
// (k_loss_prior: 125 of 300 instructions per prior), so the common ranges take a lean evaluation whose constants are operands from
// the constant bank: a few fp64 ulps of error, and whenever the fp64 value lies within FDT_CR_GUARD ulps of an fp32 rounding
// boundary -- the only place where a few ulps can change the rounded float -- the library routine decides, as it does for every
// input outside the range.  The result is therefore the library's for EVERY input, which fdt_selftest_cr_math checks exhaustively
// over all 2^32 bit patterns (tests/test_multibox_gpu.py).
constexpr int FDT_CR_GUARD = 32;
static __constant__ double FDT_EXP_C[14] = {     // 1/n!, n = 0..13
    1.0, 1.0, 0.5, 0.16666666666666666, 0.041666666666666664, 0.008333333333333333, 0.001388888888888889,
    0.0001984126984126984, 2.48015873015873e-05, 2.7557319223985893e-06, 2.755731922398589e-07, 2.505210838544172e-08,
    2.08767569878681e-09, 1.6059043836821613e-10};
static __constant__ double FDT_LOG_C[10] = {     // 2/(2n+1), n = 1..10
    0.6666666666666666, 0.4, 0.2857142857142857, 0.2222222222222222, 0.18181818181818182, 0.15384615384615385,
    0.13333333333333333, 0.11764705882352941, 0.10526315789473684, 0.09523809523809523};
static __constant__ double FDT_LN2[4] = {1.4426950408889634, 6755399441055744.0, 0.6931471803691238, 1.9082149292705877e-10};

// true when the fp64 value (low word `lo`) is at least FDT_CR_GUARD fp64 ulps away from the midpoint of two neighbouring floats
__device__ __forceinline__ bool fdt_cr_safe(int lo)
{
    return (unsigned)((lo & 0x1fffffff) - (0x10000000 - FDT_CR_GUARD)) >= 2u * FDT_CR_GUARD;
}
__device__ __forceinline__ float fdt_expf_cr(float x)
{
    if (fabsf(x) <= 87.0f) {                                 // result a normal float in (2^-126, 2^126); NaN fails
        const double xd = (double)x;
        double t = fma(xd, FDT_LN2[0], FDT_LN2[1]);          // 1.5 * 2^52 + rint(x / ln 2)
        const int k = __double2loint(t);
        t -= FDT_LN2[1];
        double r = fma(t, -FDT_LN2[2], xd);                  // exact: ln2_hi has 32 significant bits
        r = fma(t, -FDT_LN2[3], r);                          // |r| <= 0.3466
        double p = FDT_EXP_C[13];
#pragma unroll
        for (int n = 12; n >= 0; --n) p = fma(p, r, FDT_EXP_C[n]);
        const int lo = __double2loint(p);
        if (fdt_cr_safe(lo)) return (float)__hiloint2double(__double2hiint(p) + (k << 20), lo);
    }
    return (float)exp((double)x);
}
__device__ __forceinline__ float fdt_logf_cr(float s)
{
    const unsigned bits = __float_as_uint(s);
    if (bits - 0x00800000u < 0x7f000000u) {                  // positive, normal, finite
        int e = (int)(bits >> 23) - 127;
        const unsigned mb = bits & 0x007fffffu;
        const bool up = mb > 0x3504f3u;                      // mantissa above sqrt(2): use m / 2 in (0.7071, 1)
        e += up;
        const double m = (double)__uint_as_float(mb | (up ? 0x3f000000u : 0x3f800000u));
        const double f = m - 1.0, den = m + 1.0;             // both exact
        double y;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(den));
        double er = fma(-den, y, 1.0);
        y = fma(y, er, y);
        er = fma(-den, y, 1.0);
        y = fma(y, er, y);
        double u = f * y;
        u = fma(fma(-den, u, f), y, u);                      // u = f / (2 + f), |u| <= 0.1716
        const double u2 = u * u;
        double q = FDT_LOG_C[9];
#pragma unroll
        for (int n = 8; n >= 0; --n) q = fma(q, u2, FDT_LOG_C[n]);
        const double ed = (double)e;
        double res = fma(u, u2 * q, u + u);                  // log(m) = 2u + 2u^3/3 + 2u^5/5 + ...
        res = fma(ed, FDT_LN2[3], res);
        res = fma(ed, FDT_LN2[2], res);
        if (fdt_cr_safe(__double2loint(res))) return (float)res;
    }
    return (float)log((double)s);
}

// decode (layers/box_utils.py:238-258); compiled with -fmad=false so no FMA is formed
__device__ __forceinline__ float4 fdt_decode1(float4 l, float4 p, float v0, float v1)
{
    float cx = p.x + (l.x * v0) * p.z;
    float cy = p.y + (l.y * v0) * p.w;
    float w = p.z * fdt_expf_cr(l.z * v1);
    float h = p.w * fdt_expf_cr(l.w * v1);
    float x1 = cx - w / 2.0f;
    float y1 = cy - h / 2.0f;
    return make_float4(x1, y1, w + x1, h + y1);
}
// encode (layers/box_utils.py:213-234)
__device__ __forceinline__ float4 fdt_encode1(float4 m, float4 p, float v0, float v1)
{
    float4 o;
    o.x = ((m.x + m.z) / 2.0f - p.x) / (v0 * p.z);
    o.y = ((m.y + m.w) / 2.0f - p.y) / (v0 * p.w);
    o.z = fdt_logf_cr((m.z - m.x) / p.z) / v1;
    o.w = fdt_logf_cr((m.w - m.y) / p.w) / v1;
    return o;
}
