// Access to the models' per-level head maps (SURVEY 8f rank 1; fp32 / bf16 / fp16, NCHW or channels_last), shared by Detect (detect.cu) and MultiBoxLoss
// (multibox.cu).
//
// The models hand Detect the outputs of their prediction convolutions, per pyramid level and NCHW: loc_l[B,4,H,W] and the
// 4-channel max-in-out confidence conf_l[B,4,H,W] (pyramid.py:291-306).  The reference turns them into loc[B,N,4] and
// conf[B,N,2] with chunk / max / cat / permute / contiguous / view / cat and a 2-way softmax (pyramid.py:293-309, 331-332);
// the kernels read the maps directly.  Prior n of level l sits at pixel q = n - off[l] (y outer, x inner).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "fdt_common.cuh"

namespace {

// A map is read where the network wrote it: element (b, ch, q) of a level (q = y * W + x) sits at
// data + b * bs + ch * cs + q * ps elements, each of the call's element type (FDT_DTYPE_*).  Dense NCHW is (4 hw, hw, 1), dense
// channels_last (4 hw, 1, 4).  The accessors load that type and widen it to fp32 (exact), so all arithmetic is what it is on fp32
// maps; gradients are rounded to the type (round to nearest even) as they are stored.
struct HeadMap {
    const void *p;
    int64_t bs, cs, ps;
};
struct HeadGradMap {
    void *p;
    int64_t bs, cs, ps;
};
constexpr int FDT_MAX_LEVELS = 8;
struct HeadLevels {
    HeadMap conf[FDT_MAX_LEVELS];
    HeadMap loc[FDT_MAX_LEVELS];
    int hw[FDT_MAX_LEVELS];
    int off[FDT_MAX_LEVELS + 1];           // first prior of each level; off[L] = N
    int neg_max[FDT_MAX_LEVELS];           // 1: neg = max(ch0..2), pos = ch3 (pyramid.py:293-297); 0: neg = ch0, pos = max(ch1..3) (:299-304)
    int L;
    int dtype;                             // FDT_DTYPE_* of every map of the call (and of the gradient maps)
    unsigned vec;                          // bit l: conf map of level l reads a prior's 4 channels as one aligned vector; bit 8 + l: loc map
    unsigned dense;                        // bit l: conf map of level l covers [0, B * 4 * hw) exactly (NCHW or channels_last, no gaps)
    int f32_nchw;                          // every map fp32 dense NCHW: the kernels may take HEAD_F32_NCHW
};
// How a kernel instantiation addresses the maps.  HEAD_F32_NCHW: fp32 dense NCHW, a plain [B,4,hw] array per level (the maps the
// entries without `_ex` take, at the cost they always had); HEAD_ANY: element type, strides and vector loads from the descriptors.
enum { HEAD_F32_NCHW = 0, HEAD_ANY = 1 };
__device__ __forceinline__ int head_level(const HeadLevels &h, const int p)
{
    int l = 0;
#pragma unroll
    for (int q = 1; q < FDT_MAX_LEVELS; ++q) l += (q < h.L && p >= h.off[q]) ? 1 : 0;
    return l;
}
// 16-bit element -> fp32 (exact)
__device__ __forceinline__ float head_widen16(const unsigned short u, const int dtype)
{
    return dtype == FDT_DTYPE_BF16 ? __uint_as_float((unsigned)u << 16) : __half2float(__ushort_as_half(u));
}
__device__ __forceinline__ float head_elem(const void *p, const int64_t i, const int dtype)
{
    if (dtype == FDT_DTYPE_F32) return __ldg(reinterpret_cast<const float *>(p) + i);
    return head_widen16(__ldg(reinterpret_cast<const unsigned short *>(p) + i), dtype);
}
// the 4 channels of pixel q of image b: one vector load where the host found them adjacent and aligned, else 4 scalar loads
__device__ __forceinline__ float4 head_load4(const HeadMap &m, const int dtype, const bool vec, const int b, const int q)
{
    const int64_t o = (int64_t)b * m.bs + (int64_t)q * m.ps;
    if (vec) {
        if (dtype == FDT_DTYPE_F32) return __ldg(reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(m.p) + o));
        const uint2 u = __ldg(reinterpret_cast<const uint2 *>(reinterpret_cast<const unsigned short *>(m.p) + o));
        return make_float4(head_widen16((unsigned short)(u.x & 0xffffu), dtype), head_widen16((unsigned short)(u.x >> 16), dtype),
                           head_widen16((unsigned short)(u.y & 0xffffu), dtype), head_widen16((unsigned short)(u.y >> 16), dtype));
    }
    return make_float4(head_elem(m.p, o, dtype), head_elem(m.p, o + m.cs, dtype), head_elem(m.p, o + 2 * m.cs, dtype),
                       head_elem(m.p, o + 3 * m.cs, dtype));
}
__device__ __forceinline__ unsigned short head_narrow16(const float v, const int dtype)
{
    return dtype == FDT_DTYPE_BF16 ? __bfloat16_as_ushort(__float2bfloat16_rn(v)) : __half_as_ushort(__float2half_rn(v));
}
__device__ __forceinline__ void head_store4(const HeadGradMap &m, const int dtype, const bool vec, const int b, const int q, const float4 v)
{
    const int64_t o = (int64_t)b * m.bs + (int64_t)q * m.ps;
    if (dtype == FDT_DTYPE_F32) {
        float *d = reinterpret_cast<float *>(m.p) + o;
        if (vec) { *reinterpret_cast<float4 *>(d) = v; return; }
        d[0] = v.x; d[m.cs] = v.y; d[2 * m.cs] = v.z; d[3 * m.cs] = v.w;
        return;
    }
    const unsigned short a = head_narrow16(v.x, dtype), c = head_narrow16(v.y, dtype), e = head_narrow16(v.z, dtype),
                         f = head_narrow16(v.w, dtype);
    unsigned short *d = reinterpret_cast<unsigned short *>(m.p) + o;
    if (vec) { *reinterpret_cast<uint2 *>(d) = make_uint2((unsigned)a | ((unsigned)c << 16), (unsigned)e | ((unsigned)f << 16)); return; }
    d[0] = a; d[m.cs] = c; d[2 * m.cs] = e; d[3 * m.cs] = f;
}
// torch.max over a dimension propagates NaN
__device__ __forceinline__ float nanmax(const float a, const float b) { return (a > b || a != a) ? a : b; }
// the 4 channels of pixel q of image b in the conf / loc map of level l
template <int F>
__device__ __forceinline__ float4 head_map4(const HeadLevels &h, const HeadMap &m, const bool vec, const int l, const int b, const int q)
{
    if constexpr (F == HEAD_F32_NCHW) {
        const int hw = h.hw[l];
        const float *c = reinterpret_cast<const float *>(m.p) + (int64_t)b * 4 * hw + q;
        return make_float4(__ldg(c), __ldg(c + hw), __ldg(c + 2 * hw), __ldg(c + 3 * hw));
    } else {
        return head_load4(m, h.dtype, vec, b, q);
    }
}
// (neg, pos) logits of prior p of image b: the max-in-out reduction
template <int F>
__device__ __forceinline__ float2 head_logits(const HeadLevels &h, const int b, const int p)
{
    const int l = head_level(h, p);
    const float4 c = head_map4<F>(h, h.conf[l], (h.vec >> l) & 1u, l, b, p - h.off[l]);
    if (h.neg_max[l]) return make_float2(nanmax(nanmax(c.x, c.y), c.z), c.w);
    return make_float2(c.x, nanmax(nanmax(c.y, c.z), c.w));
}
// nn.Softmax(dim=-1) over (neg, pos): exp(x - max) / sum, exp evaluated in fp64 and rounded once (library convention), fp32
// sum and IEEE division.  The larger element contributes exp(0) = 1 exactly, so ONE exp is evaluated; if neither argument
// is zero a NaN or inf - inf is involved and the sum -- hence both outputs -- is NaN whatever the other term is.
__device__ __forceinline__ float2 softmax2(const float2 x)
{
    const float m = nanmax(x.x, x.y);
    const float a0 = x.x - m, a1 = x.y - m;
    const bool z0 = a0 == 0.0f, z1 = a1 == 0.0f;
    if (!z0 && !z1) return make_float2(NAN, NAN);
    const float e = fdt_expf_cr(z0 ? a1 : a0);
    const float e0 = z0 ? 1.0f : e, e1 = z0 ? e : 1.0f;
    const float sum = e0 + e1;
    return make_float2(e0 / sum, e1 / sum);
}
template <int F>
__device__ __forceinline__ float4 head_loc_row(const HeadLevels &h, const int b, const int p)
{
    const int l = head_level(h, p);
    return head_map4<F>(h, h.loc[l], (h.vec >> (8 + l)) & 1u, l, b, p - h.off[l]);
}

// Gradient routing of the max-in-out reduction: the channel (0..3) of a prior's four conf channels c that receives the gradient
// of the max-reduced logit.  torch's max(dim) backward sends it to the index max returns: the first NaN of the triple if there
// is one, else the lowest channel equal to the maximum (-0.0 == +0.0).  The other two channels of the triple get +0.0.
__device__ __forceinline__ int head_max_channel(const float4 c, const int neg_max)
{
    const float a = neg_max ? c.x : c.y, b = neg_max ? c.y : c.z, d = neg_max ? c.z : c.w;
    int k;
    if (a != a) k = 0;
    else if (b != b) k = 1;
    else if (d != d) k = 2;
    else {
        const float m = fmaxf(fmaxf(a, b), d);
        k = a == m ? 0 : (b == m ? 1 : 2);
    }
    return neg_max ? k : k + 1;
}
// the gradients with respect to the head maps: the maps' element type, each in its own layout
struct HeadGrads {
    HeadGradMap conf[FDT_MAX_LEVELS];
    HeadGradMap loc[FDT_MAX_LEVELS];
    unsigned vec;                          // as HeadLevels::vec
    int f32_nchw;                          // as HeadLevels::f32_nchw
};
// writes d/d(maps) of prior p of image b from d/d(loc row) `gl` and d/d(neg, pos) `gc` (either sink may be null)
template <int F>
__device__ __forceinline__ void head_grad_store(const HeadLevels &h, const HeadGrads &g, const int b, const int p, const float4 gl,
                                                const float2 gc)
{
    const int l = head_level(h, p);
    const int q = p - h.off[l];
    const HeadGradMap &gloc = g.loc[l], &gconf = g.conf[l];
    if (gloc.p) {
        if constexpr (F == HEAD_F32_NCHW) {
            const int hw = h.hw[l];
            float *d = reinterpret_cast<float *>(gloc.p) + (int64_t)b * 4 * hw + q;
            d[0] = gl.x; d[hw] = gl.y; d[2 * hw] = gl.z; d[3 * hw] = gl.w;
        } else {
            head_store4(gloc, h.dtype, (g.vec >> (8 + l)) & 1u, b, q, gl);
        }
    }
    if (gconf.p) {
        const int nm = h.neg_max[l];
        const int k = head_max_channel(head_map4<F>(h, h.conf[l], (h.vec >> l) & 1u, l, b, q), nm);
        const float gm = nm ? gc.x : gc.y;       // the max-reduced logit's gradient
        float d[4];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            const bool single = nm ? ch == 3 : ch == 0;
            d[ch] = single ? (nm ? gc.y : gc.x) : (ch == k ? gm : 0.0f);
        }
        if constexpr (F == HEAD_F32_NCHW) {
            const int hw = h.hw[l];
            float *o = reinterpret_cast<float *>(gconf.p) + (int64_t)b * 4 * hw + q;
            o[0] = d[0]; o[hw] = d[1]; o[2 * hw] = d[2]; o[3 * hw] = d[3];
        } else {
            head_store4(gconf, h.dtype, (g.vec >> l) & 1u, b, q, make_float4(d[0], d[1], d[2], d[3]));
        }
    }
}

// ---- host side: the per-level description of the C ABI's head-map entries
static inline int64_t head_elem_bytes(const int dtype) { return dtype == FDT_DTYPE_F32 ? 4 : 2; }
// checks one map descriptor (a null `data` is the caller's to refuse: some entries do not read every map) and tells whether a
// prior's 4 channels are one aligned vector (channels adjacent, row address a multiple of 4 elements)
static int head_map_check(const char *who, const char *what, int l, const void *data, int64_t bs, int64_t cs, int64_t ps, int dtype,
                          bool *vec)
{
    *vec = false;
    if (!data) return FDT_OK;
    FDT_REQUIRE(bs > 0 && cs > 0 && ps > 0, FDT_E_INVALID, "%s: %s %d has a non-positive stride (%lld, %lld, %lld)", who, what, l,
                (long long)bs, (long long)cs, (long long)ps);
    const int64_t e = head_elem_bytes(dtype);
    FDT_REQUIRE(fdt_aligned(data, (size_t)e), FDT_E_INVALID, "%s: %s %d data is not aligned to its %lld-byte elements", who, what, l,
                (long long)e);
    *vec = cs == 1 && bs % 4 == 0 && ps % 4 == 0 && fdt_aligned(data, (size_t)(4 * e));
    return FDT_OK;
}
static inline int head_is_nchw(int64_t bs, int64_t cs, int64_t ps, int64_t hw) { return bs == 4 * hw && cs == hw && ps == 1; }
static int heads_fill(HeadLevels &hl, const char *who, const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype,
                      const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, int64_t *N_out)
{
    FDT_REQUIRE(n_levels >= 1 && n_levels <= FDT_MAX_LEVELS, FDT_E_UNSUPPORTED, "%s: n_levels=%d outside [1,%d]", who, n_levels, FDT_MAX_LEVELS);
    FDT_REQUIRE(f_h && f_w && neg_max_h, FDT_E_INVALID, "%s: null level description", who);
    FDT_REQUIRE(dtype == FDT_DTYPE_F32 || dtype == FDT_DTYPE_BF16 || dtype == FDT_DTYPE_F16, FDT_E_INVALID, "%s: unknown dtype %d",
                who, dtype);
    int64_t off = 0;
    hl = HeadLevels{};
    hl.L = n_levels;
    hl.dtype = dtype;
    hl.f32_nchw = dtype == FDT_DTYPE_F32;
    for (int l = 0; l < n_levels; ++l) {
        FDT_REQUIRE(f_h[l] >= 1 && f_w[l] >= 1, FDT_E_INVALID, "%s: level %d is %dx%d", who, l, f_h[l], f_w[l]);
        const int64_t hw = (int64_t)f_h[l] * f_w[l];
        bool v = false;
        if (conf_maps_h) {
            const fdt_head_map &m = conf_maps_h[l];
            int rc = head_map_check(who, "conf map", l, m.data, m.batch_stride, m.channel_stride, m.pixel_stride, dtype, &v);
            if (rc != FDT_OK) return rc;
            hl.conf[l] = HeadMap{m.data, m.batch_stride, m.channel_stride, m.pixel_stride};
            hl.vec |= v ? 1u << l : 0u;
            const bool dense = m.batch_stride == 4 * hw && ((m.channel_stride == hw && m.pixel_stride == 1) ||
                                                            (m.channel_stride == 1 && m.pixel_stride == 4));
            hl.dense |= dense ? 1u << l : 0u;
            hl.f32_nchw &= head_is_nchw(m.batch_stride, m.channel_stride, m.pixel_stride, hw);
        }
        if (loc_maps_h) {
            const fdt_head_map &m = loc_maps_h[l];
            int rc = head_map_check(who, "loc map", l, m.data, m.batch_stride, m.channel_stride, m.pixel_stride, dtype, &v);
            if (rc != FDT_OK) return rc;
            hl.loc[l] = HeadMap{m.data, m.batch_stride, m.channel_stride, m.pixel_stride};
            hl.vec |= v ? 1u << (8 + l) : 0u;
            hl.f32_nchw &= head_is_nchw(m.batch_stride, m.channel_stride, m.pixel_stride, hw);
        }
        hl.hw[l] = (int)hw;
        hl.off[l] = (int)off;
        hl.neg_max[l] = neg_max_h[l] ? 1 : 0;
        off += hw;
        FDT_REQUIRE(off < (1ll << 31), FDT_E_UNSUPPORTED, "%s: more than 2^31-1 priors", who);
    }
    for (int l = n_levels; l <= FDT_MAX_LEVELS; ++l) hl.off[l] = (int)off;
    *N_out = off;
    return FDT_OK;
}
// the descriptors of fp32 dense-NCHW maps given as a host array of device pointers (the entries without `_ex`); null stays null
template <class Desc, class Ptr>
static const Desc *heads_nchw(Desc (&d)[FDT_MAX_LEVELS], Ptr const *maps_h, const int *f_h, const int *f_w, int n_levels)
{
    if (!maps_h) return nullptr;
    for (int l = 0; l < FDT_MAX_LEVELS; ++l) {
        const int64_t hw = (l < n_levels && f_h && f_w) ? (int64_t)f_h[l] * f_w[l] : 1;
        d[l].data = l < n_levels ? maps_h[l] : nullptr;
        d[l].batch_stride = 4 * hw; d[l].channel_stride = hw; d[l].pixel_stride = 1;
    }
    return d;
}

}  // namespace
