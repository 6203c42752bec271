// Access to the models' per-level NCHW head maps (SURVEY 8f rank 1), shared by Detect (detect.cu) and MultiBoxLoss
// (multibox.cu).
//
// The models hand Detect the outputs of their prediction convolutions, per pyramid level and NCHW: loc_l[B,4,H,W] and the
// 4-channel max-in-out confidence conf_l[B,4,H,W] (pyramid.py:291-306).  The reference turns them into loc[B,N,4] and
// conf[B,N,2] with chunk / max / cat / permute / contiguous / view / cat and a 2-way softmax (pyramid.py:293-309, 331-332);
// the kernels read the maps directly.  Prior n of level l sits at pixel q = n - off[l] (y outer, x inner).
#pragma once
#include "fdt_common.cuh"

namespace {

constexpr int FDT_MAX_LEVELS = 8;
struct HeadLevels {
    const float *conf[FDT_MAX_LEVELS];     // [B,4,hw] per level
    const float *loc[FDT_MAX_LEVELS];      // [B,4,hw] per level
    int hw[FDT_MAX_LEVELS];
    int off[FDT_MAX_LEVELS + 1];           // first prior of each level; off[L] = N
    int neg_max[FDT_MAX_LEVELS];           // 1: neg = max(ch0..2), pos = ch3 (pyramid.py:293-297); 0: neg = ch0, pos = max(ch1..3) (:299-304)
    int L;
};
__device__ __forceinline__ int head_level(const HeadLevels &h, const int p)
{
    int l = 0;
#pragma unroll
    for (int q = 1; q < FDT_MAX_LEVELS; ++q) l += (q < h.L && p >= h.off[q]) ? 1 : 0;
    return l;
}
// torch.max over a dimension propagates NaN
__device__ __forceinline__ float nanmax(const float a, const float b) { return (a > b || a != a) ? a : b; }
// (neg, pos) logits of prior p of image b: the max-in-out reduction
__device__ __forceinline__ float2 head_logits(const HeadLevels &h, const int b, const int p)
{
    const int l = head_level(h, p);
    const int hw = h.hw[l];
    const float *c = h.conf[l] + (int64_t)b * 4 * hw + (p - h.off[l]);
    const float c0 = __ldg(c), c1 = __ldg(c + hw), c2 = __ldg(c + 2 * hw), c3 = __ldg(c + 3 * hw);
    if (h.neg_max[l]) return make_float2(nanmax(nanmax(c0, c1), c2), c3);
    return make_float2(c0, nanmax(nanmax(c1, c2), c3));
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
__device__ __forceinline__ float4 head_loc_row(const HeadLevels &h, const int b, const int p)
{
    const int l = head_level(h, p);
    const int hw = h.hw[l];
    const float *c = h.loc[l] + (int64_t)b * 4 * hw + (p - h.off[l]);
    return make_float4(__ldg(c), __ldg(c + hw), __ldg(c + 2 * hw), __ldg(c + 3 * hw));
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
// maps of the gradients with respect to the head maps, laid out as HeadLevels' maps ([B,4,hw] per level)
struct HeadGrads {
    float *conf[FDT_MAX_LEVELS];
    float *loc[FDT_MAX_LEVELS];
};
// writes d/d(maps) of prior p of image b from d/d(loc row) `gl` and d/d(neg, pos) `gc` (either sink may be null)
__device__ __forceinline__ void head_grad_store(const HeadLevels &h, const HeadGrads &g, const int b, const int p, const float4 gl,
                                                const float2 gc)
{
    const int l = head_level(h, p);
    const int hw = h.hw[l];
    const int64_t o = (int64_t)b * 4 * hw + (p - h.off[l]);
    // (selected, not indexed: an indexed kernel-parameter array of pointers is copied to the stack)
    float *gloc = nullptr, *gconf = nullptr;
#pragma unroll
    for (int q = 0; q < FDT_MAX_LEVELS; ++q)
        if (q == l) { gloc = g.loc[q]; gconf = g.conf[q]; }
    if (gloc) {
        float *d = gloc + o;
        d[0] = gl.x; d[hw] = gl.y; d[2 * hw] = gl.z; d[3 * hw] = gl.w;
    }
    if (gconf) {
        const float *c = h.conf[l] + o;
        const int nm = h.neg_max[l];
        const int k = head_max_channel(make_float4(__ldg(c), __ldg(c + hw), __ldg(c + 2 * hw), __ldg(c + 3 * hw)), nm);
        const float gm = nm ? gc.x : gc.y;       // the max-reduced logit's gradient
        float *d = gconf + o;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
            const bool single = nm ? ch == 3 : ch == 0;
            d[ch * hw] = single ? (nm ? gc.y : gc.x) : (ch == k ? gm : 0.0f);
        }
    }
}

// host side: the per-level description of the C ABI's head-map entries
static int heads_fill(HeadLevels &hl, const char *who, const float *const *loc_maps_h, const float *const *conf_maps_h,
                      const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, int64_t *N_out)
{
    FDT_REQUIRE(n_levels >= 1 && n_levels <= FDT_MAX_LEVELS, FDT_E_UNSUPPORTED, "%s: n_levels=%d outside [1,%d]", who, n_levels, FDT_MAX_LEVELS);
    FDT_REQUIRE(f_h && f_w && neg_max_h, FDT_E_INVALID, "%s: null level description", who);
    int64_t off = 0;
    hl = HeadLevels{};
    hl.L = n_levels;
    for (int l = 0; l < n_levels; ++l) {
        FDT_REQUIRE(f_h[l] >= 1 && f_w[l] >= 1, FDT_E_INVALID, "%s: level %d is %dx%d", who, l, f_h[l], f_w[l]);
        hl.conf[l] = conf_maps_h ? conf_maps_h[l] : nullptr;
        hl.loc[l] = loc_maps_h ? loc_maps_h[l] : nullptr;
        hl.hw[l] = f_h[l] * f_w[l];
        hl.off[l] = (int)off;
        hl.neg_max[l] = neg_max_h[l] ? 1 : 0;
        off += (int64_t)f_h[l] * f_w[l];
        FDT_REQUIRE(off < (1ll << 31), FDT_E_UNSUPPORTED, "%s: more than 2^31-1 priors", who);
    }
    for (int l = n_levels; l <= FDT_MAX_LEVELS; ++l) hl.off[l] = (int)off;
    *N_out = off;
    return FDT_OK;
}

}  // namespace
