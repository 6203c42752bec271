// Elementwise / pairwise box math of layers/box_utils.py and utils/calc_performance.py, plus PriorBox.
#include "fdt_common.cuh"

namespace {

constexpr int EW_THREADS = 256;
inline unsigned ew_blocks(int64_t n) { return (unsigned)((n + EW_THREADS - 1) / EW_THREADS); }

// prior_box.py:28-44 -- fp64 arithmetic in python operand order, one rounding to fp32
struct PriorParams {
    double width, height, stride, box;
    int n_scales, n_ar, f_w, f_h;
    double box_scale[8];
    double sqrt_ar[8];
};
__global__ void k_priorbox(const PriorParams P, float4 *__restrict__ out)
{
    const int per_cell = P.n_scales * (1 + P.n_ar);
    const int64_t total = (int64_t)P.f_h * P.f_w * per_cell;
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    int v = (int)(t % per_cell);
    int64_t cell = t / per_cell;
    int j = (int)(cell % P.f_w), i = (int)(cell / P.f_w);
    int s = v / (1 + P.n_ar), a = v % (1 + P.n_ar);
    double cx = (j + 0.5) * P.stride / P.width;            // :34
    double cy = (i + 0.5) * P.stride / P.height;           // :35
    double sx = P.box * P.box_scale[s] / P.width;          // :36
    double sy = P.box * P.box_scale[s] / P.height;         // :37
    if (a > 0) { sx = sx / P.sqrt_ar[a - 1]; sy = sy * P.sqrt_ar[a - 1]; }   // :41
    out[t] = make_float4((float)cx, (float)cy, (float)sx, (float)sy);
}

__global__ void k_point_form(const float4 *__restrict__ b, int64_t n, float4 *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 p = b[i];
    float hw = p.z / 2.0f, hh = p.w / 2.0f;
    out[i] = make_float4(p.x - hw, p.y - hh, p.x + hw, p.y + hh);          // box_utils.py:15-16
}
__global__ void k_center_size(const float4 *__restrict__ b, int64_t n, float4 *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 p = b[i];
    out[i] = make_float4((p.z + p.x) / 2.0f, (p.w + p.y) / 2.0f, p.z - p.x, p.w - p.y);   // box_utils.py:27-28
}
__global__ void k_encode(const float4 *__restrict__ m, const float4 *__restrict__ p, int64_t n, float v0, float v1, float4 *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = fdt_encode1(m[i], p[i], v0, v1);
}
__global__ void k_decode(const float4 *__restrict__ l, const float4 *__restrict__ p, int64_t n, float v0, float v1, float4 *__restrict__ out)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = fdt_decode1(l[i], p[i], v0, v1);
}

// torch.min/max and np.minimum/maximum propagate NaN; fminf/fmaxf do not
template <typename T> __device__ __forceinline__ T nmin(T a, T b) { return (a != a || b != b) ? (T)NAN : (a < b ? a : b); }
template <typename T> __device__ __forceinline__ T nmax(T a, T b) { return (a != a || b != b) ? (T)NAN : (a > b ? a : b); }

// box_utils.py:58-66 / :94-100 and calc_performance.py:20-31 / :65-74 ; out[A,B], one thread per pair,
// B (priors) is the fast axis so box_b loads and the store are coalesced, box_a is a broadcast.
template <typename T, bool IOU>
__global__ void k_pairwise(const T *__restrict__ a, int64_t A, const T *__restrict__ b, int64_t B, T *__restrict__ out)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t i = blockIdx.y;
    if (j >= B) return;
    const T ax1 = a[4 * i], ay1 = a[4 * i + 1], ax2 = a[4 * i + 2], ay2 = a[4 * i + 3];
    const T bx1 = b[4 * j], by1 = b[4 * j + 1], bx2 = b[4 * j + 2], by2 = b[4 * j + 3];
    T w = nmin(ax2, bx2) - nmax(ax1, bx1);
    T h = nmin(ay2, by2) - nmax(ay1, by1);
    w = nmax(w, (T)0); h = nmax(h, (T)0);
    T inter = w * h;
    if (IOU) {
        T area_a = (ax2 - ax1) * (ay2 - ay1);
        T area_b = (bx2 - bx1) * (by2 - by1);
        T uni = area_a + area_b - inter;
        out[i * B + j] = inter / uni;
    } else {
        out[i * B + j] = inter;
    }
}

// utils/calc_performance.py:34-51 calculate_distance (float64); `dis ** 0.25` correctly rounded, as the tracker computes it
__global__ void k_pairwise_distance_f64(const double *__restrict__ a, int64_t A, const double *__restrict__ b, int64_t B, double *__restrict__ out)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t i = blockIdx.y;
    if (j >= B) return;
    const double *p = a + 4 * i, *q = b + 4 * j;
    const double adx = p[2] - p[0], ady = p[3] - p[1], bdx = q[2] - q[0], bdy = q[3] - q[1];
    const double cax = (p[2] + p[0]) / 2, cay = (p[3] + p[1]) / 2, cbx = (q[2] + q[0]) / 2, cby = (q[3] + q[1]) / 2;
    const double dx = cbx - cax, dy = cby - cay;
    const double dz = ((adx - bdx) + (ady - bdy)) / 2;
    const double dis = __dadd_rn(__dadd_rn(__dmul_rn(dz, dz), __dmul_rn(dx, dx)), __dmul_rn(dy, dy));      // no FMA, numpy operand order
    out[i * B + j] = fdt_qroot_cr(dis);
}

// utils/calc_performance.py:77-92 calc_pr: one thread per prediction, max IoU over the truth boxes (given as x, y, w, h)
__global__ void k_calc_pr(const double *__restrict__ pred, int64_t P, int stride, const double *__restrict__ truth, int64_t T,
                          double thr, int32_t *__restrict__ tf)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P) return;
    const double *q = pred + stride * j;
    double best = -INFINITY;
    bool any_nan = false;
    for (int64_t t = 0; t < T; ++t) {
        const double x1 = truth[4 * t], y1 = truth[4 * t + 1], x2 = truth[4 * t + 2] + x1, y2 = truth[4 * t + 3] + y1;      // :88
        double w = nmin(x2, q[2]) - nmax(x1, q[0]);
        double h = nmin(y2, q[3]) - nmax(y1, q[1]);
        w = nmax(w, 0.0); h = nmax(h, 0.0);
        const double inter = w * h;
        const double uni = (x2 - x1) * (y2 - y1) + (q[2] - q[0]) * (q[3] - q[1]) - inter;
        const double v = inter / uni;
        if (v != v) any_nan = true;                 // np.max propagates NaN, NaN > thr is False
        else if (v > best) best = v;
    }
    tf[j] = (!any_nan && best > thr) ? 1 : 0;       // :91
}

// Detect's consumers (My_test.py:43-57, iouTracke_cal.py:55-68): per image and class, the leading rows with score >= thr
// (the python `while` stops at the first row below thr), boxes scaled to pixels in fp32 (detections[...] * scale).
// One block per image; rows_out[b][r] = [x1*w, y1*h, x2*w, y2*h, score] in class-major order, n_rows[b] = how many.
__global__ void k_detections_to_rows(const float *__restrict__ det, int C, int top_k, float thr, float width, float height,
                                     float *__restrict__ rows_out, int32_t *__restrict__ n_rows)
{
    __shared__ int s_len, s_base;
    const int b = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int i = 0; i < C; ++i) {
        const float *plane = det + ((int64_t)(b * C + i) * top_k) * 5;
        if (tid == 0) s_len = top_k;
        __syncthreads();
        for (int j = tid; j < top_k; j += blockDim.x)
            if (!(plane[5 * j] >= thr)) atomicMin(&s_len, j);                 // first row that fails `>= thr` (NaN fails)
        __syncthreads();
        const int len = s_len, base = s_base;
        for (int j = tid; j < len; j += blockDim.x) {
            const float *r = plane + 5 * j;
            float *o = rows_out + ((int64_t)b * C * top_k + base + j) * 5;
            o[0] = r[1] * width; o[1] = r[2] * height; o[2] = r[3] * width; o[3] = r[4] * height; o[4] = r[0];
        }
        __syncthreads();
        if (tid == 0) s_base = base + len;
        __syncthreads();
    }
    if (tid == 0) n_rows[b] = s_base;
}

// Detect -> tracker without leaving the device (iouTracke_cal.py:55-84 detect_face, one image per frame): the rows of
// k_detections_to_rows divided by `shrink` (:76-80, float32) and widened to float64, frames packed back to back; a frame without a
// detection becomes the reference's dummy row [0, 0, 0, 0, 0.4] (:73-74).  Two passes: counts -> offsets, then the rows.
__device__ __forceinline__ int leading_rows(const float *__restrict__ plane, const int top_k, const float thr, int *s_len)
{
    if (threadIdx.x == 0) *s_len = top_k;
    __syncthreads();
    for (int j = threadIdx.x; j < top_k; j += blockDim.x)
        if (!(plane[5 * j] >= thr)) atomicMin(s_len, j);                      // first row that fails `>= thr` (NaN fails)
    __syncthreads();
    const int len = *s_len;
    __syncthreads();
    return len;
}
__global__ void k_frames_count(const float *__restrict__ det, int C, int top_k, float thr, int32_t *__restrict__ n_rows)
{
    __shared__ int s_len;
    const int f = blockIdx.x;
    int n = 0;
    for (int i = 0; i < C; ++i) n += leading_rows(det + ((int64_t)(f * C + i) * top_k) * 5, top_k, thr, &s_len);
    if (threadIdx.x == 0) n_rows[f] = n;
}
// frame_off[0] = 0, frame_off[f + 1] = frame_off[f] + max(n_rows[f], 1)   (one block; F in chunks of blockDim)
__global__ void k_frames_offsets(const int32_t *__restrict__ n_rows, int64_t F, int64_t *__restrict__ frame_off)
{
    __shared__ long long s_warp[33];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) { s_carry = 0; frame_off[0] = 0; }
    __syncthreads();
    for (int64_t base = 0; base < F; base += blockDim.x) {
        const int64_t f = base + threadIdx.x;
        long long v = 0;
        if (f < F) { const int n = n_rows[f]; v = n > 0 ? n : 1; }
        long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            long long w = lane < nw ? s_warp[lane] : 0, winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += t; }
            s_warp[lane] = winc - w;
            if (lane == 31) s_warp[32] = winc;
        }
        __syncthreads();
        if (f < F) frame_off[f + 1] = s_carry + s_warp[warp] + inc;
        __syncthreads();
        if (threadIdx.x == 0) s_carry += s_warp[32];
        __syncthreads();
    }
}
__global__ void k_frames_pack(const float *__restrict__ det, int C, int top_k, float thr, float width, float height, double shrink,
                              const int64_t *__restrict__ frame_off, double *__restrict__ dets)
{
    __shared__ int s_len;
    const int f = blockIdx.x;
    double *out = dets + 5 * frame_off[f];
    int base = 0;
    for (int i = 0; i < C; ++i) {
        const float *plane = det + ((int64_t)(f * C + i) * top_k) * 5;
        const int len = leading_rows(plane, top_k, thr, &s_len);
        for (int j = threadIdx.x; j < len; j += blockDim.x) {
            const float *r = plane + 5 * j;
            double *o = out + 5 * (base + j);
            // pt = detections[...] * scale in fp32 (:64); np.array keeps float32 and `/ shrink` divides in float32 (:76-79, a python
            // scalar does not promote); det0.tolist() then widens exactly (:127).  The score is a float32 too (:70).
            const float sh = (float)shrink;
            o[0] = (double)((r[1] * width) / sh); o[1] = (double)((r[2] * height) / sh);
            o[2] = (double)((r[3] * width) / sh); o[3] = (double)((r[4] * height) / sh); o[4] = (double)r[0];
        }
        base += len;
    }
    if (base == 0 && threadIdx.x == 0) { out[0] = 0.0; out[1] = 0.0; out[2] = 0.0; out[3] = 0.0; out[4] = 0.4; }     // :73-74
}

// box_utils.py:261-269: global max, then log(sum(exp(x - max))) + max per row
__global__ void k_global_max(const float *__restrict__ x, int64_t n, unsigned *__restrict__ gmax_key)
{
    float m = -INFINITY;
    bool nan = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float v = x[i];
        nan |= (v != v);
        m = fmaxf(m, v);
    }
    if (nan) m = NAN;
    unsigned k = fdt_float_key(m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) k = max(k, __shfl_xor_sync(0xffffffffu, k, o));
    if ((threadIdx.x & 31) == 0) atomicMax(gmax_key, k);
}
__global__ void k_lse_rows(const float *__restrict__ x, int64_t R, int C, const unsigned *__restrict__ gmax_key, float *__restrict__ out)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const float xmax = fdt_key_float(*gmax_key);
    float s = 0.0f;
    for (int c = 0; c < C; ++c) s += fdt_expf_cr(x[r * C + c] - xmax);
    out[r] = fdt_logf_cr(s) + xmax;
}

}  // namespace

FDT_API int fdt_priorbox(double width, double height, double stride, double box,
                         int n_scales, const double *box_scale_h, int n_ar, const double *sqrt_ar_h,
                         int f_w, int f_h, float *out, fdt_stream_t stream)
{
    FDT_REQUIRE(n_scales >= 0 && n_scales <= 8 && n_ar >= 0 && n_ar <= 8, FDT_E_UNSUPPORTED,
                "fdt_priorbox: n_scales=%d / n_ar=%d outside [0,8]", n_scales, n_ar);
    FDT_REQUIRE(f_w >= 0 && f_h >= 0, FDT_E_INVALID, "fdt_priorbox: negative feature-map size");
    int64_t total = (int64_t)f_h * f_w * n_scales * (1 + n_ar);
    if (total == 0) return FDT_OK;
    FDT_REQUIRE(out && fdt_aligned(out, 16), FDT_E_INVALID, "fdt_priorbox: out null or not 16-byte aligned");
    FDT_REQUIRE((n_scales == 0 || box_scale_h) && (n_ar == 0 || sqrt_ar_h), FDT_E_INVALID, "fdt_priorbox: null scale arrays");
    PriorParams P{};
    P.width = width; P.height = height; P.stride = stride; P.box = box;
    P.n_scales = n_scales; P.n_ar = n_ar; P.f_w = f_w; P.f_h = f_h;
    for (int s = 0; s < n_scales; ++s) P.box_scale[s] = box_scale_h[s];
    for (int a = 0; a < n_ar; ++a) P.sqrt_ar[a] = sqrt_ar_h[a];
    k_priorbox<<<ew_blocks(total), EW_THREADS, 0, (cudaStream_t)stream>>>(P, (float4 *)out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

#define FDT_EW_PROLOGUE(name, ...)                                                                         \
    FDT_REQUIRE(n >= 0, FDT_E_INVALID, name ": negative n");                                               \
    if (n == 0) return FDT_OK;                                                                             \
    { const void *ptrs_[] = {__VA_ARGS__};                                                                 \
      for (const void *q : ptrs_) FDT_REQUIRE(q && fdt_aligned(q, 16), FDT_E_INVALID, name ": null or not 16-byte aligned pointer"); }

FDT_API int fdt_point_form(const float *boxes, int64_t n, float *out, fdt_stream_t stream)
{
    FDT_EW_PROLOGUE("fdt_point_form", boxes, out)
    k_point_form<<<ew_blocks(n), EW_THREADS, 0, (cudaStream_t)stream>>>((const float4 *)boxes, n, (float4 *)out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}
FDT_API int fdt_center_size(const float *boxes, int64_t n, float *out, fdt_stream_t stream)
{
    FDT_EW_PROLOGUE("fdt_center_size", boxes, out)
    k_center_size<<<ew_blocks(n), EW_THREADS, 0, (cudaStream_t)stream>>>((const float4 *)boxes, n, (float4 *)out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}
FDT_API int fdt_encode(const float *matched, const float *priors, int64_t n, float var0, float var1, float *out, fdt_stream_t stream)
{
    FDT_EW_PROLOGUE("fdt_encode", matched, priors, out)
    k_encode<<<ew_blocks(n), EW_THREADS, 0, (cudaStream_t)stream>>>((const float4 *)matched, (const float4 *)priors, n, var0, var1, (float4 *)out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}
FDT_API int fdt_decode(const float *loc, const float *priors, int64_t n, float var0, float var1, float *out, fdt_stream_t stream)
{
    FDT_EW_PROLOGUE("fdt_decode", loc, priors, out)
    k_decode<<<ew_blocks(n), EW_THREADS, 0, (cudaStream_t)stream>>>((const float4 *)loc, (const float4 *)priors, n, var0, var1, (float4 *)out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

template <typename T, bool IOU>
static int pairwise(const char *name, const T *a, int64_t A, const T *b, int64_t B, T *out, fdt_stream_t stream)
{
    FDT_REQUIRE(A >= 0 && B >= 0 && A < 65536, FDT_E_INVALID, "%s: bad sizes A=%lld (max 65535) B=%lld", name, (long long)A, (long long)B);
    if (A == 0 || B == 0) return FDT_OK;
    FDT_REQUIRE(a && b && out, FDT_E_INVALID, "%s: null pointer", name);
    dim3 g(ew_blocks(B), (unsigned)A);
    k_pairwise<T, IOU><<<g, EW_THREADS, 0, (cudaStream_t)stream>>>(a, A, b, B, out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}
FDT_API int fdt_intersect(const float *a, int64_t A, const float *b, int64_t B, float *out, fdt_stream_t s) { return pairwise<float, false>("fdt_intersect", a, A, b, B, out, s); }
FDT_API int fdt_calculate_iou(const float *a, int64_t A, const float *b, int64_t B, float *out, fdt_stream_t s) { return pairwise<float, true>("fdt_calculate_iou", a, A, b, B, out, s); }
FDT_API int fdt_calculate_iou_f64(const double *a, int64_t A, const double *b, int64_t B, double *out, fdt_stream_t s) { return pairwise<double, true>("fdt_calculate_iou_f64", a, A, b, B, out, s); }

FDT_API int fdt_intersect_f64(const double *a, int64_t A, const double *b, int64_t B, double *out, fdt_stream_t s) { return pairwise<double, false>("fdt_intersect_f64", a, A, b, B, out, s); }

FDT_API int fdt_calculate_distance_f64(const double *a, int64_t A, const double *b, int64_t B, double *out, fdt_stream_t stream)
{
    FDT_REQUIRE(A >= 0 && B >= 0 && A < 65536, FDT_E_INVALID, "fdt_calculate_distance_f64: bad sizes");
    if (A == 0 || B == 0) return FDT_OK;
    FDT_REQUIRE(a && b && out, FDT_E_INVALID, "fdt_calculate_distance_f64: null pointer");
    dim3 g(ew_blocks(B), (unsigned)A);
    k_pairwise_distance_f64<<<g, EW_THREADS, 0, (cudaStream_t)stream>>>(a, A, b, B, out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_calc_pr(const double *predict, int64_t P, int predict_stride, const double *truth, int64_t T, double iou_thresh,
                        int32_t *tf, fdt_stream_t stream)
{
    FDT_REQUIRE(P >= 0 && T >= 0 && predict_stride >= 4, FDT_E_INVALID, "fdt_calc_pr: bad sizes");
    if (P == 0) return FDT_OK;
    FDT_REQUIRE(predict && tf && (T == 0 || truth), FDT_E_INVALID, "fdt_calc_pr: null pointer");
    k_calc_pr<<<ew_blocks(P), EW_THREADS, 0, (cudaStream_t)stream>>>(predict, P, predict_stride, truth, T, iou_thresh, tf);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_detections_to_rows(const float *detections, int B, int C, int top_k, float thresh, float width, float height,
                                   float *rows_out, int32_t *n_rows, fdt_stream_t stream)
{
    FDT_REQUIRE(B >= 0 && C >= 1 && top_k >= 1, FDT_E_INVALID, "fdt_detections_to_rows: bad sizes");
    if (B == 0) return FDT_OK;
    FDT_REQUIRE(detections && rows_out && n_rows, FDT_E_INVALID, "fdt_detections_to_rows: null pointer");
    k_detections_to_rows<<<B, 256, 0, (cudaStream_t)stream>>>(detections, C, top_k, thresh, width, height, rows_out, n_rows);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_detections_to_frames_count(const float *detections, int64_t F, int C, int top_k, float thresh,
                                           int32_t *n_rows, int64_t *frame_off, fdt_stream_t stream)
{
    FDT_REQUIRE(F >= 0 && F < (1ll << 31) && C >= 1 && top_k >= 1, FDT_E_INVALID, "fdt_detections_to_frames_count: bad sizes");
    FDT_REQUIRE(frame_off != nullptr, FDT_E_INVALID, "fdt_detections_to_frames_count: frame_off is null");
    if (F == 0) { FDT_CUDA(cudaMemsetAsync(frame_off, 0, sizeof(int64_t), (cudaStream_t)stream)); return FDT_OK; }
    FDT_REQUIRE(detections && n_rows, FDT_E_INVALID, "fdt_detections_to_frames_count: null pointer");
    k_frames_count<<<(unsigned)F, 128, 0, (cudaStream_t)stream>>>(detections, C, top_k, thresh, n_rows);
    FDT_LAUNCH_CHECK();
    k_frames_offsets<<<1, 1024, 0, (cudaStream_t)stream>>>(n_rows, F, frame_off);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_detections_to_frames_pack(const float *detections, int64_t F, int C, int top_k, float thresh, float width, float height,
                                          double shrink, const int64_t *frame_off, double *dets_out, fdt_stream_t stream)
{
    FDT_REQUIRE(F >= 0 && F < (1ll << 31) && C >= 1 && top_k >= 1, FDT_E_INVALID, "fdt_detections_to_frames_pack: bad sizes");
    if (F == 0) return FDT_OK;
    FDT_REQUIRE(detections && frame_off && dets_out, FDT_E_INVALID, "fdt_detections_to_frames_pack: null pointer");
    k_frames_pack<<<(unsigned)F, 128, 0, (cudaStream_t)stream>>>(detections, C, top_k, thresh, width, height, shrink, frame_off, dets_out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_log_sum_exp(const float *x, int64_t R, int C, float *out, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    FDT_REQUIRE(R >= 0 && C >= 1, FDT_E_INVALID, "fdt_log_sum_exp: bad sizes");
    if (R == 0) return FDT_OK;
    FDT_REQUIRE(x && out && ws && ws_bytes >= 256, FDT_E_WORKSPACE, "fdt_log_sum_exp: needs a 256-byte workspace");
    FDT_CUDA(cudaMemsetAsync(ws, 0, 4, st));
    int64_t n = R * C;
    unsigned blocks = (unsigned)((n + EW_THREADS * 8 - 1) / (EW_THREADS * 8));
    if (blocks > FDT_NUM_SMS * 8) blocks = FDT_NUM_SMS * 8;
    k_global_max<<<blocks, EW_THREADS, 0, st>>>(x, n, (unsigned *)ws);
    FDT_LAUNCH_CHECK();
    k_lse_rows<<<ew_blocks(R), EW_THREADS, 0, st>>>(x, R, C, (const unsigned *)ws, out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

// ---- self-test of fdt_expf_cr / fdt_logf_cr against the CUDA math library (fdt_common.cuh) --------------------------------------
namespace {
__global__ void k_selftest_cr_math(int which, uint32_t first, uint64_t count, unsigned long long *result)
{
    unsigned long long bad = 0, lowest = ~0ull;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t bits = first + (uint32_t)i;
        const float x = __uint_as_float(bits);
        const float a = which == 0 ? fdt_expf_cr(x) : fdt_logf_cr(x);
        const float b = which == 0 ? (float)exp((double)x) : (float)log((double)x);
        const bool same = __float_as_uint(a) == __float_as_uint(b) || (a != a && b != b);
        if (!same) { ++bad; if ((unsigned long long)bits + 1 < lowest) lowest = (unsigned long long)bits + 1; }
    }
    if (bad) { atomicAdd(&result[0], bad); atomicMin(&result[1], lowest); }
}
}  // namespace

FDT_API int fdt_selftest_cr_math(int which, uint32_t first_bits, uint64_t count, uint64_t *result, fdt_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    FDT_REQUIRE((which == 0 || which == 1) && result, FDT_E_INVALID, "fdt_selftest_cr_math: which must be 0 or 1, result non-null");
    const unsigned long long init[2] = {0ull, ~0ull};
    FDT_CUDA(cudaMemcpyAsync(result, init, sizeof(init), cudaMemcpyHostToDevice, st));
    if (count == 0) return FDT_OK;
    k_selftest_cr_math<<<FDT_NUM_SMS * 8, 256, 0, st>>>(which, first_bits, count, (unsigned long long *)result);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}
