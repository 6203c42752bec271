/*
 * fdt_b200.h -- C ABI of libfdt_b200.so: the B200 (sm_100a) SSD box pipeline.
 *
 * The reference (limacv/Face-detection-and-tracking) is pure Python and has NO FFI; its boundary
 * for this path is the Python call signatures of `layers` (SURVEY.md section 8b).  Each entry point
 * below names the reference function it replaces (file:line relative to the reference root); the
 * Python modules in face-detection-and-tracking_b200/ keep those signatures and call these symbols
 * through ctypes.  INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer owned by the caller unless the
 *     parameter is documented as host (`_h` suffix or "host");
 *   - the library allocates nothing on the device-pointer entry points: scratch comes from a caller
 *     workspace sized by the matching *_workspace_bytes(); 256-byte alignment is required;
 *   - every launch goes to `stream` (a cudaStream_t passed as void*), asynchronously; calls are
 *     reentrant across streams with distinct workspaces and CUDA-graph capturable;
 *   - a Detect workspace is STATEFUL: its first 256 bytes carry a call sequence between calls (see
 *     fdt_detect).  Use one workspace per stream, do not write into it, and do not hand the same
 *     workspace to two streams at a time; memory that never was a workspace (any content) is fine;
 *   - returns FDT_OK or a negative FDT_E_* code; fdt_last_error() gives the thread-local message;
 *     no exceptions, no exit(), no CPU fallback.
 *   - fp32 arithmetic is IEEE in the reference's operand order with FMA contraction off
 *     (-fmad=false); exp/log are evaluated in fp64 and rounded once to fp32.
 */
#ifndef FDT_B200_H
#define FDT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDT_OK             0
#define FDT_E_INVALID     -1   /* bad argument (null pointer, negative size, misaligned buffer) */
#define FDT_E_CUDA        -2   /* CUDA runtime error; message carries cudaGetErrorString */
#define FDT_E_WORKSPACE   -3   /* workspace smaller than *_workspace_bytes() */
#define FDT_E_UNSUPPORTED -4   /* size outside the kernel limits (see each function) */
#define FDT_E_DEVICE      -5   /* device is not sm_100 (B200) */

/* overlap rule of the sibling NMS implementations (fdt_nms_variant); 0 = layers/box_utils.nms */
#define FDT_NMS_SUMFIRST   1      /* union = (area_i + area_j) - inter   (numpy / FaceBoxes / MTCNN operand order) */
#define FDT_NMS_MINIMUM    2      /* overlap = inter / min(area_i, area_j)   (mode="Minimum") */
#define FDT_NMS_PLUS1      4      /* widths, heights and areas measured with "+ 1" (pixel convention) */
#define FDT_NMS_LE         8      /* a box survives iff overlap <= thresh (default: overlap < thresh) */

#define FDT_MAX_NMS_TOP_K  8000   /* candidates that can enter Detect's NMS per image/class (the reference uses 5000) */

/* sticky status bits of a Detect workspace (fdt_detect_status): a device-side wait gave up after ~4 s */
#define FDT_STATUS_TIMEOUT_LOCAL 1u   /* a call of the same workspace never completed (the kernel also traps) */
#define FDT_STATUS_TIMEOUT_PEER  2u   /* fused multi-GPU gather: a peer rank never acknowledged / never delivered its rows */

typedef void *fdt_stream_t;        /* cudaStream_t */
typedef struct fdt_ctx fdt_ctx;    /* host-buffer context: owns a stream, device + pinned staging buffers */

int         fdt_version(void);
const char *fdt_last_error(void);
/* FDT_OK iff `device` exists and is compute capability 10.0 (the only target this library is built for). */
int         fdt_device_check(int device);

/* ---- P1  PriorBoxLayer.__call__  (layers/functions/prior_box.py:28-44) --------------------------
 * One pyramid level -> out[f_h*f_w*n_scales*(1+n_ar), 4] = [cx,cy,w,h], y outer / x inner.
 * box_scale_h[n_scales] = (2**(1/3))**s and sqrt_ar_h[n_ar] = sqrt(ar) are HOST arrays evaluated by the
 * caller in python-float arithmetic (prior_box.py:33,41); fp64 on device, one rounding to fp32. */
int fdt_priorbox(double width, double height, double stride, double box,
                 int n_scales, const double *box_scale_h, int n_ar, const double *sqrt_ar_h,
                 int f_w, int f_h, float *out, fdt_stream_t stream);

/* ---- M1  point_form / center_size  (layers/box_utils.py:7-16, 19-28) ---------------------------- */
int fdt_point_form(const float *boxes, int64_t n, float *out, fdt_stream_t stream);
int fdt_center_size(const float *boxes, int64_t n, float *out, fdt_stream_t stream);

/* ---- M2/M3  intersect / calculate_iou  (layers/box_utils.py:31-67, 70-100) -> out[A,B] fp32 ------ */
int fdt_intersect(const float *box_a, int64_t A, const float *box_b, int64_t B, float *out, fdt_stream_t stream);
int fdt_calculate_iou(const float *box_a, int64_t A, const float *box_b, int64_t B, float *out, fdt_stream_t stream);
/* ---- T1  utils.calc_performance.calculate_iou (utils/calc_performance.py:54-74), float64 -------- */
int fdt_calculate_iou_f64(const double *box_a, int64_t A, const double *box_b, int64_t B, double *out, fdt_stream_t stream);

/* ---- (SURVEY 8f, Detect consumers)  utils.calc_performance.intersect / calculate_distance / calc_pr, float64 -----------------
 * (utils/calc_performance.py:4-31, 34-51, 77-92).  calculate_distance ends in x ** 0.25, correctly rounded.
 * calc_pr: predict[P, predict_stride >= 4] rows [x1,y1,x2,y2,(score..)], truth[T,4] rows [x,y,w,h] -> tf[P] int32 =
 * (max_t IoU > iou_thresh); NaN IoU makes the max NaN and the comparison false, as numpy does. */
int fdt_intersect_f64(const double *box_a, int64_t A, const double *box_b, int64_t B, double *out, fdt_stream_t stream);
int fdt_calculate_distance_f64(const double *box_a, int64_t A, const double *box_b, int64_t B, double *out, fdt_stream_t stream);
int fdt_calc_pr(const double *predict, int64_t P, int predict_stride, const double *truth, int64_t T, double iou_thresh,
                int32_t *tf, fdt_stream_t stream);

/* Detect's row read-out (My_test.py:43-57, iouTracke_cal.py:55-68): for every image, and class by class, the leading rows of
 * detections[B,C,top_k,5] with score >= thresh, scaled to pixels -> rows_out[B, C*top_k, 5] = [x1,y1,x2,y2,score], n_rows[B]. */
int fdt_detections_to_rows(const float *detections, int B, int C, int top_k, float thresh, float width, float height,
                           float *rows_out, int32_t *n_rows, fdt_stream_t stream);

/* Detect -> tracker on the device (iouTracke_cal.py:55-84 detect_face, one image per frame): the same leading rows, divided by
 * `shrink` in float32 (:76-80) and widened to float64, packed frame after frame as fdt_iou_track wants them; a frame without a detection gets
 * the reference's dummy row [0, 0, 0, 0, 0.4] (:73-74).  _count fills n_rows[F] (int32, before the dummy rule) and
 * frame_off[F+1] (int64, after it); the caller reads frame_off[F] to size dets_out[frame_off[F], 5], then calls _pack. */
int fdt_detections_to_frames_count(const float *detections, int64_t F, int C, int top_k, float thresh,
                                   int32_t *n_rows, int64_t *frame_off, fdt_stream_t stream);
int fdt_detections_to_frames_pack(const float *detections, int64_t F, int C, int top_k, float thresh, float width, float height,
                                  double shrink, const int64_t *frame_off, double *dets_out, fdt_stream_t stream);

/* ---- M6 / D1  encode / decode  (layers/box_utils.py:213-234, 238-258) --------------------------- */
int fdt_encode(const float *matched, const float *priors, int64_t n, float var0, float var1, float *out, fdt_stream_t stream);
int fdt_decode(const float *loc, const float *priors, int64_t n, float var0, float var1, float *out, fdt_stream_t stream);

/* ---- L1  log_sum_exp  (layers/box_utils.py:261-269): x[R,C] -> out[R]; global max as the reference.
 * workspace: 256 bytes. */
int fdt_log_sum_exp(const float *x, int64_t R, int C, float *out, void *ws, size_t ws_bytes, fdt_stream_t stream);

/* Self-test of the library's fp32 exp / log (the convention above: (float)exp((double)x), (float)log((double)x); the common ranges
 * take a lean fp64 evaluation and hand every value near an fp32 rounding boundary to the CUDA math library): compares both for the
 * `count` consecutive float bit patterns from `first_bits` on.  which = 0 exp, 1 log.  result (device, 2 x uint64, zeroed by the
 * call): [0] = mismatching patterns, [1] = the lowest mismatching pattern + 1 (all ones when there is none). */
int fdt_selftest_cr_math(int which, uint32_t first_bits, uint64_t count, uint64_t *result, fdt_stream_t stream);

/* ---- N1  nms  (layers/box_utils.py:275-340) ------------------------------------------------------
 * boxes[n,4], scores[n] -> keep[n] int64 zero-padded (indices into the input, descending score),
 * *count (device int64).  Sort ties: higher index first.  top_k <= 0 means n, as idx[-0:] does.
 * min(n, top_k) <= FDT_MAX_NMS_TOP_K runs in one shared-memory kernel; beyond that (the reference has no cap, :296-298) the call
 * takes the sort + pairwise-mask + reduce formulation (up to 131,072 boxes; the workspace grows with n * n / 8 bytes). */
size_t fdt_nms_workspace_bytes(int64_t n);
int fdt_nms(const float *boxes, const float *scores, int64_t n, float overlap, int64_t top_k,
            int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream);

/* ---- (SURVEY 8f rank 3) sibling decode + NMS implementations of the reference ---------------------------------------------
 * fdt_nms_variant: greedy NMS where EVERY box enters (no top_k) and the overlap rule is chosen by FDT_NMS_* flags:
 *   FACEBOX/encoderl.py:218-266 DataEncoder.nms_np, MTCNN/mtcnn/core/utils.py:62-113 nms   mode "Union":   FDT_NMS_SUMFIRST
 *                                                                                      mode "Minimum": FDT_NMS_MINIMUM
 *   MTCNN/mtcnn/core/nms.py:4-40 torch_nms            FDT_NMS_PLUS1 | FDT_NMS_LE | (FDT_NMS_SUMFIRST or FDT_NMS_MINIMUM)
 *   FACEBOX/encoderl.py:268-306 DataEncoder.nms       FDT_NMS_SUMFIRST | FDT_NMS_LE
 * keep[n] int64 zero padded = indices in keep order (descending score; ties: higher index first), *count device int64.
 * Workspace fdt_nms_workspace_bytes(n) (n > FDT_MAX_NMS_TOP_K takes the mask formulation, as fdt_nms does).
 * fdt_nms_variant_f64: the same rules in float64 -- MTCNN's `nms` runs in the dtype of its float64 `dets`
 * (core/utils.py:62-113, callers core/detect.py:314, 326, 431, 579); workspace fdt_nms_f64_workspace_bytes(n), n <= 131,072.
 * fdt_facebox_decode: the box part of DataEncoder.decode_np (encoderl.py:318-320), corner form [x1,y1,x2,y2].
 * fdt_threshold_nms: rows p of a box table with conf[p,1] > conf_thresh (conf[N,2]) enter fdt_nms_variant's NMS without a
 * host round trip; keep[N] holds table indices.  More than FDT_MAX_NMS_TOP_K candidates: keep zeroed, *count = -1. */
int fdt_nms_variant(const float *boxes, const float *scores, int64_t n, float thresh, int variant,
                    int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream);
size_t fdt_nms_f64_workspace_bytes(int64_t n);
int fdt_nms_variant_f64(const double *boxes, const double *scores, int64_t n, double thresh, int variant,
                        int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_facebox_decode(const float *loc, const float *default_boxes, int64_t n, float var0, float var1, float *out,
                       fdt_stream_t stream);
size_t fdt_threshold_nms_workspace_bytes(int64_t N);
int fdt_threshold_nms(const float *boxes, const float *conf, int64_t N, float conf_thresh, float nms_thresh, int variant,
                      int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream);

/* ---- D3  Detect.__call__  (layers/functions/detection.py:34-84) ---------------------------------
 * loc[B,N,4], conf[B,N,C] (post-softmax), priors[N,4] -> out[B,C,top_k,5] rows [score,x1,y1,x2,y2]
 * in keep order, zero padded; class-0 plane zero.  Optional: counts[B,C] int32 rows written;
 * kept_prior[B,C,top_k] int64 prior index per row (-1 padding).  Candidates: score > conf_thresh
 * (strict); exactly one candidate yields no detection (reference quirk, detection.py:66-72).
 * Limit: nms_top_k <= FDT_MAX_NMS_TOP_K (FDT_E_UNSUPPORTED beyond).  See DESIGN.md. */
size_t fdt_detect_workspace_bytes(int B, int64_t N, int C);
int fdt_detect(const float *loc, const float *conf, const float *priors,
               int B, int64_t N, int C, int top_k, int nms_top_k,
               float conf_thresh, float nms_thresh, float var0, float var1,
               float *out, int32_t *counts, int64_t *kept_prior,
               void *ws, size_t ws_bytes, fdt_stream_t stream);
/* Mixed precision (what a model under torch.autocast, or one converted with .half() / .to(torch.bfloat16), hands over): loc and conf
 * each of element type loc_dtype / conf_dtype (FDT_DTYPE_F32 / _BF16 / _F16, defined below), read in place.  Every element is widened
 * to fp32 exactly and all arithmetic is what it is on fp32 inputs, so out / counts / kept_prior are bit-identical to fdt_detect on the
 * inputs converted to fp32.  The threshold is compared in fp32 against the widened score (score > conf_thresh), not rounded to the
 * input's type first.  Each pointer must be aligned to its element size, an fp32 loc to 16 bytes; an unknown dtype or a misaligned
 * pointer is FDT_E_INVALID before any CUDA call.  fdt_detect == fdt_detect_ex with two FDT_DTYPE_F32. */
int fdt_detect_ex(const void *loc, int loc_dtype, const void *conf, int conf_dtype, const float *priors,
                  int B, int64_t N, int C, int top_k, int nms_top_k,
                  float conf_thresh, float nms_thresh, float var0, float var1,
                  float *out, int32_t *counts, int64_t *kept_prior,
                  void *ws, size_t ws_bytes, fdt_stream_t stream);
/* Overlap of consecutive calls.  A workspace of fdt_detect_workspace_bytes_depth(B, N, C, depth) bytes, depth 2..4, holds `depth`
 * slots of per-call scratch: call s uses slot s % depth, so the threshold pass of call s + 1 runs while the NMS kernel of call s is
 * still in flight and its NMS CTAs take over SMs as those of call s retire (all on ONE stream, chained by programmatic dependent
 * launch; a control block at the head of the workspace keeps the calls' completion in order, so anything enqueued after a call
 * still finds it -- and every earlier call -- complete).  Rules: the inputs of a call must be complete when the call is
 * enqueued-in-stream-order as usual; a call that writes the same out / counts / kept_prior buffer as a call still in flight waits
 * for it (use `depth` rotating output buffers to overlap).  depth 1 (fdt_detect_workspace_bytes) runs calls one after another. */
size_t fdt_detect_workspace_bytes_depth(int B, int64_t N, int C, int depth);
/* FDT_STATUS_* bits of the workspace (0 = fine); synchronises `stream`. */
int fdt_detect_status(const void *ws, fdt_stream_t stream, uint32_t *status_h);
/* Process-wide tuning / diagnostic switches (defaults come from the environment variables FDT_K3_PROFILE, FDT_K3_CLUSTER,
 * FDT_K3_PDL, FDT_DETECT_DEPTH, FDT_DETECT_FUSED, read once): "k3_profile" 0/1/2, "k3_cluster" -1 auto / 0 / 1, "k3_pdl" 0/1,
 * "detect_depth" 1..4, "detect_fused" -1 auto / 0 / 1 (1: k_sort_nms thresholds its own conf rows, no separate threshold grid). */
int fdt_set_option(const char *name, int value);

/* Stage entry points (same workspace, same semantics; fdt_detect == stage 1 then stage 2).  They let
 * tests and bench.py check / time the two kernels separately (a stage-1 call never overlaps an earlier call):
 *   stage 1  K2 threshold + compaction: conf -> per-(image,class) candidate keys + counts in `ws`
 *   stage 2  K3 select/sort + decode + NMS + output rows, consuming `ws` */
int fdt_detect_threshold_compact(const float *conf, int B, int64_t N, int C, float conf_thresh,
                                 void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_detect_sort_nms(const float *loc, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                        float nms_thresh, float var0, float var1,
                        float *out, int32_t *counts, int64_t *kept_prior,
                        void *ws, size_t ws_bytes, fdt_stream_t stream);
/* Number of candidates per (image, class>=1) list after stage 1: copies B*(C-1) int32 to counts_out (device). */
int fdt_detect_candidate_counts(const void *ws, size_t ws_bytes, int B, int64_t N, int C, int32_t *counts_out, fdt_stream_t stream);

/* Detect with the multi-GPU gather fused in (SURVEY 8e): instead of a local `out`, the detection rows of this rank's B images are
 * stored straight into the gathered block [world*B, C, top_k, 5] of n_peers destination ranks at image index image_offset + b, over
 * NVLink peer memory (16-byte vector stores, no separate collective).  peer_out_ptrs: DEVICE array of n_peers base pointers of those
 * blocks (e.g. torch symmetric memory `buffer_ptrs_dev`); the caller synchronises the ranks afterwards (a symmetric-memory
 * barrier).  The background (class 0) planes of the gathered blocks are NOT written: the caller zeroes the blocks once after
 * allocating them and they stay zero (half of the NVLink traffic of a two-class Detect). */
int fdt_detect_peers(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                     float conf_thresh, float nms_thresh, float var0, float var1,
                     const uint64_t *peer_out_ptrs, int n_peers, int64_t image_offset,
                     void *ws, size_t ws_bytes, fdt_stream_t stream);
/* The same with the completion signalling folded in (no barrier launch, nobody spins inside the NMS kernel).
 *   dest_out_ptrs     DEVICE array of n_dest block pointers: root >= 0: n_dest = 1, the root's block; root = -1: n_dest = world,
 *                     every rank's block in rank order (all-gather).  `ring` blocks alternate between calls (the caller passes
 *                     the pointer table of block epoch % ring).
 *   peer_signal_ptrs  DEVICE array of `world` pointers to every rank's uint32 signal[2 * world] array (symmetric memory, zeroed
 *                     once): [q] = last epoch whose rows from rank q have landed here, [world + q] = last call rank q has begun.
 *   epoch             call counter (>= 1), the same on every rank, increasing by one per call.
 * A source rank waits (before storing, normally long satisfied) until every destination has begun call epoch - ring + 1 -- in the
 * destination's stream that follows whatever consumed call epoch - ring, so the block is free --, stores its rows, and its last
 * CTA publishes `epoch` to the destinations (a destination to itself as well).  A destination rank additionally enqueues
 * fdt_detect_gather_await (done here), a one-block kernel that ends when all ranks have published `epoch`: what consumes the gathered block follows it in stream
 * order, while the next call is NOT held back by it.  Every rank must make the call for the destinations' streams to advance; a
 * wait that sees no progress for ~4 s gives up, sets FDT_STATUS_TIMEOUT_PEER (fdt_detect_status) and the rank stops signalling.
 * `epoch` is a launch parameter: do not replay this call from a captured CUDA graph. */
int fdt_detect_gather_signal(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                             float conf_thresh, float nms_thresh, float var0, float var1,
                             const uint64_t *dest_out_ptrs, int n_dest, const uint64_t *peer_signal_ptrs,
                             int world, int rank, int root, uint32_t epoch, int ring, int64_t image_offset,
                             void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_detect_gather_await(const uint64_t *peer_signal_ptrs, int world, int rank, uint32_t epoch, void *ws, fdt_stream_t stream);
/* The same call WITHOUT the await kernel: the destination enqueues fdt_detect_gather_await itself, on any stream -- the kernel depends
 * on nothing but the signal array (a destination's own k_sort_nms publishes `epoch` in its own slot like every source), so it needs
 * no stream order behind the call.  On a stream of its own it is not a third grid per call in the calls' stream: the destination's
 * step is 17.4 instead of 18.6 us at B = 64 (tools/peer_breakdown.py); consumers then wait for that stream (an event). */
int fdt_detect_gather_store(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                            float conf_thresh, float nms_thresh, float var0, float var1,
                            const uint64_t *dest_out_ptrs, int n_dest, const uint64_t *peer_signal_ptrs,
                            int world, int rank, int root, uint32_t epoch, int ring, int64_t image_offset,
                            void *ws, size_t ws_bytes, fdt_stream_t stream);

/* ---- (SURVEY 8f rank 1) head post-processing that feeds Detect  (pyramid.py:291-309, 331-338; same code in
 * pyramid_mobile_try1.py:297-327, pyramid_mb2_try3/4/5.py) -------------------------------------------------------------
 * The models produce, per pyramid level l, NCHW maps loc_l[B,4,H_l,W_l] and the 4-channel max-in-out confidence
 * conf_l[B,4,H_l,W_l].  The reference reduces the confidence to (neg, pos) with chunk/max/cat -- neg = max(ch0..2),
 * pos = ch3 where neg_max_h[l] != 0 (level 0, pyramid.py:293-297), else neg = ch0, pos = max(ch1..3) (:299-304; torch.max
 * propagates NaN) --, permutes both to NHWC, concatenates the levels into loc[B,N,4] / conf[B,N,2] (N = sum H_l*W_l, y
 * outer, x inner) and applies nn.Softmax(dim=-1) in the test phase (:331-332).
 *   loc_maps_h / conf_maps_h : HOST arrays of n_levels DEVICE pointers; f_h / f_w / neg_max_h : HOST int arrays.
 * fdt_heads_to_loc_conf materialises the reference's tensors (either output may be null; softmax != 0 applies the
 * softmax, the training path keeps raw logits).  fdt_detect_heads == fdt_heads_to_loc_conf(softmax) + fdt_detect with
 * nothing materialised: the threshold kernel reads the conf maps (max-in-out + softmax fused), NMS gathers the loc rows
 * it decodes from the loc maps.  Softmax: exp(x - max) in fp64 rounded once, fp32 sum and IEEE division.
 * Workspace of fdt_detect_heads: fdt_detect_workspace_bytes(B, N, 2).  Limit: n_levels <= 8.
 *
 * Mixed precision and channels_last: the `_ex` entries take each map as a descriptor -- element (b, ch, y, x) of a level is
 * data[b * batch_stride + ch * channel_stride + (y * W + x) * pixel_stride], strides in elements, all > 0 -- and one element type
 * for every map of the call (FDT_DTYPE_*).  Dense NCHW is (4*H*W, H*W, 1), dense channels_last (NHWC in memory) (4*H*W, 1, 4).
 * The kernels read the maps in place and widen each element to fp32 (exact), so every output is bit-identical to the entry without
 * `_ex` on the maps converted to fp32 NCHW.  Where a prior's four channels are adjacent and their address is a multiple of four
 * elements, they are read with one vector load.  Gradient maps (fdt_head_grad_map) have the maps' element type and their own strides;
 * a gradient is computed in fp32 as for fp32 maps and rounded to the element type (round to nearest even, overflow to +-inf).
 * An unknown dtype, a null `data` of a map the call reads or writes, a stride <= 0 or a `data` not aligned to the element size is
 * FDT_E_INVALID, checked before any CUDA call.  The entries without `_ex` are these with fp32 dense-NCHW descriptors. */
#define FDT_DTYPE_F32  0
#define FDT_DTYPE_BF16 1
#define FDT_DTYPE_F16  2
typedef struct { const void *data; int64_t batch_stride, channel_stride, pixel_stride; } fdt_head_map;
typedef struct { void *data; int64_t batch_stride, channel_stride, pixel_stride; } fdt_head_grad_map;
int fdt_heads_to_loc_conf(const float *const *loc_maps_h, const float *const *conf_maps_h,
                          const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, int B, int softmax,
                          float *loc_out, float *conf_out, fdt_stream_t stream);
int fdt_detect_heads(const float *const *loc_maps_h, const float *const *conf_maps_h,
                     const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, const float *priors,
                     int B, int top_k, int nms_top_k, float conf_thresh, float nms_thresh, float var0, float var1,
                     float *out, int32_t *counts, int64_t *kept_prior, void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_heads_to_loc_conf_ex(const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype,
                             const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, int B, int softmax,
                             float *loc_out, float *conf_out, fdt_stream_t stream);
int fdt_detect_heads_ex(const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype,
                        const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, const float *priors,
                        int B, int top_k, int nms_top_k, float conf_thresh, float nms_thresh, float var0, float var1,
                        float *out, int32_t *counts, int64_t *kept_prior, void *ws, size_t ws_bytes, fdt_stream_t stream);

/* Diagnostics (FDT_K3_PROFILE=1): per-phase clock64 deltas of CTA 0 of the last fdt_detect_sort_nms / fdt_nms launch. */
int fdt_debug_k3_profile(long long *out1024_h);  /* [0..31] phases of CTA 0, [64..319] cycles per CTA, [320..575] rounds*1e5 + k per CTA, [640..767] phase-B per warp */

/* ---- host-buffer variants (the reference-facing call when tensors live on the CPU) --------------
 * All pointers are HOST pointers.  The context owns two streams (copies / kernels), device staging slots and the resident prior
 * set; one context per host thread.  A call is cut into chunks of `host_chunk` images (fdt_set_option, default 16) whose conf
 * copies overlap the kernels of the chunk before; pinned `loc_h` is gathered in place over PCIe (never copied), pinned `out_h` is
 * written in place by the kernel.
 *   fdt_detect_host         submit + wait (returns after the results landed in out_h / counts_h / kept_prior_h)
 *   fdt_detect_host_submit  enqueues the call and returns a ticket; the host buffers must stay untouched until the wait.  Any
 *                           number of calls may be in flight; they complete in submission order.  With pageable buffers the
 *                           copies, hence the submit, block.
 *   fdt_detect_host_wait    blocks until the call of `ticket` (and every earlier one) has completed
 *   fdt_ctx_set_priors      uploads a prior set [N,4]; calls that pass priors_h == NULL use the set uploaded last (by this
 *                           function or by a call that passed priors_h), so a constant set crosses the link once */
int fdt_ctx_create(int device, fdt_ctx **ctx);
int fdt_ctx_destroy(fdt_ctx *ctx);
int fdt_ctx_set_priors(fdt_ctx *ctx, const float *priors_h, int64_t N);
int fdt_detect_host(fdt_ctx *ctx, const float *loc_h, const float *conf_h, const float *priors_h,
                    int B, int64_t N, int C, int top_k, int nms_top_k,
                    float conf_thresh, float nms_thresh, float var0, float var1,
                    float *out_h, int32_t *counts_h, int64_t *kept_prior_h);
int fdt_detect_host_submit(fdt_ctx *ctx, const float *loc_h, const float *conf_h, const float *priors_h,
                           int B, int64_t N, int C, int top_k, int nms_top_k,
                           float conf_thresh, float nms_thresh, float var0, float var1,
                           float *out_h, int32_t *counts_h, int64_t *kept_prior_h, uint64_t *ticket);
int fdt_detect_host_wait(fdt_ctx *ctx, uint64_t ticket);
/* the same on bf16 / fp16 / fp32 host tensors (as fdt_detect_ex): conf chunks cross the link at their own element size, a pinned loc_h
 * is gathered in place (8-byte aligned 16-bit rows, 16-byte fp32 rows), any other is copied at its own size.  Host buffers need only be
 * aligned to their elements.  One context serves every
 * dtype.  fdt_detect_host / _submit == these with two FDT_DTYPE_F32. */
int fdt_detect_host_ex(fdt_ctx *ctx, const void *loc_h, int loc_dtype, const void *conf_h, int conf_dtype, const float *priors_h,
                       int B, int64_t N, int C, int top_k, int nms_top_k,
                       float conf_thresh, float nms_thresh, float var0, float var1,
                       float *out_h, int32_t *counts_h, int64_t *kept_prior_h);
int fdt_detect_host_submit_ex(fdt_ctx *ctx, const void *loc_h, int loc_dtype, const void *conf_h, int conf_dtype, const float *priors_h,
                              int B, int64_t N, int C, int top_k, int nms_top_k,
                              float conf_thresh, float nms_thresh, float var0, float var1,
                              float *out_h, int32_t *counts_h, int64_t *kept_prior_h, uint64_t *ticket);

/* ---- M4/M5  match_default / match_ensure_max_prior (layers/box_utils.py:165-210, 103-162) -------
 * Batched over images: gt[total_gt,5] rows [x1,y1,x2,y2,label], gt_off[B+1] int64 (device).
 * -> loc_t[B,N,4], conf_t[B,N] int64; optional best_truth_idx[B,N] int32, best_truth_overlap[B,N].
 * Images with zero GT (the reference raises) are defined as all-background, loc_t = 0. */
size_t fdt_match_workspace_bytes(int B, int64_t N, int64_t total_gt);
int fdt_match_encode(const float *priors, const float *gt, const int64_t *gt_off, int64_t total_gt, int B, int64_t N,
                     float threshold, float var0, float var1, int bipartite,
                     float *loc_t, int64_t *conf_t, int32_t *best_truth_idx, float *best_truth_overlap,
                     void *ws, size_t ws_bytes, fdt_stream_t stream);

/* ---- L2  hard-negative mining  (layers/modules/multibox_loss.py:112-116) -------------------------
 * loss_c[B,N] (zero at positives), pos[B,N] uint8 -> neg[B,N] uint8 = rank < min(ratio*num_pos, N-1).
 * Ties at the boundary: lower prior index first (stable descending). */
size_t fdt_mine_workspace_bytes(int B, int64_t N);
int fdt_hard_negative_mine(const float *loss_c, const uint8_t *pos, int B, int64_t N, int negpos_ratio,
                           uint8_t *neg, void *ws, size_t ws_bytes, fdt_stream_t stream);

/* ---- L2  MultiBoxLoss.forward / backward  (layers/modules/multibox_loss.py:48-136) ---------------
 * forward: match+encode, smooth-L1 over positives, per-prior CE, mining, CE over pos U neg.
 * losses[2] (device) = {loss_l/N, loss_c/N}; norm[1] (device) = N.  loc_t/conf_t/sel are outputs the
 * backward pass reuses (sel[B,N] uint8 = pos | neg).  loc_t holds the encoded target at the POSITIVE priors
 * (conf_t > 0) and zeros elsewhere: the reference encodes every prior (box_utils.py:208) but its loss only reads
 * the positives (multibox_loss.py:96-101) and never returns the tensor; fdt_match_encode fills all rows.
 * The forward is three kernels on `stream` (prepare -> match + loss terms -> mining + selection + final division) with no memset
 * node; the workspace content does not matter before a call and is re-initialised by every call.  Limits: B <= 65535,
 * N <= 65535 * 256; conf needs 8-byte alignment when C == 2.  loss_c_all (optional, [B,N]) receives the mining input
 * log_sum_exp(conf) - conf[label] with zeros at the positives (multibox_loss.py:104-110).
 * backward: grad_loc[B,N,4], grad_conf[B,N,C] for upstream gradients g_l, g_c (host scalars). */
size_t fdt_multibox_workspace_bytes(int B, int64_t N, int C, int64_t total_gt);
int fdt_multibox_loss_forward(const float *loc, const float *conf, const float *priors,
                              const float *gt, const int64_t *gt_off, int64_t total_gt, int B, int64_t N, int C,
                              float threshold, int negpos_ratio, int bipartite, float var0, float var1,
                              float *losses, float *norm, float *loc_t, int64_t *conf_t, uint8_t *sel,
                              float *loss_c_all, void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_multibox_loss_backward(const float *loc, const float *conf, const float *loc_t, const int64_t *conf_t,
                               const uint8_t *sel, const float *norm, float g_l, float g_c,
                               int B, int64_t N, int C, float *grad_loc, float *grad_conf, fdt_stream_t stream);
/* the same with the upstream gradients as DEVICE scalars (what autograd hands over): no host synchronisation, graph capturable */
int fdt_multibox_loss_backward_dev(const float *loc, const float *conf, const float *loc_t, const int64_t *conf_t,
                                   const uint8_t *sel, const float *norm, const float *g_l_dev, const float *g_c_dev,
                                   int B, int64_t N, int C, float *grad_loc, float *grad_conf, fdt_stream_t stream);
/* Mixed precision: loc / conf of element types loc_dtype / conf_dtype (FDT_DTYPE_*), read in place, each pointer aligned to its element
 * size (an fp32 loc to 16 bytes; the forward's fp32 conf with C == 2 to 8, as before); the outputs are bit-identical to the entries above on the inputs
 * converted to fp32.  grad_loc / grad_conf have the element types of loc / conf: the fp32 gradients rounded to nearest even.  An
 * unknown dtype or a misaligned pointer is FDT_E_INVALID before any CUDA call.  The entries above are these with FDT_DTYPE_F32. */
int fdt_multibox_loss_forward_ex(const void *loc, int loc_dtype, const void *conf, int conf_dtype, const float *priors,
                                 const float *gt, const int64_t *gt_off, int64_t total_gt, int B, int64_t N, int C,
                                 float threshold, int negpos_ratio, int bipartite, float var0, float var1,
                                 float *losses, float *norm, float *loc_t, int64_t *conf_t, uint8_t *sel,
                                 float *loss_c_all, void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_multibox_loss_backward_dev_ex(const void *loc, int loc_dtype, const void *conf, int conf_dtype, const float *loc_t,
                                      const int64_t *conf_t, const uint8_t *sel, const float *norm, const float *g_l_dev,
                                      const float *g_c_dev, int B, int64_t N, int C, void *grad_loc, void *grad_conf, fdt_stream_t stream);

/* ---- training from head maps (SURVEY 8f rank 1; replaces pyramid.py:291-309 + MyTrain_repo.py:170-171 and their autograd backward)
 * Map arguments as fdt_heads_to_loc_conf (HOST arrays of n_levels DEVICE pointers, NCHW [B,4,H_l,W_l]; the `_ex` entries: HOST arrays
 * of descriptors, any element type and layout fdt_heads_to_loc_conf_ex accepts); N = sum H_l*W_l, C = 2.
 * Gradient maps have the maps' layout.  The gradient of a max-reduced logit goes to the channel torch's max(dim) backward picks: the
 * first NaN of the three channels if there is one, else the lowest channel equal to their maximum (-0.0 == +0.0); the other two
 * channels of the three receive +0.0.
 * fdt_heads_to_loc_conf_backward: the backward of fdt_heads_to_loc_conf.  grad_loc[B,N,4] / grad_conf[B,N,2] may each be null, and
 *   then the matching map gradients are not written (nor read: their array may be null); otherwise every element of them is written.
 *   softmax != 0 applies the 2-way softmax's backward y * (g - (g0*y0 + g1*y1)) first, y recomputed from conf_maps_h.
 * fdt_multibox_loss_forward_heads == fdt_heads_to_loc_conf(softmax = 0) + fdt_multibox_loss_forward(C = 2), with the same outputs
 *   and nothing materialised: the kernels read the maps.  priors[N,4]; workspace fdt_multibox_workspace_bytes(B, N, 2, total_gt).
 * fdt_multibox_loss_backward_heads_dev == fdt_multibox_loss_backward_dev + fdt_heads_to_loc_conf_backward(softmax = 0), bit-identical,
 *   writing the map gradients directly (either gradient array may be null: not written).  Device scalars, graph capturable. */
int fdt_heads_to_loc_conf_backward(const float *const *conf_maps_h, const int *f_h, const int *f_w, const int *neg_max_h,
                                   int n_levels, int B, int softmax, const float *grad_loc, const float *grad_conf,
                                   float *const *grad_loc_maps_h, float *const *grad_conf_maps_h, fdt_stream_t stream);
int fdt_multibox_loss_forward_heads(const float *const *loc_maps_h, const float *const *conf_maps_h, const int *f_h, const int *f_w,
                                    const int *neg_max_h, int n_levels, const float *priors, const float *gt, const int64_t *gt_off,
                                    int64_t total_gt, int B, float threshold, int negpos_ratio, int bipartite, float var0, float var1,
                                    float *losses, float *norm, float *loc_t, int64_t *conf_t, uint8_t *sel, float *loss_c_all,
                                    void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_multibox_loss_backward_heads_dev(const float *const *loc_maps_h, const float *const *conf_maps_h, const int *f_h,
                                         const int *f_w, const int *neg_max_h, int n_levels, const float *loc_t,
                                         const int64_t *conf_t, const uint8_t *sel, const float *norm, const float *g_l_dev,
                                         const float *g_c_dev, int B, float *const *grad_loc_maps_h,
                                         float *const *grad_conf_maps_h, fdt_stream_t stream);
/* the same on map descriptors (see fdt_heads_to_loc_conf_ex) */
int fdt_heads_to_loc_conf_backward_ex(const fdt_head_map *conf_maps_h, int dtype, const int *f_h, const int *f_w, const int *neg_max_h,
                                      int n_levels, int B, int softmax, const float *grad_loc, const float *grad_conf,
                                      const fdt_head_grad_map *grad_loc_maps_h, const fdt_head_grad_map *grad_conf_maps_h,
                                      fdt_stream_t stream);
int fdt_multibox_loss_forward_heads_ex(const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype, const int *f_h,
                                       const int *f_w, const int *neg_max_h, int n_levels, const float *priors, const float *gt,
                                       const int64_t *gt_off, int64_t total_gt, int B, float threshold, int negpos_ratio, int bipartite,
                                       float var0, float var1, float *losses, float *norm, float *loc_t, int64_t *conf_t, uint8_t *sel,
                                       float *loss_c_all, void *ws, size_t ws_bytes, fdt_stream_t stream);
int fdt_multibox_loss_backward_heads_dev_ex(const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype, const int *f_h,
                                            const int *f_w, const int *neg_max_h, int n_levels, const float *loc_t,
                                            const int64_t *conf_t, const uint8_t *sel, const float *norm, const float *g_l_dev,
                                            const float *g_c_dev, int B, const fdt_head_grad_map *grad_loc_maps_h,
                                            const fdt_head_grad_map *grad_conf_maps_h, fdt_stream_t stream);

/* ---- T2  IoU tracker association  (iouTracke_cal.py:126-155 loop, :174-176 flush) ----------------
 * dets[total,5] float64 rows [x1,y1,x2,y2,score]; frame_off[F+1] int64 (device); frames are 1-based in
 * the output.  Outputs (device): n_tracks[1] int64; track_off[total+1] int64 CSR offsets into
 * track_dets[total] int64 (global det rows in append order); track_start[total] int64;
 * track_max[total] float64 -- entries [0, n_tracks) are valid, in the reference's finishing order.
 * max_dets_per_frame must be at least every frame's row count; at most 864 rows per frame (the frame state of
 * cap = 32 * ceil(max_dets_per_frame / 32) rows lives in shared memory), more return FDT_E_UNSUPPORTED before any CUDA call and
 * fdt_iou_track_workspace_bytes returns 0 for them. */
#define FDT_TRACK_IOU       0   /* use_iou = True:  calculate_iou, argmax, matched iff > sigma_iou   (iouTracke_cal.py:131-134) */
#define FDT_TRACK_DISTANCE  1   /* use_iou = False: calculate_distance, argmin, matched iff < sigma_dis (iouTracke_cal.py:135-138) */
size_t fdt_iou_track_workspace_bytes(int64_t F, int64_t total, int64_t max_dets_per_frame);
int fdt_iou_track(const double *dets, const int64_t *frame_off, int64_t F, int64_t total, int64_t max_dets_per_frame,
                  double sigma_iou, double sigma_h, int64_t t_min,
                  int64_t *n_tracks, int64_t *track_off, int64_t *track_dets, int64_t *track_start, double *track_max,
                  void *ws, size_t ws_bytes, fdt_stream_t stream);
/* the same with the association rule of the reference's `use_iou` switch: metric FDT_TRACK_IOU (sigma = sigma_iou) or
 * FDT_TRACK_DISTANCE (sigma = sigma_dis; utils/calc_performance.py:34-51, `** 0.25` correctly rounded). */
int fdt_iou_track_metric(const double *dets, const int64_t *frame_off, int64_t F, int64_t total, int64_t max_dets_per_frame,
                         int metric, double sigma, double sigma_h, int64_t t_min,
                         int64_t *n_tracks, int64_t *track_off, int64_t *track_dets, int64_t *track_start, double *track_max,
                         void *ws, size_t ws_bytes, fdt_stream_t stream);

/* ---- T2  online multi-stream tracker: each step advances V independent videos by one frame (iouTracke_cal.py:117-155
 * inside the video loop), with every stream's active tracks kept on the device in a caller-owned `state` buffer (256-byte
 * aligned).  No call synchronises with the host, so a Detect -> step chain can be captured in a CUDA graph.  For every stream,
 * its steps followed by its flush give exactly fdt_iou_track_metric on that stream's frames.
 *   cap = 32 * ceil(max_dets_per_frame / 32) (max_dets_per_frame <= 864, as offline; the size queries
 *   return 0 above it).  Every call repeats V and
 *   max_dets_per_frame; a call whose values differ from the state's sets FDT_STATUS_TRACK_MISMATCH and changes nothing.
 *   Track ids are stream-local, in creation order from 0 (new tracks of a frame in detection order), below 2^31.
 *   Finish records, [V, cap] each, entries [0, fin_count[v]) valid, in the reference's finishing order: fin_index = the
 *   track's index in tracks_finished (the offline "track ID"), fin_track = its id, fin_start (1-based frame), fin_len, fin_max. */
#define FDT_STATUS_TRACK_OVERFLOW 4u   /* a stream's frame had more than cap rows: that frame was skipped (state unchanged, ids -1) */
#define FDT_STATUS_TRACK_MISMATCH 8u   /* a call's V / max_dets_per_frame differ from the state's (or it was never initialised) */
size_t fdt_track_stream_state_bytes(int64_t V, int64_t max_dets_per_frame);
size_t fdt_track_stream_workspace_bytes(int64_t V, int64_t max_dets_per_frame);      /* candidate rows of one step */
/* metric / sigma as fdt_iou_track_metric; every stream starts a new video */
int fdt_track_stream_init(void *state, size_t state_bytes, int64_t V, int64_t max_dets_per_frame,
                          int metric, double sigma, double sigma_h, int64_t t_min, fdt_stream_t stream);
/* One frame per stream: dets = packed float64 rows, frame_off[V+1] (device; what fdt_detections_to_frames_count/_pack write for a
 * [V,C,top_k,5] Detect output).  advance[V] (NULL = all): 0 = the stream has no frame this call, its state is untouched -- not the
 * same as an empty frame (D = 0: every active track is silently dropped).  row_track[frame_off[V]] = the id of the track each row
 * joined or started (-1 for the rows of a stream that was not advanced or whose frame was over capacity). */
int fdt_track_stream_step(void *state, int64_t V, int64_t max_dets_per_frame, const double *dets, const int64_t *frame_off,
                          const uint8_t *advance, int64_t *row_track, int32_t *fin_count, int64_t *fin_index,
                          int64_t *fin_track, int64_t *fin_start, int64_t *fin_len, double *fin_max,
                          void *ws, size_t ws_bytes, fdt_stream_t stream);
/* end of video (iouTracke_cal.py:174-176: len >= t_min) for the streams with streams[v] != 0 (NULL = all), the same records
 * (fin_count[v] = 0 elsewhere); those slots then start a new video */
int fdt_track_stream_flush(void *state, int64_t V, int64_t max_dets_per_frame, const uint8_t *streams, int32_t *fin_count,
                           int64_t *fin_index, int64_t *fin_track, int64_t *fin_start, int64_t *fin_len, double *fin_max,
                           fdt_stream_t stream);
/* sticky FDT_STATUS_TRACK_* bits of the state (0 = fine); synchronises `stream`. */
int fdt_track_stream_status(const void *state, fdt_stream_t stream, uint32_t *status_h);

#ifdef __cplusplus
}
#endif
#endif /* FDT_B200_H */
