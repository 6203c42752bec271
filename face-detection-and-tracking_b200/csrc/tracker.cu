// IoU tracker association (iouTracke_cal.py:126-155 per-frame loop, :174-176 flush) for sm_100a, float64.
//
// Every active track's last box is a detection of the previous frame (a track that is not extended in a
// frame is finished or dropped at once), so the active list after frame f is a permutation of frame f's
// detections.  That splits the problem:
//
//   k_track_mask     all frame pairs in parallel, one warp per previous-frame detection: float64 IoU
//                    (utils/calc_performance.py:54-74 operand order) against every detection of the next
//                    frame -> bit rows "IoU > sigma_iou" (+ a per-row NaN flag).  This is the O(sum D^2)
//                    part and it is embarrassingly parallel.
//   k_track_resolve  one CTA walks the frames in order (the greedy chain is inherently serial across
//                    frames).  Inside a frame the reference's "for track in tracks_active: take the best
//                    remaining detection" is a serial dictatorship in track order; it is evaluated as a
//                    parallel deferred-acceptance fixed point (each track proposes to its best not-yet-
//                    refused candidate, a detection keeps the lowest-order proposer), which reaches exactly
//                    the sequential result.  Frames that contain a NaN IoU (0/0: zero-area boxes such as the
//                    reference's dummy detection [0,0,0,0,0.4], :73-74) take an exact warp-sequential path
//                    that mirrors numpy's argmax-picks-first-NaN behaviour.
//   k_track_scatter  detections -> CSR track_dets via (head, position) recorded during resolve.
//
// Online (fdt_track_stream_*): the state k_track_resolve carries from one frame to the next lives per stream in a caller-owned
// buffer; a step is k_track_mask<StreamRows> (one warp per stream and active track) + k_track_step (one CTA per stream), which
// runs the same per-frame body (track_frame) and flush (track_flush) as k_track_resolve.
#include <cstdlib>
#include <climits>
#include "fdt_common.cuh"

namespace {

constexpr int TR_THREADS = 1024;
constexpr int OFF_CHUNK = 512;

__device__ __forceinline__ double dmin_nan(double a, double b) { return (a != a || b != b) ? (double)NAN : (a < b ? a : b); }
__device__ __forceinline__ double dmax_nan(double a, double b) { return (a != a || b != b) ? (double)NAN : (a > b ? a : b); }

// calc_performance.py:20-31, 65-74 with box_a = detection, box_b = the track's last box
__device__ __forceinline__ double iou_f64(const double *a, const double *b)
{
    double w = dmin_nan(a[2], b[2]) - dmax_nan(a[0], b[0]);
    double h = dmin_nan(a[3], b[3]) - dmax_nan(a[1], b[1]);
    w = dmax_nan(w, 0.0); h = dmax_nan(h, 0.0);
    double inter = w * h;
    double area_a = (a[2] - a[0]) * (a[3] - a[1]);
    double area_b = (b[2] - b[0]) * (b[3] - b[1]);
    double uni = area_a + area_b - inter;
    return inter / uni;
}

// utils/calc_performance.py:34-51 calculate_distance(box_a = detection, box_b = the track's last box): numpy operand order, no FMA,
// `dis ** 0.25` correctly rounded (fdt_qroot_cr), so ties and `< sigma_dis` at equality are decided like the reference.  Not inlined:
// inlined into track_frame's re-rank and sequential path it made k_track_resolve and k_track_step spill.
__device__ __noinline__ double distance_f64(const double *a, const double *b)
{
    const double adx = a[2] - a[0], ady = a[3] - a[1], bdx = b[2] - b[0], bdy = b[3] - b[1];
    const double cax = (a[2] + a[0]) / 2, cay = (a[3] + a[1]) / 2, cbx = (b[2] + b[0]) / 2, cby = (b[3] + b[1]) / 2;
    const double dx = cbx - cax, dy = cby - cay;
    const double dz = ((adx - bdx) + (ady - bdy)) / 2;
    const double dis = __dadd_rn(__dadd_rn(__dmul_rn(dz, dz), __dmul_rn(dx, dx)), __dmul_rn(dy, dy));
    return fdt_qroot_cr(dis);
}
// association value, larger = better: the IoU (iouTracke_cal.py:131-134, matched iff > sigma_iou) or minus the distance
// (:135-138: argmin, matched iff < sigma_dis  <=>  -distance > -sigma_dis).  First index on ties and first NaN wins either way.
__device__ __forceinline__ double track_value(const double *a, const double *b, const int metric)
{
    return metric == 0 ? iou_f64(a, b) : -distance_f64(a, b);
}

__global__ void k_track_frame_of(const int64_t *__restrict__ frame_off, int64_t F, int32_t *__restrict__ frame_of)
{
    int64_t f = blockIdx.x;
    for (int64_t g = frame_off[f] + threadIdx.x; g < frame_off[f + 1]; g += blockDim.x) frame_of[g] = (int32_t)f;
}

// Row layout (uint32 words) per previous-frame detection: [0, W) bits "IoU > sigma_iou" over the next frame's detections,
// [W] NaN flag, [W+1], [W+2] the 4 best candidates as uint16 (best first: IoU descending, lower index first on ties = numpy's
// argmax order; 0xffff = none), [W+3] number of candidates.  The ranking is done here, for all frame pairs in parallel, so the
// serial resolve kernel normally never evaluates an IoU.
constexpr int ROW_EXTRA = 4;

// dynamic shared memory of k_track_resolve (and of k_track_step: prefetch = 0) for cap = 32 * W rows per frame
constexpr size_t resolve_smem(int W, int prefetch)
{
    const size_t cap = (size_t)W * 32;
    size_t s = ((prefetch ? 2 : 1) * cap * (W + ROW_EXTRA) * 4 + 15) / 16 * 16;
    s += sizeof(double) * ((prefetch ? 3 : 2) * cap * 5 + 2 * cap);
    s += sizeof(int32_t) * 10 * cap;
    return s;
}
constexpr size_t TR_SMEM_LIMIT = (size_t)FDT_SMEM_MAX - 1024;
constexpr int tr_max_w()
{
    int W = 1;
    while (resolve_smem(W + 1, 0) <= TR_SMEM_LIMIT) ++W;
    return W;
}
// The one limit on rows per frame, offline and online: the largest cap whose frame state fits in shared memory (W = 27:
// 224,640 B).  Frames of up to 608 rows (W = 19) also fit the prefetch layout.
constexpr int TR_MAX_D = 32 * tr_max_w();
static_assert(TR_MAX_D == 864 && TR_MAX_D <= TR_THREADS, "one thread per track / detection");

// Where row g of k_track_mask takes its track box and its candidate frame from: row() returns false for a warp without a row,
// otherwise it loads tb (the track's last box) and sets n0, D (the candidate rows dets[n0 .. n0 + D)); it may replace the rule.
// The row's WR words are mask[g * WR ..].
struct OfflineRows {           // row g = detection g of frame f (f < F-1) against frame f+1
    __device__ __forceinline__ bool row(int64_t g, const double *__restrict__ dets, const int64_t *__restrict__ frame_off,
                                        const int32_t *__restrict__ frame_of, int64_t F, int64_t total, double (&tb)[4],
                                        int64_t &n0, int &D, int &, double &) const
    {
        if (g >= total) return false;
        const int64_t f = frame_of[g];
        if (f + 1 >= F) return false;
        n0 = frame_off[f + 1];
        D = (int)(frame_off[f + 2] - n0);
#pragma unroll
        for (int k = 0; k < 4; ++k) tb[k] = dets[5 * g + k];
        return true;
    }
};
struct StreamRows;             // row v * cap + i = active track of stream v whose last box is row i of its previous frame (below)

// one warp per row (see the sources)
template <class Src>
__global__ void __launch_bounds__(256)
k_track_mask(const double *__restrict__ dets, const int64_t *__restrict__ frame_off, const int32_t *__restrict__ frame_of,
             int64_t F, int64_t total, int W, int metric, double sigma_iou, uint32_t *__restrict__ mask, const Src src)
{
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    double tb[4];
    int64_t n0;
    int D;
    if (!src.row(g, dets, frame_off, frame_of, F, total, tb, n0, D, metric, sigma_iou)) return;
    const int WR = W + ROW_EXTRA;
    bool any_nan = false;
    int count = 0;
    double cv[4] = {0.0, 0.0, 0.0, 0.0};        // lane-local best candidates (IoU descending, index ascending)
    int cj[4] = {-1, -1, -1, -1};
    int nc = 0;
    for (int c = 0; c * 32 < D && c < W; ++c) {
        const int j = c * 32 + lane;
        bool over = false, isn = false;
        double v = 0.0;
        if (j < D) {
            double db[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) db[k] = dets[5 * (n0 + j) + k];
            v = track_value(db, tb, metric);
            over = v > sigma_iou;                                  // iouTracke_cal.py:134 / :138 (sigma_iou = -sigma_dis there)
            isn = v != v;
        }
        const unsigned bits = __ballot_sync(0xffffffffu, over);
        any_nan |= __any_sync(0xffffffffu, isn);
        count += __popc(bits);
        if (lane == 0) mask[g * WR + c] = bits;
        if (over) {
            int p = nc < 4 ? nc : 4;
#pragma unroll
            for (int q = 3; q >= 0; --q) if (q < nc && cv[q] < v) p = q;
#pragma unroll
            for (int q = 3; q >= 1; --q) if (q > p) { cv[q] = cv[q - 1]; cj[q] = cj[q - 1]; }
#pragma unroll
            for (int q = 0; q < 4; ++q) if (q == p) { cv[q] = v; cj[q] = j; }
            if (nc < 4) ++nc;
        }
    }
    // the warp's 4 best: four rounds of "every lane offers its head, the best one is taken"
    unsigned packed[2] = {0xffffffffu, 0xffffffffu};
    if (count > 0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            double bv = nc > 0 ? cv[0] : -INFINITY;                // nothing to offer (bj == INT_MAX decides)
            int bj = nc > 0 ? cj[0] : INT_MAX;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
                const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
                if (oj != INT_MAX && (bj == INT_MAX || ov > bv || (ov == bv && oj < bj))) { bv = ov; bj = oj; }
            }
            if (bj != INT_MAX) {
                if (nc > 0 && cj[0] == bj) {                       // this lane's head was taken: pop it
#pragma unroll
                    for (int q = 0; q < 3; ++q) { cv[q] = cv[q + 1]; cj[q] = cj[q + 1]; }
                    --nc;
                }
                packed[r >> 1] = (packed[r >> 1] & ~(0xffffu << (16 * (r & 1)))) | ((unsigned)bj << (16 * (r & 1)));
            }
        }
    }
    if (lane == 0) {
        mask[g * WR + W] = any_nan ? 1u : 0u;
        mask[g * WR + W + 1] = packed[0];
        mask[g * WR + W + 2] = packed[1];
        mask[g * WR + W + 3] = (unsigned)count;
    }
}

// exclusive scan of one int per thread over the block; returns (exclusive prefix, total)
__device__ __forceinline__ int block_excl_scan(int v, int *s_warp, int &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
    __syncthreads();
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0, winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += n; }
        s_warp[lane] = winc - w;
        if (lane == 31) s_warp[32] = winc;
    }
    __syncthreads();
    total = s_warp[32];
    return inc - v + s_warp[warp];
}

// exclusive scan of a 64-bit value per thread over the block (two packed counters); returns (exclusive prefix, total)
__device__ __forceinline__ long long block_excl_scan64(long long v, long long *s_warp64, long long &total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { long long n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
    __syncthreads();
    if (lane == 31) s_warp64[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        long long w = lane < (int)(blockDim.x >> 5) ? s_warp64[lane] : 0, winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { long long n = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += n; }
        s_warp64[lane] = winc - w;
        if (lane == 31) s_warp64[32] = winc;
    }
    __syncthreads();
    total = s_warp64[32];
    return inc - v + s_warp64[warp];
}

// the association rule (iouTracke_cal.py:22-28, :131-147); k_track_resolve passes its ResolveParams, which has the same fields
struct TrackRule {
    double sigma_iou, sigma_h; int64_t t_min;      // sigma_iou: threshold on the association value (-sigma_dis in distance mode)
    int metric;                                    // 0 IoU, 1 distance
    int force_slow;
};

// Shared-memory views of one frame step: the detections of frame f (box, and the per-detection track state written for them)
// and the tracks active before it (pbox .. pord: their last boxes and state, indexed by their detection of frame f-1).
struct FrameBufs {
    const double *box, *pbox;
    uint32_t *rows;                              // candidate row of each active track, indexed like pbox (see k_track_mask)
    double *maxs; const double *pmaxs;
    int32_t *head, *len, *start, *ord;
    const int32_t *phead, *plen, *pstart, *pord;  // pord[t] = detection of frame f-1 of the t-th active track
    int32_t *owner, *match;                      // [cap]: owner[] = INT_MAX and match[] = -1 on entry, synchronised
};

// One frame of iouTracke_cal.py:126-155 for the T active tracks against the D detections in B.box (D <= cap = blockDim.x).  The
// sink receives what the frame decides: finish(id, first_row, head, len, start, max) for a finished track (id = its index in
// tracks_finished, first_row = the number of rows finished before it), extend(j, head, pos) for detection j appended to a track,
// new_head(j, k) / begin(j, head) for detection j starting the k-th new track of the frame, created(n) once.  f = 0-based frame.
template <class Rule, class Sink>
__device__ __forceinline__ void track_frame(const FrameBufs &B, const Rule &R, const int D, const int64_t f, const int W,
                                            int &T, int64_t &n_fin, int64_t &fin_rows, Sink &out,
                                            int *s_warp, long long *s_warp64, int *s_slow)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W1 = W + ROW_EXTRA;
    const double *box = B.box, *pbox = B.pbox, *pmaxs = B.pmaxs;
    const int32_t *phead = B.phead, *plen = B.plen, *pstart = B.pstart, *pord = B.pord;
    int32_t *owner = B.owner, *match = B.match, *ord = B.ord;
    const int Wd = (D + 31) >> 5;
    const int my = tid < T ? pord[tid] : 0;                       // this thread's track = detection `my` of frame f-1
    uint32_t *row = B.rows + my * W1;
    const bool slow = __syncthreads_or((tid < T && row[W] != 0) || (R.force_slow && T > 0));

    int n_upd = 0;                 // tracks continued into this frame (uniform after the paths below)
    if (!slow) {
        // ---- deferred acceptance == serial dictatorship in track order (see header).  Each track ranks its
        //      candidates once (the 4 best are cached; more are re-ranked only if all 4 get refused).
        const double *tb = pbox + 5 * my;
        double cv[4] = {0.0, 0.0, 0.0, 0.0};
        int cj[4] = {-1, -1, -1, -1};
        int nc = 0;
        auto rank_candidates = [&]() {
            nc = 0;
            int nbits = 0, only = -1;
            for (int c = 0; c < Wd; ++c) { const uint32_t bits = row[c]; if (bits) { nbits += __popc(bits); only = c * 32 + __ffs(bits) - 1; } }
            if (nbits == 1) { cj[0] = only; nc = 1; return; }        // a single detection above sigma_iou: nothing to rank
            if (nbits == 0) return;
            for (int c = 0; c < Wd; ++c) {
                uint32_t bits = row[c];
                while (bits) {
                    const int j = c * 32 + __ffs(bits) - 1;
                    bits &= bits - 1;
                    const double v = track_value(box + 5 * j, tb, R.metric);
                    int p = nc < 4 ? nc : 4;                       // first slot with a smaller value (ties keep the lower j first)
#pragma unroll
                    for (int q = 3; q >= 0; --q) if (q < nc && cv[q] < v) p = q;
#pragma unroll
                    for (int q = 3; q >= 1; --q) if (q > p) { cv[q] = cv[q - 1]; cj[q] = cj[q - 1]; }
#pragma unroll
                    for (int q = 0; q < 4; ++q) if (q == p) { cv[q] = v; cj[q] = j; }
                    ++nc;
                }
            }
        };
        const bool active = tid < T && D > 0;
        if (active) {                          // preference list precomputed by k_track_mask
            const uint32_t p0 = row[W + 1], p1 = row[W + 2];
            cj[0] = (int)(p0 & 0xffffu); cj[1] = (int)(p0 >> 16); cj[2] = (int)(p1 & 0xffffu); cj[3] = (int)(p1 >> 16);
            nc = (int)row[W + 3];
        }
        int ptr = 0, prop = -1;
        for (;;) {
            prop = -1;
            if (active) {
                if (ptr >= 4 && nc > 4) { rank_candidates(); ptr = 0; }      // refused bits were cleared from the row
#pragma unroll
                for (int q = 0; q < 4; ++q) if (q == ptr && q < nc) prop = cj[q];
                if (prop >= 0) atomicMin(&owner[prop], tid);
            }
            __syncthreads();
            const bool refused = prop >= 0 && owner[prop] != tid;           // a lower-order track holds it
            if (refused) { row[prop >> 5] &= ~(1u << (prop & 31)); ++ptr; }
            if (!__syncthreads_or(refused)) break;
        }
        const int matched = (active && prop >= 0) ? 1 : 0;
        if (matched) match[tid] = prop;
        int tot;
        const int before = block_excl_scan(matched, s_warp, tot);
        n_upd = tot;
        // a track whose turn comes after all D detections are taken is dropped, not finished (:130, Q5)
        const bool had_dets = D > 0 && before < D;
        int fin = 0;
        if (tid < T && !matched && had_dets) fin = (pmaxs[my] > R.sigma_h && (int64_t)plen[my] > R.t_min) ? 1 : 0;   // :147 strict >
        if (matched) ord[before] = prop;
        long long ptot;
        const long long pb = block_excl_scan64(fin ? ((1ll << 32) | (long long)plen[my]) : 0ll, s_warp64, ptot);   // (count << 32) | rows
        if (fin) out.finish(n_fin + (pb >> 32), fin_rows + (pb & 0xffffffffll), phead[my], plen[my], pstart[my], pmaxs[my]);
        n_fin += ptot >> 32; fin_rows += ptot & 0xffffffffll;
    } else {
        // ---- exact sequential path (warp 0), mirrors the python loop including NaN argmax
        if (warp == 0) {
            int n_alive = D, nu = 0;
            int64_t nf = n_fin, fr = fin_rows;
            for (int t = 0; t < T; ++t) {
                const int i = pord[t];
                if (n_alive <= 0) continue;                                  // :130 silently dropped
                const double *tb = pbox + 5 * i;
                double bv = 0.0; int bj = INT_MAX; int bn = 0;               // lane-local: value, index, is-NaN
                for (int j = lane; j < D; j += 32) {
                    if (owner[j] != INT_MAX) continue;                       // already deleted from dets (:145)
                    const double v = track_value(box + 5 * j, tb, R.metric);
                    const int vn = v != v;
                    if (bj == INT_MAX) { bv = v; bj = j; bn = vn; }
                    else if (!bn && (vn || v > bv)) { bv = v; bj = j; bn = vn; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {                           // first NaN, else first max
                    const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
                    const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
                    const int on = __shfl_xor_sync(0xffffffffu, bn, o);
                    if (oj == INT_MAX) continue;
                    bool take;
                    if (bj == INT_MAX) take = true;
                    else if (bn != on) take = on != 0;
                    else if (bn) take = oj < bj;
                    else take = (ov > bv) || (ov == bv && oj < bj);
                    if (take) { bv = ov; bj = oj; bn = on; }
                }
                const bool matched = !bn && bv > R.sigma_iou;                // :134
                if (matched) {
                    if (lane == 0) { owner[bj] = t; match[t] = bj; ord[nu] = bj; }
                    ++nu; --n_alive;
                } else if (pmaxs[i] > R.sigma_h && (int64_t)plen[i] > R.t_min) {
                    if (lane == 0) out.finish(nf, fr, phead[i], plen[i], pstart[i], pmaxs[i]);
                    ++nf; fr += plen[i];
                }
                __syncwarp();
            }
            if (lane == 0) { s_slow[0] = nu; s_slow[1] = (int)(nf - n_fin); s_slow[2] = (int)(fr - fin_rows); }
        }
        __syncthreads();
        n_upd = s_slow[0]; n_fin += s_slow[1]; fin_rows += s_slow[2];
        __syncthreads();
    }

    // ---- state of the continued tracks (:141-143) ...
    if (tid < T && match[tid] >= 0) {
        const int j = match[tid];
        const double sc = box[5 * j + 4];
        B.head[j] = phead[my];
        B.len[j] = plen[my] + 1;
        B.start[j] = pstart[my];
        B.maxs[j] = sc > pmaxs[my] ? sc : pmaxs[my];                        // python max(a, b)
        out.extend(j, phead[my], plen[my]);
    }
    // ---- ... and new tracks from the detections left over, in detection order (:150-154)
    {
        const int is_new = (tid < D && owner[tid] == INT_MAX) ? 1 : 0;
        int tot;
        const int before = block_excl_scan(is_new, s_warp, tot);
        if (is_new) {
            const int j = tid;
            const int32_t h = out.new_head(j, before);
            ord[n_upd + before] = j;
            B.head[j] = h;
            B.len[j] = 1;
            B.start[j] = (int32_t)(f + 1);                                   // frame_num is 1-based (:118)
            B.maxs[j] = box[5 * j + 4];
            out.begin(j, h);
        }
        T = n_upd + tot;                                                     // :155
        out.created(tot);
    }
    __syncthreads();
}

// End of the video (:174-175): the T active tracks with max_score > sigma_h and len >= t_min finish, in active order.  The
// state pointers may be shared or global memory.
template <class Rule, class Sink>
__device__ __forceinline__ void track_flush(const double *pmaxs, const int32_t *phead, const int32_t *plen, const int32_t *pstart,
                                            const int32_t *pord, const Rule &R, const int T, int64_t &n_fin, int64_t &fin_rows,
                                            Sink &out, long long *s_warp64)
{
    const int tid = threadIdx.x;
    int fin = 0, i = 0;
    if (tid < T) { i = pord[tid]; fin = (pmaxs[i] > R.sigma_h && (int64_t)plen[i] >= R.t_min) ? 1 : 0; }
    long long ptot;
    const long long pb = block_excl_scan64(fin ? ((1ll << 32) | (long long)plen[i]) : 0ll, s_warp64, ptot);
    if (fin) out.finish(n_fin + (pb >> 32), fin_rows + (pb & 0xffffffffll), phead[i], plen[i], pstart[i], pmaxs[i]);
    n_fin += ptot >> 32; fin_rows += ptot & 0xffffffffll;
}

struct ResolveParams {
    const double *dets; const int64_t *frame_off; int64_t F; int W; int cap;   // cap = W * 32 >= max detections per frame
    const uint32_t *mask;                        // [total][W + ROW_EXTRA], see k_track_mask
    double sigma_iou, sigma_h; int64_t t_min;      // sigma_iou: threshold on the association value (-sigma_dis in distance mode)
    int metric;                                    // 0 IoU, 1 distance
    int32_t *det_head, *det_pos, *fin_id;        // [total]
    int64_t *n_tracks, *track_off, *track_start; double *track_max;
    int force_slow;
    int prefetch;                                // 1: stage frame f+1 while frame f is resolved (needs the larger smem layout)
};

// offline outputs: a track's head is the global row of its first detection; k_track_scatter turns (head, position) into track_dets
struct OfflineSink {
    const ResolveParams &P; int64_t g0;
    __device__ __forceinline__ void finish(int64_t id, int64_t row0, int32_t head, int32_t, int32_t start, double mx) const
    {
        P.fin_id[head] = (int32_t)id; P.track_off[id] = row0; P.track_start[id] = start; P.track_max[id] = mx;
    }
    __device__ __forceinline__ void extend(int j, int32_t head, int32_t pos) const { P.det_head[g0 + j] = head; P.det_pos[g0 + j] = pos; }
    __device__ __forceinline__ int32_t new_head(int j, int) const { return (int32_t)(g0 + j); }
    __device__ __forceinline__ void begin(int j, int32_t head) const { P.det_head[g0 + j] = head; P.det_pos[g0 + j] = 0; }
    __device__ __forceinline__ void created(int) const {}
};

// async global -> shared copies (LDGSTS) used to stage frame f+1 while frame f is being resolved
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__global__ void __launch_bounds__(TR_THREADS, 1)
k_track_resolve(const ResolveParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    // layout: rows[NR][cap*(W+1)] u32 | boxes[NBX][cap*5] f64 | maxs[2][cap] f64 | int arrays   (NR, NBX = 2, 3 with prefetch; 1, 2 without)
    const int W1 = P.W + ROW_EXTRA, CAP = P.cap;      // W1 = words per row
    const int PF = P.prefetch, NR = PF ? 2 : 1, NBX = PF ? 3 : 2;
    uint32_t *rowbuf = reinterpret_cast<uint32_t *>(smem);
    double *boxbuf = reinterpret_cast<double *>(smem + ((size_t)NR * CAP * W1 * 4 + 15) / 16 * 16);
    double *maxbuf = boxbuf + NBX * CAP * 5;
    int32_t *ibase = reinterpret_cast<int32_t *>(maxbuf + 2 * CAP);
    int32_t *headbuf = ibase, *lenbuf = ibase + 2 * CAP, *startbuf = ibase + 4 * CAP;
    int32_t *order = ibase + 6 * CAP;        // [2][CAP] local det index of each active track, in order
    int32_t *owner = ibase + 8 * CAP;        // [CAP]
    int32_t *match = ibase + 9 * CAP;        // [CAP] det matched to track t (or -1)
    __shared__ int s_warp[33];
    __shared__ long long s_warp64[33];
    __shared__ int s_slow[4];
    __shared__ int64_t s_off[OFF_CHUNK + 3];       // frame_off[c0 .. c0 + OFF_CHUNK + 2]: no global-latency chain at the top of a frame

    const int tid = threadIdx.x, NT = blockDim.x;   // NT = cap: one thread per track / detection
    int64_t off_c0 = 0;
    auto load_offsets = [&](int64_t c0) {
        off_c0 = c0;
        for (int i = tid; i < OFF_CHUNK + 3; i += NT) s_off[i] = P.frame_off[min(c0 + i, P.F)];
        __syncthreads();
    };
    auto foff = [&](int64_t fr) -> int64_t { return s_off[fr - off_c0]; };
    load_offsets(0);
    int cur = 0;                       // parity of the frame being processed (rows / per-det state double buffers)
    int T = 0;                         // active tracks = |order[prev]|
    int64_t n_fin = 0, fin_rows = 0;   // finished tracks so far, and their total length (uniform across threads)

    // async staging: boxes of frame fr -> boxbuf[fr % NBX]; candidate rows of the detections of frame g (they belong to the
    // tracks that are active while frame g+1 is resolved) -> rowbuf[PF ? g & 1 : 0]
    auto stage_boxes = [&](int64_t fr) {
        const int64_t a0 = foff(fr);
        const int Dn = min((int)(foff(fr + 1) - a0), CAP);
        double *bdst = boxbuf + (fr % NBX) * CAP * 5;
        for (int i = tid; i < Dn * 5; i += NT) cp_async8(bdst + i, P.dets + 5 * a0 + i);
    };
    auto stage_rows = [&](int64_t g) {
        const int64_t a0 = foff(g);
        const int Dn = min((int)(foff(g + 1) - a0), CAP);
        uint32_t *rdst = rowbuf + (PF ? (g & 1) : 0) * CAP * W1;
        for (int i = tid; i < Dn * W1; i += NT) cp_async4(rdst + i, P.mask + a0 * W1 + i);
    };
    if (PF && P.F > 0) { stage_boxes(0); cp_async_commit(); }

    for (int64_t f = 0; f < P.F; ++f, cur ^= 1) {
        const int prv = cur ^ 1;
        if (f - off_c0 >= OFF_CHUNK) load_offsets(f - 1);            // keeps f-1 .. f+2 addressable (stage_rows(f-1) without prefetch)
        const int64_t g0 = foff(f);
        const int D = min((int)(foff(f + 1) - g0), CAP);            // host guarantees D <= cap; clamp keeps memory safe
        const FrameBufs B{boxbuf + (f % NBX) * CAP * 5, boxbuf + ((f + NBX - 1) % NBX) * CAP * 5,
                          rowbuf + (PF ? prv : 0) * CAP * W1,      // rows of frame f-1's detections = of the active tracks
                          maxbuf + cur * CAP, maxbuf + prv * CAP,
                          headbuf + cur * CAP, lenbuf + cur * CAP, startbuf + cur * CAP, order + cur * CAP,
                          headbuf + prv * CAP, lenbuf + prv * CAP, startbuf + prv * CAP, order + prv * CAP,
                          owner, match};

        // ---- with prefetch this frame was staged one iteration ago and the next one is staged behind the resolution
        if (!PF) { stage_boxes(f); if (f > 0) stage_rows(f - 1); cp_async_commit(); }
        cp_async_wait_all();
        if (tid < D) owner[tid] = INT_MAX;
        if (tid < CAP) match[tid] = -1;
        __syncthreads();
        if (PF && f + 1 < P.F) { stage_boxes(f + 1); stage_rows(f); cp_async_commit(); }
        OfflineSink out{P, g0};
        track_frame(B, P, D, f, P.W, T, n_fin, fin_rows, out, s_warp, s_warp64, s_slow);
    }

    {
        const int prv = cur ^ 1;
        OfflineSink out{P, 0};
        track_flush(maxbuf + prv * CAP, headbuf + prv * CAP, lenbuf + prv * CAP, startbuf + prv * CAP, order + prv * CAP, P, T,
                    n_fin, fin_rows, out, s_warp64);
        if (tid == 0) { *P.n_tracks = n_fin; P.track_off[n_fin] = fin_rows; }
    }
}

__global__ void k_track_scatter(const int32_t *__restrict__ det_head, const int32_t *__restrict__ det_pos,
                                const int32_t *__restrict__ fin_id, const int64_t *__restrict__ track_off, int64_t total,
                                int64_t *__restrict__ track_dets)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    const int32_t id = fin_id[det_head[g]];
    if (id >= 0) track_dets[track_off[id] + det_pos[g]] = g;
}

struct TrackWs { uint32_t *mask; int32_t *frame_of, *det_head, *det_pos, *fin_id; size_t bytes; };
TrackWs plan_track_ws(void *ws, int64_t total, int W)
{
    TrackWs t;
    char *p = (char *)ws;
    size_t o = 0;
    const size_t n = (size_t)(total > 0 ? total : 1);
    t.mask = (uint32_t *)(p + o); o += fdt_align256(n * (W + ROW_EXTRA) * 4);
    t.frame_of = (int32_t *)(p + o); o += fdt_align256(n * 4);
    t.det_head = (int32_t *)(p + o); o += fdt_align256(n * 4);
    t.det_pos = (int32_t *)(p + o); o += fdt_align256(n * 4);
    t.fin_id = (int32_t *)(p + o); o += fdt_align256(n * 4);
    t.bytes = o;
    return t;
}


// ---- online, multi-stream tracking: one frame per stream and call, the state carried between calls in a caller-owned buffer.
// State = StreamHeader (256 bytes) + V slots.  A slot holds what k_track_resolve carries from frame f to frame f+1: the previous
// frame's rows (boxes), per row the track id / length / start frame / max score of the track it belongs to, the active order and
// T, the frame counter, the finished-track counter and the next track id.  A track's "head" is its stream-local id here.
constexpr uint32_t STREAM_MAGIC = 0x46445453u;      // "FDTS"
struct StreamHeader {
    uint32_t magic, status;                          // status: sticky FDT_STATUS_TRACK_* bits
    int32_t V, cap, metric, pad;
    double sigma_iou, sigma_h; int64_t t_min;        // sigma_iou: threshold on the association value (-sigma_dis in distance mode)
};
struct SlotHead { int32_t T, pad; int64_t frame, n_fin, next_id; };
constexpr size_t STREAM_HDR_BYTES = 256;

size_t stream_slot_bytes(int cap) { return fdt_align256(sizeof(SlotHead) + (size_t)cap * (6 * sizeof(double) + 4 * sizeof(int32_t))); }

struct SlotView {
    SlotHead *h; double *box, *maxs; int32_t *head, *len, *start, *ord;
};
__device__ __forceinline__ SlotView slot_view(void *state, int64_t v, int cap, size_t slot_bytes)
{
    char *p = (char *)state + STREAM_HDR_BYTES + (size_t)v * slot_bytes;
    SlotView s;
    s.h = (SlotHead *)p;
    s.box = (double *)(p + sizeof(SlotHead)); s.maxs = s.box + 5 * cap;
    s.head = (int32_t *)(s.maxs + cap); s.len = s.head + cap; s.start = s.len + cap; s.ord = s.start + cap;
    return s;
}
__device__ __forceinline__ bool header_ok(const StreamHeader *hd, int64_t V, int cap)
{
    return hd->magic == STREAM_MAGIC && hd->V == V && hd->cap == cap;
}

struct StreamRows {
    void *state; size_t slot_bytes; int cap; int64_t V; const uint8_t *advance;
    __device__ __forceinline__ bool row(int64_t g, const double *__restrict__, const int64_t *__restrict__ frame_off,
                                        const int32_t *__restrict__, int64_t, int64_t, double (&tb)[4],
                                        int64_t &n0, int &D, int &metric, double &sigma_iou) const
    {
        const int64_t v = g / cap;
        const int i = (int)(g - v * cap);
        if (v >= V) return false;
        const StreamHeader *hd = (const StreamHeader *)state;
        if (!header_ok(hd, V, cap) || (advance && !advance[v])) return false;
        const SlotView s = slot_view(state, v, cap, slot_bytes);
        if (i >= s.h->T) return false;
        n0 = frame_off[v];
        D = (int)(frame_off[v + 1] - n0);
        if (D < 0 || D > cap) return false;                             // over capacity: k_track_step skips the frame
#pragma unroll
        for (int k = 0; k < 4; ++k) tb[k] = s.box[5 * i + k];
        metric = hd->metric; sigma_iou = hd->sigma_iou;
        return true;
    }
};

// streaming outputs: row ids, and per finished track a record at position k of this call's [cap] block
struct StreamSink {
    int64_t *row_track; int64_t g0, fin_base, next_id;
    int64_t *fin_index, *fin_track, *fin_start, *fin_len; double *fin_max;
    __device__ __forceinline__ void finish(int64_t id, int64_t, int32_t head, int32_t len, int32_t start, double mx) const
    {
        const int64_t k = id - fin_base;
        fin_index[k] = id; fin_track[k] = head; fin_start[k] = start; fin_len[k] = len; fin_max[k] = mx;
    }
    __device__ __forceinline__ void extend(int j, int32_t head, int32_t) const { row_track[g0 + j] = head; }
    __device__ __forceinline__ int32_t new_head(int, int k) const { return (int32_t)(next_id + k); }
    __device__ __forceinline__ void begin(int j, int32_t head) const { row_track[g0 + j] = head; }
    __device__ __forceinline__ void created(int n) { next_id += n; }
};

struct StreamOut {
    int32_t *fin_count; int64_t *fin_index, *fin_track, *fin_start, *fin_len; double *fin_max;   // [V], [V, cap] x 5
};

__global__ void k_track_stream_init(void *state, int64_t V, int cap, size_t slot_bytes, int metric, double sigma_iou, double sigma_h,
                                    int64_t t_min)
{
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v == 0) {
        StreamHeader *hd = (StreamHeader *)state;
        hd->magic = STREAM_MAGIC; hd->status = 0; hd->V = (int32_t)V; hd->cap = cap; hd->metric = metric; hd->pad = 0;
        hd->sigma_iou = sigma_iou; hd->sigma_h = sigma_h; hd->t_min = t_min;
    }
    if (v < V) *slot_view(state, v, cap, slot_bytes).h = SlotHead{0, 0, 0, 0, 0};
}

// one CTA (cap threads) per stream: load the slot into k_track_resolve's shared layout (no prefetch buffers), run one frame, store
__global__ void __launch_bounds__(TR_THREADS, 1)
k_track_step(void *state, size_t slot_bytes, int64_t V, int W, const double *__restrict__ dets, const int64_t *__restrict__ frame_off,
             const uint8_t *__restrict__ advance, const uint32_t *__restrict__ mask, int64_t *__restrict__ row_track, StreamOut O,
             int force_slow)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int W1 = W + ROW_EXTRA, CAP = blockDim.x, tid = threadIdx.x;
    const int64_t v = blockIdx.x;
    StreamHeader *hd = (StreamHeader *)state;
    if (!header_ok(hd, V, CAP)) {                                        // the call does not describe this state: change nothing
        if (v == 0 && tid == 0) atomicOr(&hd->status, FDT_STATUS_TRACK_MISMATCH);
        return;
    }
    const int64_t g0 = frame_off[v];
    const int64_t Dg = frame_off[v + 1] - g0;
    const bool adv = advance == nullptr || advance[v] != 0;
    if (!adv || Dg < 0 || Dg > CAP) {                                    // no frame, or one over capacity: the slot is untouched
        for (int64_t r = tid; r < Dg; r += CAP) row_track[g0 + r] = -1;
        if (tid == 0) {
            O.fin_count[v] = 0;
            if (adv) atomicOr(&hd->status, FDT_STATUS_TRACK_OVERFLOW);
        }
        return;
    }
    const int D = (int)Dg;
    uint32_t *rowbuf = reinterpret_cast<uint32_t *>(smem);
    double *boxbuf = reinterpret_cast<double *>(smem + ((size_t)CAP * W1 * 4 + 15) / 16 * 16);
    double *maxbuf = boxbuf + 2 * CAP * 5;
    int32_t *ibase = reinterpret_cast<int32_t *>(maxbuf + 2 * CAP);
    int32_t *headbuf = ibase, *lenbuf = ibase + 2 * CAP, *startbuf = ibase + 4 * CAP;
    int32_t *order = ibase + 6 * CAP, *owner = ibase + 8 * CAP, *match = ibase + 9 * CAP;
    __shared__ int s_warp[33];
    __shared__ long long s_warp64[33];
    __shared__ int s_slow[4];

    const SlotView s = slot_view(state, v, CAP, slot_bytes);
    const SlotHead sh = *s.h;
    int T = sh.T;
    const TrackRule R{hd->sigma_iou, hd->sigma_h, hd->t_min, hd->metric, force_slow};
    // cur = 0 (this frame), prv = 1 (the slot)
    const FrameBufs B{boxbuf, boxbuf + CAP * 5, rowbuf, maxbuf, maxbuf + CAP,
                      headbuf, lenbuf, startbuf, order, headbuf + CAP, lenbuf + CAP, startbuf + CAP, order + CAP, owner, match};
    for (int i = tid; i < D * 5; i += CAP) boxbuf[i] = dets[5 * g0 + i];
    for (int i = tid; i < T * 5; i += CAP) boxbuf[CAP * 5 + i] = s.box[i];
    for (int i = tid; i < T * W1; i += CAP) rowbuf[i] = mask[(size_t)v * CAP * W1 + i];
    if (tid < T) {
        maxbuf[CAP + tid] = s.maxs[tid]; headbuf[CAP + tid] = s.head[tid]; lenbuf[CAP + tid] = s.len[tid];
        startbuf[CAP + tid] = s.start[tid]; order[CAP + tid] = s.ord[tid];
    }
    if (tid < D) owner[tid] = INT_MAX;
    match[tid] = -1;
    __syncthreads();

    int64_t n_fin = sh.n_fin, fin_rows = 0;
    StreamSink out{row_track, g0, sh.n_fin, sh.next_id, O.fin_index + v * CAP, O.fin_track + v * CAP, O.fin_start + v * CAP,
                   O.fin_len + v * CAP, O.fin_max + v * CAP};
    track_frame(B, R, D, sh.frame, W, T, n_fin, fin_rows, out, s_warp, s_warp64, s_slow);

    // every detection of this frame now is the last box of exactly one active track (T == D)
    for (int i = tid; i < D * 5; i += CAP) s.box[i] = boxbuf[i];
    if (tid < D) { s.maxs[tid] = maxbuf[tid]; s.head[tid] = headbuf[tid]; s.len[tid] = lenbuf[tid]; s.start[tid] = startbuf[tid]; }
    if (tid < T) s.ord[tid] = order[tid];
    if (tid == 0) {
        *s.h = SlotHead{T, 0, sh.frame + 1, n_fin, out.next_id};
        O.fin_count[v] = (int32_t)(n_fin - sh.n_fin);
    }
}

// end of video for the selected streams: the flush records, then the slot starts over (frame 0, no tracks, ids from 0)
__global__ void __launch_bounds__(TR_THREADS, 1)
k_track_stream_flush(void *state, size_t slot_bytes, int64_t V, const uint8_t *__restrict__ sel, StreamOut O)
{
    __shared__ long long s_warp64[33];
    const int CAP = blockDim.x, tid = threadIdx.x;
    const int64_t v = blockIdx.x;
    StreamHeader *hd = (StreamHeader *)state;
    if (!header_ok(hd, V, CAP)) {
        if (v == 0 && tid == 0) atomicOr(&hd->status, FDT_STATUS_TRACK_MISMATCH);
        return;
    }
    if (sel && !sel[v]) {
        if (tid == 0) O.fin_count[v] = 0;
        return;
    }
    const SlotView s = slot_view(state, v, CAP, slot_bytes);
    const SlotHead sh = *s.h;
    const TrackRule R{hd->sigma_iou, hd->sigma_h, hd->t_min, hd->metric, 0};
    int64_t n_fin = sh.n_fin, fin_rows = 0;
    StreamSink out{nullptr, 0, sh.n_fin, sh.next_id, O.fin_index + v * CAP, O.fin_track + v * CAP, O.fin_start + v * CAP,
                   O.fin_len + v * CAP, O.fin_max + v * CAP};
    track_flush(s.maxs, s.head, s.len, s.start, s.ord, R, sh.T, n_fin, fin_rows, out, s_warp64);   // (synchronises the block)
    if (tid == 0) {
        O.fin_count[v] = (int32_t)(n_fin - sh.n_fin);
        *s.h = SlotHead{0, 0, 0, 0, 0};
    }
}

int stream_cap(int64_t max_dets_per_frame) { return 32 * (int)(max_dets_per_frame > 0 ? (max_dets_per_frame + 31) / 32 : 1); }

// host-side checks shared by the stream entry points
int stream_check(const char *fn, const void *state, int64_t V, int64_t max_dets_per_frame)
{
    FDT_REQUIRE(state, FDT_E_INVALID, "%s: null state", fn);
    FDT_REQUIRE(fdt_aligned(state, 256), FDT_E_INVALID, "%s: state needs 256-byte alignment", fn);
    FDT_REQUIRE(V >= 1 && max_dets_per_frame >= 0, FDT_E_INVALID, "%s: V=%lld, max_dets_per_frame=%lld", fn, (long long)V,
                (long long)max_dets_per_frame);
    FDT_REQUIRE(V <= INT_MAX, FDT_E_UNSUPPORTED, "%s: V=%lld exceeds 2^31-1 streams", fn, (long long)V);
    FDT_REQUIRE(max_dets_per_frame <= TR_MAX_D, FDT_E_UNSUPPORTED,
                "%s: %lld detections in one frame exceed the limit of %d (shared memory)", fn, (long long)max_dets_per_frame, TR_MAX_D);
    return FDT_OK;
}

}  // namespace

FDT_API size_t fdt_iou_track_workspace_bytes(int64_t F, int64_t total, int64_t max_dets_per_frame)
{
    (void)F;
    if (total < 0 || max_dets_per_frame < 0 || max_dets_per_frame > TR_MAX_D) return 0;     // what fdt_iou_track_metric refuses
    int W = (int)((max_dets_per_frame + 31) / 32);
    if (W < 1) W = 1;
    return plan_track_ws(nullptr, total, W).bytes;
}

FDT_API int fdt_iou_track(const double *dets, const int64_t *frame_off, int64_t F, int64_t total, int64_t max_dets_per_frame,
                          double sigma_iou, double sigma_h, int64_t t_min,
                          int64_t *n_tracks, int64_t *track_off, int64_t *track_dets, int64_t *track_start, double *track_max,
                          void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return fdt_iou_track_metric(dets, frame_off, F, total, max_dets_per_frame, FDT_TRACK_IOU, sigma_iou, sigma_h, t_min,
                                n_tracks, track_off, track_dets, track_start, track_max, ws, ws_bytes, stream);
}

FDT_API int fdt_iou_track_metric(const double *dets, const int64_t *frame_off, int64_t F, int64_t total, int64_t max_dets_per_frame,
                                 int metric, double sigma, double sigma_h, int64_t t_min,
                                 int64_t *n_tracks, int64_t *track_off, int64_t *track_dets, int64_t *track_start, double *track_max,
                                 void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    FDT_REQUIRE(metric == FDT_TRACK_IOU || metric == FDT_TRACK_DISTANCE, FDT_E_INVALID, "fdt_iou_track: unknown metric %d", metric);
    const double sigma_iou = metric == FDT_TRACK_IOU ? sigma : -sigma;
    FDT_REQUIRE(F >= 0 && total >= 0 && max_dets_per_frame >= 0, FDT_E_INVALID, "fdt_iou_track: negative size");
    FDT_REQUIRE(n_tracks && track_off, FDT_E_INVALID, "fdt_iou_track: null output pointer");
    FDT_REQUIRE(total < (1ll << 31), FDT_E_UNSUPPORTED, "fdt_iou_track: total=%lld exceeds 2^31-1", (long long)total);
    FDT_REQUIRE(max_dets_per_frame <= TR_MAX_D, FDT_E_UNSUPPORTED,
                "fdt_iou_track: %lld detections in one frame exceed the limit of %d (shared memory)", (long long)max_dets_per_frame,
                TR_MAX_D);
    if (F == 0 || total == 0) {
        FDT_CUDA(cudaMemsetAsync(n_tracks, 0, sizeof(int64_t), st));
        FDT_CUDA(cudaMemsetAsync(track_off, 0, sizeof(int64_t), st));
        return FDT_OK;
    }
    FDT_REQUIRE(dets && frame_off && track_dets && track_start && track_max && ws, FDT_E_INVALID, "fdt_iou_track: null pointer argument");
    FDT_REQUIRE(fdt_aligned(ws, 256), FDT_E_INVALID, "fdt_iou_track: workspace needs 256-byte alignment");
    int W = (int)((max_dets_per_frame + 31) / 32);
    if (W < 1) W = 1;
    TrackWs t = plan_track_ws(ws, total, W);
    FDT_REQUIRE(ws_bytes >= t.bytes, FDT_E_WORKSPACE, "fdt_iou_track: workspace %zu < %zu bytes", ws_bytes, t.bytes);
    const int prefetch = resolve_smem(W, 1) <= TR_SMEM_LIMIT;
    const size_t smem = resolve_smem(W, prefetch);       // <= TR_SMEM_LIMIT: W <= TR_MAX_D / 32 (checked above, before any CUDA call)

    FDT_CUDA(cudaMemsetAsync(t.fin_id, 0xff, (size_t)total * 4, st));
    k_track_frame_of<<<(unsigned)F, 128, 0, st>>>(frame_off, F, t.frame_of);
    FDT_LAUNCH_CHECK();
    k_track_mask<<<(unsigned)((total + 7) / 8), 256, 0, st>>>(dets, frame_off, t.frame_of, F, total, W, metric, sigma_iou, t.mask,
                                                              OfflineRows{});
    FDT_LAUNCH_CHECK();
    ResolveParams P{};
    P.dets = dets; P.frame_off = frame_off; P.F = F; P.W = W; P.cap = W * 32; P.mask = t.mask;
    P.sigma_iou = sigma_iou; P.sigma_h = sigma_h; P.t_min = t_min; P.metric = metric;
    P.det_head = t.det_head; P.det_pos = t.det_pos; P.fin_id = t.fin_id;
    P.n_tracks = n_tracks; P.track_off = track_off; P.track_start = track_start; P.track_max = track_max;
    const char *env = getenv("FDT_TRACK_FORCE_SLOW");
    P.force_slow = (env && env[0] == '1') ? 1 : 0;
    P.prefetch = prefetch;
    FDT_CUDA(cudaFuncSetAttribute(k_track_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_track_resolve<<<1, P.cap, smem, st>>>(P);      // cap = multiple of 32 >= max detections per frame, <= TR_MAX_D
    FDT_LAUNCH_CHECK();
    k_track_scatter<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(t.det_head, t.det_pos, t.fin_id, track_off, total, track_dets);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API size_t fdt_track_stream_state_bytes(int64_t V, int64_t max_dets_per_frame)
{
    if (V < 0 || max_dets_per_frame < 0 || max_dets_per_frame > TR_MAX_D) return 0;
    return STREAM_HDR_BYTES + (size_t)V * stream_slot_bytes(stream_cap(max_dets_per_frame));
}

FDT_API size_t fdt_track_stream_workspace_bytes(int64_t V, int64_t max_dets_per_frame)
{
    if (V < 0 || max_dets_per_frame < 0 || max_dets_per_frame > TR_MAX_D) return 0;
    const int cap = stream_cap(max_dets_per_frame);
    return fdt_align256((size_t)(V > 0 ? V : 1) * cap * (cap / 32 + ROW_EXTRA) * 4);
}

FDT_API int fdt_track_stream_init(void *state, size_t state_bytes, int64_t V, int64_t max_dets_per_frame, int metric, double sigma,
                                  double sigma_h, int64_t t_min, fdt_stream_t stream)
{
    const int rc = stream_check("fdt_track_stream_init", state, V, max_dets_per_frame);
    if (rc != FDT_OK) return rc;
    FDT_REQUIRE(metric == FDT_TRACK_IOU || metric == FDT_TRACK_DISTANCE, FDT_E_INVALID, "fdt_track_stream_init: unknown metric %d", metric);
    const size_t need = fdt_track_stream_state_bytes(V, max_dets_per_frame);
    FDT_REQUIRE(state_bytes >= need, FDT_E_WORKSPACE, "fdt_track_stream_init: state %zu < %zu bytes", state_bytes, need);
    const int cap = stream_cap(max_dets_per_frame);
    const unsigned blocks = (unsigned)((V + 255) / 256);
    k_track_stream_init<<<blocks, 256, 0, (cudaStream_t)stream>>>(state, V, cap, stream_slot_bytes(cap), metric,
                                                                  metric == FDT_TRACK_IOU ? sigma : -sigma, sigma_h, t_min);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_track_stream_step(void *state, int64_t V, int64_t max_dets_per_frame, const double *dets, const int64_t *frame_off,
                                  const uint8_t *advance, int64_t *row_track, int32_t *fin_count, int64_t *fin_index,
                                  int64_t *fin_track, int64_t *fin_start, int64_t *fin_len, double *fin_max, void *ws, size_t ws_bytes,
                                  fdt_stream_t stream)
{
    const int rc = stream_check("fdt_track_stream_step", state, V, max_dets_per_frame);
    if (rc != FDT_OK) return rc;
    FDT_REQUIRE(dets && frame_off && row_track && fin_count && fin_index && fin_track && fin_start && fin_len && fin_max && ws,
                FDT_E_INVALID, "fdt_track_stream_step: null pointer argument");
    FDT_REQUIRE(fdt_aligned(ws, 256), FDT_E_INVALID, "fdt_track_stream_step: workspace needs 256-byte alignment");
    const size_t need = fdt_track_stream_workspace_bytes(V, max_dets_per_frame);
    FDT_REQUIRE(ws_bytes >= need, FDT_E_WORKSPACE, "fdt_track_stream_step: workspace %zu < %zu bytes", ws_bytes, need);
    cudaStream_t st = (cudaStream_t)stream;
    const int cap = stream_cap(max_dets_per_frame), W = cap / 32;
    const size_t slot = stream_slot_bytes(cap);
    const int64_t rows = V * cap;
    k_track_mask<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(dets, frame_off, nullptr, V, rows, W, 0, 0.0, (uint32_t *)ws,
                                                             StreamRows{state, slot, cap, V, advance});
    FDT_LAUNCH_CHECK();
    const char *env = getenv("FDT_TRACK_FORCE_SLOW");
    const int force_slow = (env && env[0] == '1') ? 1 : 0;
    const size_t smem = resolve_smem(W, 0);
    FDT_CUDA(cudaFuncSetAttribute(k_track_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_track_step<<<(unsigned)V, cap, smem, st>>>(state, slot, V, W, dets, frame_off, advance, (const uint32_t *)ws, row_track,
                                                  StreamOut{fin_count, fin_index, fin_track, fin_start, fin_len, fin_max}, force_slow);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_track_stream_flush(void *state, int64_t V, int64_t max_dets_per_frame, const uint8_t *streams, int32_t *fin_count,
                                   int64_t *fin_index, int64_t *fin_track, int64_t *fin_start, int64_t *fin_len, double *fin_max,
                                   fdt_stream_t stream)
{
    const int rc = stream_check("fdt_track_stream_flush", state, V, max_dets_per_frame);
    if (rc != FDT_OK) return rc;
    FDT_REQUIRE(fin_count && fin_index && fin_track && fin_start && fin_len && fin_max, FDT_E_INVALID,
                "fdt_track_stream_flush: null pointer argument");
    const int cap = stream_cap(max_dets_per_frame);
    k_track_stream_flush<<<(unsigned)V, cap, 0, (cudaStream_t)stream>>>(state, stream_slot_bytes(cap), V, streams,
                                                                      StreamOut{fin_count, fin_index, fin_track, fin_start, fin_len, fin_max});
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_track_stream_status(const void *state, fdt_stream_t stream, uint32_t *status_h)
{
    FDT_REQUIRE(state && status_h, FDT_E_INVALID, "fdt_track_stream_status: null pointer argument");
    cudaStream_t st = (cudaStream_t)stream;
    FDT_CUDA(cudaMemcpyAsync(status_h, (const char *)state + offsetof(StreamHeader, status), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    FDT_CUDA(cudaStreamSynchronize(st));
    return FDT_OK;
}
