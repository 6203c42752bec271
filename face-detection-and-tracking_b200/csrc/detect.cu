// Detect (layers/functions/detection.py:34-84) and nms (layers/box_utils.py:275-340) for sm_100a.
//
// Three launches per call chained by programmatic dependent launch, no host synchronisation, CUDA-graph capturable:
//   --  k_zero_counters     : clears the per-list counters; resident behind the previous call's K3, releases K2 once that ended.
//   K2  k_threshold_compact : streams conf once (HBM-bound), strict `score > conf_thresh`, warp-ballot + block-aggregated
//                             compaction into unordered 64-bit keys (score_key << 32 | prior) + the list's score range.
//       k_heads_threshold_compact : the same from the models' per-level NCHW head maps (max-in-out + softmax fused).
//   K3  k_sort_nms          : one 1024-thread CTA -- or a 2-CTA thread-block cluster when the batch leaves SMs idle -- per
//                             (image, class) list, launched with programmatic stream serialization behind K2:
//         stage 1  top-nms_top_k selection by a bucket (counting) sort of the keys in shared memory
//                  (exact radix-select / bitonic fallbacks for degenerate score distributions);
//         stage 2  lazy greedy NMS over windows of <= 1024 sorted candidates: exact in-bucket order, decode of exactly those
//                  rows, a multi-level uniform grid (CSR) over the window, then
//                    A  drop candidates suppressed by boxes kept in earlier windows,
//                    B  collect, per survivor, the earlier survivors that suppress it (each pair examined once),
//                    C  resolve by parallel sweeps (dead iff a suppressor is kept, kept iff all are dead),
//                  stopping as soon as top_k boxes are kept (Detect reads only keep[:top_k], detection.py:80-81, so the
//                  output equals the reference's run-to-completion loop);
//         stage 3  output rows -- locally, or straight into the gathered block of a root rank / of every rank over NVLink peer
//                  memory, optionally publishing / awaiting the cross-rank completion signals itself.
// MODE_NMS runs the same kernel for layers/box_utils.nms and, with FDT_NMS_* flags, for the FaceBoxes / MTCNN NMS variants.
//
// Tie rule (unspecified in the reference, torch.sort is unstable): keys are unique, descending key order = descending score,
// higher prior index first among equal scores.  DESIGN.md section 4 has the exactness arguments.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <mutex>
#include <string>
#include <cooperative_groups.h>
#include "fdt_common.cuh"
#include "heads.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int K2_THREADS = 256;
constexpr int K2_PER_THREAD = 8;
constexpr int K2_TILE = K2_THREADS * K2_PER_THREAD;

constexpr int K3_THREADS = 1024;
constexpr int WIN = K3_THREADS;                 // sorted candidates examined per NMS round: one thread each
constexpr int NB = 2048;                        // score buckets of the shared-memory bucket sort
constexpr int BIG_BUCKET = 512;                 // a larger bucket inside the top-k range -> full bitonic sort fallback
constexpr int NLEV = 6;                         // grid levels: 32, 16, 8, 4, 2, 1 cells per side
constexpr int NCELLS = 1024 + 256 + 64 + 16 + 4 + 1;
constexpr int BIGCELL = NCELLS;                 // pseudo-cell: boxes the grid cannot index (see box_regular)
constexpr int NCELLX = NCELLS + 1;
constexpr int DEPS = 8;                         // stored earlier-suppressors per survivor (more -> re-query path)
constexpr int KEPT_ROW_BYTES = 28;              // box 16 + key 8 + area 4
constexpr int SEG_SLOTS = 8;                    // phase B: row segments a lane can queue (more -> visited in place)

enum { MODE_DETECT = 0, MODE_NMS = 1 };

// ------------------------------------------------------------------------------------------- head maps (SURVEY 8f rank 1)
// HeadLevels, head_logits, head_loc_row, softmax2: heads.cuh.

// Materialises the reference's tensors: loc_out[B,N,4] and conf_out[B,N,2] (softmax applied iff `softmax`; the training
// path keeps raw logits, pyramid.py:339-346).  Either output may be null.
template <int F>
__global__ void __launch_bounds__(256)
k_heads_to_loc_conf(const HeadLevels h, const int N, const int softmax, float *__restrict__ loc_out, float *__restrict__ conf_out)
{
    const int b = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    if (conf_out) {
        float2 x = head_logits<F>(h, b, p);
        if (softmax) x = softmax2(x);
        reinterpret_cast<float2 *>(conf_out)[(int64_t)b * N + p] = x;
    }
    if (loc_out) reinterpret_cast<float4 *>(loc_out)[(int64_t)b * N + p] = head_loc_row<F>(h, b, p);
}

// ------------------------------------------------------------------------------------------- call sequencing
// The first 256 bytes of a Detect workspace hold a control block that lives across calls; the rest is a ring of R >= 1 slots
// (per-list counters + candidate keys + spilled kept rows), R = how many the caller's workspace has room for.  Call number s
// (1, 2, ...) of a workspace uses slot s % R, so with R >= 2 nothing call s + 1 writes before its NMS is read by call s: its
// counter clear and K2 run UNDER the previous call's k_sort_nms (on the SMs that kernel leaves idle), and its k_sort_nms CTAs take
// over SMs as the previous call's CTAs retire -- consecutive calls on one stream overlap on the device.  Everything is chained by
// programmatic dependent launch; the hazards that stream order no longer covers are covered here:
//   * k_detect_begin(s) runs while k_sort_nms(s - 1) may still be in flight (that kernel triggers at its start).  If NO call of
//     this workspace is in flight (done == seq) whatever precedes us in the stream may be a foreign kernel, e.g. the producer of
//     `conf`: full dependency wait.  If one is in flight it IS our predecessor (a foreign kernel launched after it would have
//     waited for its completion, which publishes done == seq): nothing to wait for, the inputs were complete before it began.
//   * slot reuse: wait until call s - R has completed (done >= s - R).
//   * the same `out` / `counts` / `kept_prior` buffer as one of the calls still in flight: wait until done == s - 1.
//   * completion in order: the last CTA of k_sort_nms(s) publishes done = s only after done == s - 1, so a kernel that waits for
//     k_sort_nms(s) (normal stream order) also finds every earlier call complete.
// seq, k3s and done are sequence numbers (wrapping uint32, compared by signed difference).
//
// Inside a call the three kernels depend on each other through FLAGS in the slot, not through griddepcontrol.wait: that
// instruction waits for EVERY earlier grid of the stream (grids retire in order), i.e. also for the previous call's k_sort_nms --
// measured with tools/pdl_probe.cu: with hardware waits a chain of calls runs strictly one after another, without them the
// stream runs up to 8 grids ahead of its oldest incomplete one.  So: k_detect_begin publishes begin_seq = s once the slot's counters
// are cleared, every K2 block waits for that before its first atomic and counts itself in k2_done when its keys are written
// (fence + atomic), and every k_sort_nms CTA waits until k2_done has reached the number of K2 blocks.  A waiting grid was launched
// after ALL blocks of the grid it waits for had started (programmatic launch completion), so the producers are resident and the
// spins cannot deadlock.  Keys and counters written by another grid still in flight are read with ld.global.cg (L2).
//
// Slot header: int32 counters[3 * lists] | k2_done | begin_seq.
constexpr unsigned long long FDT_CTL_MAGIC = 0x4644543262303031ull;      // "FDT2b001"
// FDT_DETECT_MAX_DEPTH (fdt_common.cuh) = 4 slots at most                // (a power of two: ticket index = seq & 3)
struct DetectCtl {
    unsigned long long magic;          // FDT_CTL_MAGIC ^ geometry hash; anything else: first call on this memory
    unsigned seq;                      // calls begun
    unsigned k3s;                      // latest call whose k_sort_nms has started
    unsigned done;                     // latest call whose k_sort_nms has completed (in order)
    unsigned error;                    // sticky FDT_STATUS_* bits (a wait timed out)
    unsigned check;                    // ~seq ^ (unsigned)magic: guards against foreign writes into a recycled buffer
    unsigned pad;
    unsigned ticket[FDT_DETECT_MAX_DEPTH];     // completion ticket per slot: writer CTAs of k_sort_nms count themselves out, the last one resets it
    unsigned long long outs[FDT_DETECT_MAX_DEPTH][3];      // out / counts / kept_prior of the last R calls
};
static_assert(sizeof(DetectCtl) <= 256, "control block is 256 bytes");
constexpr int FDT_GATHER_RING_MAX = 8;
struct DetectSlots {
    DetectCtl *ctl;                    // null: no sequencing (fdt_nms), `base` is the only slot
    int32_t *gather_rows;              // [FDT_GATHER_RING_MAX][lists]: rows this rank left in gathered block (epoch % ring) of the destinations
    int gather_n;                      // FDT_GATHER_RING_MAX * lists
    char *base;                        // slot 0
    size_t stride;                     // bytes per slot
    size_t keys_off, kept_off;         // inside a slot: counters | keys | kept rows
    int depth;                         // R
};
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned *p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
constexpr int SLOT_K2_DONE = 0, SLOT_BEGIN_SEQ = 1, SLOT_EXTRA = 4;     // after counters[3 * lists]
// spins until (int)(*p - target) >= 0; false after ~4 s (a bug or a dead peer must not hang the GPU for ever)
__device__ __forceinline__ bool spin_until_reached(const unsigned *p, const unsigned target)
{
    const long long t0 = clock64();
    while ((int)(ld_acquire_u32(p) - target) < 0) {
        if (clock64() - t0 > (1ll << 33)) return false;
        __nanosleep(64);
    }
    return true;
}

// First kernel of every call: sequencing (see above) + clears the call's per-list counters.  A kernel rather than
// cudaMemsetAsync so that K2 can be launched behind it with programmatic stream serialization.
__global__ void __launch_bounds__(256)
k_detect_begin(const DetectSlots S, const unsigned long long magic, const int lists, const int serialize,
               const unsigned long long out0, const unsigned long long out1, const unsigned long long out2)
{
    __shared__ unsigned s_slot, s_seqv;
    DetectCtl *ctl = S.ctl;
    if (threadIdx.x == 0) {
        const int R = S.depth;
        volatile DetectCtl *v = ctl;
        unsigned seq = v->seq, k3s = v->k3s, done = ld_acquire_u32(&ctl->done);
        bool fresh = v->magic != magic || v->check != (~seq ^ (unsigned)magic) || (int)(seq - done) < 0 || (int)(seq - done) > R ||
                     (int)(seq - k3s) < 0 || (int)(k3s - done) < 0;
        bool waited = false;
        if (fresh || done == seq || serialize) {              // nothing of ours in flight: the predecessor may be anybody
            cudaGridDependencySynchronize();
            waited = true;
        }
        if (fresh) {
            // sequence numbers start from an arbitrary value: a stale begin_seq / k2_done pair left in recycled memory cannot match
            seq = k3s = done = (unsigned)(clock64() >> 3) * 2654435761u;
            for (int q = 0; q < FDT_DETECT_MAX_DEPTH; ++q) { v->outs[q][0] = 0; v->outs[q][1] = 0; v->outs[q][2] = 0; }
            v->error = 0; v->k3s = seq; v->done = seq;
            for (int q = 0; q < FDT_DETECT_MAX_DEPTH; ++q) v->ticket[q] = 0;
            for (int q = 0; q < S.gather_n; ++q) S.gather_rows[q] = 0;          // (the destinations' gathered blocks start zeroed)
        } else {
            if (k3s != seq) {
                // the previous call never launched its k_sort_nms (stage 1 alone): it is void.  Its K2 is our predecessor.
                if (!waited) { cudaGridDependencySynchronize(); waited = true; }
                if (!spin_until_reached(&ctl->done, k3s)) { atomicOr(&ctl->error, FDT_STATUS_TIMEOUT_LOCAL); __trap(); }
                v->k3s = seq; v->done = seq; done = seq;
            }
            // an output buffer of a call that may still be running is about to be written again: take turns
            bool alias = serialize != 0;
            for (int q = 1; q < R && !alias; ++q) {
                if ((int)((seq + 1 - q) - done) <= 0) break;                  // call seq + 1 - q has completed
                const int sl = (seq + 1 - q) % R;
                alias = (out0 && v->outs[sl][0] == out0) || (out1 && v->outs[sl][1] == out1) || (out2 && v->outs[sl][2] == out2);
            }
            const unsigned need = alias ? seq : seq + 1 - (unsigned)R;        // slot reuse: call s - R has completed
            if ((int)(done - need) < 0 && !spin_until_reached(&ctl->done, need)) { atomicOr(&ctl->error, FDT_STATUS_TIMEOUT_LOCAL); __trap(); }
            if (alias && !waited) { cudaGridDependencySynchronize(); waited = true; }     // and its stores have landed
        }
        seq += 1;
        const int sl = seq % R;
        v->outs[sl][0] = out0; v->outs[sl][1] = out1; v->outs[sl][2] = out2;
        v->magic = magic; v->check = ~seq ^ (unsigned)magic;
        v->seq = seq;
        s_slot = (unsigned)sl; s_seqv = seq;
        __threadfence();
    }
    __syncthreads();
    cudaTriggerProgrammaticLaunchCompletion();           // K2 may be scheduled: its blocks wait for begin_seq below
    int32_t *counters = reinterpret_cast<int32_t *>(S.base + (size_t)s_slot * S.stride);
    for (int i = threadIdx.x; i < 3 * lists + SLOT_BEGIN_SEQ; i += blockDim.x) counters[i] = 0;       // counters, k2_done
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) st_release_u32(reinterpret_cast<unsigned *>(counters) + 3 * lists + SLOT_BEGIN_SEQ, s_seqv);
}
__device__ __forceinline__ bool spin_until_equal(const unsigned *p, const unsigned target)
{
    const long long t0 = clock64();
    while (ld_acquire_u32(p) != target) {
        if (clock64() - t0 > (1ll << 33)) return false;
        __nanosleep(32);
    }
    return true;
}
// K2 side of the flags: wait until k_detect_begin has cleared this call's slot (thread 0; callers follow with a barrier), and count
// the block in once its keys and counters are written
__device__ __forceinline__ void k2_wait_slot_ready(const int32_t *counters, const int lists, const unsigned seq, DetectCtl *ctl)
{
    if (threadIdx.x == 0 && !spin_until_equal(reinterpret_cast<const unsigned *>(counters) + 3 * lists + SLOT_BEGIN_SEQ, seq)) {
        atomicOr(&ctl->error, FDT_STATUS_TIMEOUT_LOCAL); __trap();
    }
}
__device__ __forceinline__ void k2_block_done(int32_t *counters, const int lists)
{
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(counters + 3 * lists + SLOT_K2_DONE, 1);
}
// slot of the call this kernel belongs to, read by every K2 / k_sort_nms CTA BEFORE it lets its dependents be scheduled: the
// next call's k_detect_begin (which advances seq) cannot start until every CTA of this grid has triggered.
__device__ __forceinline__ unsigned detect_call_seq(const DetectSlots &S, unsigned *s_seq)
{
    if (threadIdx.x == 0) *s_seq = *reinterpret_cast<volatile unsigned *>(&S.ctl->seq);
    __syncthreads();
    return *s_seq;
}

// K2 for head maps (fdt_detect_heads): max-in-out + softmax + threshold + compaction.  The exact softmax costs an fp64 exp,
// so a block first screens its tile with the logit gap alone (pos - neg > logit(thr) - margin: a superset of the
// candidates, ~1/4 of the priors on the headline workload) while parking the logits in shared memory, lists the survivors
// densely, and only those get the exact score, the exact `score > thr` test and a key.  One global atomic per block, as in K2.
// 9 priors per thread: 15 tiles per 640x640 image, so that B = 64 is a single wave at 7 blocks per SM.
constexpr int K2H_PER_THREAD = 9;
constexpr int K2H_TILE = K2_THREADS * K2H_PER_THREAD;
template <int F>
__global__ void __launch_bounds__(K2_THREADS, 7)
k_heads_threshold_compact(const HeadLevels hl, const int64_t N, const float thr, const float dcut,
                          const DetectSlots S, long long *prof)
{
    unsigned long long gt0 = 0;
    if (prof && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0));
    __shared__ unsigned s_seq;
    const unsigned my_seq = detect_call_seq(S, &s_seq);
    char *slot = S.base + (size_t)(my_seq % (unsigned)S.depth) * S.stride;
    cudaTriggerProgrammaticLaunchCompletion();
    int32_t *__restrict__ counters = reinterpret_cast<int32_t *>(slot);
    uint64_t *__restrict__ keys = reinterpret_cast<uint64_t *>(slot + S.keys_off);
    const int b = blockIdx.y, lists = gridDim.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t base = (int64_t)blockIdx.x * K2H_TILE;
    __shared__ int s_warp[K2_THREADS / 32];
    __shared__ unsigned s_wmax[K2_THREADS / 32], s_wminv[K2_THREADS / 32];
    __shared__ int s_base, s_total;
    __shared__ uint16_t s_i[K2H_TILE];                   // tile-local indices of the screened priors, dense
    __shared__ unsigned long long s_x[K2H_TILE];         // (neg, pos) logits per tile slot; then the key of a candidate (0: rejected)

    // ---- screen
    unsigned bal[K2H_PER_THREAD];
    int wtotal = 0;
#pragma unroll
    for (int u = 0; u < K2H_PER_THREAD; ++u) {
        const int64_t p = base + u * K2_THREADS + tid;
        bool maybe = false;
        if (p < N) {
            const float2 lg = head_logits<F>(hl, b, (int)p);
            maybe = (lg.y - lg.x) > dcut;
            s_x[u * K2_THREADS + tid] = ((unsigned long long)__float_as_uint(lg.y) << 32) | __float_as_uint(lg.x);
        }
        bal[u] = __ballot_sync(0xffffffffu, maybe);
        wtotal += __popc(bal[u]);
    }
    if (lane == 0) s_warp[warp] = wtotal;
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
#pragma unroll
        for (int w = 0; w < K2_THREADS / 32; ++w) { const int c = s_warp[w]; s_warp[w] = tot; tot += c; }
        s_total = tot;
    }
    __syncthreads();
    {
        int off = s_warp[warp];
#pragma unroll
        for (int u = 0; u < K2H_PER_THREAD; ++u) {
            if ((bal[u] >> lane) & 1u) s_i[off + __popc(bal[u] & ((1u << lane) - 1u))] = (uint16_t)(u * K2_THREADS + tid);
            off += __popc(bal[u]);
        }
    }
    __syncthreads();
    // ---- exact score of the screened priors (dense lanes); each listed slot belongs to exactly one entry
    const int M = s_total;
    int mine = 0;
    unsigned kmx = 0u, kmnv = 0u;
    for (int e = tid; e < M; e += K2_THREADS) {
        const int sl = s_i[e];
        const unsigned long long x = s_x[sl];
        const float sc = softmax2(make_float2(__uint_as_float((unsigned)x), __uint_as_float((unsigned)(x >> 32)))).y;
        unsigned long long key = 0ull;
        if (sc > thr) {                                              // detection.py:64 strict gt
            const unsigned kk = fdt_float_key(sc);
            key = ((unsigned long long)kk << 32) | (unsigned)(base + sl);
            kmx = max(kmx, kk); kmnv = max(kmnv, ~kk);
            ++mine;
        }
        s_x[sl] = key;                                               // a key is never 0: its score half has the sign bit set
    }
    // ---- block-exclusive scan of the per-thread candidate counts, one atomic, scatter
    int inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
    kmx = __reduce_max_sync(0xffffffffu, kmx); kmnv = __reduce_max_sync(0xffffffffu, kmnv);
    __syncthreads();                                                 // s_warp (screen offsets) is free again
    if (lane == 31) s_warp[warp] = inc;
    if (lane == 0) { s_wmax[warp] = kmx; s_wminv[warp] = kmnv; }
    k2_wait_slot_ready(counters, lists, my_seq, S.ctl);              // k_detect_begin has cleared the slot
    __syncthreads();
    if (tid == 0) {
        int tot = 0;
        unsigned bmx = 0u, bmnv = 0u;
#pragma unroll
        for (int w = 0; w < K2_THREADS / 32; ++w) {
            const int c = s_warp[w]; s_warp[w] = tot; tot += c;
            bmx = max(bmx, s_wmax[w]); bmnv = max(bmnv, s_wminv[w]);
        }
        s_base = tot ? atomicAdd(&counters[b], tot) : 0;
        if (tot) {
            atomicMax(reinterpret_cast<unsigned *>(counters) + lists + b, bmx);
            atomicMax(reinterpret_cast<unsigned *>(counters) + 2 * lists + b, bmnv);
        }
    }
    __syncthreads();
    {
        uint64_t *kl = keys + (int64_t)b * N + s_base + s_warp[warp] + (inc - mine);
        for (int e = tid; e < M; e += K2_THREADS) {
            const unsigned long long key = s_x[s_i[e]];
            if (key) *kl++ = key;
        }
    }
    k2_block_done(counters, lists);
    if (prof && threadIdx.x == 0) {
        unsigned long long gt1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
        atomicMin((unsigned long long *)&prof[44], gt0); atomicMax((unsigned long long *)&prof[45], gt1);
    }
}

// score of prior i, class cl, of a 16-bit (bf16 / fp16) conf[B,N,C], widened to fp32 (exact); row0 = element (b, 0, 0).  pair: C == 2 and
// row0 4-byte aligned, so the (background, face) pair of a prior is one 32-bit word whose high half is the face score -- bf16 widens
// with one AND.
__device__ __forceinline__ float conf16_score(const unsigned short *row0, const int64_t i, const int C, const int cl, const int dtype,
                                              const bool pair)
{
    if (pair) {
        const unsigned w = __ldg(reinterpret_cast<const unsigned *>(row0) + i);
        return dtype == FDT_DTYPE_BF16 ? __uint_as_float(w & 0xffff0000u) : __half2float(__ushort_as_half((unsigned short)(w >> 16)));
    }
    return head_widen16(__ldg(row0 + i * C + cl), dtype);
}

// SRC 0: conf[B,N,C] with C > 2; 1: conf[B,N,2]; 2: 16-bit conf[B,N,C] of element type hl.dtype (hl.vec bit 0: conf16_score's pair)
#ifndef FDT_K2_MINBLOCKS
#define FDT_K2_MINBLOCKS 6
#endif
template <int SRC>
__global__ void __launch_bounds__(K2_THREADS, FDT_K2_MINBLOCKS)
k_threshold_compact(const float *__restrict__ conf, const HeadLevels hl, int64_t N, int C, float thr,
                    const DetectSlots S, long long *prof)
{
    unsigned long long gt0 = 0;
    if (prof && threadIdx.x == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0));
    const int b = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t base = (int64_t)blockIdx.x * K2_TILE;
    const float *cb = conf + (int64_t)b * N * C;
    __shared__ int s_warp[K2_THREADS / 32];
    __shared__ unsigned s_wmax[K2_THREADS / 32], s_wminv[K2_THREADS / 32];
    __shared__ int s_base;
    __shared__ unsigned s_seq;
    const int lists = gridDim.y * (C - 1);
    int32_t *__restrict__ counters = nullptr;
    uint64_t *__restrict__ keys = nullptr;
    unsigned my_seq = 0;

    for (int cl = 1; cl < C; ++cl) {
        float sc[K2_PER_THREAD];
        unsigned bal[K2_PER_THREAD];
        int wtotal = 0;
        unsigned kmx = 0u, kmnv = 0u;                    // max key and max ~key (= ~min key) of this thread's candidates
        if constexpr (SRC == 2) {
            // the dtype / pair choice is uniform: taken once per tile, not per prior (a branch per load cost a third of this kernel)
            const unsigned short *c16 = reinterpret_cast<const unsigned short *>(conf) + (int64_t)b * N * C;
            const bool bf = hl.dtype == FDT_DTYPE_BF16;
            if (hl.vec & 1u) {
#pragma unroll
                for (int u = 0; u < K2_PER_THREAD; ++u) {
                    const int64_t p = base + u * K2_THREADS + tid;
                    const unsigned w = p < N ? __ldg(reinterpret_cast<const unsigned *>(c16) + p) : 0u;
                    sc[u] = bf ? __uint_as_float(w & 0xffff0000u) : __half2float(__ushort_as_half((unsigned short)(w >> 16)));
                }
            } else {
#pragma unroll
                for (int u = 0; u < K2_PER_THREAD; ++u) {
                    const int64_t p = base + u * K2_THREADS + tid;
                    sc[u] = p < N ? head_widen16(__ldg(c16 + p * C + cl), hl.dtype) : 0.0f;
                }
            }
        } else {
#pragma unroll
        for (int u = 0; u < K2_PER_THREAD; ++u) {        // the tile's loads are in flight before anything below waits
            const int64_t p = base + u * K2_THREADS + tid;
            float s = 0.0f;
            if (p < N) {
                if (SRC == 1) s = __ldg(reinterpret_cast<const float2 *>(cb) + p).y;
                else s = __ldg(cb + p * C + cl);
            }
            sc[u] = s;
        }
        }
        if (cl == 1) {
            my_seq = detect_call_seq(S, &s_seq);
            char *slot = S.base + (size_t)(my_seq % (unsigned)S.depth) * S.stride;
            counters = reinterpret_cast<int32_t *>(slot);
            keys = reinterpret_cast<uint64_t *>(slot + S.keys_off);
            // programmatic dependent launch: let k_sort_nms be scheduled while this grid drains (it waits for our completion itself)
            cudaTriggerProgrammaticLaunchCompletion();
        }
#pragma unroll
        for (int u = 0; u < K2_PER_THREAD; ++u) {
            const int64_t p = base + u * K2_THREADS + tid;
            const bool in = p < N;
            const float s = sc[u];
            const bool cand = in && s > thr;                         // detection.py:64 strict gt
            bal[u] = __ballot_sync(0xffffffffu, cand);
            wtotal += __popc(bal[u]);
            if (cand) {
                const unsigned kk = fdt_float_key(s); kmx = max(kmx, kk); kmnv = max(kmnv, ~kk);
            }
        }
        kmx = __reduce_max_sync(0xffffffffu, kmx); kmnv = __reduce_max_sync(0xffffffffu, kmnv);
        if (lane == 0) { s_warp[warp] = wtotal; s_wmax[warp] = kmx; s_wminv[warp] = kmnv; }
        if (cl == 1) k2_wait_slot_ready(counters, lists, my_seq, S.ctl);    // k_detect_begin has cleared the slot (the conf loads were issued before the wait)
        __syncthreads();
        const int list = b * (C - 1) + (cl - 1);
        if (tid == 0) {
            int tot = 0;
            unsigned bmx = 0u, bmnv = 0u;
#pragma unroll
            for (int w = 0; w < K2_THREADS / 32; ++w) {
                int c = s_warp[w]; s_warp[w] = tot; tot += c;
                bmx = max(bmx, s_wmax[w]); bmnv = max(bmnv, s_wminv[w]);
            }
            s_base = tot ? atomicAdd(&counters[list], tot) : 0;
            if (tot) {           // score range of the list for k_sort_nms' bucket map: counters[lists + list] = max key, [2 lists + list] = ~min key
                atomicMax(reinterpret_cast<unsigned *>(counters) + lists + list, bmx);
                atomicMax(reinterpret_cast<unsigned *>(counters) + 2 * lists + list, bmnv);
            }
        }
        __syncthreads();
        int off = s_base + s_warp[warp];
        uint64_t *kl = keys + (int64_t)list * N;
#pragma unroll
        for (int u = 0; u < K2_PER_THREAD; ++u) {
            if ((bal[u] >> lane) & 1u) {
                int64_t p = base + u * K2_THREADS + tid;
                kl[off + __popc(bal[u] & ((1u << lane) - 1u))] = ((uint64_t)fdt_float_key(sc[u]) << 32) | (uint32_t)p;
            }
            off += __popc(bal[u]);
        }
        __syncthreads();
    }
    k2_block_done(counters, lists);
    if (prof && threadIdx.x == 0) {      // diagnostics (FDT_K3_PROFILE=1): first block start / last block end on the global timer
        unsigned long long gt1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
        atomicMin((unsigned long long *)&prof[44], gt0); atomicMax((unsigned long long *)&prof[45], gt1);
    }
}

__global__ void k_build_keys(const float *__restrict__ scores, int64_t n, uint64_t *__restrict__ keys)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = ((uint64_t)fdt_float_key(scores[i]) << 32) | (uint32_t)i;
}

// ------------------------------------------------------------------------------------------- K3
// Shared-memory layout of k_sort_nms.  Everything whose size does not depend on the call sits at a COMPILE-TIME offset (the
// addresses fold into the LDS/STS immediates; with run-time offsets ~15 % of the kernel's instructions were address
// arithmetic); the key array and the kept-box arrays follow at run-time offsets.
constexpr int up16c(int x) { return (x + 15) / 16 * 16; }
constexpr int SM_HIST = 0;                                          // sort: fill[NB] | start[NB]
constexpr int SM_SEGS = SM_HIST + 2 * NB * 4;                       // [32 warps][SEG_SLOTS * 32] phase-B row segments
constexpr int SM_SBOX = SM_SEGS + K3_THREADS * SEG_SLOTS * 4;       // [WIN] window boxes in cell (CSR) order
constexpr int SM_SAREA = SM_SBOX + WIN * 16;
constexpr int SM_SDEPS = SM_SAREA + WIN * 4;                        // [WIN][DEPS] earlier suppressors per window candidate
constexpr int SM_SNDEP = SM_SDEPS + WIN * DEPS * 2;                 // [WIN] how many were found (may exceed DEPS)
constexpr int SM_WSTART = SM_SNDEP + WIN * 4;                       // [NCELLX + 1] CSR over the window
constexpr int SM_KSTART = SM_WSTART + up16c((NCELLX + 1) * 4);      // [NCELLX + 1] CSR over the kept boxes
constexpr int SM_KCUR = SM_KSTART + up16c((NCELLX + 1) * 4);        // [NCELLX + 1] fill cursors
constexpr int SM_WPOS = SM_KCUR + up16c((NCELLX + 1) * 4);          // [WIN] CSR position of each window candidate
constexpr int SM_WCELL = SM_WPOS + WIN * 2;                         // [WIN] grid cell of each window candidate
constexpr int SM_WITEMS = SM_WCELL + WIN * 2;                       // [WIN] window candidates sorted by cell
constexpr int SM_STATUS = SM_WITEMS + WIN * 2;                      // [WIN] 0 undecided, 1 kept, 2 dead
constexpr int SM_KEYS = SM_STATUS + WIN;                            // [key_cap] bucket-ordered, then sorted per window
struct SmemPlan {
    int key_cap;                                   // entries of the key array (power of two >= kcap + 64)
    int off_kitems, off_kcell;
    int off_kbox, off_karea, off_kkey;             // < 0: kept arrays live in the global workspace
    int total;
};

struct SortNmsParams {
    DetectSlots S;              // S.ctl != null: keys / counters / kept rows come from the call's workspace slot (sequenced calls)
    const uint64_t *keys;       // [lists, key_stride]            (S.ctl == null)
    const int32_t *counters;    // [3][lists] (MODE_DETECT): candidate count, max key, ~min key; null: P.n candidates   (S.ctl == null)
    int use_counters;           // S.ctl != null: the slot's counters hold the candidate count
    int k2_blocks;              // S.ctl != null: blocks of the call's K2 grid (k_sort_nms waits until all have counted themselves in)
    int64_t key_stride;
    const float *conf;          // [B,N,C]  (FUSED: the kernel thresholds its own list)
    float conf_thresh;
    const float *loc;           // [B,N,4]  (MODE_DETECT); null: gather the rows from the head maps `hl`
    int loc_prefetch;           // loc is device memory: prefetch the rows of the first window into L2 during the scatter
    const float *priors;        // [N,4]    (MODE_DETECT)
    const float *boxes;         // [n,4]    (MODE_NMS)
    int64_t N;
    int C;
    int nms_top_k;              // candidates that enter NMS
    int max_keep;               // stop after this many kept
    int top_k;                  // output rows (MODE_DETECT)
    float nms_thresh, v0, v1;
    float *out;                 // [B,C,top_k,5]
    int32_t *counts;            // [B,C] or null
    int64_t *kept_prior;        // [B,C,top_k] or null
    int64_t *keep;              // [n] (MODE_NMS)
    int64_t *count_out;         // [1] (MODE_NMS)
    int64_t n;                  // MODE_NMS list length
    int variant;                // MODE_NMS: FDT_NMS_* flags (0 = layers/box_utils.nms)
    const unsigned long long *peer_out;   // device array of n_peers output base pointers (this GPU's and its NVLink peers'), or null
    int n_peers;
    int64_t img_offset;         // image index of this rank's first image inside the peers' gathered blocks
    // signalled gather to a root rank (fdt_detect_sort_nms_gather_signal): no barrier launch
    const unsigned long long *peer_sig;   // device array of `world` pointers to every rank's uint32 signal[world + 1] (or null)
    int world, my_rank, root;
    unsigned epoch;             // call counter, the same on every rank, >= 1
    int ring;                   // gathered blocks that alternate (epoch % ring)
    int kept_global;            // kept arrays live in global memory (per list stride max_keep): sm.off_kbox < 0
    float4 *g_kbox;             // (S.ctl == null; else carved from the slot)
    float *g_karea;
    uint64_t *g_kkey;
    SmemPlan sm;
    HeadLevels hl;              // per-level NCHW loc maps (MODE_DETECT with loc == null)
    long long *prof;            // diagnostics: per-phase clock64 of CTA 0 (null unless FDT_K3_PROFILE=1 / 2)
    int prof_all;               // FDT_K3_PROFILE=2: every CTA of every launch ADDS its phase clocks (steady-state averages; [30] counts CTAs)
    int conf_dtype;             // FUSED with HT = 1: FDT_DTYPE_* of `conf` (the pointer then addresses elements of that type)
    int conf_pair;              // ... 16-bit, C == 2, 4-byte aligned: conf16_score's pair load
};

// "i (kept, higher score) suppresses j": box_utils.py:322-339, union = (area_j - inter) + area_i,
// survive iff IoU < overlap, so NaN suppresses.
__device__ __forceinline__ bool fdt_suppresses(const float4 bi, const float area_i, const float4 bj, const float area_j,
                                               const float thr)
{
    float xx1 = fmaxf(bj.x, bi.x), yy1 = fmaxf(bj.y, bi.y);
    float xx2 = fminf(bj.z, bi.z), yy2 = fminf(bj.w, bi.w);
    float w = fmaxf(xx2 - xx1, 0.0f), h = fmaxf(yy2 - yy1, 0.0f);
    float inter = w * h;
    float uni = (area_j - inter) + area_i;
    if (inter > 0.0f) return !(inter / uni < thr);
    return (!(uni > 0.0f) && !(uni < 0.0f)) || !(0.0f < thr);      // 0/uni is NaN iff uni is 0 or NaN, else 0 (survives iff 0 < thr)
}

// Same predicate, division only when the quotient is within 2^-20 of thr: with p = fl(thr * uni) and uni > 0,
// inter < p (1 - 2^-20) implies fl(inter / uni) < thr and inter > p (1 + 2^-20) implies fl(inter / uni) >= thr (the rounding
// errors of p and of the scaled bounds are <= 2^-23 each).  NaNs and uni <= 0 fall through to the exact form.
__device__ __forceinline__ bool fdt_suppresses_fast(const float4 bi, const float area_i, const float4 bj, const float area_j,
                                                    const float thr)
{
    float xx1 = fmaxf(bj.x, bi.x), yy1 = fmaxf(bj.y, bi.y);
    float xx2 = fminf(bj.z, bi.z), yy2 = fminf(bj.w, bi.w);
    float w = fmaxf(xx2 - xx1, 0.0f), h = fmaxf(yy2 - yy1, 0.0f);
    float inter = w * h;
    float uni = (area_j - inter) + area_i;
    const float p = thr * uni;
    if (p > 1e-30f) {                                  // normal range (no underflow in p); false for NaN and uni <= 0
        if (inter < p * 0.99999905f) return false;
        if (inter > p * 1.00000095f) return true;
    }
    if (inter > 0.0f) return !(inter / uni < thr);
    return (!(uni > 0.0f) && !(uni < 0.0f)) || !(0.0f < thr);
}


// ---- sibling NMS implementations of the reference (SURVEY 8f rank 3), selected by FDT_NMS_* flags (include/fdt_b200.h):
//   FACEBOX/encoderl.py:218-266 nms_np and MTCNN/mtcnn/core/utils.py:62-113 nms: union = (area_i + area_j) - inter  [SUMFIRST],
//     mode "Minimum": inter / min(area_i, area_j)  [MINIMUM], survive iff ovr < thr;
//   MTCNN/mtcnn/core/nms.py:4-40 torch_nms: widths, heights and areas with "+ 1"  [PLUS1], survive iff ovr <= thr  [LE];
//   FACEBOX/encoderl.py:268-306 DataEncoder.nms: SUMFIRST | LE.
// i = the kept (higher-score) box, j = the candidate.  numpy / torch min-max propagate NaN; here a NaN coordinate always
// makes the box's area NaN, which reaches the quotient through the denominator, so the plain fminf/fmaxf below suffice
// (MINIMUM takes the NaN-propagating minimum explicitly).
__device__ __forceinline__ float box_area_v(const float4 b, const int variant)
{
    if (variant & FDT_NMS_PLUS1) return ((b.z - b.x) + 1.0f) * ((b.w - b.y) + 1.0f);
    return (b.z - b.x) * (b.w - b.y);
}
__device__ __forceinline__ bool fdt_suppresses_v(const float4 bi, const float area_i, const float4 bj, const float area_j,
                                                 const float thr, const int variant)
{
    const float xx1 = fmaxf(bi.x, bj.x), yy1 = fmaxf(bi.y, bj.y);
    const float xx2 = fminf(bi.z, bj.z), yy2 = fminf(bi.w, bj.w);
    float dw = xx2 - xx1, dh = yy2 - yy1;
    if (variant & FDT_NMS_PLUS1) { dw += 1.0f; dh += 1.0f; }
    const float inter = fmaxf(0.0f, dw) * fmaxf(0.0f, dh);
    float den;
    if (variant & FDT_NMS_MINIMUM) den = (area_i != area_i || area_j != area_j) ? NAN : fminf(area_i, area_j);
    else if (variant & FDT_NMS_SUMFIRST) den = (area_i + area_j) - inter;
    else den = (area_j - inter) + area_i;
    const float ovr = inter / den;
    return (variant & FDT_NMS_LE) ? !(ovr <= thr) : !(ovr < thr);
}
// the box the spatial grid sees: PLUS1 measures [x1, x2 + 1] x [y1, y2 + 1]
__device__ __forceinline__ float4 grid_box(const float4 b, const int variant)
{
    if (variant & FDT_NMS_PLUS1) return make_float4(b.x, b.y, b.z + 1.0f, b.w + 1.0f);
    return b;
}
// Boxes the spatial grid may index: finite, not inverted, 0 < area < inf.  For two such boxes inter <= min(area_i,
// area_j) holds exactly in fp32 (rounding is monotone), so union >= area_i > 0 and IoU is a finite number bounded by
// the ratio of the longer sides; they can only suppress each other if they intersect.  Everything else (NaN/inf
// coordinates, inverted or zero-area boxes -- 0/0 = NaN suppresses at ANY distance, box_utils.py:337-339) lives in a
// pseudo-cell that every query scans and is itself tested against everything.
__device__ __forceinline__ bool box_regular(const float4 b)
{
    const float a = (b.z - b.x) * (b.w - b.y);
    return (b.z >= b.x) && (b.w >= b.y) && fabsf(b.x) < INFINITY && fabsf(b.y) < INFINITY && fabsf(b.z) < INFINITY &&
           fabsf(b.w) < INFINITY && a > 0.0f && a < INFINITY;
}

// Multi-level uniform grid over the extent of the first window's boxes, stored CSR-style (items sorted by cell).
// Level l has (32 >> l)^2 cells of size c_l = extent / (32 >> l).  A regular box lives at the smallest level whose
// cell is at least as long as the box's longer side, in the cell of its min corner (clamped: the cell map is monotone
// in the coordinate, which is all the proof below needs).  A box j can only reach IoU >= thr with boxes whose longer
// side is within a factor thr of its own (IoU <= side ratio), so a query visits only the levels that can hold such
// boxes, and at level l' only rows/columns [cell(x1_j - (1.01 - q) c_l'), cell(x2_j - q w_j)], q = 0.97 min(thr, 1):
// IoU <= ox / max(w_i, w_j) (ox = overlap along x: inter <= ox min(h) and union >= each area), so reaching thr needs
// ox >= thr max(w_i, w_j); then x1_i <= x2_j - ox <= x2_j - thr w_j and x1_i >= x1_j - (w_i - ox) >= x1_j - (1 - thr) c_l'.
// The 3 % margin on thr and 1 % on c cover the fp32 rounding of the IoU, of the widths and of these bounds (plus an
// absolute slack of a few ulps of the coordinates for boxes that are tiny relative to their position); same along y.
// Cells of one row are consecutive in the CSR array, so each visited row is ONE contiguous item segment.
struct GridGeom {
    float x0, y0;          // origin = min corner
    float inv0;            // cells per unit length at level 0 (32 / extent)
    float c0;              // cell size at level 0
    int ok;                // 0: degenerate extent -> every box sits in the pseudo-cell
};
__device__ __forceinline__ int grid_off(int lev) { return lev == 0 ? 0 : lev == 1 ? 1024 : lev == 2 ? 1280 : lev == 3 ? 1344 : lev == 4 ? 1360 : 1364; }
__device__ __forceinline__ int cell_of(float x, float origin, float inv, int G)
{
    int c = __float2int_rd((x - origin) * inv);
    return max(0, min(G - 1, c));
}
__device__ __forceinline__ int reg_cell(const GridGeom &gg, const float4 bx, const float side, const bool valid)
{
    if (!valid) return -1;
    if (!gg.ok || !box_regular(bx)) return BIGCELL;
    float c = gg.c0;
    int lev = 0;
#pragma unroll
    for (; lev < NLEV; ++lev, c *= 2.0f) if (side <= c) break;
    if (lev >= NLEV) return BIGCELL;
    const int G = 32 >> lev;
    const float inv = gg.inv0 / (float)(1 << lev);
    return grid_off(lev) + cell_of(bx.y, gg.y0, inv, G) * G + cell_of(bx.x, gg.x0, inv, G);
}
// visit(t) is called with CSR positions t (item = items[t]) and returns true to stop; returns true iff the visitor stopped.
// `start` has NCELLX + 1 entries.
// query ranges before the per-level pad: (x1_j - slack, y1_j - slack, x2_j - q w_j + slack, y2_j - q h_j + slack)
__device__ __forceinline__ float4 query_range(const float4 bj, const float tq)
{
    const float sx = 2e-6f * fmaxf(fabsf(bj.x), fabsf(bj.z)), sy = 2e-6f * fmaxf(fabsf(bj.y), fabsf(bj.w));
    return make_float4(bj.x - sx, bj.y - sy, (bj.z - tq * (bj.z - bj.x)) + sx, (bj.w - tq * (bj.w - bj.y)) + sy);
}
template <typename F>
__device__ __forceinline__ bool csr_query(const GridGeom &gg, const int *start, const float4 bj, const float sj,
                                          const float prune, const float tq, F &&visit)
{
    float c = gg.c0, inv = gg.inv0, cprev = 0.0f;
    int G = 32, base = 0;
    const float4 qr = query_range(bj, tq);
    const float padf = 1.01f - tq;
#pragma unroll 1
    for (int lev = 0; lev < NLEV; ++lev, cprev = c, c *= 2.0f, inv *= 0.5f, base += G * G, G >>= 1) {
        if (c < prune * sj) continue;                    // every box of this level is too small to reach thr
        if (cprev * prune > sj) break;                   // this and all coarser levels only hold boxes too large
        if (start[base + G * G] == start[base]) continue;
        const float pad = padf * c;
        const int cx0 = cell_of(qr.x - pad, gg.x0, inv, G), cx1 = cell_of(qr.z, gg.x0, inv, G);
        const int cy0 = cell_of(qr.y - pad, gg.y0, inv, G), cy1 = cell_of(qr.w, gg.y0, inv, G);
        for (int cy = cy0; cy <= cy1; ++cy) {
            const int t1 = start[base + cy * G + cx1 + 1];
            for (int t = start[base + cy * G + cx0]; t < t1; ++t)
                if (visit(t)) return true;
        }
    }
    const int t1 = start[BIGCELL + 1];
    for (int t = start[BIGCELL]; t < t1; ++t)
        if (visit(t)) return true;
    return false;
}

// Forward half of csr_query for the window grid, as row segments: emits the non-empty CSR ranges [t0, t1) that lie AFTER
// `own_t` (own level: the rest of the own row and the rows below; coarser levels: everything in range; finer levels:
// nothing).  Every pair of window candidates that csr_query would find from either side is found by exactly one of the two
// forward queries (the one with the lower CSR position), because each side's full query finds the other.
// `part` of `nparts` (1, 2 or 4 lanes share a candidate): the lanes take grid rows round-robin; part 0 takes the pseudo-cell.
template <typename F>
__device__ __forceinline__ void csr_segments_forward(const GridGeom &gg, const int *start, const float4 bj, const float sj,
                                                     const float prune, const float tq, const int own_cell, const int own_t, const int part, const int nparts, F &&emit)
{
    float c = gg.c0, inv = gg.inv0, cprev = 0.0f;
    int G = 32, base = 0;
    const float4 qr = query_range(bj, tq);
    const float padf = 1.01f - tq;
#pragma unroll 1
    for (int lev = 0; lev < NLEV; ++lev, cprev = c, c *= 2.0f, inv *= 0.5f, base += G * G, G >>= 1) {
        if (own_cell >= base + G * G) continue;          // finer than the own level: those candidates look forward to us
        if (c < prune * sj) continue;
        if (cprev * prune > sj) break;
        if (start[base + G * G] == start[base]) continue;
        const float pad = padf * c;
        const int cx0 = cell_of(qr.x - pad, gg.x0, inv, G), cx1 = cell_of(qr.z, gg.x0, inv, G);
        int cy0 = cell_of(qr.y - pad, gg.y0, inv, G);
        const int cy1 = cell_of(qr.w, gg.y0, inv, G);
        const bool own_level = own_cell >= base;         // (own_cell < base + G*G holds here)
        const int own_cy = own_level ? (own_cell - base) >> (5 - lev) : -1;      // G = 32 >> lev
        if (own_level) cy0 = max(cy0, own_cy);
        for (int cy = cy0 + part; cy <= cy1; cy += nparts) {
            const int t1 = start[base + cy * G + cx1 + 1];
            int t = start[base + cy * G + cx0];
            if (cy == own_cy) t = max(t, own_t + 1);
            if (t < t1) emit(t, t1);
        }
    }
    if (part == 0) {
        const int t1 = start[BIGCELL + 1];
        const int t = max(start[BIGCELL], own_t + 1);
        if (t < t1) emit(t, t1);
    }
}

// clock64 that cannot be read before a preceding barrier has released: BAR.SYNC is deferred-blocking, the shared-memory
// load below is the first instruction that really waits for it, and the clock read takes the loaded value as an input.
__device__ __forceinline__ long long fdt_clock_after(const int *smem_word)
{
    int v = *reinterpret_cast<const volatile int *>(smem_word);
    long long t;
    asm volatile("{ .reg .b32 z; and.b32 z, %1, 0; mov.u64 %0, %%clock64; }" : "=l"(t) : "r"(v) : "memory");
    return t;
}

// exclusive prefix sum of one int per thread over the 1024-thread block; `total` = block sum
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
        int w = s_warp[lane], winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += n; }
        s_warp[lane] = winc - w;
        if (lane == 31) s_warp[32] = winc;
    }
    __syncthreads();
    total = s_warp[32];
    return inc - v + s_warp[warp];
}
// in-place inclusive scan of a[0 .. NCELLX] (a[0] stays 0): counts at a[c + 1] become CSR starts
__device__ __forceinline__ void csr_scan(int *a, int *s_warp)
{
    const int i0 = 2 * threadIdx.x, i1 = i0 + 1;
    const int v0 = i0 <= NCELLX ? a[i0] : 0, v1 = i1 <= NCELLX ? a[i1] : 0;
    int tot;
    const int ex = block_excl_scan(v0 + v1, s_warp, tot);
    if (i0 <= NCELLX) a[i0] = ex + v0;
    if (i1 <= NCELLX) a[i1] = ex + v0 + v1;
    __syncthreads();
}

// CL = CTAs per list: 1, or 2 as a thread-block cluster when the batch leaves SMs idle.  With CL = 2 both CTAs run every stage
// redundantly and deterministically (identical shared-memory state) except phase B -- the dominant one -- whose candidates they
// split; the partial dependency lists are merged through distributed shared memory.
// FUSED (MODE_DETECT, CL = 1): no K2, no candidate keys in global memory -- the CTA thresholds its own list of `conf` itself:
// one pass for the bucket histogram (which also counts the candidates), one for the scatter (served by L2), the rare exact
// fallbacks re-scan the row.  With consecutive calls overlapping on the device what counts is SM time, not latency: the ~1,350
// SM-microseconds per B = 64 call that a separate K2 grid and the hand-over to this kernel cost shrink to the two row scans.
#ifndef FDT_K3_MAXREG
#define FDT_K3_MAXREG 64
#endif
#if FDT_K3_MAXREG < 64
#define K3_BOUNDS __maxnreg__(FDT_K3_MAXREG)
#else
#define K3_BOUNDS __launch_bounds__(K3_THREADS, 1)
#endif
// HT = 1: MODE_DETECT with the loc rows gathered from head maps other than fp32 dense NCHW (HEAD_ANY, heads.cuh): in the
// instantiations above their loads and widening would cost the 64-register kernel extra spill traffic.  A flat loc[B,N,4] of a
// 16-bit type is such a map (one level, hw = N, strides (4N, 1, 4)).  FUSED with HT = 1 is the fused kernel for flat inputs of which
// at least one is 16-bit: loc through its one-level map (any element type), conf of element type P.conf_dtype widened as it is read.
template <int MODE, int CL, bool FUSED, int HT = 0>
__global__ void K3_BOUNDS
k_sort_nms(const SortNmsParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ unsigned s_seq;
    // Sequenced call: which call of the workspace this is (hence its slot) must be read before the trigger below lets the NEXT
    // call's k_detect_begin be scheduled; block 0 also records that this call's k_sort_nms exists (see k_detect_begin).
    unsigned my_seq = 0;
    const uint64_t *keys_base = P.keys;
    const int32_t *counters = P.counters;
    int *ticket = nullptr;
    const int *slot_hdr = nullptr;
    char *slot_kept = nullptr;
    if (P.S.ctl) {
        my_seq = detect_call_seq(P.S, &s_seq);
        if (blockIdx.x == 0 && threadIdx.x == 0) { *reinterpret_cast<volatile unsigned *>(&P.S.ctl->k3s) = my_seq; __threadfence(); }
        // (tickets are indexed by seq & 3: calls s and s + 4 are never in flight together, k_detect_begin(s + 4) waits for done >= s)
        ticket = reinterpret_cast<int *>(&P.S.ctl->ticket[my_seq & (FDT_DETECT_MAX_DEPTH - 1)]);
        if (!FUSED || P.sm.off_kbox < 0) {                     // the fused kernel only needs its slot for spilled kept rows
            char *slot = P.S.base + (size_t)(my_seq % (unsigned)P.S.depth) * P.S.stride;
            keys_base = reinterpret_cast<const uint64_t *>(slot + P.S.keys_off);
            counters = P.use_counters ? reinterpret_cast<const int32_t *>(slot) : nullptr;
            slot_hdr = reinterpret_cast<const int *>(slot) + 3 * (int)(gridDim.x / CL);
            slot_kept = slot + P.S.kept_off;
        }
        if (MODE == MODE_DETECT && P.peer_sig && blockIdx.x == 0 && (P.root < 0 || P.root == P.my_rank) &&
            threadIdx.x < P.world && (int)threadIdx.x != P.my_rank) {
            // destination of a fused gather: "call `epoch` has begun here" -> the blocks of epochs <= epoch - 1 have been consumed
            unsigned *dst = reinterpret_cast<unsigned *>(P.peer_sig[threadIdx.x]) + P.world + P.my_rank;
            asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(dst), "r"(P.epoch) : "memory");
        }
    }
    // lets the NEXT Detect call's k_detect_begin / K2 be scheduled behind this grid: with a deep enough workspace ring they run
    // while this grid is still in NMS (see "call sequencing")
    cudaTriggerProgrammaticLaunchCompletion();
    uint64_t *skeys = reinterpret_cast<uint64_t *>(smem + SM_KEYS);
    int *s_hist = reinterpret_cast<int *>(smem + SM_HIST);
    int *s_start = s_hist + NB;
    uint16_t *wpos = reinterpret_cast<uint16_t *>(smem + SM_WPOS);
    uint32_t *segs = reinterpret_cast<uint32_t *>(smem + SM_SEGS);
    uint16_t *wcell = reinterpret_cast<uint16_t *>(smem + SM_WCELL);
    unsigned char *status = smem + SM_STATUS;
    uint16_t *witems = reinterpret_cast<uint16_t *>(smem + SM_WITEMS);
    int *wstart = reinterpret_cast<int *>(smem + SM_WSTART);
    float4 *sbox = reinterpret_cast<float4 *>(smem + SM_SBOX);
    float *sarea = reinterpret_cast<float *>(smem + SM_SAREA);
    uint16_t *sdeps = reinterpret_cast<uint16_t *>(smem + SM_SDEPS);
    int *sndep = reinterpret_cast<int *>(smem + SM_SNDEP);
    int *kstart = reinterpret_cast<int *>(smem + SM_KSTART);
    int *kcur = reinterpret_cast<int *>(smem + SM_KCUR);
    uint16_t *kitems = reinterpret_cast<uint16_t *>(smem + P.sm.off_kitems);     // [max_keep]
    uint16_t *kcell = reinterpret_cast<uint16_t *>(smem + P.sm.off_kcell);       // [max_keep]
    const int list = blockIdx.x / CL;
    const int crank = CL == 2 ? (int)(blockIdx.x & 1) : 0;     // cluster dims (2,1,1): rank = blockIdx.x % 2
    float4 *kbox; float *karea; uint64_t *kkey;
    if (P.sm.off_kbox >= 0) {
        kbox = reinterpret_cast<float4 *>(smem + P.sm.off_kbox);
        karea = reinterpret_cast<float *>(smem + P.sm.off_karea);
        kkey = reinterpret_cast<uint64_t *>(smem + P.sm.off_kkey);
    } else {
        // kept rows in global memory: [lists][max_keep] boxes | keys | areas, carved from the slot (or passed by fdt_nms)
        const size_t nl = gridDim.x / CL;
        float4 *gb = slot_kept ? reinterpret_cast<float4 *>(slot_kept) : P.g_kbox;
        uint64_t *gk = slot_kept ? reinterpret_cast<uint64_t *>(slot_kept + nl * (size_t)P.max_keep * 16) : P.g_kkey;
        float *ga = slot_kept ? reinterpret_cast<float *>(slot_kept + nl * (size_t)P.max_keep * 24) : P.g_karea;
        kbox = gb + (int64_t)list * P.max_keep; kkey = gk + (int64_t)list * P.max_keep; karea = ga + (int64_t)list * P.max_keep;
    }

    __shared__ int s_sel[3];
    __shared__ int s_placed, s_maxb, s_next;
    __shared__ unsigned s_kmin, s_kmax;
    __shared__ int s_hist8[256];
    __shared__ int s_warp[33];
    __shared__ unsigned s_ext[4];          // extent of the regular boxes as order-preserving keys

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = (MODE == MODE_DETECT) ? list / (P.C - 1) : 0;
    const int cl = (MODE == MODE_DETECT) ? 1 + list % (P.C - 1) : 0;
    const uint64_t *gkeys = keys_base + (int64_t)list * P.key_stride;

    // Output that does not depend on the producer kernel goes first: the all-zero background plane (detection.py:48, :63)
    // is written while k_threshold_compact still runs (programmatic dependent launch).
    // (Peer-gather launches skip it: the caller zeroes the gathered blocks once and nothing ever writes their background planes.)
    if (MODE == MODE_DETECT && crank == 0 && cl == 1 && P.n_peers == 0) {
        const int ndst = P.n_peers > 0 ? P.n_peers : 1;
        const int nq = (P.top_k * 5) >> 2;                       // whole float4s; planes are 16-byte aligned iff top_k * 5 % 4 == 0
        const bool vec = ((P.top_k * 5) & 3) == 0;
        for (int pr = 0; pr < ndst; ++pr) {
            float *base = P.n_peers > 0 ? reinterpret_cast<float *>(P.peer_out[pr]) + (P.img_offset * P.C) * (int64_t)P.top_k * 5 : P.out;
            float *o0 = base + ((int64_t)(b * P.C) * P.top_k) * 5;
            if (vec && ((uintptr_t)o0 & 15) == 0) for (int t = tid; t < nq; t += K3_THREADS) reinterpret_cast<float4 *>(o0)[t] = make_float4(0.f, 0.f, 0.f, 0.f);
            else for (int t = tid; t < P.top_k * 5; t += K3_THREADS) o0[t] = 0.0f;
        }
        if (P.kept_prior) {
            int64_t *kp = P.kept_prior + (int64_t)(b * P.C) * P.top_k;
            for (int r = tid; r < P.top_k; r += K3_THREADS) kp[r] = -1;
        }
        if (P.counts && tid == 0) P.counts[b * P.C] = 0;
    }
    if (FUSED) {
        // nothing to wait for: k_detect_begin lets this grid be scheduled only after its sequencing (which includes the full
        // dependency wait when the predecessor may be the producer of conf / loc) is done
    } else if (P.S.ctl) {
        // K2 of this call has written the slot: every one of its blocks has counted itself in (see "call sequencing")
        if (tid == 0) {
            const unsigned *hdr = reinterpret_cast<const unsigned *>(slot_hdr);
            // (begin_seq first: until k_detect_begin has cleared the slot, k2_done still holds what call seq - depth left there)
            if (!spin_until_equal(hdr + SLOT_BEGIN_SEQ, my_seq) || !spin_until_reached(hdr + SLOT_K2_DONE, (unsigned)P.k2_blocks)) {
                atomicOr(&P.S.ctl->error, FDT_STATUS_TIMEOUT_LOCAL); __trap();
            }
        }
        __syncthreads();
    } else {
        cudaGridDependencySynchronize();  // fdt_nms: behind k_build_keys; a no-op unless launched with programmatic stream serialization
    }
    int n_c = FUSED ? 0 : (counters ? __ldcg(counters + list) : (int)P.n);
    if (MODE == MODE_DETECT && n_c == 1) n_c = 0;            // detection.py:66-72: one candidate -> `continue`
    int k = min(n_c, P.nms_top_k);                           // box_utils.py:299 idx[-top_k:]   (FUSED: known after the first row scan)
    const bool prof = P.prof != nullptr && (blockIdx.x == 0 || P.prof_all) && tid == 0;
    const bool writer = crank == 0;                              // only one CTA of a cluster writes the results
    // Profiling state of thread 0 lives in shared memory: held in registers across the whole kernel, its clocks and per-phase
    // accumulators made ptxas spill under the 64-register cap in every build, profiled or not.
    __shared__ long long s_prof[10];                         // [0] last stamp, [1] CTA start clock, [2] CTA start globaltimer, [3 + q] phase q
    long long *const pacc = s_prof + 3;
    if (P.prof && tid == 0) {
        unsigned long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        s_prof[0] = s_prof[1] = clock64(); s_prof[2] = (long long)g;
        for (int q = 0; q < 7; ++q) pacc[q] = 0;
    }
#define K3_STAMP(slot) do { if (P.prof) __syncthreads(); if (prof) { long long now_ = fdt_clock_after(s_warp); atomicAdd((unsigned long long *)&P.prof[slot], (unsigned long long)(now_ - s_prof[0])); s_prof[0] = now_; } } while (0)
#define K3_ACC(slot) do { if (P.prof) __syncthreads(); if (prof) { long long now_ = fdt_clock_after(s_warp); pacc[slot] += now_ - s_prof[0]; s_prof[0] = now_; } } while (0)

    // =========================================================== stage 1: top-k selection by bucket (counting) sort
    // Monotone score -> bucket map; counting sort by bucket, descending; only buckets that can reach rank < k are
    // materialised (bucket-contiguous, unordered inside a bucket).  Exact order inside buckets is produced lazily per
    // NMS window.  Keys stay in registers across the three passes when the list has <= 8192 entries.
    bool presorted = false;
    int placed = 0;
    unsigned kmin = 0;
    float binv = 0.0f;
    auto bucket = [&](uint64_t key) -> int { return min(NB - 1, (int)((float)((unsigned)(key >> 32) - kmin) * binv)); };
    // FUSED: the candidates of this list are the priors i with conf[b, i, cl] > conf_thresh (detection.py:64, strict), read from the row
    const float *crow = FUSED ? P.conf + ((int64_t)b * P.N) * P.C + cl : nullptr;
    const float cthr = P.conf_thresh;
    const int n_scan = FUSED ? (int)P.N : n_c;               // entries a full pass looks at
    // FUSED: the windows usually stop long before nms_top_k (the headline keeps its 750 boxes within the first ~900 of 5,000 candidates),
    // so stage 1 selects and scatters the k_all = min(candidates, nms_top_k) best keys in chunks of at most two first windows.  When the
    // windows have consumed a chunk without reaching max_keep, the next chunk is selected the same way among the keys below `tmax`, the
    // last key processed, by a re-scan of the row in place (the queues are window arrays by then).  Chunks follow score order, so the
    // windows see exactly the sequence of the unchunked selection.  What the windows carry from one chunk to the next waits in shared
    // memory (`s_ck`), so that none of it occupies registers during stage 1.
    struct ChunkState {
        uint64_t tmax;                                       // only keys below it take part (later chunks)
        int chunk, k_all, done_k;                            // chunk number, min(candidates, nms_top_k), candidates of earlier chunks
        int nkept, rounds, sweeps, win_cap;
        GridGeom gg;
    };
    __shared__ ChunkState s_ck;
    if (tid == 0) {
        s_ck.tmax = ~0ull; s_ck.chunk = 0; s_ck.k_all = k; s_ck.done_k = 0;
        s_ck.nkept = 0; s_ck.rounds = 0; s_ck.sweeps = 0;
        // Window size.  Detect stops at max_keep kept boxes, so a window only needs the candidates that get it there: the first one takes
        // 1.2 x max_keep (+16) of them, later ones what the keep rate of the previous window predicts (+1/8 + 32) -- at least one whole
        // bucket more than the largest bucket of the range (BIG_BUCKET), at most WIN.  Windows are consumed in score order whatever their
        // size, so the result does not depend on it; a short window leaves warps idle in every phase of the round.
        s_ck.win_cap = MODE == MODE_DETECT ? min(WIN, max(BIG_BUCKET + 64, (P.max_keep * 6) / 5 + 16)) : WIN;
        s_ck.gg.ok = 0; s_ck.gg.x0 = s_ck.gg.y0 = s_ck.gg.inv0 = s_ck.gg.c0 = 0.0f;
    }
    int nkept_out = 0, rounds_out = 0, sweeps_out = 0;
    for (;;) {
    presorted = false;
    if (FUSED || k > 0) {
        constexpr int KREG = FUSED ? 1 : 8;
        const bool cached = !FUSED && n_c <= KREG * K3_THREADS;
        uint64_t kreg[KREG];
        if (cached) {
#pragma unroll
            for (int u = 0; u < KREG; ++u) { const int i = tid + u * K3_THREADS; kreg[u] = i < n_c ? __ldcg(gkeys + i) : 0; }
        }
        // FUSED: the first U x 1024 priors of the row (34 x 1024 covers the 34,125 priors of a 640 x 640 image) are loaded with all
        // U loads of a thread in flight together, and each warp compacts its candidates (ballot order) into its own queue in the
        // shared memory that only the NMS windows use later.  The histogram / scatter passes then run over DENSE queue entries:
        // one shared-memory atomic instruction per 32 candidates instead of one per 32 priors (a candidate density of ~1/5 made the
        // atomics of the sparse form the most expensive part of the kernel).  What does not fit -- a warp with more than WQ_CAP
        // candidates, rows longer than U x 1024 -- is visited in place on every pass: the scores of the first round stay in registers,
        // later rounds are re-read (L2).
        constexpr int U = FUSED ? 36 : 3;                    // 36 x 1024 priors per scan (a 640 x 640 image has 34,125)
        constexpr int WQ_CAP = (SM_WSTART - SM_SEGS) / 8 / (K3_THREADS / 32);          // 288 keys per warp
        int wq_n = 0;                                        // warp-uniform: queue length
        bool scanned = false, wq_ovf = false;                // wq_ovf: the warp's candidates did not fit, it visits its priors in place
        uint64_t *wq = reinterpret_cast<uint64_t *>(smem + SM_SEGS) + warp * WQ_CAP;
        const int Nn = (int)P.N, Cc = P.C;
        auto key_of = [&](const float sc, const int i) -> uint64_t { return ((uint64_t)fdt_float_key(sc) << 32) | (uint32_t)i; };
        // HT = 1: score of prior i of the list, of element type P.conf_dtype, widened to fp32 (exact) before any compare
        auto conf_any = [&](const int i) -> float {
            if (P.conf_dtype == FDT_DTYPE_F32) return __ldg(reinterpret_cast<const float *>(P.conf) + ((int64_t)b * Nn + i) * Cc + cl);
            return conf16_score(reinterpret_cast<const unsigned short *>(P.conf) + (int64_t)b * Nn * Cc, i, Cc, cl, P.conf_dtype,
                                P.conf_pair != 0);
        };
        auto for_each_key = [&](auto &&body) {
            if (FUSED) {
                if (!scanned) {
                    scanned = true;
                    // Compaction into the warp's queue, one group of UG priors at a time: each thread counts its candidates, one warp
                    // scan gives every thread its first queue position, and its candidates go to consecutive entries (thread-major
                    // order inside a group; keys are unique, so the order inside the queue is free).  A group that would take the
                    // queue past WQ_CAP is not stored: the warp then visits ALL its priors in place on every pass.  The U loads are
                    // issued in NG groups, group g + 1 before group g is compacted: two groups in flight hide the HBM latency
                    // without the register spills of all U at once.
                    constexpr int NG = FUSED ? 4 : 3, UG = U / NG;
                    const float qnan = __int_as_float(0x7fc00000);                          // never a candidate
                    const uint32_t qaddr = (uint32_t)__cvta_generic_to_shared(wq);
                    int run = 0;
                    float sv[NG][UG];
                    auto load_group = [&](const int g) {
                        const int i0 = tid + g * UG * K3_THREADS;
                        const bool whole = (g + 1) * UG * K3_THREADS <= Nn;                  // (uniform) no prior of the group is past the row
                        if constexpr (HT == 1) {
                            if (P.conf_pair) {          // (uniform) the prior's 32-bit (background, face) word, addresses folded
                                const unsigned *w0 = reinterpret_cast<const unsigned *>(P.conf) + (int64_t)b * Nn + i0;
                                const bool bf = P.conf_dtype == FDT_DTYPE_BF16;
#pragma unroll
                                for (int u = 0; u < UG; ++u) {
                                    const unsigned w = (whole || i0 + u * K3_THREADS < Nn) ? __ldg(w0 + u * K3_THREADS) : 0x7fc00000u;
                                    sv[g][u] = bf ? __uint_as_float(w & 0xffff0000u) : __half2float(__ushort_as_half((unsigned short)(w >> 16)));
                                }
                            } else if (P.conf_dtype == FDT_DTYPE_F32 && Cc == 2) {     // (uniform) fp32 conf beside a 16-bit loc
                                const float *p0 = reinterpret_cast<const float *>(P.conf) + ((int64_t)b * Nn + i0) * 2 + cl;
#pragma unroll
                                for (int u = 0; u < UG; ++u) sv[g][u] = (whole || i0 + u * K3_THREADS < Nn) ? __ldg(p0 + 2 * u * K3_THREADS) : qnan;
                            } else {
#pragma unroll
                                for (int u = 0; u < UG; ++u) {
                                    const int i = i0 + u * K3_THREADS;
                                    sv[g][u] = (whole || i < Nn) ? conf_any(i) : qnan;
                                }
                            }
                        } else if (Cc == 2) {                                                // (addresses fold into the load immediates)
                            const float *p0 = crow + 2 * i0;
                            if (whole) {
#pragma unroll
                                for (int u = 0; u < UG; ++u) sv[g][u] = __ldg(p0 + 2 * u * K3_THREADS);
                            } else {
#pragma unroll
                                for (int u = 0; u < UG; ++u) sv[g][u] = i0 + u * K3_THREADS < Nn ? __ldg(p0 + 2 * u * K3_THREADS) : qnan;
                            }
                        } else {
#pragma unroll
                            for (int u = 0; u < UG; ++u) {
                                const int i = i0 + u * K3_THREADS;
                                sv[g][u] = (whole || i < Nn) ? __ldg(crow + (int64_t)i * Cc) : qnan;
                            }
                        }
                    };
                    // POS: conf_thresh >= 0, so every candidate is a positive float and its key is its bits with the sign bit set
                    auto compact = [&](auto pos_thr) {
                        constexpr bool POS = decltype(pos_thr)::value;
                        load_group(0);
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            if (g + 1 < NG) load_group(g + 1);
                            // detection.py:64 strict gt; set.s32 gives -1 / 0, the count folds into 3-input adds and the stores
                            // below re-test each score where it is stored (fewer predicate registers live than priors in a group)
                            int cnt = 0;
#pragma unroll
                            for (int u = 0; u < UG; ++u) {
                                int m;
                                asm("set.gt.s32.f32 %0, %1, %2;" : "=r"(m) : "f"(sv[g][u]), "f"(cthr));
                                cnt -= m;
                            }
                            int inc = cnt;
#pragma unroll
                            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
                            const int tot = __shfl_sync(0xffffffffu, inc, 31);
                            if (run + tot <= WQ_CAP) {                                          // (warp-uniform)
                                uint32_t a = qaddr + 8u * (uint32_t)(run + inc - cnt);
                                const uint32_t i0 = (uint32_t)(tid + g * UG * K3_THREADS);
#pragma unroll
                                for (int u = 0; u < UG; ++u) {
                                    const uint32_t kk = POS ? (__float_as_uint(sv[g][u]) | 0x80000000u) : fdt_float_key(sv[g][u]);
                                    // predicated store and advance, no branch: a divergent `if` costs a BSSY / BRA / BSYNC triple per prior
                                    asm volatile("{ .reg .pred p; setp.gt.f32 p, %1, %2; @p st.shared.v2.u32 [%0], {%3, %4}; @p add.u32 %0, %0, 8; }"
                                                 : "+r"(a) : "f"(sv[g][u]), "f"(cthr), "r"(i0 + u * K3_THREADS), "r"(kk) : "memory");
                                }
                            }
                            run += tot;
                        }
                    };
                    if (cthr >= 0.0f) compact(std::true_type{});
                    else compact(std::false_type{});
                    wq_ovf = run > WQ_CAP;
                    wq_n = wq_ovf ? 0 : run;
                    __syncwarp();
                }
                for (int e = lane; e < wq_n; e += 32) body(wq[e]);
                // in place (re-read, L2): the whole first round of a warp whose queue overflowed, and every prior beyond it
                for (int i = (wq_ovf ? 0 : U * K3_THREADS) + tid; i < Nn; i += K3_THREADS) {
                    float sc;
                    if constexpr (HT == 1) sc = conf_any(i);
                    else sc = __ldg(crow + (int64_t)i * Cc);
                    if (sc > cthr) {
                        const uint64_t kq = key_of(sc, i);
                        if (!FUSED || kq < s_ck.tmax) body(kq);
                    }
                }
            } else if (cached) {
#pragma unroll
                for (int u = 0; u < KREG; ++u) { if (tid + u * K3_THREADS < n_c) body(kreg[u]); }
            } else {
                for (int i = tid; i < n_c; i += K3_THREADS) body(__ldcg(gkeys + i));
            }
        };
        if (tid == 0) { s_kmin = 0xffffffffu; s_kmax = 0u; s_maxb = 0; }
        for (int i = tid; i < 2 * NB; i += K3_THREADS) s_hist[i] = 0;
        __syncthreads();
        if (FUSED && s_ck.chunk > 0) { scanned = true; wq_ovf = true; }      // (uniform) the queues are gone: in place
        unsigned kmax;
        if (FUSED) {
            // the score range is known beforehand: every candidate is above conf_thresh, softmax outputs end at 1.  Anything beyond
            // lands in the top bucket (the map clamps) and is handled exactly by the fallbacks below.
            kmin = fdt_float_key(cthr);
            kmax = max(fdt_float_key(1.0f), kmin);
        } else if (MODE == MODE_DETECT) {   // k_threshold_compact already reduced the score range of the list
            const int lists = (int)(gridDim.x / CL);
            kmax = (unsigned)__ldcg(counters + lists + list);
            kmin = ~(unsigned)__ldcg(counters + 2 * lists + list);
        } else {
            unsigned lo = 0xffffffffu, hi = 0u;
            for_each_key([&](uint64_t key) { unsigned k32 = (unsigned)(key >> 32); lo = min(lo, k32); hi = max(hi, k32); });
            lo = __reduce_min_sync(0xffffffffu, lo); hi = __reduce_max_sync(0xffffffffu, hi);
            if (lane == 0) { atomicMin(&s_kmin, lo); atomicMax(&s_kmax, hi); }
            __syncthreads();
            kmin = s_kmin; kmax = s_kmax;
        }
        K3_STAMP(0);
        binv = (float)NB / ((float)(kmax - kmin) + 1.0f);
        uint64_t tmin = 0;                                   // after the fallback select: only keys >= tmin take part
        for (int attempt = 0; attempt < 2; ++attempt) {
            if (tmin == 0) for_each_key([&](uint64_t key) { atomicAdd(&s_hist[bucket(key)], 1); });          // (the common case, no 64-bit compare)
            else for_each_key([&](uint64_t key) { if (key >= tmin) atomicAdd(&s_hist[bucket(key)], 1); });
            __syncthreads();
            // descending exclusive scan: start[b] = number of keys in higher buckets
            int c[NB / K3_THREADS], sum = 0;
#pragma unroll
            for (int q = 0; q < NB / K3_THREADS; ++q) { c[q] = s_hist[NB - 1 - (tid * (NB / K3_THREADS) + q)]; sum += c[q]; }
            int inc = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
            if (lane == 31) s_warp[warp] = inc;
            if (tid == 0) { s_placed = 0; s_maxb = 0; }
            __syncthreads();
            if (warp == 0) {
                int w = s_warp[lane], winc = w;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, winc, o); if (lane >= o) winc += v; }
                s_warp[lane] = winc - w;
                if (lane == 31) s_warp[32] = winc;               // histogram total
            }
            __syncthreads();
            if (FUSED && attempt == 0) {                         // the first row scan counted the candidates
                if (s_ck.chunk == 0) {
                    n_c = s_warp[32];
                    if (MODE == MODE_DETECT && n_c == 1) n_c = 0;    // detection.py:66-72: one candidate -> `continue`
                    k = min(n_c, P.nms_top_k);
                    if (tid == 0) s_ck.k_all = k;                // (read after the windows' barriers only)
                } else {
                    k = s_ck.k_all - s_ck.done_k;
                }
                k = min(k, 2 * s_ck.win_cap);
                if (k == 0) break;                               // (uniform)
            }
            int run = inc - sum + s_warp[warp], mb = 0;
#pragma unroll
            for (int q = 0; q < NB / K3_THREADS; ++q) {
                const int bq = NB - 1 - (tid * (NB / K3_THREADS) + q);
                s_start[bq] = run;
                s_hist[bq] = 0;                              // becomes the fill counter of the scatter pass
                if (run < k) mb = max(mb, c[q]);
                if (run < k && run + c[q] >= k) s_placed = run + c[q];      // exactly one bucket straddles rank k
                run += c[q];
            }
            if (mb > BIG_BUCKET) atomicMax(&s_maxb, mb);
            __syncthreads();
            if (s_placed <= P.sm.key_cap || attempt == 1) break;
            // Degenerate score distribution (the straddling bucket does not fit): exact MSB radix select of the k-th
            // largest key, then bucket only the k keys >= that threshold.
            uint64_t prefix = 0, pmask = 0;
            int need = k;
            for (int shift = 56; shift >= 0; shift -= 8) {
                if (tid < 256) s_hist8[tid] = 0;
                __syncthreads();
                for (int base = 0; base < n_scan; base += K3_THREADS) {
                    int i = base + tid;
                    int d = 256;
                    if (i < n_scan) {
                        uint64_t key;
                        bool cand = true;
                        if (FUSED) {
                            float sc;
                            if constexpr (HT == 1) sc = conf_any(i);
                            else sc = __ldg(crow + (int64_t)i * P.C);
                            key = ((uint64_t)fdt_float_key(sc) << 32) | (uint32_t)i;
                            cand = sc > cthr && key < s_ck.tmax;
                        } else key = __ldcg(gkeys + i);
                        if (cand && (key & pmask) == prefix) d = (int)((key >> shift) & 0xff);
                    }
                    unsigned peers = __match_any_sync(0xffffffffu, d);
                    if (d < 256 && lane == __ffs(peers) - 1) atomicAdd(&s_hist8[d], __popc(peers));
                }
                __syncthreads();
                if (warp == 0) {
                    int cc = 0;
#pragma unroll
                    for (int q = 0; q < 8; ++q) cc += s_hist8[255 - 8 * lane - q];
                    int cum = cc;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, cum, o); if (lane >= o) cum += v; }
                    unsigned hit = __ballot_sync(0xffffffffu, cum >= need);
                    int first = __ffs(hit) - 1;
                    if (lane == first) {
                        int rem = need - (cum - cc);
                        for (int q = 0; q < 8; ++q) {
                            int hcount = s_hist8[255 - 8 * lane - q];
                            if (hcount >= rem) { s_sel[0] = 255 - 8 * lane - q; s_sel[1] = rem; s_sel[2] = hcount; break; }
                            rem -= hcount;
                        }
                    }
                }
                __syncthreads();
                prefix |= (uint64_t)s_sel[0] << shift;
                pmask |= (uint64_t)0xff << shift;
                need = s_sel[1];
                const bool done = (s_sel[2] == need);
                __syncthreads();
                if (done) break;
            }
            tmin = prefix;                                   // exactly k keys are >= prefix (keys are unique)
        }
        K3_STAMP(1);
        if (k > 0) {
        // scatter into bucket-contiguous order (arbitrary order inside a bucket)
        for_each_key([&](uint64_t key) {
            if (key >= tmin) {
                const int bq = bucket(key);
                const int st = s_start[bq];
                if (st < k) skeys[st + atomicAdd(&s_hist[bq], 1)] = key;
                if (MODE == MODE_DETECT && st < WIN && P.loc_prefetch) {
                    // will be decoded by the first NMS window: start pulling its loc / prior rows into L2 now
                    const uint32_t pp = (uint32_t)key;
                    asm volatile("prefetch.global.L2 [%0];" :: "l"(reinterpret_cast<const float4 *>(P.loc) + ((int64_t)b * P.N + pp)));
                    asm volatile("prefetch.global.L2 [%0];" :: "l"(reinterpret_cast<const float4 *>(P.priors) + pp));
                }
            }
        });
        __syncthreads();
        placed = min(s_placed, P.sm.key_cap);
        if (s_maxb > BIG_BUCKET) {
            // A bucket too large for the per-window ranking (e.g. thousands of equal scores): sort everything that was
            // placed with a bitonic network (descending, padded with the minimum key).  Rare, slow, exact.
            int P2 = 2;
            while (P2 < placed) P2 <<= 1;
            for (int i = placed + tid; i < P2; i += K3_THREADS) skeys[i] = 0;
            __syncthreads();
            for (int size = 2; size <= P2; size <<= 1)
                for (int stride = size >> 1; stride > 0; stride >>= 1) {
                    for (int t = tid; t < (P2 >> 1); t += K3_THREADS) {
                        int i = 2 * t - (t & (stride - 1));
                        int j = i + stride;
                        uint64_t a = skeys[i], c2 = skeys[j];
                        bool desc = (i & size) == 0;
                        if ((a < c2) == desc) { skeys[i] = c2; skeys[j] = a; }
                    }
                    __syncthreads();
                }
            presorted = true;
        }
        }
        K3_STAMP(2);
    } else {
        __syncthreads();                                     // (no candidates, not fused) publishes s_ck
    }

    // =========================================================== stage 2: lazy greedy NMS over windows of sorted candidates
    // Each round takes the next <= 1024 candidates (whole score buckets), orders them exactly, decodes their boxes and
    //   A  drops those suppressed by a box kept in an earlier round            (query of the kept-box grid),
    //   B  finds, for every survivor, the earlier survivors that suppress it   (query of the window grid),
    //   C  resolves: dead iff one of those is kept, kept iff all are dead      (parallel sweeps; the earliest undecided
    //      survivor always resolves, statuses never change once set -> exactly the sequential greedy result),
    // and stops once top_k boxes are kept: Detect only reads keep[:top_k] (detection.py:80-81).
    // In phases A-C thread t works on the t-th candidate IN CELL ORDER, so the lanes of a warp walk the same grid rows.
    const float thr = P.nms_thresh;
    const int variant = (MODE == MODE_NMS) ? P.variant : 0;
    // "Minimum" overlap (inter / smaller area) is not bounded by the side ratio nor by the overlap / width ratio: every
    // intersecting pair at every coarser level has to be looked at
    const float prune = (variant & FDT_NMS_MINIMUM) ? 0.0f : 0.99f * thr;
    const float tq = (variant & FDT_NMS_MINIMUM) ? 0.0f : 0.97f * fminf(thr, 1.0f);          // query-range tightening, see the grid comment
    auto suppresses = [&](const float4 bi, const float ai, const float4 bj2, const float aj2) -> bool {
        if (MODE == MODE_NMS && variant != 0) return fdt_suppresses_v(bi, ai, bj2, aj2, thr, variant);
        return fdt_suppresses_fast(bi, ai, bj2, aj2, thr);
    };
    auto suppresses_exact = [&](const float4 bi, const float ai, const float4 bj2, const float aj2) -> bool {
        if (MODE == MODE_NMS && variant != 0) return fdt_suppresses_v(bi, ai, bj2, aj2, thr, variant);
        return fdt_suppresses(bi, ai, bj2, aj2, thr);
    };
    const int max_keep = P.max_keep;
    int nkept = s_ck.nkept, rounds = s_ck.rounds, sweeps = s_ck.sweeps;        // (s_ck: see stage 1)
    GridGeom gg = s_ck.gg;
    int win_cap = s_ck.win_cap;
    for (int lo = 0; lo < k && nkept < max_keep; ++rounds) {
        // ---- window [lo, hi): whole buckets, at most win_cap candidates
        int hi;
        if (presorted) hi = min(lo + win_cap, k);
        else {
            const int e = min(lo + win_cap, placed);
            if (e == placed) hi = placed;
            else {
                const int bq = bucket(skeys[e - 1]);
                const int bend = s_start[bq] + s_hist[bq];
                hi = (bend == e) ? e : s_start[bq];          // buckets in range are <= BIG_BUCKET < win_cap, so hi > lo
            }
        }
        for (int i = tid; i <= NCELLX; i += K3_THREADS) { wstart[i] = 0; kstart[i] = 0; }
        sndep[tid] = 0;
        if (tid == 0) s_next = 0;
        if (tid == 0) { s_ext[0] = 0xffffffffu; s_ext[1] = 0xffffffffu; s_ext[2] = 0u; s_ext[3] = 0u; }
        // ---- exact order inside the window: rank = bucket start + number of larger keys in the same bucket.  The thread that
        //      holds the key at (unsorted) position lo + tid issues the loads of that candidate's loc / prior rows first, ranks
        //      the key while they are in flight, and then owns window position `wi` = rank - lo up to the CSR build.
        const int j = lo + tid;
        int wi = -1;
        float4 ld0 = make_float4(0.f, 0.f, 0.f, 0.f), ld1 = ld0;
        {
            uint64_t key = 0;
            int r = -1;
            if (j < hi) {
                key = skeys[j];
                const uint32_t p = (uint32_t)key;
                if (MODE == MODE_DETECT) {
                    if constexpr (HT == 1) ld0 = head_loc_row<HEAD_ANY>(P.hl, b, (int)p);
                    else ld0 = P.loc ? __ldg(reinterpret_cast<const float4 *>(P.loc) + ((int64_t)b * P.N + p)) : head_loc_row<HEAD_F32_NCHW>(P.hl, b, (int)p);
                    ld1 = __ldg(reinterpret_cast<const float4 *>(P.priors) + p);
                } else {
                    ld0 = __ldg(reinterpret_cast<const float4 *>(P.boxes) + p);
                }
                if (!presorted) {
                    const int bq = bucket(key);
                    const int blo = s_start[bq], bhi = blo + s_hist[bq];
                    int g = 0;
                    for (int t = blo; t < bhi; ++t) g += skeys[t] > key;
                    r = blo + g;
                } else r = j;
                wi = r - lo;
            }
            __syncthreads();                 // every key of the window is read (and the zeroed grid counters are visible)
            if (!presorted && r >= 0) skeys[r] = key;
        }
        K3_ACC(0);
        // ---- boxes of the window (decode only what NMS looks at); grid geometry from the first window
        const bool valid = wi >= 0 && lo + wi < k;
        const int nvalid = min(hi, k) - lo;
        {
            float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) bx = (MODE == MODE_DETECT) ? fdt_decode1(ld0, ld1, P.v0, P.v1) : ld0;      // detection.py:55
            const float4 gb = grid_box(bx, variant);
            const float side = fmaxf(gb.z - gb.x, gb.w - gb.y);
            if (rounds == 0) {
                const bool reg = valid && box_regular(gb);
                float x0 = reg ? gb.x : INFINITY, y0 = reg ? gb.y : INFINITY, x1 = reg ? gb.z : -INFINITY, y1 = reg ? gb.w : -INFINITY;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    x0 = fminf(x0, __shfl_xor_sync(0xffffffffu, x0, o)); y0 = fminf(y0, __shfl_xor_sync(0xffffffffu, y0, o));
                    x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, o)); y1 = fmaxf(y1, __shfl_xor_sync(0xffffffffu, y1, o));
                }
                if (lane == 0) {      // float min/max through the order-preserving integer map
                    atomicMin(&s_ext[0], fdt_float_key(x0)); atomicMin(&s_ext[1], fdt_float_key(y0));
                    atomicMax(&s_ext[2], fdt_float_key(x1)); atomicMax(&s_ext[3], fdt_float_key(y1));
                }
                __syncthreads();
                const float ex0 = fdt_key_float(s_ext[0]), ey0 = fdt_key_float(s_ext[1]);
                const float ex1 = fdt_key_float(s_ext[2]), ey1 = fdt_key_float(s_ext[3]);
                const float ext = fmaxf(ex1 - ex0, ey1 - ey0);
                gg.ok = (ext > 0.0f) && (ext < INFINITY) && (thr > 0.0f);     // thr <= 0 (or NaN): every pair suppresses, at any distance
                gg.x0 = ex0; gg.y0 = ey0;
                gg.inv0 = gg.ok ? 32.0f / ext : 0.0f;
                gg.c0 = gg.ok ? ext / 32.0f : 0.0f;
                if (!(gg.inv0 > 0.0f && gg.inv0 < INFINITY && gg.c0 > 0.0f)) gg.ok = 0;
            }
            K3_ACC(1);
            // ---- window grid and (from the second round on) kept-box grid, CSR: count per cell, scan, place
            const int cell = reg_cell(gg, gb, side, valid);
            if (wi >= 0) wcell[wi] = (uint16_t)(cell < 0 ? BIGCELL : cell);
            const int slot = cell >= 0 ? atomicAdd(&wstart[cell + 1], 1) : 0;
            if (rounds > 0)
                for (int i = tid; i < nkept; i += K3_THREADS) atomicAdd(&kstart[kcell[i] + 1], 1);
            __syncthreads();
            csr_scan(wstart, s_warp);
            if (cell >= 0) { const int ps = wstart[cell] + slot; witems[ps] = (uint16_t)wi; wpos[wi] = (uint16_t)ps; sbox[ps] = bx; sarea[ps] = box_area_v(bx, variant); }
            if (CL == 2) {
                // Both CTAs of the cluster must see the SAME CSR array (they split it by position): order every cell by window
                // position instead of by atomic arrival.
                __syncthreads();
                int np = -1;
                uint16_t it = 0;
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                float ar = 0.0f;
                if (tid < nvalid) {
                    it = witems[tid]; b4 = sbox[tid]; ar = sarea[tid];
                    const int c2 = wcell[it];
                    const int s0 = wstart[c2], s1 = wstart[c2 + 1];
                    int r = 0;
                    for (int t2 = s0; t2 < s1; ++t2) r += witems[t2] < it;
                    np = s0 + r;
                }
                __syncthreads();
                if (np >= 0) { witems[np] = it; wpos[it] = (uint16_t)np; sbox[np] = b4; sarea[np] = ar; }
            }
            if (rounds > 0) {
                csr_scan(kstart, s_warp);
                for (int i = tid; i <= NCELLX; i += K3_THREADS) kcur[i] = kstart[i];
                __syncthreads();
                for (int i = tid; i < nkept; i += K3_THREADS) kitems[atomicAdd(&kcur[kcell[i]], 1)] = (uint16_t)i;
            }
        }
        __syncthreads();
        K3_ACC(2);

        // ---- from here on this thread owns candidate `id` = the tid-th window candidate in cell order
        const bool have = tid < nvalid;
        const int id = have ? witems[tid] : 0;
        const float4 bj = sbox[have ? tid : 0];
        const float4 gj = grid_box(bj, variant);
        const float aj = sarea[have ? tid : 0], sj = fmaxf(gj.z - gj.x, gj.w - gj.y);
        const bool chk = nkept > 0;          // only then can a window candidate already be dead (phase A)
        const bool in_grid = have && wcell[id] != BIGCELL;
        // ---- phase A: against the boxes kept in earlier rounds
        bool alive = have;
        if (have && nkept > 0) {
            auto hit = [&](int t) -> bool { const int slot = kitems[t]; return suppresses(kbox[slot], karea[slot], bj, aj); };
            if (in_grid) alive = !csr_query(gg, kstart, gj, sj, prune, tq, hit);
            else for (int t = 0; t < nkept && alive; ++t) if (suppresses_exact(kbox[t], karea[t], bj, aj)) alive = false;
        }
        if (have) status[id] = alive ? 0 : 2;
        K3_ACC(3);
        __syncthreads();
        // ---- phase B: suppression pairs among the survivors of this window, each unordered pair examined once (forward
        //      queries); "a suppresses b" (a earlier in score order) is recorded in b's list with shared-memory atomics.
        //      B1: 1, 2 or 4 lanes share a candidate and walk its grid rows (round-robin), queueing the non-empty CSR row
        //          segments in the warp's own shared-memory region (no item is touched yet);
        //      B2: the warp flattens its segments into (candidate, item) pairs -- 32 pairs per step whatever the segment
        //          lengths are (prefix sum + ballot/REDUX owner search) -- so the IoU tests run without divergence.
        {
            const int share = (nvalid + CL - 1) / CL;                                            // candidates this CTA queries
            const int lpc = share > K3_THREADS / 2 ? 1 : share > K3_THREADS / 4 ? 2 : 4;        // lanes per candidate
            const int per_chunk = 32 / lpc;
            const int part = lane % lpc, sub = lane / lpc;
            const bool wprof = P.prof != nullptr && blockIdx.x == 0;
            const long long wb0 = wprof ? clock64() : 0;
            int nvis = 0;
            uint32_t *wseg = segs + warp * (SEG_SLOTS * 32);
            auto pair = [&](const int tc, const int t2) {       // CSR positions: candidate, item (tc < t2)
                if (wprof) ++nvis;
                const int cid = witems[tc], other = witems[t2];
                if (chk && status[other] == 2) return;
                const float4 cb = sbox[tc], bo = sbox[t2];
                const float ca = sarea[tc], ao = sarea[t2];
                const bool me_first = cid < other;           // window index = score order
                // the intersection is symmetric in the two boxes (max / min commute bit for bit); only the union's operand order
                // depends on which box is the kept one: one evaluation with the areas swapped instead of two divergent ones
                const bool sup = suppresses(cb, me_first ? ca : ao, bo, me_first ? ao : ca);
                if (sup) {
                    const int later = me_first ? other : cid, earlier = me_first ? cid : other;
                    const int sl = atomicAdd(&sndep[later], 1);
                    if (sl < DEPS) sdeps[later * DEPS + sl] = (uint16_t)earlier;
                }
            };
            // one chunk of 32 / lpc candidates per warp (the cluster's CTAs take alternate chunks), from the end of the CSR
            // array: 32 * CL chunks cover the window for every lpc
            const int t = nvalid - 1 - ((CL * warp + crank) * per_chunk + sub);
            int nseg = 0;
            if (t >= 0) {
                const int cid = witems[t];
                if (status[cid] != 2) {                         // else: suppressed in phase A
                    auto emit = [&](const int t0, const int t1) {
                        if (nseg < SEG_SLOTS) { wseg[nseg * 32 + lane] = (uint32_t)t | ((uint32_t)t0 << 10) | ((uint32_t)(t1 - t0) << 20); ++nseg; }
                        else for (int t2 = t0; t2 < t1; ++t2) pair(t, t2);
                    };
                    if (wcell[cid] != BIGCELL) {
                        const float4 cb = grid_box(sbox[t], variant);
                        csr_segments_forward(gg, wstart, cb, fmaxf(cb.z - cb.x, cb.w - cb.y), prune, tq, (int)wcell[cid], t, part, lpc, emit);
                    } else if (part == 0) {
                        // irregular boxes sit last in CSR order: every regular candidate's forward query reaches them; they
                        // only pair among themselves
                        const int t1 = wstart[BIGCELL + 1];
                        if (t + 1 < t1) emit(t + 1, t1);
                    }
                }
            }
            // compact the lanes' segment queues into one list (in place: position excl + k <= own slot k * 32 + lane ... read first)
            uint32_t mine[SEG_SLOTS];
#pragma unroll
            for (int q = 0; q < SEG_SLOTS; ++q) mine[q] = q < nseg ? wseg[q * 32 + lane] : 0u;
            int inc = nseg;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
            const int S = __shfl_sync(0xffffffffu, inc, 31);
            __syncwarp();
#pragma unroll
            for (int q = 0; q < SEG_SLOTS; ++q) if (q < nseg) wseg[inc - nseg + q] = mine[q];
            __syncwarp();
            for (int b0 = 0; b0 < S; b0 += 32) {
                const uint32_t sg = b0 + lane < S ? wseg[b0 + lane] : 0u;
                const int len = (int)(sg >> 20);
                int e = len;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, e, o); if (lane >= o) e += v; }
                const int T = __shfl_sync(0xffffffffu, e, 31);
                e -= len;                                        // exclusive: strictly increasing over the valid lanes, T beyond
                for (int ib = 0; ib < T; ib += 32) {
                    // owner of pair i = ib + lane: the last segment with e <= i
                    const unsigned below = __ballot_sync(0xffffffffu, e < ib);
                    const unsigned M = __reduce_or_sync(0xffffffffu, (e >= ib && e < ib + 32) ? 1u << (e - ib) : 0u);
                    const int owner = min(31, max(0, __popc(below) + __popc(M & (0xffffffffu >> (31 - lane))) - 1));
                    const uint32_t so = __shfl_sync(0xffffffffu, sg, owner);
                    const int eo = __shfl_sync(0xffffffffu, e, owner);
                    const int i = ib + lane;
                    if (i < T) pair((int)(so & 1023u), (int)((so >> 10) & 1023u) + (i - eo));
                }
            }
            if (wprof) {
                const long long wb1 = clock64();
                const int vsum = __reduce_add_sync(0xffffffffu, nvis), vmax = __reduce_max_sync(0xffffffffu, nvis);
                if (lane == 0) { P.prof[640 + warp] = wb1 - wb0; P.prof[672 + warp] = vsum; P.prof[704 + warp] = vmax; P.prof[736 + warp] = S; }
            }
        }
        __syncthreads();                                   // dependency lists complete
        if (CL == 2) {
            // merge the other CTA's partial lists (distributed shared memory): read them, cluster barrier, then append
            cg::cluster_group cluster = cg::this_cluster();
            cluster.sync();
            const int *r_ndep = cluster.map_shared_rank(sndep, crank ^ 1);
            const uint16_t *r_deps = cluster.map_shared_rank(sdeps, crank ^ 1);
            const int nrem = r_ndep[tid];
            uint16_t rd[DEPS];
#pragma unroll
            for (int d = 0; d < DEPS; ++d) rd[d] = (d < nrem) ? r_deps[tid * DEPS + d] : (uint16_t)0;
            cluster.sync();
            const int nloc = sndep[tid];
            int w = min(nloc, DEPS);
#pragma unroll
            for (int d = 0; d < DEPS; ++d)
                if (d < nrem && w < DEPS) sdeps[tid * DEPS + w++] = rd[d];
            sndep[tid] = nloc + nrem;
            __syncthreads();
        }
        K3_ACC(4);
        // ---- phase C: resolve
        {
            int st = alive ? 0 : 2;
            const int nfound = have ? sndep[id] : 0;             // published by the barrier of K3_ACC / first sweep below
            const int nd = min(nfound, DEPS);
            const bool ovf = nfound > DEPS;
            for (;;) {
                if (prof) ++sweeps;
                if (st == 0) {
                    bool any_kept = false, pend = false;
                    for (int d = 0; d < nd; ++d) { const int s2 = status[sdeps[id * DEPS + d]]; any_kept |= (s2 == 1); pend |= (s2 == 0); }
                    if (ovf && !any_kept && !pend) {  // the DEPS earliest suppressors are all dead: look at the others
                        if (in_grid) {
                            auto look = [&](int t) -> bool {
                                const int a = witems[t];
                                if (a < id && status[a] != 2 && suppresses(sbox[t], sarea[t], bj, aj)) {
                                    if (status[a] == 1) { any_kept = true; return true; }
                                    pend = true;
                                }
                                return false;
                            };
                            csr_query(gg, wstart, gj, sj, prune, tq, look);
                        } else {
                            for (int a = 0; a < id && !any_kept; ++a)
                                if (status[a] != 2 && suppresses_exact(sbox[wpos[a]], sarea[wpos[a]], bj, aj)) {
                                    if (status[a] == 1) any_kept = true; else pend = true;
                                }
                        }
                    }
                    if (any_kept) { st = 2; status[id] = 2; }
                    else if (!pend) { st = 1; status[id] = 1; }
                }
                if (!__syncthreads_or(st == 0)) break;       // one barrier per sweep; it also publishes the status bytes
                if (prof && sweeps <= 4) { long long now_ = clock64(); P.prof[20 + sweeps] = now_ - s_prof[0]; }
            }
        }
        K3_ACC(5);
        // ---- append the newly kept boxes in score order (thread <-> window position again)
        {
            const int mine = (tid < nvalid && status[tid] == 1) ? 1 : 0;     // thread <-> window position
            int tot;
            const int before = block_excl_scan(mine, s_warp, tot);
            const int slot = nkept + before;
            if (mine && slot < max_keep) {
                const int ps = wpos[tid];
                kbox[slot] = sbox[ps]; karea[slot] = sarea[ps]; kkey[slot] = skeys[j]; kcell[slot] = wcell[tid];
            }
            nkept = min(nkept + tot, max_keep);
            if (MODE == MODE_DETECT) {
                const int est = (int)(((long long)(max_keep - nkept) * nvalid) / max(tot, 1));
                win_cap = min(WIN, max(BIG_BUCKET + 64, est + (est >> 3) + 32));
            }
        }
        __syncthreads();
        K3_ACC(6);
        lo = hi;
    }
    nkept_out = nkept; rounds_out = rounds; sweeps_out = sweeps;
    if (!FUSED || nkept >= max_keep || s_ck.done_k + k >= s_ck.k_all) break;      // (uniform)
    // next chunk: the last key of this one is in exact order (its window ranked it); once every thread has evaluated the test above,
    // thread 0 records the state, and the first barrier of stage 1 publishes it
    __syncthreads();
    if (tid == 0) {
        s_ck.tmax = skeys[k - 1]; s_ck.done_k += k; s_ck.chunk += 1;
        s_ck.nkept = nkept; s_ck.rounds = rounds; s_ck.sweeps = sweeps; s_ck.win_cap = win_cap; s_ck.gg = gg;
    }
    }
    const int nkept = nkept_out, rounds = rounds_out, sweeps = sweeps_out;
    if (FUSED) k = s_ck.k_all;
    if (prof) {
        for (int q = 0; q < 6; ++q) atomicAdd((unsigned long long *)&P.prof[5 + q], (unsigned long long)pacc[q]);
        atomicAdd((unsigned long long *)&P.prof[16], (unsigned long long)pacc[6]);
        atomicAdd((unsigned long long *)&P.prof[12], (unsigned long long)nkept); atomicAdd((unsigned long long *)&P.prof[13], (unsigned long long)k);
        atomicAdd((unsigned long long *)&P.prof[14], (unsigned long long)rounds); atomicAdd((unsigned long long *)&P.prof[15], (unsigned long long)sweeps);
        atomicAdd((unsigned long long *)&P.prof[30], 1ull);
        atomicAdd((unsigned long long *)&P.prof[31], (unsigned long long)(clock64() - s_prof[1]));
    }

    // =========================================================== stage 3: outputs
    if (P.prof && tid == 0 && blockIdx.x < 256) { unsigned long long gt1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1)); atomicMin((unsigned long long *)&P.prof[40], (unsigned long long)s_prof[2]); atomicMax((unsigned long long *)&P.prof[41], (unsigned long long)s_prof[2]); atomicMin((unsigned long long *)&P.prof[42], gt1); atomicMax((unsigned long long *)&P.prof[43], gt1); P.prof[64 + blockIdx.x] = clock64() - s_prof[1]; P.prof[320 + blockIdx.x] = (long long)rounds * 100000 + k; }
    if (!writer) return;
    const bool gather = MODE == MODE_DETECT && P.peer_sig != nullptr;
    // Completion ticket (see the end of the kernel).  Fused call, local output, kept rows in shared memory: `done` only has to say
    // that every CTA is past its NMS, so the ticket is taken HERE and its round trip to L2 overlaps the output stores instead of
    // holding the SM (and its 200 KB of shared memory) at the very end.
    const bool early_ticket = FUSED && !gather && P.S.ctl != nullptr && P.sm.off_kbox >= 0;
    int my_ticket = -1;
    if (early_ticket && tid == 0) my_ticket = atomicAdd(ticket, 1);
    bool peer_ok = true;
    if (gather) {
        // Rows of epoch e go into block e % ring of every destination rank: that rank must be done with what epoch e - ring left
        // there.  A destination acknowledges "call x has begun" (which, in its stream, follows the consumer of call x - 1) in
        // slot [world + its rank] of every source's signal array at the start of its own k_sort_nms: wait for e - ring + 1.
        bool bad = false;
        if (tid < P.world && tid != P.my_rank && (P.root < 0 || tid == P.root)) {
            const unsigned *ack = reinterpret_cast<const unsigned *>(P.peer_sig[P.my_rank]) + P.world + tid;
            const unsigned need = P.epoch - (unsigned)P.ring + 1u;
            const long long t0 = clock64();
            unsigned v;
            for (;;) {
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(ack) : "memory");
                if ((int)(v - need) >= 0) break;
                if (clock64() - t0 > (1ll << 33)) { bad = true; break; }       // ~4 s: a dead peer must not hang the GPU
                __nanosleep(200);
            }
        }
        peer_ok = !__syncthreads_or(bad);
        if (!peer_ok && tid == 0) atomicOr(&P.S.ctl->error, FDT_STATUS_TIMEOUT_PEER);
    }
    if (MODE == MODE_DETECT) {
        const int top_k = P.top_k;
        const int cnt = min(nkept, top_k);                                   // detection.py:80
        // The plane [top_k, 5] is composed in shared memory (the phase-B segment queues are dead) and stored with 16-byte
        // vector stores -- to the local output, a pinned host tensor, or (fused gather) the gathered blocks of the destination
        // ranks over NVLink peer memory.  The staging buffer starts at the same 16-byte phase as the destination.
        constexpr int CH = 1600;                                             // rows per chunk: 32,000 bytes
        float *stage0 = reinterpret_cast<float *>(smem + SM_SEGS);
        const int ndst = P.n_peers > 0 ? P.n_peers : 1;
        // Signalled gather: the destination blocks start zeroed and only this protocol writes them, so a plane only needs its `cnt`
        // rows plus zeros over whatever the epoch that used the same ring block last (epoch - ring) left beyond them -- real images
        // have a few detections, not top_k: the NVLink traffic follows the detections, not the padding.
        int rows_w = top_k;
        if (gather && peer_ok && P.ring <= FDT_GATHER_RING_MAX) {
            int32_t *left = P.S.gather_rows + (size_t)(P.epoch % (unsigned)P.ring) * (gridDim.x / CL) + list;
            rows_w = max(cnt, min(top_k, *left));
            __syncthreads();                                                 // everybody has read the old value
            if (tid == 0) *left = cnt;
        }
        for (int r0 = 0; r0 < rows_w && peer_ok; r0 += CH) {
            const int nr = min(CH, rows_w - r0), nf = nr * 5;
            int staged_ph = -1;
            for (int pr = 0; pr < ndst; ++pr) {
                float *base = P.n_peers > 0 ? reinterpret_cast<float *>(P.peer_out[pr]) + (P.img_offset * P.C) * (int64_t)top_k * 5 : P.out;
                float *o = base + ((int64_t)(b * P.C + cl) * top_k + r0) * 5;
                const int ph = (int)(((uintptr_t)o >> 2) & 3);                // floats past a 16-byte boundary
                float *stage = stage0 + ph;
                if (ph != staged_ph) {                                       // (every destination block has the same alignment in practice)
                    if (staged_ph >= 0) __syncthreads();
                    staged_ph = ph;
                    for (int r = tid; r < nr; r += K3_THREADS) {
                        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f, v4 = 0.f;
                        if (r0 + r < cnt) {
                            const float4 bx = kbox[r0 + r];
                            v0 = fdt_key_float((uint32_t)(kkey[r0 + r] >> 32)); v1 = bx.x; v2 = bx.y; v3 = bx.z; v4 = bx.w;
                        }
                        float *d = stage + 5 * r;                            // stride 5 words: conflict-free
                        d[0] = v0; d[1] = v1; d[2] = v2; d[3] = v3; d[4] = v4;       // detection.py:82
                    }
                    __syncthreads();
                }
                const int lead = min(nf, (4 - ph) & 3);                      // scalar floats up to the first 16-byte boundary
                const int nq = (nf - lead) >> 2;
                if (tid < lead) o[tid] = stage[tid];
                const float4 *s4 = reinterpret_cast<const float4 *>(stage + lead);
                float4 *o4 = reinterpret_cast<float4 *>(o + lead);
                for (int t = tid; t < nq; t += K3_THREADS) o4[t] = s4[t];
                const int tail0 = lead + 4 * nq;
                if (tid < nf - tail0) o[tail0 + tid] = stage[tail0 + tid];
            }
            if (r0 + CH < rows_w) __syncthreads();
        }
        if (P.kept_prior) {
            int64_t *kp = P.kept_prior + (int64_t)(b * P.C + cl) * top_k;
            for (int r = tid; r < top_k; r += K3_THREADS) kp[r] = r < cnt ? (int64_t)(uint32_t)kkey[r] : -1;
        }
        if (P.counts && tid == 0) P.counts[b * P.C + cl] = cnt;
    } else {
        for (int64_t t = tid; t < P.n; t += K3_THREADS)
            P.keep[t] = t < nkept ? (int64_t)(uint32_t)kkey[t] : 0;           // box_utils.py:289 zero-initialised
        if (tid == 0) *P.count_out = nkept;
    }
    if (P.S.ctl) {
        // Completion.  Every writer CTA takes a ticket after a device-scope fence; the last one
        //   * (fused gather) publishes `epoch` in slot [rank] of every destination's signal array -- its system-scope fence is
        //     cumulative over all rows it has observed through the ticket chain; nobody waits here, the destination's
        //     k_gather_await does;
        //   * publishes done = seq once the previous call has completed (in-order completion, see "call sequencing").
        // (fused, local output: `done` only has to say that every CTA has reached its end -- grids retire in stream order, and a
        // call that writes the same buffers again takes the full dependency wait -- so the stores need not be fenced here)
        if (!early_ticket) {
            if (!FUSED || gather) __threadfence();
            __syncthreads();
            if (tid == 0) my_ticket = atomicAdd(ticket, 1);
        }
        if (tid == 0) {
            const int writers = (int)(gridDim.x / CL);
            if (my_ticket == writers - 1) {
                *ticket = 0;                                   // (a stage-2 launch may be repeated on the same slot)
                DetectCtl *ctl = P.S.ctl;
                if (gather) {
                    __threadfence_system();
                    const bool ok = *reinterpret_cast<volatile unsigned *>(&ctl->error) == 0;      // a timed-out wait: never signal
                    // (a destination publishes in its OWN array too: "my rows of this call are in my block" -- k_gather_await then
                    // needs no stream order behind this kernel and may run on any stream)
                    for (int q = 0; q < P.world && ok; ++q) {
                        if (!(P.root < 0 || q == P.root)) continue;
                        unsigned *dst = reinterpret_cast<unsigned *>(P.peer_sig[q]) + P.my_rank;
                        asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(dst), "r"(P.epoch) : "memory");
                    }
                }
                if (!spin_until_reached(&ctl->done, my_seq - 1u)) { atomicOr(&ctl->error, FDT_STATUS_TIMEOUT_LOCAL); __trap(); }
                st_release_u32(&ctl->done, my_seq);
            }
        }
    }
    K3_STAMP(11);
#undef K3_STAMP
#undef K3_ACC
}

SmemPlan plan_smem(int kcap, int max_keep, bool kept_in_smem)
{
    auto up16 = [](int x) { return (x + 15) / 16 * 16; };
    SmemPlan s;
    s.key_cap = 64;
    while (s.key_cap < kcap + 64) s.key_cap <<= 1;
    int off = SM_KEYS + s.key_cap * 8;
    s.off_kitems = off; off += up16(max_keep * 2);
    s.off_kcell = off; off += up16(max_keep * 2);
    s.off_kbox = s.off_karea = s.off_kkey = -1;
    if (kept_in_smem) {
        s.off_kbox = off; off += up16(max_keep * 16);
        s.off_karea = off; off += up16(max_keep * 4);
        s.off_kkey = off; off += up16(max_keep * 8);
    }
    s.total = off;
    return s;
}

constexpr int K3_STATIC_SMEM = 2 * 1024;         // small arrays declared __shared__ in k_sort_nms

// ---- process-wide options: read from the environment once, overridable through fdt_set_option (tests, tools)
struct Options {
    std::atomic<int> k3_profile, k3_cluster, k3_pdl, detect_depth, detect_fused, detect_prefetch, host_chunk;
    Options()
    {
        auto env_int = [](const char *name, int dflt) { const char *e = getenv(name); return e && *e ? atoi(e) : dflt; };
        k3_profile = env_int("FDT_K3_PROFILE", 0);
        k3_cluster = env_int("FDT_K3_CLUSTER", -1);          // -1: automatic
        k3_pdl = env_int("FDT_K3_PDL", 1);
        detect_depth = env_int("FDT_DETECT_DEPTH", FDT_DETECT_MAX_DEPTH);
        detect_fused = env_int("FDT_DETECT_FUSED", -1);      // -1: automatic
        detect_prefetch = env_int("FDT_DETECT_PREFETCH", 1);
        host_chunk = env_int("FDT_HOST_CHUNK", 16);          // images per copy/compute chunk of fdt_detect_host (0: no chunking)
    }
};
static Options &options() { static Options o; return o; }

static std::mutex g_prof_mutex;
static long long *g_prof_dev = nullptr;
static bool g_prof_armed = false;       // the producer launch already cleared the buffer (keeps K2 -> K3 adjacent in the stream)

static int prof_arm(cudaStream_t st)
{
    if (!g_prof_dev) { FDT_CUDA(cudaMalloc(&g_prof_dev, 1024 * sizeof(long long))); }
    FDT_CUDA(cudaMemsetAsync(g_prof_dev, 0, 1024 * sizeof(long long), st));
    FDT_CUDA(cudaMemsetAsync(g_prof_dev + 40, 0xff, sizeof(long long), st));
    FDT_CUDA(cudaMemsetAsync(g_prof_dev + 42, 0xff, sizeof(long long), st));
    FDT_CUDA(cudaMemsetAsync(g_prof_dev + 44, 0xff, sizeof(long long), st));
    return FDT_OK;
}

// cudaFuncSetAttribute is per device and not free: remember what was set per (kernel, device)
struct FuncAttrCache {
    std::mutex m;
    int smem[16] = {0};          // largest dynamic shared-memory size set so far, per device
};
template <typename K>
static int ensure_dyn_smem(K kernel, FuncAttrCache &c, int bytes)
{
    int dev = 0;
    FDT_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> g(c.m);
    if (dev < 0 || dev >= 16 || c.smem[dev] < bytes) {
        FDT_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        if (dev >= 0 && dev < 16) c.smem[dev] = bytes;
    }
    return FDT_OK;
}

// `P.S.ctl == null` (fdt_nms): kept_ws = global memory for the kept arrays (28 bytes per kept row and list) used when they do not
// fit in shared memory; sequenced calls carve them from the workspace slot (kept_ws_bytes = what a slot reserves for them).
template <int MODE>
int launch_sort_nms(SortNmsParams &P, int lists, int kcap, void *kept_ws, size_t kept_ws_bytes, cudaStream_t st)
{
    Options &opt = options();
    if (opt.k3_profile.load() == 2) {                    // accumulate over launches; cleared by fdt_debug_k3_profile
        std::lock_guard<std::mutex> g(g_prof_mutex);
        if (!g_prof_dev) { int rc = prof_arm(st); if (rc != FDT_OK) return rc; FDT_CUDA(cudaStreamSynchronize(st)); }
        P.prof = g_prof_dev; P.prof_all = 1;
    } else if (opt.k3_profile.load() == 1) {
        std::lock_guard<std::mutex> g(g_prof_mutex);
        if (!g_prof_armed) { int rc = prof_arm(st); if (rc != FDT_OK) return rc; }
        g_prof_armed = false;
        P.prof = g_prof_dev;
    }
    FDT_REQUIRE(kcap <= FDT_MAX_NMS_TOP_K, FDT_E_UNSUPPORTED, "nms_top_k=%d exceeds %d", kcap, FDT_MAX_NMS_TOP_K);
    const int limit = FDT_SMEM_MAX - K3_STATIC_SMEM;
    const bool fused = MODE == MODE_DETECT && P.conf != nullptr;
    // the fused kernel selects at most two first windows (<= 2 x WIN keys) per chunk: its key array need not hold nms_top_k keys
    const int kslot = fused ? std::min(kcap, 2 * WIN) : kcap;
    SmemPlan sp = plan_smem(kslot, P.max_keep, true);
    if (sp.total > limit) {
        sp = plan_smem(kslot, P.max_keep, false);
        const size_t need = (size_t)lists * P.max_keep * KEPT_ROW_BYTES;
        FDT_REQUIRE(kept_ws_bytes >= need && (kept_ws != nullptr || P.S.ctl != nullptr), FDT_E_WORKSPACE,
                    "kept rows (%d per list) do not fit in shared memory and the workspace lacks %zu bytes for them", P.max_keep, need);
        if (kept_ws) {
            char *p = (char *)kept_ws;
            P.g_kbox = (float4 *)p; p += (size_t)lists * P.max_keep * 16;
            P.g_kkey = (uint64_t *)p; p += (size_t)lists * P.max_keep * 8;
            P.g_karea = (float *)p;
        }
    }
    FDT_REQUIRE(sp.total <= limit, FDT_E_UNSUPPORTED,
                "nms_top_k=%d / max_keep=%d need %d bytes of shared memory (limit %d)", kcap, P.max_keep, sp.total, limit);
    P.sm = sp;
    // Two CTAs per list as a thread-block cluster (phase B split, dependency lists merged through DSMEM): shortens an isolated
    // call when the batch leaves SMs idle.  Back-to-back calls overlap on the device (workspace ring), where total SM time
    // counts: the cluster repeats every stage but phase B in both CTAs, so it is only used when the workspace has a single slot.
    // Kept rows in global memory (large max_keep) stay on the single-CTA path.
    const int want = opt.k3_cluster.load();
    const bool fits = lists * 2 <= FDT_NUM_SMS && sp.off_kbox >= 0;
    const bool cluster = !fused && fits && (want < 0 ? (P.S.ctl == nullptr || P.S.depth == 1) : want == 1);
    const bool pdl = opt.k3_pdl.load() == 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(lists * (cluster ? 2 : 1))); cfg.blockDim = dim3(K3_THREADS);
    cfg.dynamicSmemBytes = (size_t)sp.total; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (cluster) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = 2; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
        ++na;
    }
    if (pdl) {      // overlap this kernel's launch latency with the tail of the producer (k_threshold_compact / k_build_keys)
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = attr; cfg.numAttrs = na;
    static FuncAttrCache cache_cl, cache_1, cache_f, cache_cl_any, cache_1_any, cache_f_any;
    const bool head_any = MODE == MODE_DETECT && P.loc == nullptr && !P.hl.f32_nchw;
    if (fused && (P.loc == nullptr || P.conf_dtype != FDT_DTYPE_F32)) {         // flat inputs, at least one of them 16-bit
        int rc = ensure_dyn_smem(k_sort_nms<MODE_DETECT, 1, true, 1>, cache_f_any, sp.total); if (rc != FDT_OK) return rc;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_sort_nms<MODE_DETECT, 1, true, 1>, P));
    } else if (head_any && cluster) {
        int rc = ensure_dyn_smem(k_sort_nms<MODE_DETECT, 2, false, 1>, cache_cl_any, sp.total); if (rc != FDT_OK) return rc;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_sort_nms<MODE_DETECT, 2, false, 1>, P));
    } else if (head_any) {
        int rc = ensure_dyn_smem(k_sort_nms<MODE_DETECT, 1, false, 1>, cache_1_any, sp.total); if (rc != FDT_OK) return rc;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_sort_nms<MODE_DETECT, 1, false, 1>, P));
    } else if (fused) {
        int rc = ensure_dyn_smem(k_sort_nms<MODE_DETECT, 1, true>, cache_f, sp.total); if (rc != FDT_OK) return rc;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_sort_nms<MODE_DETECT, 1, true>, P));
    } else if (cluster) {
        int rc = ensure_dyn_smem(k_sort_nms<MODE, 2, false>, cache_cl, sp.total); if (rc != FDT_OK) return rc;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_sort_nms<MODE, 2, false>, P));
    } else {
        int rc = ensure_dyn_smem(k_sort_nms<MODE, 1, false>, cache_1, sp.total); if (rc != FDT_OK) return rc;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_sort_nms<MODE, 1, false>, P));
    }
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

// Workspace of the Detect family: [control block 256 B][slot 0][slot 1] ... ; slot = int32 [3][lists] (candidate count, max key,
// ~min key) + 1 completion ticket | uint64 keys[lists][N] | kept rows (only used when top_k rows exceed shared memory).
struct DetectWsPlan {
    size_t head_bytes;                 // control block + gather_rows
    size_t counters_bytes, keys_bytes, kept_bytes, slot_bytes;
    int lists;
};
static DetectWsPlan detect_ws_plan(int B, int64_t N, int C)
{
    DetectWsPlan w;
    w.lists = B * (C - 1);
    const size_t lists = (size_t)w.lists;
    const size_t kept_rows = (size_t)(N < FDT_MAX_NMS_TOP_K ? N : FDT_MAX_NMS_TOP_K);
    w.counters_bytes = fdt_align256((3 * lists + SLOT_EXTRA) * sizeof(int32_t));
    w.keys_bytes = fdt_align256(lists * (size_t)N * sizeof(uint64_t));
    w.kept_bytes = fdt_align256(lists * kept_rows * KEPT_ROW_BYTES);
    w.slot_bytes = w.counters_bytes + w.keys_bytes + w.kept_bytes;
    w.head_bytes = 256 + fdt_align256((size_t)FDT_GATHER_RING_MAX * lists * sizeof(int32_t));
    return w;
}
static DetectSlots detect_slots(void *ws, size_t ws_bytes, const DetectWsPlan &w)
{
    DetectSlots S;
    S.ctl = (DetectCtl *)ws;
    S.gather_rows = (int32_t *)((char *)ws + 256);
    S.gather_n = FDT_GATHER_RING_MAX * w.lists;
    S.base = (char *)ws + w.head_bytes;
    S.stride = w.slot_bytes;
    S.keys_off = w.counters_bytes;
    S.kept_off = w.counters_bytes + w.keys_bytes;
    size_t fit = (ws_bytes - w.head_bytes) / w.slot_bytes;
    int cap = options().detect_depth.load();
    if (cap < 1) cap = 1;
    if (cap > FDT_DETECT_MAX_DEPTH) cap = FDT_DETECT_MAX_DEPTH;
    S.depth = (int)(fit < (size_t)cap ? fit : (size_t)cap);
    return S;
}
static int k2_grid_x(int64_t N, bool heads) { const int tile = heads ? K2H_TILE : K2_TILE; return (int)((N + tile - 1) / tile); }
static unsigned long long detect_geometry_magic(int B, int64_t N, int C, int depth)
{
    unsigned long long h = 0x9e3779b97f4a7c15ull;
    for (unsigned long long v : {(unsigned long long)B, (unsigned long long)N, (unsigned long long)C, (unsigned long long)depth}) {
        h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
        h *= 0xff51afd7ed558ccdull;
    }
    return FDT_CTL_MAGIC ^ h;
}

}  // namespace

int fdt_option_host_chunk() { return options().host_chunk.load(); }

// =============================================================================================== C ABI
FDT_API size_t fdt_detect_workspace_bytes_depth(int B, int64_t N, int C, int depth)
{
    if (B <= 0 || N <= 0 || C <= 1) return 256;
    if (depth < 1) depth = 1;
    if (depth > FDT_DETECT_MAX_DEPTH) depth = FDT_DETECT_MAX_DEPTH;
    const DetectWsPlan w = detect_ws_plan(B, N, C);
    return w.head_bytes + (size_t)depth * w.slot_bytes;
}
FDT_API size_t fdt_detect_workspace_bytes(int B, int64_t N, int C) { return fdt_detect_workspace_bytes_depth(B, N, C, 1); }

FDT_API int fdt_set_option(const char *name, int value)
{
    FDT_REQUIRE(name != nullptr, FDT_E_INVALID, "fdt_set_option: null name");
    Options &o = options();
    const std::string n(name);
    if (n == "k3_profile") o.k3_profile = value;
    else if (n == "k3_cluster") o.k3_cluster = value;
    else if (n == "k3_pdl") o.k3_pdl = value;
    else if (n == "detect_depth") o.detect_depth = value;
    else if (n == "detect_fused") o.detect_fused = value;
    else if (n == "detect_prefetch") o.detect_prefetch = value;
    else if (n == "host_chunk") o.host_chunk = value;
    else { fdt_set_error("fdt_set_option: unknown option '%s'", name); return FDT_E_INVALID; }
    return FDT_OK;
}

static int detect_check_common(const char *who, int B, int64_t N, int C, const void *ws, size_t ws_bytes)
{
    FDT_REQUIRE(B >= 0 && N >= 0 && C >= 1, FDT_E_INVALID, "%s: bad sizes B=%d N=%lld C=%d", who, B, (long long)N, C);
    FDT_REQUIRE(N < (1ll << 31), FDT_E_UNSUPPORTED, "%s: N=%lld exceeds 2^31-1", who, (long long)N);
    if (B == 0 || C == 1 || N == 0) return FDT_OK;
    FDT_REQUIRE(ws && fdt_aligned(ws, 256), FDT_E_INVALID, "%s: workspace null or not 256-byte aligned", who);
    FDT_REQUIRE(ws_bytes >= fdt_detect_workspace_bytes(B, N, C), FDT_E_WORKSPACE,
                "%s: workspace %zu < %zu bytes", who, ws_bytes, fdt_detect_workspace_bytes(B, N, C));
    return FDT_OK;
}

// out0..2: the buffers the call's k_sort_nms will write (k_detect_begin serialises a call behind an in-flight one that shares
// them); the stage entry point does not know them and serialises instead.
static int threshold_compact_impl(const float *conf, const HeadLevels *heads, int B, int64_t N, int C, float conf_thresh,
                                  void *ws, size_t ws_bytes, fdt_stream_t stream,
                                  const void *out0, const void *out1, const void *out2, int serialize, bool begin_only = false,
                                  int conf_dtype = FDT_DTYPE_F32)
{
    cudaStream_t st = (cudaStream_t)stream;
    int rc = detect_check_common("fdt_detect_threshold_compact", B, N, C, ws, ws_bytes);
    if (rc != FDT_OK) return rc;
    const int lists = B * (C - 1);
    if (lists == 0 || N == 0) return FDT_OK;
    const bool c16 = conf_dtype != FDT_DTYPE_F32;
    FDT_REQUIRE(heads || (conf && fdt_aligned(conf, c16 ? 2 : 4)), FDT_E_INVALID, "fdt_detect: conf null or not aligned to its elements");
    FDT_REQUIRE(heads || begin_only || c16 || C != 2 || fdt_aligned(conf, 8), FDT_E_INVALID, "fdt_detect_threshold_compact: conf not 8-byte aligned");
    const DetectWsPlan w = detect_ws_plan(B, N, C);
    const DetectSlots S = detect_slots(ws, ws_bytes, w);
    long long *prof = nullptr;
    if (options().k3_profile.load() == 1) {
        std::lock_guard<std::mutex> g(g_prof_mutex);
        int rc2 = prof_arm(st); if (rc2 != FDT_OK) return rc2;
        g_prof_armed = true; prof = g_prof_dev;
    }
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(1); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cfg.attrs = attr; cfg.numAttrs = 1;
        FDT_CUDA(cudaLaunchKernelEx(&cfg, k_detect_begin, S, detect_geometry_magic(B, N, C, S.depth), lists, serialize,
                                    (unsigned long long)(uintptr_t)out0, (unsigned long long)(uintptr_t)out1, (unsigned long long)(uintptr_t)out2));
    }
    FDT_LAUNCH_CHECK();
    if (begin_only) return FDT_OK;             // fused call: k_sort_nms thresholds its own rows
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)k2_grid_x(N, heads != nullptr), (unsigned)B);
        cfg.blockDim = dim3(K2_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cfg.attrs = attr; cfg.numAttrs = 1;
        const int64_t N_ = N;
        HeadLevels hl{};
        if (heads) hl = *heads;
        if (heads) {
            // screening cut on the logit gap: sigmoid(gap) > thr needs gap > logit(thr); 1e-3 covers every rounding on either side
            float dcut = -INFINITY;
            if (conf_thresh > 1e-4f && conf_thresh < 1.0f - 1e-4f) dcut = logf(conf_thresh / (1.0f - conf_thresh)) - 1e-3f;
            else if (conf_thresh >= 1.0f - 1e-4f) dcut = 9.0f;          // sigmoid(9) < 1 - 1e-4: nothing at or below can pass
            if (hl.f32_nchw) FDT_CUDA(cudaLaunchKernelEx(&cfg, k_heads_threshold_compact<HEAD_F32_NCHW>, hl, N_, conf_thresh, dcut, S, prof));
            else             FDT_CUDA(cudaLaunchKernelEx(&cfg, k_heads_threshold_compact<HEAD_ANY>, hl, N_, conf_thresh, dcut, S, prof));
        }
        else if (c16) {
            hl.dtype = conf_dtype;
            hl.vec = (C == 2 && fdt_aligned(conf, 4)) ? 1u : 0u;
            FDT_CUDA(cudaLaunchKernelEx(&cfg, k_threshold_compact<2>, conf, hl, N_, C, conf_thresh, S, prof));
        }
        else if (C == 2) FDT_CUDA(cudaLaunchKernelEx(&cfg, k_threshold_compact<1>, conf, hl, N_, C, conf_thresh, S, prof));
        else             FDT_CUDA(cudaLaunchKernelEx(&cfg, k_threshold_compact<0>, conf, hl, N_, C, conf_thresh, S, prof));
    }
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_detect_threshold_compact(const float *conf, int B, int64_t N, int C, float conf_thresh,
                                         void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return threshold_compact_impl(conf, nullptr, B, N, C, conf_thresh, ws, ws_bytes, stream, nullptr, nullptr, nullptr, 1);
}

__global__ void k_copy_candidate_counts(const DetectSlots S, const int n, int32_t *__restrict__ out)
{
    const int32_t *c = reinterpret_cast<const int32_t *>(S.base + (size_t)(S.ctl->seq % (unsigned)S.depth) * S.stride);
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = c[i];
}

FDT_API int fdt_detect_candidate_counts(const void *ws, size_t ws_bytes, int B, int64_t N, int C, int32_t *counts_out, fdt_stream_t stream)
{
    FDT_REQUIRE(ws && counts_out && B >= 0 && C >= 1 && N >= 0, FDT_E_INVALID, "fdt_detect_candidate_counts: bad arguments");
    if (B * (C - 1) == 0 || N == 0) return FDT_OK;
    int rc = detect_check_common("fdt_detect_candidate_counts", B, N, C, ws, ws_bytes);
    if (rc != FDT_OK) return rc;
    const DetectSlots S = detect_slots((void *)ws, ws_bytes, detect_ws_plan(B, N, C));
    k_copy_candidate_counts<<<1, 256, 0, (cudaStream_t)stream>>>(S, B * (C - 1), counts_out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

// Sticky status of a Detect workspace (FDT_STATUS_* bits; 0 = fine): synchronises `stream`.
FDT_API int fdt_detect_status(const void *ws, fdt_stream_t stream, uint32_t *status_h)
{
    FDT_REQUIRE(ws && status_h, FDT_E_INVALID, "fdt_detect_status: null argument");
    FDT_CUDA(cudaMemcpyAsync(status_h, &((const DetectCtl *)ws)->error, sizeof(uint32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    FDT_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return FDT_OK;
}

struct GatherArgs {
    const unsigned long long *dest_out = nullptr;     // device array of n_dest destination block pointers
    int n_dest = 0;
    int64_t img_offset = 0;
    const unsigned long long *peer_sig = nullptr;
    int world = 0, rank = 0, root = 0, ring = 2;
    unsigned epoch = 0;
};

static int detect_sort_nms_impl(const float *loc, const HeadLevels *heads, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                                float nms_thresh, float var0, float var1,
                                float *out, int32_t *counts, int64_t *kept_prior,
                                const GatherArgs &G, void *ws, size_t ws_bytes, fdt_stream_t stream,
                                const float *fused_conf = nullptr, float conf_thresh = 0.0f, unsigned flags = 0,
                                int conf_dtype = FDT_DTYPE_F32, bool flat = false)
{
    // flat: `heads` describes a flat loc[B,N,4] (flat_loc_levels), and stage 1 was the flat K2 (its grid counts K2_TILE priors per block)
    cudaStream_t st = (cudaStream_t)stream;
    int rc = detect_check_common("fdt_detect_sort_nms", B, N, C, ws, ws_bytes);
    if (rc != FDT_OK) return rc;
    FDT_REQUIRE(top_k >= 1, FDT_E_INVALID, "fdt_detect_sort_nms: top_k=%d", top_k);
    FDT_REQUIRE(nms_top_k >= 1 && nms_top_k <= FDT_MAX_NMS_TOP_K, FDT_E_UNSUPPORTED,
                "fdt_detect: nms_top_k=%d outside [1,%d]", nms_top_k, FDT_MAX_NMS_TOP_K);
    FDT_REQUIRE(nms_thresh > 0.0f, FDT_E_INVALID, "fdt_detect: nms_thresh must be > 0 (detection.py:28-29)");
    if (B == 0) return FDT_OK;
    const int n_peers = G.n_dest;
    FDT_REQUIRE(out != nullptr || n_peers > 0, FDT_E_INVALID, "fdt_detect: out is null");
    const int lists = B * (C - 1);
    if (lists == 0 || N == 0) {
        FDT_REQUIRE(n_peers == 0, FDT_E_UNSUPPORTED, "fdt_detect_sort_nms_peers: needs C >= 2 and N > 0");
        FDT_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * C * top_k * 5, st));
        if (counts) FDT_CUDA(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)B * C, st));
        if (kept_prior) FDT_CUDA(cudaMemsetAsync(kept_prior, 0xff, sizeof(int64_t) * (size_t)B * C * top_k, st));
        return FDT_OK;
    }
    FDT_REQUIRE((heads || (loc && fdt_aligned(loc, 16))) && priors && fdt_aligned(priors, 16), FDT_E_INVALID,
                "fdt_detect: loc/priors null or not 16-byte aligned");
    const DetectWsPlan w = detect_ws_plan(B, N, C);
    SortNmsParams P{};
    P.S = detect_slots(ws, ws_bytes, w); P.use_counters = 1; P.key_stride = N; P.k2_blocks = k2_grid_x(N, heads != nullptr && !flat) * B;
    P.loc = heads ? nullptr : loc; P.priors = priors; P.N = N; P.C = C;
    P.loc_prefetch = (!heads && !(flags & FDT_FLAG_LOC_HOST_MAPPED) && options().detect_prefetch.load() == 1) ? 1 : 0;
    P.conf = fused_conf; P.conf_thresh = conf_thresh;
    P.conf_dtype = conf_dtype; P.conf_pair = conf_dtype != FDT_DTYPE_F32 && C == 2 && fdt_aligned(fused_conf, 4);
    if (heads) P.hl = *heads;
    P.nms_top_k = nms_top_k; P.max_keep = top_k < nms_top_k ? top_k : nms_top_k; P.top_k = top_k;
    P.nms_thresh = nms_thresh; P.v0 = var0; P.v1 = var1;
    P.out = out; P.counts = counts; P.kept_prior = kept_prior;
    P.peer_out = G.dest_out; P.n_peers = n_peers; P.img_offset = G.img_offset;
    P.peer_sig = G.peer_sig; P.world = G.world; P.my_rank = G.rank; P.root = G.root; P.epoch = G.epoch; P.ring = G.ring;
    int kcap = (int)((int64_t)nms_top_k < N ? nms_top_k : N);
    if (P.max_keep > kcap) P.max_keep = kcap;
    return launch_sort_nms<MODE_DETECT>(P, lists, kcap, nullptr, w.kept_bytes, st);
}

FDT_API int fdt_detect_sort_nms(const float *loc, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                                float nms_thresh, float var0, float var1,
                                float *out, int32_t *counts, int64_t *kept_prior,
                                void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return detect_sort_nms_impl(loc, nullptr, priors, B, N, C, top_k, nms_top_k, nms_thresh, var0, var1, out, counts, kept_prior,
                                GatherArgs{}, ws, ws_bytes, stream);
}

// One whole Detect call: sequencing + (K2 +) k_sort_nms.  Plain `conf` input takes the fused kernel (no K2); head maps and
// fdt_set_option("detect_fused", 0) take K2 + k_sort_nms.
// a flat loc[B,N,4] as a one-level loc map (heads.cuh): hw = N, strides (4N, 1, 4), one vector load per row where aligned
static HeadLevels flat_loc_levels(const void *loc, int64_t N, int dtype)
{
    HeadLevels hl{};
    hl.L = 1;
    hl.dtype = dtype;
    hl.hw[0] = (int)N;
    hl.loc[0] = HeadMap{loc, 4 * N, 1, 4};
    for (int l = 1; l <= FDT_MAX_LEVELS; ++l) hl.off[l] = (int)N;
    hl.vec = fdt_aligned(loc, (size_t)(4 * head_elem_bytes(dtype))) ? 1u << 8 : 0u;
    return hl;
}

static int detect_call(const void *loc, const void *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                       float conf_thresh, float nms_thresh, float var0, float var1,
                       float *out, int32_t *counts, int64_t *kept_prior, const GatherArgs &G, const void *alias0,
                       void *ws, size_t ws_bytes, fdt_stream_t stream, unsigned flags = 0,
                       int loc_dtype = FDT_DTYPE_F32, int conf_dtype = FDT_DTYPE_F32)
{
    // Fused pays when one wave of CTAs holds every list (what counts then is SM time per list, and consecutive calls fill the
    // other SMs); with several waves of lists the chip-wide K2 streams conf at a higher rate than 148 CTAs scanning their own rows,
    // and rows much longer than the per-warp candidate queues (34 x 1024 priors per round) would mostly be visited in place.
    const int want = options().detect_fused.load();
    const bool fused = want < 0 ? ((int64_t)B * (C - 1) <= FDT_NUM_SMS && N <= 40960) : want == 1;
    // before anything is enqueued: a null loc read through its one-level map (16-bit inputs) would be gathered from address 0
    FDT_REQUIRE(B <= 0 || N <= 0 || C < 2 || (loc && priors), FDT_E_INVALID, "fdt_detect: loc / priors is null");
    const float *conf32 = (const float *)conf;
    int rc = threshold_compact_impl(conf32, nullptr, B, N, C, conf_thresh, ws, ws_bytes, stream, alias0, counts, kept_prior, 0, fused,
                                    conf_dtype);
    if (rc != FDT_OK) return rc;
    if (loc_dtype == FDT_DTYPE_F32 && conf_dtype == FDT_DTYPE_F32)
        return detect_sort_nms_impl((const float *)loc, nullptr, priors, B, N, C, top_k, nms_top_k, nms_thresh, var0, var1, out, counts,
                                    kept_prior, G, ws, ws_bytes, stream, fused ? conf32 : nullptr, conf_thresh, flags);
    // 16-bit input(s): a 16-bit loc is gathered through its one-level map by the HT = 1 instantiations (fused or not); the fused kernel for
    // 16-bit conf (k_sort_nms<MODE_DETECT, 1, true, 1>) reads loc through that map whatever its type.  An fp32 loc with K2 keeps P.loc.
    const bool via_map = loc_dtype != FDT_DTYPE_F32 || fused;
    const HeadLevels hl = flat_loc_levels(loc, N, loc_dtype);
    return detect_sort_nms_impl((const float *)loc, via_map ? &hl : nullptr, priors, B, N, C, top_k, nms_top_k, nms_thresh, var0, var1,
                                out, counts, kept_prior, G, ws, ws_bytes, stream, fused ? conf32 : nullptr, conf_thresh, flags,
                                conf_dtype, true);
}

// The element types and alignments of flat loc / conf (checked before any CUDA call): FDT_DTYPE_*, each pointer aligned to its
// elements, an fp32 loc to f32_loc_align bytes.  Null pointers are the caller's to refuse (each entry knows when it reads them).
int fdt_flat_inputs_ok(const char *who, const void *loc, int loc_dtype, const void *conf, int conf_dtype, size_t f32_loc_align)
{
    for (int d : {loc_dtype, conf_dtype})
        FDT_REQUIRE(d == FDT_DTYPE_F32 || d == FDT_DTYPE_BF16 || d == FDT_DTYPE_F16, FDT_E_INVALID, "%s: unknown dtype %d", who, d);
    const size_t la = loc_dtype == FDT_DTYPE_F32 ? f32_loc_align : 2;
    FDT_REQUIRE(!loc || fdt_aligned(loc, la), FDT_E_INVALID, "%s: loc is not aligned to %d bytes", who, (int)la);
    FDT_REQUIRE(!conf || fdt_aligned(conf, (size_t)head_elem_bytes(conf_dtype)), FDT_E_INVALID, "%s: conf is not aligned to its elements",
                who);
    return FDT_OK;
}

// Destination side of the signalled gather: ends when every rank -- this one included -- has published `epoch` in this rank's signal
// array (its rows of that call have landed in this rank's block).  It depends on nothing but those signals, so it may be enqueued
// behind the call on the same stream (launched with programmatic serialization and triggering at once, the NEXT call is not held
// back) or, better, on a stream of its own: in the calls' stream it is a third grid per call in the in-order window of grids the
// stream runs ahead by (measured: +1.3 us per call on the destination).  Whatever consumes the gathered block follows it in stream
// order.  A source that does not show up within ~4 s sets FDT_STATUS_TIMEOUT_PEER in the workspace status.
__global__ void k_gather_await(const unsigned long long *peer_sig, const int world, const int my_rank, const unsigned epoch, DetectCtl *ctl)
{
    cudaTriggerProgrammaticLaunchCompletion();
    cudaGridDependencySynchronize();
    const int q = threadIdx.x;
    if (q < world) {
        const unsigned *mine = reinterpret_cast<const unsigned *>(peer_sig[my_rank]) + q;
        const long long t0 = clock64();
        unsigned v;
        for (;;) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
            if ((int)(v - epoch) >= 0) break;
            if (clock64() - t0 > (1ll << 33)) { atomicOr(&ctl->error, FDT_STATUS_TIMEOUT_PEER); break; }
            __nanosleep(200);
        }
    }
}

FDT_API int fdt_detect_gather_await(const uint64_t *peer_signal_ptrs, int world, int rank, uint32_t epoch, void *ws, fdt_stream_t stream)
{
    FDT_REQUIRE(peer_signal_ptrs && ws && world >= 1 && world <= 1024 && rank >= 0 && rank < world && epoch >= 1, FDT_E_INVALID,
                "fdt_detect_gather_await: bad arguments");
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1); cfg.blockDim = dim3((unsigned)((world + 31) / 32 * 32)); cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    FDT_CUDA(cudaLaunchKernelEx(&cfg, k_gather_await, (const unsigned long long *)peer_signal_ptrs, world, rank, (unsigned)epoch, (DetectCtl *)ws));
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_detect_peers(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                             float conf_thresh, float nms_thresh, float var0, float var1,
                             const uint64_t *peer_out_ptrs, int n_peers, int64_t image_offset,
                             void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    FDT_REQUIRE(peer_out_ptrs != nullptr && n_peers >= 1 && image_offset >= 0, FDT_E_INVALID, "fdt_detect_peers: bad peer arguments");
    GatherArgs G;
    G.dest_out = (const unsigned long long *)peer_out_ptrs; G.n_dest = n_peers; G.img_offset = image_offset;
    return detect_call(loc, conf, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1, nullptr, nullptr, nullptr,
                       G, peer_out_ptrs, ws, ws_bytes, stream);
}

static int gather_call(const char *who, const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                       float conf_thresh, float nms_thresh, float var0, float var1,
                       const uint64_t *dest_out_ptrs, int n_dest, const uint64_t *peer_signal_ptrs,
                       int world, int rank, int root, uint32_t epoch, int ring, int64_t image_offset,
                       void *ws, size_t ws_bytes, fdt_stream_t stream, bool await)
{
    FDT_REQUIRE(dest_out_ptrs && peer_signal_ptrs && world >= 1 && world <= K3_THREADS && rank >= 0 && rank < world && root >= -1 && root < world &&
                image_offset >= 0 && epoch >= 1 && ring >= 1 && (root >= 0 ? n_dest == 1 : n_dest == world), FDT_E_INVALID,
                "%s: bad arguments", who);
    FDT_REQUIRE(B > 0 && N > 0 && C >= 2, FDT_E_UNSUPPORTED, "%s: needs B > 0, N > 0, C >= 2", who);
    GatherArgs G;
    G.dest_out = (const unsigned long long *)dest_out_ptrs; G.n_dest = n_dest; G.img_offset = image_offset;
    G.peer_sig = (const unsigned long long *)peer_signal_ptrs; G.world = world; G.rank = rank; G.root = root; G.epoch = epoch; G.ring = ring;
    int rc = detect_call(loc, conf, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1, nullptr, nullptr, nullptr,
                         G, dest_out_ptrs, ws, ws_bytes, stream);
    if (rc != FDT_OK) return rc;
    if (await && (root < 0 || root == rank)) return fdt_detect_gather_await(peer_signal_ptrs, world, rank, epoch, ws, stream);
    return FDT_OK;
}

FDT_API int fdt_detect_gather_signal(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                                     float conf_thresh, float nms_thresh, float var0, float var1,
                                     const uint64_t *dest_out_ptrs, int n_dest, const uint64_t *peer_signal_ptrs,
                                     int world, int rank, int root, uint32_t epoch, int ring, int64_t image_offset,
                                     void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return gather_call("fdt_detect_gather_signal", loc, conf, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1, dest_out_ptrs,
                       n_dest, peer_signal_ptrs, world, rank, root, epoch, ring, image_offset, ws, ws_bytes, stream, true);
}

FDT_API int fdt_detect_gather_store(const float *loc, const float *conf, const float *priors, int B, int64_t N, int C, int top_k, int nms_top_k,
                                    float conf_thresh, float nms_thresh, float var0, float var1,
                                    const uint64_t *dest_out_ptrs, int n_dest, const uint64_t *peer_signal_ptrs,
                                    int world, int rank, int root, uint32_t epoch, int ring, int64_t image_offset,
                                    void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return gather_call("fdt_detect_gather_store", loc, conf, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1, dest_out_ptrs,
                       n_dest, peer_signal_ptrs, world, rank, root, epoch, ring, image_offset, ws, ws_bytes, stream, false);
}

int fdt_detect_flags(const void *loc, int loc_dtype, const void *conf, int conf_dtype, const float *priors,
                     int B, int64_t N, int C, int top_k, int nms_top_k,
                     float conf_thresh, float nms_thresh, float var0, float var1,
                     float *out, int32_t *counts, int64_t *kept_prior,
                     void *ws, size_t ws_bytes, fdt_stream_t stream, unsigned flags)
{
    return detect_call(loc, conf, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1, out, counts, kept_prior,
                       GatherArgs{}, out, ws, ws_bytes, stream, flags, loc_dtype, conf_dtype);
}

FDT_API int fdt_detect_ex(const void *loc, int loc_dtype, const void *conf, int conf_dtype, const float *priors,
                          int B, int64_t N, int C, int top_k, int nms_top_k,
                          float conf_thresh, float nms_thresh, float var0, float var1,
                          float *out, int32_t *counts, int64_t *kept_prior,
                          void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    int rc = fdt_flat_inputs_ok("fdt_detect", loc, loc_dtype, conf, conf_dtype, 16);
    if (rc != FDT_OK) return rc;
    return fdt_detect_flags(loc, loc_dtype, conf, conf_dtype, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1,
                            out, counts, kept_prior, ws, ws_bytes, stream, 0);
}

FDT_API int fdt_detect(const float *loc, const float *conf, const float *priors,
                       int B, int64_t N, int C, int top_k, int nms_top_k,
                       float conf_thresh, float nms_thresh, float var0, float var1,
                       float *out, int32_t *counts, int64_t *kept_prior,
                       void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return fdt_detect_ex(loc, FDT_DTYPE_F32, conf, FDT_DTYPE_F32, priors, B, N, C, top_k, nms_top_k, conf_thresh, nms_thresh, var0, var1,
                         out, counts, kept_prior, ws, ws_bytes, stream);
}

// ---- head maps -> Detect (SURVEY 8f rank 1; pyramid.py:291-309, 331-338)
FDT_API int fdt_heads_to_loc_conf_ex(const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype,
                                     const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, int B, int softmax,
                                     float *loc_out, float *conf_out, fdt_stream_t stream)
{
    HeadLevels hl;
    int64_t N = 0;
    int rc = heads_fill(hl, "fdt_heads_to_loc_conf", loc_maps_h, conf_maps_h, dtype, f_h, f_w, neg_max_h, n_levels, &N);
    if (rc != FDT_OK) return rc;
    FDT_REQUIRE(B >= 0, FDT_E_INVALID, "fdt_heads_to_loc_conf: B=%d", B);
    if (B == 0 || (!loc_out && !conf_out)) return FDT_OK;
    for (int l = 0; l < n_levels; ++l) {
        FDT_REQUIRE(!loc_out || hl.loc[l].p, FDT_E_INVALID, "fdt_heads_to_loc_conf: loc map %d is null", l);
        FDT_REQUIRE(!conf_out || hl.conf[l].p, FDT_E_INVALID, "fdt_heads_to_loc_conf: conf map %d is null", l);
    }
    FDT_REQUIRE((!loc_out || fdt_aligned(loc_out, 16)) && (!conf_out || fdt_aligned(conf_out, 8)), FDT_E_INVALID,
                "fdt_heads_to_loc_conf: outputs need 16 / 8-byte alignment");
    dim3 g((unsigned)((N + 255) / 256), (unsigned)B);
    if (hl.f32_nchw) k_heads_to_loc_conf<HEAD_F32_NCHW><<<g, 256, 0, (cudaStream_t)stream>>>(hl, (int)N, softmax, loc_out, conf_out);
    else             k_heads_to_loc_conf<HEAD_ANY><<<g, 256, 0, (cudaStream_t)stream>>>(hl, (int)N, softmax, loc_out, conf_out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

FDT_API int fdt_heads_to_loc_conf(const float *const *loc_maps_h, const float *const *conf_maps_h,
                                  const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, int B, int softmax,
                                  float *loc_out, float *conf_out, fdt_stream_t stream)
{
    fdt_head_map lm[FDT_MAX_LEVELS], cm[FDT_MAX_LEVELS];
    return fdt_heads_to_loc_conf_ex(heads_nchw(lm, loc_maps_h, f_h, f_w, n_levels), heads_nchw(cm, conf_maps_h, f_h, f_w, n_levels),
                                    FDT_DTYPE_F32, f_h, f_w, neg_max_h, n_levels, B, softmax, loc_out, conf_out, stream);
}

FDT_API int fdt_detect_heads_ex(const fdt_head_map *loc_maps_h, const fdt_head_map *conf_maps_h, int dtype,
                                const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, const float *priors,
                                int B, int top_k, int nms_top_k, float conf_thresh, float nms_thresh, float var0, float var1,
                                float *out, int32_t *counts, int64_t *kept_prior, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    HeadLevels hl;
    int64_t N = 0;
    int rc = heads_fill(hl, "fdt_detect_heads", loc_maps_h, conf_maps_h, dtype, f_h, f_w, neg_max_h, n_levels, &N);
    if (rc != FDT_OK) return rc;
    FDT_REQUIRE(loc_maps_h && conf_maps_h, FDT_E_INVALID, "fdt_detect_heads: null map arrays");
    for (int l = 0; l < n_levels; ++l)
        FDT_REQUIRE(hl.loc[l].p && hl.conf[l].p, FDT_E_INVALID, "fdt_detect_heads: map %d is null", l);
    rc = threshold_compact_impl(nullptr, &hl, B, N, 2, conf_thresh, ws, ws_bytes, stream, out, counts, kept_prior, 0);
    if (rc != FDT_OK) return rc;
    return detect_sort_nms_impl(nullptr, &hl, priors, B, N, 2, top_k, nms_top_k, nms_thresh, var0, var1, out, counts, kept_prior,
                                GatherArgs{}, ws, ws_bytes, stream);
}

FDT_API int fdt_detect_heads(const float *const *loc_maps_h, const float *const *conf_maps_h,
                             const int *f_h, const int *f_w, const int *neg_max_h, int n_levels, const float *priors,
                             int B, int top_k, int nms_top_k, float conf_thresh, float nms_thresh, float var0, float var1,
                             float *out, int32_t *counts, int64_t *kept_prior, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    fdt_head_map lm[FDT_MAX_LEVELS], cm[FDT_MAX_LEVELS];
    return fdt_detect_heads_ex(heads_nchw(lm, loc_maps_h, f_h, f_w, n_levels), heads_nchw(cm, conf_maps_h, f_h, f_w, n_levels),
                               FDT_DTYPE_F32, f_h, f_w, neg_max_h, n_levels, priors, B, top_k, nms_top_k, conf_thresh, nms_thresh,
                               var0, var1, out, counts, kept_prior, ws, ws_bytes, stream);
}

// Diagnostics: with FDT_K3_PROFILE=1 in the environment, CTA 0 of k_sort_nms records clock64 deltas per phase:
// [0] key min/max, [1] histogram+scan(+select), [2] scatter, [3] rank+permute, [4] decode+extent, [5..9] summed over
// rounds: phase A, compaction, phase B pairs, resolve, insert; [10] rounds, [11] output, [12] kept, [13] k, [14] big list.
FDT_API int fdt_debug_k3_profile(long long *out640_h /* 1024 entries */)
{
    FDT_REQUIRE(out640_h != nullptr, FDT_E_INVALID, "fdt_debug_k3_profile: null output");
    FDT_REQUIRE(g_prof_dev != nullptr, FDT_E_INVALID, "fdt_debug_k3_profile: run with FDT_K3_PROFILE=1 first");
    FDT_CUDA(cudaDeviceSynchronize());
    FDT_CUDA(cudaMemcpy(out640_h, g_prof_dev, 1024 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (options().k3_profile.load() == 2) { int rc = prof_arm(nullptr); if (rc != FDT_OK) return rc; FDT_CUDA(cudaDeviceSynchronize()); }
    return FDT_OK;
}

FDT_API size_t fdt_nms_workspace_bytes(int64_t n)
{
    size_t nn = (size_t)(n > 0 ? n : 1);
    size_t kept_rows = nn < FDT_MAX_NMS_TOP_K ? nn : FDT_MAX_NMS_TOP_K;
    size_t own = fdt_align256(nn * sizeof(uint64_t)) + fdt_align256(kept_rows * KEPT_ROW_BYTES);
    if (n > FDT_MAX_NMS_TOP_K) {                  // more candidates than k_sort_nms holds may enter: the mask formulation (nms_generic.cu)
        const size_t gen = fdt_nms_generic_workspace_bytes(n);
        if (gen > own) own = gen;
    }
    return own;
}

static int nms_impl(const float *boxes, const float *scores, int64_t n, float overlap, int64_t top_k, int variant,
                    int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    FDT_REQUIRE(n >= 0 && n < (1ll << 31), FDT_E_INVALID, "fdt_nms: bad n=%lld", (long long)n);
    FDT_REQUIRE(count != nullptr, FDT_E_INVALID, "fdt_nms: count is null");
    if (n == 0) { FDT_CUDA(cudaMemsetAsync(count, 0, sizeof(int64_t), st)); return FDT_OK; }   // box_utils.py:290-291
    FDT_REQUIRE(boxes && scores && keep && ws, FDT_E_INVALID, "fdt_nms: null pointer argument");
    FDT_REQUIRE(fdt_aligned(boxes, 16) && fdt_aligned(ws, 256), FDT_E_INVALID, "fdt_nms: boxes need 16-byte, workspace 256-byte alignment");
    FDT_REQUIRE(ws_bytes >= fdt_nms_workspace_bytes(n), FDT_E_WORKSPACE, "fdt_nms: workspace %zu < %zu bytes", ws_bytes, fdt_nms_workspace_bytes(n));
    int64_t k = (top_k <= 0 || top_k > n) ? n : top_k;         // idx[-top_k:]; idx[-0:] is the whole list
    if (k > FDT_MAX_NMS_TOP_K)                                 // box_utils.nms has no cap (:296-298): sort + pairwise mask + reduce, any n
        return fdt_nms_generic<float>(boxes, scores, n, overlap, top_k, variant, keep, count, ws, ws_bytes, st);
    uint64_t *keys = (uint64_t *)ws;
    k_build_keys<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(scores, n, keys);
    FDT_LAUNCH_CHECK();
    SortNmsParams P{};
    P.keys = keys; P.key_stride = n; P.boxes = boxes; P.n = n; P.N = n; P.C = 2;
    P.nms_top_k = (int)k; P.max_keep = (int)k; P.nms_thresh = overlap; P.variant = variant;
    P.keep = keep; P.count_out = count;
    char *kept_ws = (char *)ws + fdt_align256((size_t)n * sizeof(uint64_t));
    size_t kept_rows = (size_t)(n < FDT_MAX_NMS_TOP_K ? n : FDT_MAX_NMS_TOP_K);
    return launch_sort_nms<MODE_NMS>(P, 1, (int)k, kept_ws, fdt_align256(kept_rows * KEPT_ROW_BYTES), st);
}

FDT_API int fdt_nms(const float *boxes, const float *scores, int64_t n, float overlap, int64_t top_k,
                    int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    return nms_impl(boxes, scores, n, overlap, top_k, 0, keep, count, ws, ws_bytes, stream);
}

// ---- sibling NMS implementations (SURVEY 8f rank 3): every box enters (no top_k), overlap rule per `variant`
FDT_API int fdt_nms_variant(const float *boxes, const float *scores, int64_t n, float thresh, int variant,
                            int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    FDT_REQUIRE(variant >= 0 && variant < 16, FDT_E_INVALID, "fdt_nms_variant: unknown variant flags %d", variant);
    return nms_impl(boxes, scores, n, thresh, 0, variant, keep, count, ws, ws_bytes, stream);
}

// FaceBoxes DataEncoder.decode_np, box part (FACEBOX/encoderl.py:318-320):
//   cxcy = loc[:, :2] * 0.1 * d[:, 2:] + d[:, :2];  wh = exp(loc[:, 2:] * 0.2) * d[:, 2:];  boxes = [cxcy - wh/2, cxcy + wh/2]
__global__ void k_facebox_decode(const float4 *__restrict__ loc, const float4 *__restrict__ dbox, int64_t n, float v0, float v1,
                                 float4 *__restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 l = __ldg(loc + i), d = __ldg(dbox + i);
    const float cx = (l.x * v0) * d.z + d.x, cy = (l.y * v0) * d.w + d.y;
    const float w = fdt_expf_cr(l.z * v1) * d.z, h = fdt_expf_cr(l.w * v1) * d.w;
    out[i] = make_float4(cx - w / 2.0f, cy - h / 2.0f, cx + w / 2.0f, cy + h / 2.0f);
}

FDT_API int fdt_facebox_decode(const float *loc, const float *default_boxes, int64_t n, float var0, float var1, float *out,
                               fdt_stream_t stream)
{
    FDT_REQUIRE(n >= 0, FDT_E_INVALID, "fdt_facebox_decode: n=%lld", (long long)n);
    if (n == 0) return FDT_OK;
    FDT_REQUIRE(loc && default_boxes && out && fdt_aligned(loc, 16) && fdt_aligned(default_boxes, 16) && fdt_aligned(out, 16),
                FDT_E_INVALID, "fdt_facebox_decode: null or not 16-byte aligned pointer");
    k_facebox_decode<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const float4 *)loc, (const float4 *)default_boxes, n, var0, var1, (float4 *)out);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}

// Threshold + NMS over a box table: the boxes p with conf[p, 1] > conf_thresh enter NMS (all of them, at most
// FDT_MAX_NMS_TOP_K -- more is FDT_E_UNSUPPORTED at run time: then keep is all zero and *count = -1), no host round trip:
// K2 compacts the candidates, k_sort_nms reads the count on the device.  keep[N] = table indices in keep order.
FDT_API size_t fdt_threshold_nms_workspace_bytes(int64_t N) { return fdt_detect_workspace_bytes(1, N, 2); }

__global__ void k_threshold_nms_guard(const DetectSlots S, int64_t *keep, int64_t *count, int64_t N, int limit)
{
    // more candidates than NMS admits: k_sort_nms would silently keep only the `limit` best (idx[-top_k:] semantics)
    const int32_t *counters = reinterpret_cast<const int32_t *>(S.base + (size_t)(S.ctl->seq % (unsigned)S.depth) * S.stride);
    if (counters[0] <= limit) return;
    for (int64_t i = threadIdx.x; i < N; i += blockDim.x) keep[i] = 0;
    if (threadIdx.x == 0) *count = -1;
}

FDT_API int fdt_threshold_nms(const float *boxes, const float *conf, int64_t N, float conf_thresh, float nms_thresh, int variant,
                              int64_t *keep, int64_t *count, void *ws, size_t ws_bytes, fdt_stream_t stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    FDT_REQUIRE(variant >= 0 && variant < 16, FDT_E_INVALID, "fdt_threshold_nms: unknown variant flags %d", variant);
    FDT_REQUIRE(N >= 0 && N < (1ll << 31) && count != nullptr, FDT_E_INVALID, "fdt_threshold_nms: bad arguments");
    if (N == 0) { FDT_CUDA(cudaMemsetAsync(count, 0, sizeof(int64_t), st)); return FDT_OK; }
    FDT_REQUIRE(boxes && conf && keep && fdt_aligned(boxes, 16), FDT_E_INVALID, "fdt_threshold_nms: null or misaligned pointer");
    int rc = threshold_compact_impl(conf, nullptr, 1, N, 2, conf_thresh, ws, ws_bytes, stream, keep, count, nullptr, 0);
    if (rc != FDT_OK) return rc;
    const DetectWsPlan w = detect_ws_plan(1, N, 2);
    const int kcap = (int)(N < FDT_MAX_NMS_TOP_K ? N : FDT_MAX_NMS_TOP_K);
    SortNmsParams P{};
    P.S = detect_slots(ws, ws_bytes, w); P.use_counters = 1; P.k2_blocks = k2_grid_x(N, false); P.key_stride = N; P.boxes = boxes; P.n = N; P.N = N; P.C = 2;
    P.nms_top_k = kcap; P.max_keep = kcap; P.nms_thresh = nms_thresh; P.variant = variant;
    P.keep = keep; P.count_out = count;
    rc = launch_sort_nms<MODE_NMS>(P, 1, kcap, nullptr, w.kept_bytes, st);
    if (rc != FDT_OK) return rc;
    k_threshold_nms_guard<<<1, 256, 0, st>>>(P.S, keep, count, N, kcap);
    FDT_LAUNCH_CHECK();
    return FDT_OK;
}
