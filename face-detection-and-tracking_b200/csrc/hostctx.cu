// Host-buffer entry points: the reference-facing call when the caller's tensors live in host memory
// (the reference's Detect builds its output with torch.zeros on the default device, detection.py:48).
//
// A batch is bound by the host-to-device copy of `conf` (17.5 MB per 64 images at 640 x 640: ~0.33 ms on PCIe 5 x16, twenty times
// the kernel time), so the context is a small copy/compute pipeline:
//   * a call is split into chunks of `host_chunk` images (16).  The chunk's `conf` block is copied on the context's COPY stream into
//     one of four staging slots; the kernels of the chunk run on the SLOT's own stream behind an event (one stream per slot: an event
//     wait between two kernels of ONE stream would hold the second until the first has drained, and a kernel that gathers `loc` over
//     PCIe is latency-bound, ~0.1 ms).  The copy of chunk i + 1 (and of the next call's first chunk) overlaps the kernels of chunk i,
//     the kernels of up to four chunks overlap each other, and only the last chunk's kernel is exposed at the end of a call.
//   * fdt_detect_host_submit returns a ticket as soon as everything is enqueued, fdt_detect_host_wait blocks until that call's results
//     landed in the caller's buffers; with two calls in flight the link never idles.  fdt_detect_host = submit + wait.
//   * Detect only decodes the candidates NMS actually looks at (<= 1024 rows of `loc` per image and round), so a pinned `loc_h`
//     (page-locked, hence mapped into the unified address space) is NOT copied: k_sort_nms gathers those 16-byte rows straight from
//     host memory over PCIe -- ~1 MB instead of 35 MB per batch of 64.  A pinned `out_h` is likewise written in place: the output
//     stage of k_sort_nms stores the rows over PCIe (posted writes) and the device-to-host copy of [B,C,top_k,5] disappears.
//   * the prior set is a constant of the model: it stays resident in the context (two buffers, so an upload never waits for the
//     kernels still reading the previous set) and `priors_h == NULL` means "the set uploaded last".
#include <cstdlib>
#include <cstring>
#include "fdt_common.cuh"

namespace {
constexpr int HOST_SLOTS = 4;      // chunk staging slots
constexpr int HOST_CALLS = 8;      // completion events kept (tickets older than that have completed: slots are reused in order)

struct HostSlot {
    cudaStream_t st;               // the chunk's kernels and device-to-host copies
    cudaEvent_t copied, done;
    bool used;
};
struct HostPlan {                  // layout of the staging allocation, a function of (Bc, N, C, top_k)
    int Bc, C, top_k;
    int64_t N;
    size_t ws_bytes, slot_stride, so_conf, so_loc, so_out, so_cnt, so_kept, total;
};

HostPlan make_plan(int Bc, int64_t N, int C, int top_k)
{
    HostPlan p;
    p.Bc = Bc; p.C = C; p.top_k = top_k; p.N = N;
    // per slot: a single-slot Detect workspace (the Bc geometry also holds the remainder chunk's), then the staging buffers, sized for
    // fp32 inputs so that one layout serves every element type (a 16-bit conf / loc chunk fills the first half of its buffer)
    p.ws_bytes = fdt_align256(fdt_detect_workspace_bytes_depth(Bc, N, C, 1));
    size_t o = p.ws_bytes;
    p.so_conf = o; o += fdt_align256((size_t)Bc * N * C * 4);
    p.so_loc = o; o += fdt_align256((size_t)Bc * N * 16);
    p.so_out = o; o += fdt_align256((size_t)Bc * C * top_k * 20);
    p.so_cnt = o; o += fdt_align256((size_t)Bc * C * 4);
    p.so_kept = o; o += fdt_align256((size_t)Bc * C * top_k * 8);
    p.slot_stride = o;
    p.total = HOST_SLOTS * p.slot_stride;
    return p;
}

// device view of a pinned (mapped) host pointer whose device address is `align`-byte aligned, or null
template <typename T>
T *mapped_view(T *host, size_t align = 16)
{
    if (!host) return nullptr;
    cudaPointerAttributes attr;
    cudaError_t e = cudaPointerGetAttributes(&attr, (const void *)host);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }   // pageable memory on old drivers reports an error: ignore
    if (attr.type == cudaMemoryTypeHost && attr.devicePointer && fdt_aligned(attr.devicePointer, align)) return (T *)attr.devicePointer;
    return nullptr;
}
}  // namespace

struct fdt_ctx {
    int device;
    cudaStream_t stream;           // joins the slots' streams: completion of a call
    cudaStream_t copy;             // host-to-device copies
    void *buf;
    size_t cap;
    HostPlan plan;
    bool planned;
    HostSlot slot[HOST_SLOTS];
    cudaEvent_t call_done[HOST_CALLS];
    uint64_t chunks, calls;
    // resident prior sets
    void *pri_buf[2];
    size_t pri_cap[2];
    cudaEvent_t pri_copied;
    uint64_t pri_last_call[2];     // last call (ticket) that reads the buffer
    int pri_cur;                   // buffer holding the current set
    int64_t pri_n;                 // its size (0: none uploaded)
    uint64_t pri_uploads;
};

static int ctx_drain(fdt_ctx *c)
{
    FDT_CUDA(cudaStreamSynchronize(c->copy));
    for (int s = 0; s < HOST_SLOTS; ++s) FDT_CUDA(cudaStreamSynchronize(c->slot[s].st));
    FDT_CUDA(cudaStreamSynchronize(c->stream));
    return FDT_OK;
}

static int ctx_plan(fdt_ctx *c, int Bc, int64_t N, int C, int top_k)
{
    if (c->planned && c->plan.Bc == Bc && c->plan.N == N && c->plan.C == C && c->plan.top_k == top_k) return FDT_OK;
    int rc = ctx_drain(c);                                       // the layout changes under everything in flight
    if (rc != FDT_OK) return rc;
    const HostPlan p = make_plan(Bc, N, C, top_k);
    if (p.total > c->cap) {
        if (c->buf) { FDT_CUDA(cudaFree(c->buf)); c->buf = nullptr; c->cap = 0; }
        const size_t want = p.total + p.total / 4;
        FDT_CUDA(cudaMalloc(&c->buf, want));
        c->cap = want;
    }
    // the Detect workspaces are stateful: start from zeroed memory (a fresh workspace) rather than from the previous layout's bytes
    for (int s = 0; s < HOST_SLOTS; ++s) {
        FDT_CUDA(cudaMemsetAsync((char *)c->buf + s * p.slot_stride, 0, p.ws_bytes, c->slot[s].st));
        c->slot[s].used = false;
    }
    c->plan = p;
    c->planned = true;
    return FDT_OK;
}

FDT_API int fdt_ctx_create(int device, fdt_ctx **out)
{
    FDT_REQUIRE(out != nullptr, FDT_E_INVALID, "fdt_ctx_create: out is null");
    int rc = fdt_device_check(device);
    if (rc != FDT_OK) return rc;
    FDT_CUDA(cudaSetDevice(device));
    fdt_ctx *c = (fdt_ctx *)calloc(1, sizeof(fdt_ctx));
    FDT_REQUIRE(c != nullptr, FDT_E_INVALID, "fdt_ctx_create: out of host memory");
    c->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking);
    for (int s = 0; s < HOST_SLOTS && e == cudaSuccess; ++s) {
        e = cudaStreamCreateWithFlags(&c->slot[s].st, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->slot[s].copied, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->slot[s].done, cudaEventDisableTiming);
    }
    for (int s = 0; s < HOST_CALLS && e == cudaSuccess; ++s) e = cudaEventCreateWithFlags(&c->call_done[s], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->pri_copied, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        fdt_set_error("fdt_ctx_create: %s", cudaGetErrorString(e));
        fdt_ctx_destroy(c);
        return FDT_E_CUDA;
    }
    *out = c;
    return FDT_OK;
}

FDT_API int fdt_ctx_destroy(fdt_ctx *c)
{
    if (!c) return FDT_OK;
    cudaSetDevice(c->device);
    if (c->copy) cudaStreamSynchronize(c->copy);
    for (int s = 0; s < HOST_SLOTS; ++s) if (c->slot[s].st) cudaStreamSynchronize(c->slot[s].st);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (int s = 0; s < HOST_SLOTS; ++s) {
        if (c->slot[s].st) cudaStreamDestroy(c->slot[s].st);
        if (c->slot[s].copied) cudaEventDestroy(c->slot[s].copied);
        if (c->slot[s].done) cudaEventDestroy(c->slot[s].done);
    }
    for (int s = 0; s < HOST_CALLS; ++s) if (c->call_done[s]) cudaEventDestroy(c->call_done[s]);
    if (c->pri_copied) cudaEventDestroy(c->pri_copied);
    if (c->buf) cudaFree(c->buf);
    for (int s = 0; s < 2; ++s) if (c->pri_buf[s]) cudaFree(c->pri_buf[s]);
    if (c->copy) cudaStreamDestroy(c->copy);
    if (c->stream) cudaStreamDestroy(c->stream);
    (void)cudaGetLastError();
    free(c);
    return FDT_OK;
}

// Upload a prior set [N,4] (host pointer): it becomes the set of every later call that passes priors_h == NULL.  Asynchronous when
// `priors_h` is pinned; earlier calls keep reading the set they were submitted with.
FDT_API int fdt_ctx_set_priors(fdt_ctx *c, const float *priors_h, int64_t N)
{
    FDT_REQUIRE(c != nullptr && priors_h != nullptr && N > 0, FDT_E_INVALID, "fdt_ctx_set_priors: null context / pointer or N <= 0");
    FDT_CUDA(cudaSetDevice(c->device));
    const int b = c->pri_n ? 1 - c->pri_cur : 0;
    const size_t bytes = (size_t)N * 16;
    // the buffer's previous set may still be read by a call in flight (an event re-recorded since belongs to a later call: covers it)
    if (c->pri_last_call[b]) FDT_CUDA(cudaStreamWaitEvent(c->copy, c->call_done[(c->pri_last_call[b] - 1) % HOST_CALLS], 0));
    if (c->pri_cap[b] < bytes) {
        if (c->pri_buf[b]) {
            if (c->pri_last_call[b]) { int rc = ctx_drain(c); if (rc != FDT_OK) return rc; }
            FDT_CUDA(cudaFree(c->pri_buf[b]));
            c->pri_buf[b] = nullptr; c->pri_cap[b] = 0;
        }
        FDT_CUDA(cudaMalloc(&c->pri_buf[b], fdt_align256(bytes)));
        c->pri_cap[b] = fdt_align256(bytes);
    }
    FDT_CUDA(cudaMemcpyAsync(c->pri_buf[b], priors_h, bytes, cudaMemcpyHostToDevice, c->copy));
    FDT_CUDA(cudaEventRecord(c->pri_copied, c->copy));       // (the chunk copies that follow on the copy stream are behind it anyway)
    c->pri_cur = b;
    c->pri_n = N;
    c->pri_last_call[b] = 0;
    ++c->pri_uploads;
    return FDT_OK;
}

FDT_API int fdt_detect_host_submit_ex(fdt_ctx *c, const void *loc_h, int loc_dtype, const void *conf_h, int conf_dtype,
                                      const float *priors_h, int B, int64_t N, int C, int top_k, int nms_top_k,
                                      float conf_thresh, float nms_thresh, float var0, float var1,
                                      float *out_h, int32_t *counts_h, int64_t *kept_prior_h, uint64_t *ticket)
{
    FDT_REQUIRE(c != nullptr && ticket != nullptr, FDT_E_INVALID, "fdt_detect_host_submit: null context / ticket");
    FDT_REQUIRE(B >= 0 && N >= 0 && C >= 1 && top_k >= 1, FDT_E_INVALID, "fdt_detect_host_submit: bad sizes");
    // host buffers: element alignment only -- a loc_h that is not a 16-byte (fp32) / 8-byte (16-bit) aligned pinned buffer is copied
    int rc = fdt_flat_inputs_ok("fdt_detect_host_submit", loc_h, loc_dtype, conf_h, conf_dtype, 4);
    if (rc != FDT_OK) return rc;
    const size_t le = loc_dtype == FDT_DTYPE_F32 ? 4 : 2, ce = conf_dtype == FDT_DTYPE_F32 ? 4 : 2;      // element sizes
    FDT_CUDA(cudaSetDevice(c->device));
    if (B == 0) {                                                          // nothing to do: completes with the previous call
        FDT_CUDA(cudaEventRecord(c->call_done[c->calls % HOST_CALLS], c->stream));
        *ticket = ++c->calls;
        return FDT_OK;
    }
    FDT_REQUIRE(loc_h && conf_h && out_h, FDT_E_INVALID, "fdt_detect_host_submit: null pointer argument");
    FDT_REQUIRE(priors_h || c->pri_n == N, FDT_E_INVALID,
                "fdt_detect_host_submit: priors_h is null and the context holds %lld priors, not %lld", (long long)c->pri_n, (long long)N);
    if (priors_h && (rc = fdt_ctx_set_priors(c, priors_h, N)) != FDT_OK) return rc;
    const char *loc_view = mapped_view((const char *)loc_h, 4 * le);
    float *out_view = mapped_view(out_h);

    int chunk = fdt_option_host_chunk();
    if (chunk <= 0 || chunk > B) chunk = B;
    const int Bc = chunk, nchunks = (B + Bc - 1) / Bc, Br = B - (nchunks - 1) * Bc == Bc ? 0 : B - (nchunks - 1) * Bc;
    if ((rc = ctx_plan(c, Bc, N, C, top_k)) != FDT_OK) return rc;
    const HostPlan &p = c->plan;
    const float *d_pri = (const float *)c->pri_buf[c->pri_cur];
    const size_t row_out = (size_t)C * top_k;                              // output rows per image
    for (int i = 0; i < nchunks; ++i) {
        const int b0 = i * Bc, nb = (i == nchunks - 1 && Br) ? Br : Bc;
        HostSlot &s = c->slot[c->chunks % HOST_SLOTS];
        char *base = (char *)c->buf + (c->chunks % HOST_SLOTS) * p.slot_stride;
        char *d_conf = base + p.so_conf;
        char *d_locs = base + p.so_loc;
        float *d_outs = (float *)(base + p.so_out);
        int32_t *d_cnt = (int32_t *)(base + p.so_cnt);
        int64_t *d_kept = (int64_t *)(base + p.so_kept);
        if (s.used) FDT_CUDA(cudaStreamWaitEvent(c->copy, s.done, 0));     // the slot's previous chunk has been consumed
        FDT_CUDA(cudaMemcpyAsync(d_conf, (const char *)conf_h + (size_t)b0 * N * C * ce, (size_t)nb * N * C * ce, cudaMemcpyHostToDevice,
                                 c->copy));
        if (!loc_view)
            FDT_CUDA(cudaMemcpyAsync(d_locs, (const char *)loc_h + (size_t)b0 * N * 4 * le, (size_t)nb * N * 4 * le, cudaMemcpyHostToDevice,
                                     c->copy));
        FDT_CUDA(cudaEventRecord(s.copied, c->copy));                      // (behind the prior upload, if this call made one)
        FDT_CUDA(cudaStreamWaitEvent(s.st, s.copied, 0));
        // rows in place only where the chunk's block is 16-byte aligned in the caller's buffer
        float *o_view = out_view ? out_view + (size_t)b0 * row_out * 5 : nullptr;
        if (o_view && !fdt_aligned(o_view, 16)) o_view = nullptr;
        rc = fdt_detect_flags(loc_view ? loc_view + (size_t)b0 * N * 4 * le : d_locs, loc_dtype, d_conf, conf_dtype, d_pri, nb, N, C, top_k,
                              nms_top_k, conf_thresh, nms_thresh, var0, var1, o_view ? o_view : d_outs, counts_h ? d_cnt : nullptr,
                              kept_prior_h ? d_kept : nullptr, base, p.ws_bytes, s.st, loc_view ? FDT_FLAG_LOC_HOST_MAPPED : 0u);
        if (rc != FDT_OK) return rc;
        if (!o_view)
            FDT_CUDA(cudaMemcpyAsync(out_h + (size_t)b0 * row_out * 5, d_outs, (size_t)nb * row_out * 20, cudaMemcpyDeviceToHost, s.st));
        if (counts_h) FDT_CUDA(cudaMemcpyAsync(counts_h + (size_t)b0 * C, d_cnt, (size_t)nb * C * 4, cudaMemcpyDeviceToHost, s.st));
        if (kept_prior_h)
            FDT_CUDA(cudaMemcpyAsync(kept_prior_h + (size_t)b0 * row_out, d_kept, (size_t)nb * row_out * 8, cudaMemcpyDeviceToHost, s.st));
        FDT_CUDA(cudaEventRecord(s.done, s.st));
        FDT_CUDA(cudaStreamWaitEvent(c->stream, s.done, 0));               // the call's completion event covers every chunk
        s.used = true;
        ++c->chunks;
    }
    FDT_CUDA(cudaEventRecord(c->call_done[c->calls % HOST_CALLS], c->stream));
    *ticket = ++c->calls;
    c->pri_last_call[c->pri_cur] = *ticket;
    return FDT_OK;
}

FDT_API int fdt_detect_host_wait(fdt_ctx *c, uint64_t ticket)
{
    FDT_REQUIRE(c != nullptr, FDT_E_INVALID, "fdt_detect_host_wait: null context");
    FDT_REQUIRE(ticket >= 1 && ticket <= c->calls, FDT_E_INVALID, "fdt_detect_host_wait: ticket %llu was never issued (last: %llu)",
                (unsigned long long)ticket, (unsigned long long)c->calls);
    FDT_CUDA(cudaSetDevice(c->device));
    // completion is in submission order; an event that has since been re-recorded belongs to a later call and covers this one
    FDT_CUDA(cudaEventSynchronize(c->call_done[(ticket - 1) % HOST_CALLS]));
    return FDT_OK;
}

FDT_API int fdt_detect_host_submit(fdt_ctx *c, const float *loc_h, const float *conf_h, const float *priors_h,
                                   int B, int64_t N, int C, int top_k, int nms_top_k,
                                   float conf_thresh, float nms_thresh, float var0, float var1,
                                   float *out_h, int32_t *counts_h, int64_t *kept_prior_h, uint64_t *ticket)
{
    return fdt_detect_host_submit_ex(c, loc_h, FDT_DTYPE_F32, conf_h, FDT_DTYPE_F32, priors_h, B, N, C, top_k, nms_top_k, conf_thresh,
                                     nms_thresh, var0, var1, out_h, counts_h, kept_prior_h, ticket);
}

FDT_API int fdt_detect_host_ex(fdt_ctx *c, const void *loc_h, int loc_dtype, const void *conf_h, int conf_dtype, const float *priors_h,
                               int B, int64_t N, int C, int top_k, int nms_top_k,
                               float conf_thresh, float nms_thresh, float var0, float var1,
                               float *out_h, int32_t *counts_h, int64_t *kept_prior_h)
{
    uint64_t t = 0;
    int rc = fdt_detect_host_submit_ex(c, loc_h, loc_dtype, conf_h, conf_dtype, priors_h, B, N, C, top_k, nms_top_k, conf_thresh,
                                       nms_thresh, var0, var1, out_h, counts_h, kept_prior_h, &t);
    if (rc != FDT_OK) return rc;
    return fdt_detect_host_wait(c, t);
}

FDT_API int fdt_detect_host(fdt_ctx *c, const float *loc_h, const float *conf_h, const float *priors_h,
                            int B, int64_t N, int C, int top_k, int nms_top_k,
                            float conf_thresh, float nms_thresh, float var0, float var1,
                            float *out_h, int32_t *counts_h, int64_t *kept_prior_h)
{
    return fdt_detect_host_ex(c, loc_h, FDT_DTYPE_F32, conf_h, FDT_DTYPE_F32, priors_h, B, N, C, top_k, nms_top_k, conf_thresh,
                              nms_thresh, var0, var1, out_h, counts_h, kept_prior_h);
}
