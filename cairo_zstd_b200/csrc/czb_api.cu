// czb_api.cu -- host side of the C ABI: context, workspace planning, batch entry points.
// (The FrameDecoder handle mirror lives in czb_handle.cu.)
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "czb_host.h"
#include "czb_internal.cuh"
#include "czb_parse.cuh"

namespace czb {
int setup_huff_attributes();
int setup_fse_attributes();
int setup_exec_attributes();
int setup_exec_flow_attributes();
}  // namespace czb

using namespace czb;

#define CZB_CUDA(ctx, call)                                                                   \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            (ctx)->last_error = std::string(#call) + ": " + cudaGetErrorString(e__);          \
            return CZS_CUDA_ERROR;                                                            \
        }                                                                                     \
    } while (0)

template <typename T>
static int ensure(czb_context* ctx, DevBuf<T>& b, uint64_t n) {
    if (n <= b.cap) return CZS_OK;
    uint64_t want = std::max<uint64_t>(n, b.cap + b.cap / 2);
    if (b.p) CZB_CUDA(ctx, cudaFree(b.p));  // cudaFree synchronises the device: no kernel still uses it
    b.p = nullptr; b.cap = 0;
    CZB_CUDA(ctx, cudaMalloc(reinterpret_cast<void**>(&b.p), want * sizeof(T)));
    b.cap = want;
    return CZS_OK;
}

// ---- guard mode (CZB_GUARD=1): compute-sanitizer is not available on every pool, so the scratch buffers can carry guard
// zones instead.  Before a wave's kernels run, the 64 bytes behind the part of each scratch buffer that the wave may use
// (exact totals from the scan) are filled with a pattern; after the wave a small kernel checks them.  A kernel that
// writes past its slice of the literal / sequence / block scratch shows up in czb_debug_guard_faults.
constexpr uint8_t kGuardByte = 0xA5;
constexpr uint64_t kGuardBytes = 64;
__global__ void k_check_guards(const uint8_t* a, const uint8_t* b, const uint8_t* c, unsigned long long* faults) {
    const unsigned t = threadIdx.x;  // 3 x 64 guard bytes, one thread each
    const uint8_t* p = t < 64 ? a : (t < 128 ? b : c);
    if (p && p[t & 63] != kGuardByte) atomicAdd(faults, 1ull);
}

extern "C" int czb_abi_version(void) { return CZB_ABI_VERSION; }

extern "C" int czb_context_create(int device, uint64_t budget, czb_context** out) {
    if (!out) return CZS_BAD_ARGUMENT;
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0 || device < 0 || device >= n_dev) return CZS_CUDA_ERROR;
    czb_context* ctx = new czb_context();
    ctx->device = device;
    ctx->budget = budget ? budget : (24ull << 30);
    ctx->wave_frames = 262144;  // 131072 / 262144 / 524288 frames per wave: 295.9 / 298.3 / 298.6 GB/s on config 2 (fewer kernel tails)
    if (const char* e = getenv("CZB_WAVE_FRAMES")) ctx->wave_frames = (uint64_t)atoll(e) > 128 ? (uint64_t)atoll(e) : 128;  // tuning knobs
    ctx->wave_frames = (ctx->wave_frames + 127) / 128 * 128;  // k_scan_frames / k_fill_blocks: a warp or CTA never straddles two waves
    if (const char* e = getenv("CZB_BUDGET_GB")) ctx->budget = (uint64_t)atoll(e) << 30;
    // Wave pipelining over two streams is opt-in (CZB_OVERLAP=1): measured on B200 it gains ~1 % because the
    // entropy kernels and k_exec contend for the same issue slots and registers, and it makes the per-kernel
    // event times overlap.  Default: one stream, every kernel alone, exact per-kernel timings.
    ctx->no_overlap = getenv("CZB_OVERLAP") == nullptr;
    if (const char* e = getenv("CZB_HOST_CHUNK_MB")) ctx->host_chunk_bytes = (uint64_t)atoll(e) << 20;  // measurement aid: run every kernel alone
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return CZS_CUDA_ERROR; }
    if (setup_huff_attributes() != 0 || setup_fse_attributes() != 0 || setup_exec_attributes() != 0 || setup_exec_flow_attributes() != 0) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    // frames whose compressed size is at least 2^big_cls bytes get a whole CTA in sequence execution (k_exec_big)
    // and whose sequences are sparse (at least big_seq_bytes compressed bytes per sequence; 0 = any).  Knobs for tests.
    if (const char* e = getenv("CZB_GUARD")) ctx->guard = atoi(e) != 0;
    if (const char* e = getenv("CZB_FLOW_WIDE")) ctx->flow_wide_forced = atoi(e) != 0;
    if (const char* e = getenv("CZB_BIG_FLOW")) ctx->big_flow = atoi(e) != 0;  // 0: the round-1 in-order executor (k_exec_big), for A/B
    if (const char* e = getenv("CZB_BIG_CLS")) ctx->big_cls = atoi(e);
    if (const char* e = getenv("CZB_BIG_SEQ_BYTES")) ctx->big_seq_bytes = atoi(e);
    if (const char* e = getenv("CZB_SHARE_CLS")) ctx->share_cls = atoi(e);
    if (const char* e = getenv("CZB_BIG_SHARE")) ctx->big_share = atoi(e) > 0 ? atoi(e) : 1;
    if (ctx->share_cls > ctx->big_cls) ctx->share_cls = ctx->big_cls;
    {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        ctx->sm_count = sms;
        ctx->flow_max = 2ull * (uint64_t)sms;  // k_exec_flow CTAs that fit the machine at once
        if (const char* e = getenv("CZB_FLOW_MAX")) ctx->flow_max = (uint64_t)atoll(e);
        ctx->big_resident = 7 * sms;  // k_exec_big CTAs that fit the machine at once (72 registers x 128 threads)
    }
    // Planning read-back buffer: host memory mapped into the device address space.  A kernel writes the
    // per-wave totals straight into it, so the read-back never queues behind a large device-to-host
    // copy on the copy engine (that serialised decode behind the previous chunk's output transfer).
    if (cudaHostAlloc(reinterpret_cast<void**>(&ctx->totals_h), sizeof(WaveTotals) * kMaxWaves, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->totals_h_dev), ctx->totals_h, 0) != cudaSuccess) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    if (cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->exec_stream, cudaStreamNonBlocking) != cudaSuccess) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    for (int s = 0; s < 2; s++)
        if (cudaEventCreateWithFlags(&ctx->ev_entropy[s], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_exec[s], cudaEventDisableTiming) != cudaSuccess) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    if (cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_scratch_free, cudaEventDisableTiming) != cudaSuccess) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    for (int s = 0; s < czb_context::kHostSlots; s++)
        if (cudaEventCreateWithFlags(&ctx->ev_in[s], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_dec[s], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_out[s], cudaEventDisableTiming) != cudaSuccess) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    {
        int lo = 0, hi = 0;  // k_exec_big's CTAs first: the largest frames are the long pole of a wave
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&ctx->big_stream, cudaStreamNonBlocking, hi) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_big_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_big_join, cudaEventDisableTiming) != cudaSuccess) { czb_context_destroy(ctx); return CZS_CUDA_ERROR; }
    }
    *out = ctx;
    return CZS_OK;
}

extern "C" void czb_context_destroy(czb_context* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    cudaFree(ctx->infos.p); cudaFree(ctx->totals_d.p); cudaFree(ctx->guard_faults.p); cudaFree(ctx->huf_big.p);
    for (int s = 0; s < 2; s++) {
        cudaFree(ctx->exec_order[s].p); cudaFree(ctx->huf_cls0[s].p); cudaFree(ctx->huf_cls1[s].p); cudaFree(ctx->huf_recs[s].p);
        cudaFree(ctx->blocks[s].p); cudaFree(ctx->huf_items[s].p); cudaFree(ctx->fse_items[s].p); cudaFree(ctx->lit[s].p);
        cudaFree(ctx->seq[s].p); cudaFree(ctx->counters[s].p);
        if (ctx->ev_entropy[s]) cudaEventDestroy(ctx->ev_entropy[s]);
        if (ctx->ev_exec[s]) cudaEventDestroy(ctx->ev_exec[s]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_scratch_free) cudaEventDestroy(ctx->ev_scratch_free);
    for (int s = 0; s < czb_context::kHostSlots; s++) {
        if (ctx->ev_in[s]) cudaEventDestroy(ctx->ev_in[s]);
        if (ctx->ev_dec[s]) cudaEventDestroy(ctx->ev_dec[s]);
        if (ctx->ev_out[s]) cudaEventDestroy(ctx->ev_out[s]);
    }
    if (ctx->ev_big_fork) cudaEventDestroy(ctx->ev_big_fork);
    if (ctx->ev_big_join) cudaEventDestroy(ctx->ev_big_join);
    if (ctx->big_stream) cudaStreamDestroy(ctx->big_stream);
    if (ctx->exec_stream) cudaStreamDestroy(ctx->exec_stream);
    cudaFree(ctx->h_descs.p); cudaFree(ctx->h_results.p);
    for (int s = 0; s < czb_context::kHostSlots; s++) { cudaFree(ctx->h_src[s].p); cudaFree(ctx->h_dst[s].p); }
    if (ctx->totals_h) cudaFreeHost(ctx->totals_h);
    if (ctx->pin_a) cudaFreeHost(ctx->pin_a);
    if (ctx->pin_b) cudaFreeHost(ctx->pin_b);
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    if (ctx->compute) cudaStreamDestroy(ctx->compute);
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    delete ctx;
}

extern "C" const char* czb_last_error(const czb_context* ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
extern "C" uint64_t czb_kernel_launches(const czb_context* ctx) { return ctx ? ctx->launches : 0; }

// ---- per-kernel profiling ----------------------------------------------------------------------
static size_t prof_event(czb_context* ctx, cudaStream_t st) {
    if (ctx->ev_used == ctx->ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ctx->ev_pool.push_back(e); }
    cudaEventRecord(ctx->ev_pool[ctx->ev_used], st);
    return ctx->ev_used++;
}
struct ProfScope {
    czb_context* ctx; cudaStream_t st; int cls; size_t e0 = 0;
    ProfScope(czb_context* c, cudaStream_t s, int k) : ctx(c), st(s), cls(k) { if (ctx->profiling) e0 = prof_event(ctx, st); }
    ~ProfScope() { if (ctx->profiling) { size_t e1 = prof_event(ctx, st); ctx->prof.push_back({cls, e0, e1}); } }
};
extern "C" int czb_profile_enable(czb_context* ctx, int on) {
    if (!ctx) return CZS_BAD_ARGUMENT;
    ctx->profiling = on != 0;
    return CZS_OK;
}
extern "C" int czb_profile_collect(czb_context* ctx, double* ms, uint64_t* launches) {
    if (!ctx || !ms || !launches) return CZS_BAD_ARGUMENT;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    for (const auto& r : ctx->prof) {
        CZB_CUDA(ctx, cudaEventSynchronize(ctx->ev_pool[r.e1]));
        float t = 0;
        CZB_CUDA(ctx, cudaEventElapsedTime(&t, ctx->ev_pool[r.e0], ctx->ev_pool[r.e1]));
        if (r.cls >= 0 && r.cls < CZB_PROFILE_CLASSES) { ms[r.cls] += t; launches[r.cls] += 1; }
    }
    ctx->prof.clear(); ctx->ev_used = 0;
    return CZS_OK;
}

static uint64_t wave_scratch_bytes(const WaveTotals& t) {
    return t.n_blocks * sizeof(BlockDesc) + t.lit_bytes + t.n_seq * sizeof(Seq) + (t.n_huf + t.n_fse) * 4 + t.n_huf * (sizeof(HufRec) + 8);
}

constexpr uint32_t kFlagSizesOnly = 0x80000000u;  // internal: scan + block walk + k_fse, then k_frame_sizes (czb_frame_sizes_*)

// The hot path.  descs/results are device arrays.  `resume` (device array, one entry per frame, or nullptr) is the handle's
// way of continuing frames whose first blocks were executed by earlier calls (czb_handle.cu).
struct czb_batch_plan {   // what the planning read-back of a batch call produces (czb_plan_batch_device)
    uint64_t n = 0, W = 0, n_waves = 0;
    std::vector<WaveTotals> totals;
};

static int decode_batch_impl(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n, uint32_t flags,
                             void* stream_v, const FrameResume* resume, const czb_batch_plan* plan, czb_batch_plan* plan_out);

int czb_decode_batch_device_resume(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n,
                                   uint32_t flags, void* stream_v, const FrameResume* resume) {
    return decode_batch_impl(ctx, descs, results, n, flags, stream_v, resume, nullptr, nullptr);
}

// plan != nullptr: the wave split and the per-wave totals come from an earlier czb_plan_batch_device of the same frames, so
// nothing is read back and the host never waits: every kernel is only enqueued (graph capture, pipelining).
// plan_out != nullptr: only plan (scan + read-back), decode nothing.
static int decode_batch_impl(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n, uint32_t flags,
                             void* stream_v, const FrameResume* resume, const czb_batch_plan* plan, czb_batch_plan* plan_out) {
    if (!ctx || (n && (!descs || (!results && !plan_out)))) return CZS_BAD_ARGUMENT;
    if (n == 0) return CZS_OK;
    if (n > 0xFFFFFF00ull) { ctx->last_error = "more than 2^32 frames per call"; return CZS_BAD_ARGUMENT; }
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
    LaunchCtx lc{stream, &ctx->launches};
    int rc;
    // The per-context scratch (infos, totals, counters, blocks, literal and sequence scratch, work lists) is reused by
    // every call: a call on another stream must not start overwriting it while the previous call's kernels still read it.
    cudaStreamCaptureStatus cap_st = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &cap_st);
    const bool capturing = cap_st != cudaStreamCaptureStatusNone;  // a captured call is ordered by the graph it becomes part of
    if (ctx->scratch_in_use && !capturing) CZB_CUDA(ctx, cudaStreamWaitEvent(stream, ctx->ev_scratch_free, 0));
    if (plan && plan->n != n) { ctx->last_error = "plan was made for a different batch"; return CZS_BAD_ARGUMENT; }
    if ((rc = ensure(ctx, ctx->infos, n))) return rc;
    if ((rc = ensure(ctx, ctx->totals_d, kMaxWaves))) return rc;
    if (!ctx->huf_big.p) {  // scratch for Huffman-weight FSE tables with an accuracy log above 9 (global memory, one warp at a time)
        if ((rc = ensure(ctx, ctx->huf_big, huff_big_scratch_bytes()))) return rc;
        CZB_CUDA(ctx, cudaMemsetAsync(ctx->huf_big.p, 0, 64, stream));  // the lock word
    }

    // ---- plan: scan every frame, then size waves so that scratch fits the budget ----
    uint64_t W = std::min<uint64_t>((n + 127) / 128 * 128, ctx->wave_frames);
    while ((n + W - 1) / W > kMaxWaves) W *= 2;
    uint64_t n_waves = 0;
    const WaveTotals* totals_host = ctx->totals_h;
    if (plan) {  // scan with the planned wave size (device-side totals and size classes for k_fill_blocks), no read-back
        W = plan->W; n_waves = plan->n_waves; totals_host = plan->totals.data();
        CZB_CUDA(ctx, cudaMemsetAsync(ctx->totals_d.p, 0, n_waves * sizeof(WaveTotals), stream));
        { ProfScope ps(ctx, stream, 0); launch_scan_frames(lc, descs, ctx->infos.p, n, W, ctx->totals_d.p, resume); }
    }
    // A retry (a wave's scratch over the budget) scans again with the smaller wave size: the scan is the only code that
    // produces wave totals, so a retried wave's totals are the ones a call starting at that wave size would see.
    while (!plan) {
        n_waves = (n + W - 1) / W;
        CZB_CUDA(ctx, cudaMemsetAsync(ctx->totals_d.p, 0, n_waves * sizeof(WaveTotals), stream));
        { ProfScope ps(ctx, stream, 0); launch_scan_frames(lc, descs, ctx->infos.p, n, W, ctx->totals_d.p, resume); }
        launch_publish_totals(lc, ctx->totals_d.p, ctx->totals_h_dev, n_waves);
        CZB_CUDA(ctx, cudaStreamSynchronize(stream));
        uint64_t worst = 0;
        for (uint64_t w = 0; w < n_waves; w++) worst = std::max(worst, wave_scratch_bytes(ctx->totals_h[w]));
        if ((ctx->no_overlap ? 1 : 2) * worst <= ctx->budget || W <= 128 || (n + W / 2 - 1) / (W / 2) > kMaxWaves) break;
        W = std::max<uint64_t>(128, (W / 2 + 127) / 128 * 128);
    }
    if (plan_out) {
        plan_out->n = n; plan_out->W = W; plan_out->n_waves = n_waves;
        plan_out->totals.assign(ctx->totals_h, ctx->totals_h + n_waves);
    }
    WaveTotals mx{};
    for (uint64_t w = 0; w < n_waves; w++) {
        const WaveTotals& t = totals_host[w];
        mx.n_blocks = std::max(mx.n_blocks, t.n_blocks); mx.lit_bytes = std::max(mx.lit_bytes, t.lit_bytes);
        mx.n_seq = std::max(mx.n_seq, t.n_seq); mx.n_huf = std::max(mx.n_huf, t.n_huf); mx.n_fse = std::max(mx.n_fse, t.n_fse);
        if (t.n_blocks > 0xFFFFFF00ull) { ctx->last_error = "too many blocks in one wave"; return CZS_UNSUPPORTED; }
    }
    const int n_sets = (n_waves > 1 && !ctx->no_overlap) ? 2 : 1;
    for (int s = 0; s < n_sets; s++) {
        if ((rc = ensure(ctx, ctx->counters[s], 1))) return rc;
        if ((rc = ensure(ctx, ctx->blocks[s], mx.n_blocks + 2))) return rc;
        if ((rc = ensure(ctx, ctx->huf_items[s], mx.n_huf + 1))) return rc;
        if ((rc = ensure(ctx, ctx->exec_order[s], W + 1))) return rc;
        if ((rc = ensure(ctx, ctx->huf_cls0[s], mx.n_huf + 1))) return rc;
        if ((rc = ensure(ctx, ctx->huf_cls1[s], mx.n_huf + 1))) return rc;
        if ((rc = ensure(ctx, ctx->huf_recs[s], mx.n_huf + 1))) return rc;
        if ((rc = ensure(ctx, ctx->fse_items[s], mx.n_fse + 1))) return rc;
        if ((rc = ensure(ctx, ctx->lit[s], mx.lit_bytes + 64 + kGuardBytes))) return rc;
        if ((rc = ensure(ctx, ctx->seq[s], mx.n_seq + 2 + kGuardBytes / sizeof(Seq)))) return rc;
    }

    if (plan_out) return CZS_OK;  // scratch is sized, nothing else to do
    { ProfScope ps(ctx, stream, 6); launch_header_results(lc, ctx->infos.p, results, n); }
    // Two-stage pipeline over waves: the entropy stage (fill, Huffman, FSE: shared-memory bound, few
    // warps per SM) runs on `stream`; sequence execution (many warps, almost no shared memory) runs
    // on exec_stream and overlaps the entropy stage of the next wave.  Scratch is double-buffered.
    const bool overlap = n_waves > 1 && !ctx->no_overlap;
    cudaStream_t xs = overlap ? ctx->exec_stream : stream;
    LaunchCtx lx{xs, &ctx->launches};
    if (overlap) {
        CZB_CUDA(ctx, cudaEventRecord(ctx->ev_fork, stream));
        CZB_CUDA(ctx, cudaStreamWaitEvent(xs, ctx->ev_fork, 0));
    }
    for (uint64_t w = 0; w < n_waves; w++) {
        const int s = overlap ? (int)(w & 1) : 0;
        const uint64_t first = w * W, count = std::min<uint64_t>(W, n - first);
        const WaveTotals& t = totals_host[w];
        uint32_t n_exec = 0, n_big = 0;
        for (int c = 0; c < 32; c++) { n_exec += t.frame_cls[c]; if (c >= ctx->share_cls) n_big += t.frame_cls[c]; }
        // Share rule of k_exec_big (see frame_is_big): frames that hold at least 1/big_share of the wave's compressed bytes.
        // A CTA per frame only pays while the CTAs all fit the machine at once (seven per SM): with more frames than that
        // in the wave, only frames well above the mean qualify, so a large batch of equal frames stays with k_exec
        // (4096 equal 256 KiB frames: 2.4 ms one warp each, 5.3 ms one CTA each; 1024 of them: 1.6 against 1.4 ms).
        uint64_t share_bytes = 0;  // big_seq_bytes == 0 (test knob): every frame of the class
        if (ctx->big_seq_bytes) {
            share_bytes = (uint64_t)t.src_bytes / (uint64_t)ctx->big_share + 1;
            if (count > (uint64_t)ctx->big_resident) share_bytes = std::max<uint64_t>(share_bytes, (uint64_t)t.src_bytes * 3 / (2 * count) + 1);
        }
        // Which CTA-per-frame executor: k_exec_flow gives one frame 16 warps and moves it ~1.8x faster than k_exec_big's four, but only
        // two of its CTAs fit an SM against seven.  With more large frames in the wave than flow CTAs fit the machine at once the
        // aggregate rate is what counts, and k_exec_big's is higher (mixed 1 KiB..4 MiB batch: 149 against 106 GB/s).
        bool use_flow = ctx->big_flow, flow_wide = false;
        if (use_flow && !ctx->big_seq_bytes) flow_wide = ctx->flow_wide_forced;  // test knob: every frame through one shape
        if (use_flow && ctx->big_seq_bytes) {
            const uint32_t share_c = share_bytes > 1 ? size_class(share_bytes - 1) : 0u;
            const uint32_t lo_c = std::min<uint32_t>((uint32_t)ctx->big_cls, std::max<uint32_t>((uint32_t)ctx->share_cls, share_c));
            uint64_t est = 0;
            for (uint32_t c = lo_c; c < 32; c++) est += t.frame_cls[c];
            use_flow = est <= ctx->flow_max;
            flow_wide = est <= (uint64_t)ctx->sm_count;  // at most one large frame per SM: the 32-warp shape with the 128 KiB window
        }
        if (overlap && w >= 2) CZB_CUDA(ctx, cudaStreamWaitEvent(stream, ctx->ev_exec[s], 0));  // scratch set s is free again
        if (ctx->guard) {
            if ((rc = ensure(ctx, ctx->guard_faults, 1))) return rc;
            if (!ctx->guard_zeroed) { CZB_CUDA(ctx, cudaMemsetAsync(ctx->guard_faults.p, 0, sizeof(unsigned long long), stream)); ctx->guard_zeroed = true; }
            CZB_CUDA(ctx, cudaMemsetAsync(ctx->lit[s].p + t.lit_bytes, kGuardByte, kGuardBytes, stream));
            CZB_CUDA(ctx, cudaMemsetAsync(reinterpret_cast<uint8_t*>(ctx->seq[s].p + t.n_seq), kGuardByte, kGuardBytes, stream));
            CZB_CUDA(ctx, cudaMemsetAsync(reinterpret_cast<uint8_t*>(ctx->blocks[s].p + t.n_blocks), kGuardByte, kGuardBytes, stream));
        }
        CZB_CUDA(ctx, cudaMemsetAsync(ctx->counters[s].p, 0, sizeof(WaveCounters), stream));
        { ProfScope ps(ctx, stream, 1); launch_fill_blocks(lc, descs, ctx->infos.p, first, count, ctx->blocks[s].p, ctx->huf_items[s].p, ctx->fse_items[s].p, ctx->counters[s].p, ctx->totals_d.p + w, ctx->exec_order[s].p, resume); }
        if (!(flags & kFlagSizesOnly)) { ProfScope ps(ctx, stream, 2); launch_huff(lc, descs + first, ctx->blocks[s].p, ctx->huf_items[s].p, ctx->counters[s].p, (uint32_t)t.n_huf, ctx->lit[s].p, ctx->huf_recs[s].p, ctx->huf_cls0[s].p, ctx->huf_cls1[s].p, ctx->huf_big.p); }
        { ProfScope ps(ctx, stream, 3); launch_fse(lc, descs + first, ctx->blocks[s].p, ctx->fse_items[s].p, ctx->counters[s].p, (uint32_t)t.n_fse, ctx->seq[s].p); }
        if (overlap) {
            CZB_CUDA(ctx, cudaEventRecord(ctx->ev_entropy[s], stream));
            CZB_CUDA(ctx, cudaStreamWaitEvent(xs, ctx->ev_entropy[s], 0));
        }
        if (flags & kFlagSizesOnly) { ProfScope ps(ctx, xs, 7); launch_frame_sizes(lx, ctx->infos.p, first, count, ctx->blocks[s].p, results); }
        else { ProfScope ps(ctx, xs, 4); launch_exec(lx, ExecSide{ctx->big_stream, ctx->ev_big_fork, ctx->ev_big_join, use_flow, flow_wide, resume}, ctx->sm_count, descs, ctx->infos.p, first, count, n_big, n_exec, BigRule{(uint32_t)ctx->big_cls, (uint32_t)ctx->big_seq_bytes, (uint32_t)ctx->share_cls, share_bytes}, ctx->counters[s].p, ctx->exec_order[s].p, ctx->blocks[s].p, ctx->lit[s].p, ctx->seq[s].p, results); }
        if ((flags & CZB_FLAG_VERIFY_CHECKSUM) && !(flags & kFlagSizesOnly)) { ProfScope ps(ctx, xs, 5); launch_xxh64(lx, descs, results, first, count); }
        if (ctx->guard)
            k_check_guards<<<1, 192, 0, xs>>>(ctx->lit[s].p + t.lit_bytes, reinterpret_cast<const uint8_t*>(ctx->seq[s].p + t.n_seq),
                                              reinterpret_cast<const uint8_t*>(ctx->blocks[s].p + t.n_blocks), ctx->guard_faults.p);
        if (overlap) CZB_CUDA(ctx, cudaEventRecord(ctx->ev_exec[s], xs));
        ctx->last_wave = t; ctx->last_wave_first = first; ctx->last_wave_count = count; ctx->last_set = s;
    }
    if (overlap) {  // join: later work on `stream` sees every result
        CZB_CUDA(ctx, cudaStreamWaitEvent(stream, ctx->ev_exec[(n_waves - 1) & 1], 0));
        if (n_waves > 1) CZB_CUDA(ctx, cudaStreamWaitEvent(stream, ctx->ev_exec[(n_waves - 2) & 1], 0));
    }
    if (!capturing) {
        CZB_CUDA(ctx, cudaEventRecord(ctx->ev_scratch_free, stream));  // after the join: every kernel of this call is ordered before it
        ctx->scratch_in_use = true;
    }
    CZB_CUDA(ctx, cudaGetLastError());
    return CZS_OK;
}

extern "C" int czb_decode_batch_device(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n,
                                       uint32_t flags, void* stream_v) {
    return czb_decode_batch_device_resume(ctx, descs, results, n, flags & ~kFlagSizesOnly, stream_v, nullptr);
}

extern "C" int czb_plan_batch_device(czb_context* ctx, const czb_frame_desc* descs, uint64_t n, void* stream_v, czb_batch_plan** out) {
    if (!ctx || !out || (n && !descs)) return CZS_BAD_ARGUMENT;
    *out = nullptr;
    czb_batch_plan* p = new czb_batch_plan();
    const int rc = n ? decode_batch_impl(ctx, descs, nullptr, n, 0, stream_v, nullptr, nullptr, p) : CZS_OK;
    if (rc != CZS_OK) { delete p; return rc; }
    *out = p;
    return CZS_OK;
}
extern "C" void czb_plan_destroy(czb_batch_plan* plan) { delete plan; }
extern "C" int czb_decode_batch_device_planned(czb_context* ctx, const czb_batch_plan* plan, const czb_frame_desc* descs,
                                               czb_frame_result* results, uint64_t n, uint32_t flags, void* stream_v) {
    if (!plan) return CZS_BAD_ARGUMENT;
    if (n == 0) return CZS_OK;
    return decode_batch_impl(ctx, descs, results, n, flags & ~kFlagSizesOnly, stream_v, nullptr, plan, nullptr);
}

extern "C" int czb_frame_sizes_device(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n, void* stream_v) {
    return czb_decode_batch_device_resume(ctx, descs, results, n, kFlagSizesOnly, stream_v, nullptr);
}

// ---- host-pointer forms ---------------------------------------------------------------------
static int ensure_pinned(czb_context* ctx, uint8_t*& p, uint64_t& cap, uint64_t n) {
    if (n <= cap) return CZS_OK;
    if (p) CZB_CUDA(ctx, cudaFreeHost(p));
    p = nullptr; cap = 0;
    CZB_CUDA(ctx, cudaMallocHost(reinterpret_cast<void**>(&p), n));
    cap = n;
    return CZS_OK;
}

extern "C" int czb_decode_batch_host(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n,
                                     uint32_t flags) {
    if (!ctx || (n && (!descs || !results))) return CZS_BAD_ARGUMENT;
    if (n == 0) return CZS_OK;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    // gather sources into one pinned staging buffer (16-byte aligned per frame), one H2D copy
    std::vector<uint64_t> soff(n + 1), doff(n + 1);
    uint64_t stot = 0, dtot = 0;
    for (uint64_t i = 0; i < n; i++) {
        soff[i] = stot; doff[i] = dtot;
        stot += (descs[i].src_len + 15) & ~15ull;
        dtot += (descs[i].dst_cap + 15) & ~15ull;
    }
    soff[n] = stot; doff[n] = dtot;
    int rc;
    if ((rc = ensure_pinned(ctx, ctx->pin_a, ctx->pin_a_cap, stot + 16))) return rc;
    if ((rc = ensure_pinned(ctx, ctx->pin_b, ctx->pin_b_cap, std::max<uint64_t>(n * sizeof(czb_frame_desc), n * sizeof(czb_frame_result))))) return rc;
    if ((rc = ensure(ctx, ctx->h_src[0], stot + 16))) return rc;
    if ((rc = ensure(ctx, ctx->h_dst[0], dtot + 16))) return rc;
    if ((rc = ensure(ctx, ctx->h_descs, n))) return rc;
    if ((rc = ensure(ctx, ctx->h_results, n))) return rc;
    for (uint64_t i = 0; i < n; i++)
        if (descs[i].src_len) memcpy(ctx->pin_a + soff[i], descs[i].src, descs[i].src_len);
    czb_frame_desc* hd = reinterpret_cast<czb_frame_desc*>(ctx->pin_b);
    for (uint64_t i = 0; i < n; i++) {
        hd[i].src = ctx->h_src[0].p + soff[i]; hd[i].src_len = descs[i].src_len;
        hd[i].dst = ctx->h_dst[0].p + doff[i]; hd[i].dst_cap = descs[i].dst_cap;
    }
    cudaStream_t st = ctx->compute;
    CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_src[0].p, ctx->pin_a, stot, cudaMemcpyHostToDevice, st));
    CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_descs.p, hd, n * sizeof(czb_frame_desc), cudaMemcpyHostToDevice, st));
    if ((rc = czb_decode_batch_device(ctx, ctx->h_descs.p, ctx->h_results.p, n, flags, st))) return rc;
    CZB_CUDA(ctx, cudaMemcpyAsync(ctx->pin_b, ctx->h_results.p, n * sizeof(czb_frame_result), cudaMemcpyDeviceToHost, st));
    CZB_CUDA(ctx, cudaStreamSynchronize(st));
    memcpy(results, ctx->pin_b, n * sizeof(czb_frame_result));
    // copy back only what was produced, frame by frame for small batches, else one span
    uint64_t produced_end = 0;
    for (uint64_t i = 0; i < n; i++) if (results[i].status == CZS_OK && results[i].bytes_written) produced_end = doff[i] + results[i].bytes_written;
    if (produced_end) {
        if ((rc = ensure_pinned(ctx, ctx->pin_a, ctx->pin_a_cap, produced_end))) return rc;
        CZB_CUDA(ctx, cudaMemcpyAsync(ctx->pin_a, ctx->h_dst[0].p, produced_end, cudaMemcpyDeviceToHost, st));
        CZB_CUDA(ctx, cudaStreamSynchronize(st));
        for (uint64_t i = 0; i < n; i++)
            if (results[i].status == CZS_OK && results[i].bytes_written) memcpy(descs[i].dst, ctx->pin_a + doff[i], results[i].bytes_written);
    }
    return CZS_OK;
}

// Packed form: chunked, transfers overlapped with decoding (three streams, two staging slots).
extern "C" int czb_decode_batch_host_packed(czb_context* ctx, const uint8_t* src_base, const uint64_t* src_off, uint8_t* dst_base,
                                            const uint64_t* dst_off, czb_frame_result* results, uint64_t n, uint32_t flags) {
    if (!ctx || (n && (!src_base || !src_off || !dst_base || !dst_off || !results))) return CZS_BAD_ARGUMENT;
    if (n == 0) return CZS_OK;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    // chunk boundaries: bounded staging (src + dst bytes per chunk) and bounded frame count
    const uint64_t kChunkBytes = ctx->host_chunk_bytes;
    std::vector<uint64_t> cuts{0};
    {
        uint64_t i = 0;
        while (i < n) {
            uint64_t j = i + 1;
            while (j < n && j - i < 65536 && (src_off[j + 1] - src_off[i]) + (dst_off[j + 1] - dst_off[i]) <= kChunkBytes) j++;
            cuts.push_back(j);
            i = j;
        }
    }
    const uint64_t n_chunks = cuts.size() - 1;
    uint64_t max_src = 0, max_dst = 0, max_frames = 0;
    for (uint64_t c = 0; c < n_chunks; c++) {
        max_src = std::max(max_src, src_off[cuts[c + 1]] - src_off[cuts[c]]);
        max_dst = std::max(max_dst, dst_off[cuts[c + 1]] - dst_off[cuts[c]]);
        max_frames = std::max(max_frames, cuts[c + 1] - cuts[c]);
    }
    int rc;
    constexpr int NS = czb_context::kHostSlots;
    for (int s = 0; s < NS; s++) {
        if ((rc = ensure(ctx, ctx->h_src[s], max_src + 64))) return rc;
        if ((rc = ensure(ctx, ctx->h_dst[s], max_dst + 64))) return rc;
    }
    if ((rc = ensure(ctx, ctx->h_descs, NS * max_frames))) return rc;
    if ((rc = ensure(ctx, ctx->h_results, NS * max_frames))) return rc;
    if ((rc = ensure_pinned(ctx, ctx->pin_b, ctx->pin_b_cap, NS * max_frames * sizeof(czb_frame_desc)))) return rc;
    cudaEvent_t* ev_in = ctx->ev_in; cudaEvent_t* ev_dec = ctx->ev_dec; cudaEvent_t* ev_out = ctx->ev_out;  // owned by the context: nothing to leak on an early return
    const bool dbg = getenv("CZB_E2E_DEBUG") != nullptr;
    std::vector<cudaEvent_t> tev;  // debug: 6 timing events per chunk (h2d begin/end, decode begin/end, d2h begin/end)
    cudaEvent_t t0ev = nullptr;
    auto tmark = [&](cudaStream_t st) { if (dbg) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev.push_back(e); } };
    if (dbg) { cudaEventCreate(&t0ev); cudaEventRecord(t0ev, ctx->copy_in); }
    auto now_ms = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    auto enqueue_in = [&](uint64_t c) -> int {
        const int s = (int)(c % NS);
        const uint64_t f0 = cuts[c], f1 = cuts[c + 1], nf = f1 - f0;
        // slot s is free once chunk c-NS's outputs have been copied out
        if (c >= (uint64_t)NS) CZB_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_in, ev_out[s], 0));
        // the aligned base keeps each frame's alignment relative to src_base
        const uint64_t sb = src_off[f0], mis = sb & 15;
        tmark(ctx->copy_in);
        CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_src[s].p + mis, src_base + sb, src_off[f1] - sb, cudaMemcpyHostToDevice, ctx->copy_in));
        tmark(ctx->copy_in);
        czb_frame_desc* hd = reinterpret_cast<czb_frame_desc*>(ctx->pin_b) + (uint64_t)s * max_frames;
        const uint64_t db = dst_off[f0], dmis = db & 15;
        for (uint64_t i = 0; i < nf; i++) {
            hd[i].src = ctx->h_src[s].p + mis + (src_off[f0 + i] - sb); hd[i].src_len = src_off[f0 + i + 1] - src_off[f0 + i];
            hd[i].dst = ctx->h_dst[s].p + dmis + (dst_off[f0 + i] - db); hd[i].dst_cap = dst_off[f0 + i + 1] - dst_off[f0 + i];
        }
        CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_descs.p + (uint64_t)s * max_frames, hd, nf * sizeof(czb_frame_desc), cudaMemcpyHostToDevice, ctx->copy_in));
        CZB_CUDA(ctx, cudaEventRecord(ev_in[s], ctx->copy_in));
        return CZS_OK;
    };
    const double t_begin = now_ms();
    if ((rc = enqueue_in(0))) return rc;
    for (uint64_t c = 0; c < n_chunks; c++) {
        const double t_iter = now_ms();
        const int s = (int)(c % NS);
        const uint64_t f0 = cuts[c], f1 = cuts[c + 1], nf = f1 - f0;
        if (c + 1 < n_chunks) {
            // pin_b's descriptor part for that slot is reused: its previous H2D (chunk c+1-NS) completed long ago,
            // because that chunk's decode (which waited on it) was planned with a stream sync.
            if ((rc = enqueue_in(c + 1))) return rc;
        }
        CZB_CUDA(ctx, cudaStreamWaitEvent(ctx->compute, ev_in[s], 0));
        tmark(ctx->compute);
        if ((rc = czb_decode_batch_device(ctx, ctx->h_descs.p + (uint64_t)s * max_frames, ctx->h_results.p + (uint64_t)s * max_frames, nf,
                                          flags, ctx->compute))) return rc;
        tmark(ctx->compute);
        CZB_CUDA(ctx, cudaEventRecord(ev_dec[s], ctx->compute));
        CZB_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_out, ev_dec[s], 0));
        const uint64_t db = dst_off[f0], dmis = db & 15;
        tmark(ctx->copy_out);
        CZB_CUDA(ctx, cudaMemcpyAsync(dst_base + db, ctx->h_dst[s].p + dmis, dst_off[f1] - db, cudaMemcpyDeviceToHost, ctx->copy_out));
        tmark(ctx->copy_out);
        CZB_CUDA(ctx, cudaMemcpyAsync(results + f0, ctx->h_results.p + (uint64_t)s * max_frames, nf * sizeof(czb_frame_result),
                                      cudaMemcpyDeviceToHost, ctx->copy_out));
        CZB_CUDA(ctx, cudaEventRecord(ev_out[s], ctx->copy_out));
        if (dbg) fprintf(stderr, "[e2e] chunk %llu frames %llu: iter start %.1f ms, iter took %.1f ms\n", (unsigned long long)c,
                         (unsigned long long)nf, t_iter - t_begin, now_ms() - t_iter);
    }
    CZB_CUDA(ctx, cudaStreamSynchronize(ctx->copy_out));
    if (dbg) {
        fprintf(stderr, "[e2e] total %.1f ms\n", now_ms() - t_begin);
        cudaDeviceSynchronize();
        // event order per chunk c: enqueue_in(c) pushes 2 (h2d), then the loop body pushes 2 (decode) + 2 (d2h);
        // enqueue_in(c+1) is called before chunk c's decode, so sort by kind using the push pattern.
        std::vector<float> t(tev.size());
        for (size_t i = 0; i < tev.size(); i++) cudaEventElapsedTime(&t[i], t0ev, tev[i]);
        for (size_t i = 0; i + 1 < tev.size(); i += 2) fprintf(stderr, "[e2e-gpu] op %zu: [%.1f, %.1f] ms (%.1f)\n", i / 2, t[i], t[i + 1], t[i + 1] - t[i]);
        for (auto e : tev) cudaEventDestroy(e);
        cudaEventDestroy(t0ev);
    }
    CZB_CUDA(ctx, cudaStreamSynchronize(ctx->compute));
    return CZS_OK;
}

extern "C" int czb_frame_sizes_host(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n) {
    if (!ctx || (n && (!descs || !results))) return CZS_BAD_ARGUMENT;
    if (n == 0) return CZS_OK;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<uint64_t> soff(n + 1);
    uint64_t stot = 0;
    for (uint64_t i = 0; i < n; i++) { soff[i] = stot; stot += (descs[i].src_len + 15) & ~15ull; }
    int rc;
    if ((rc = ensure_pinned(ctx, ctx->pin_a, ctx->pin_a_cap, stot + 16))) return rc;
    if ((rc = ensure_pinned(ctx, ctx->pin_b, ctx->pin_b_cap, std::max<uint64_t>(n * sizeof(czb_frame_desc), n * sizeof(czb_frame_result))))) return rc;
    if ((rc = ensure(ctx, ctx->h_src[0], stot + 16))) return rc;
    if ((rc = ensure(ctx, ctx->h_descs, n))) return rc;
    if ((rc = ensure(ctx, ctx->h_results, n))) return rc;
    czb_frame_desc* hd = reinterpret_cast<czb_frame_desc*>(ctx->pin_b);
    for (uint64_t i = 0; i < n; i++) {
        if (descs[i].src_len) memcpy(ctx->pin_a + soff[i], descs[i].src, descs[i].src_len);
        hd[i].src = ctx->h_src[0].p + soff[i]; hd[i].src_len = descs[i].src_len; hd[i].dst = nullptr; hd[i].dst_cap = 0;
    }
    cudaStream_t st = ctx->compute;
    CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_src[0].p, ctx->pin_a, stot, cudaMemcpyHostToDevice, st));
    CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_descs.p, hd, n * sizeof(czb_frame_desc), cudaMemcpyHostToDevice, st));
    if ((rc = czb_decode_batch_device_resume(ctx, ctx->h_descs.p, ctx->h_results.p, n, kFlagSizesOnly, st, nullptr))) return rc;
    CZB_CUDA(ctx, cudaMemcpyAsync(ctx->pin_b, ctx->h_results.p, n * sizeof(czb_frame_result), cudaMemcpyDeviceToHost, st));
    CZB_CUDA(ctx, cudaStreamSynchronize(st));
    memcpy(results, ctx->pin_b, n * sizeof(czb_frame_result));
    return CZS_OK;
}

// ---- batch splitter (SURVEY.md section 8 row f2) ------------------------------------------------
extern "C" int czb_split_frames_host(const uint8_t* buf, uint64_t len, czb_frame_span* spans, uint64_t cap, uint64_t* n_frames,
                                     uint64_t* n_skipped, uint64_t* consumed) {
    if ((!buf && len) || (!spans && cap) || !n_frames) return CZS_BAD_ARGUMENT;
    uint64_t n = 0, sk = 0, pos = 0;
    const int32_t st = split_frames_walk(buf, len, spans, cap, n, sk, pos);
    *n_frames = n;
    if (n_skipped) *n_skipped = sk;
    if (consumed) *consumed = pos;
    return st;
}
extern "C" int czb_split_frames_device(czb_context* ctx, const uint8_t* buf, uint64_t len, czb_frame_span* spans, uint64_t cap,
                                       uint64_t* counts, void* stream_v) {
    if (!ctx || (!buf && len) || (!spans && cap) || !counts) return CZS_BAD_ARGUMENT;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    LaunchCtx lc{static_cast<cudaStream_t>(stream_v), &ctx->launches};
    launch_split_frames(lc, buf, len, spans, cap, reinterpret_cast<unsigned long long*>(counts));
    CZB_CUDA(ctx, cudaGetLastError());
    return CZS_OK;
}

// ---- one host batch over several GPUs (SURVEY.md section 8e) --------------------------------------
extern "C" int czb_partition_frames(const uint64_t* cost, uint64_t n, uint32_t n_shards, uint32_t* shard_of, uint64_t* shard_load) {
    if (!n_shards || (n && (!cost || !shard_of))) return CZS_BAD_ARGUMENT;
    std::vector<uint64_t> order(n), load(n_shards, 0);
    for (uint64_t i = 0; i < n; i++) order[i] = i;
    std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return cost[a] != cost[b] ? cost[a] > cost[b] : a < b; });
    // largest first onto the least loaded shard (ties: lowest shard index); a heap keeps it O(n log shards)
    using Slot = std::pair<uint64_t, uint32_t>;
    std::vector<Slot> heap;
    for (uint32_t sI = 0; sI < n_shards; sI++) heap.push_back({0, sI});
    auto worse = [](const Slot& a, const Slot& b) { return a.first != b.first ? a.first > b.first : a.second > b.second; };
    std::make_heap(heap.begin(), heap.end(), worse);
    for (uint64_t k = 0; k < n; k++) {
        std::pop_heap(heap.begin(), heap.end(), worse);
        Slot& sl = heap.back();
        shard_of[order[k]] = sl.second;
        sl.first += cost[order[k]]; load[sl.second] = sl.first;
        std::push_heap(heap.begin(), heap.end(), worse);
    }
    if (shard_load) for (uint32_t sI = 0; sI < n_shards; sI++) shard_load[sI] = load[sI];
    return CZS_OK;
}

struct czb_multi {
    std::vector<czb_context*> ctxs;
    std::vector<int> devices;
};
extern "C" int czb_multi_create(const int* devices, int n_devices, uint64_t budget, czb_multi** out) {
    if (!out || !devices || n_devices <= 0) return CZS_BAD_ARGUMENT;
    *out = nullptr;
    czb_multi* m = new czb_multi();
    for (int d = 0; d < n_devices; d++) {
        czb_context* c = nullptr;
        const int rc = czb_context_create(devices[d], budget, &c);
        if (rc != CZS_OK) { czb_multi_destroy(m); return rc; }
        m->ctxs.push_back(c); m->devices.push_back(devices[d]);
    }
    *out = m;
    return CZS_OK;
}
extern "C" void czb_multi_destroy(czb_multi* m) {
    if (!m) return;
    for (auto c : m->ctxs) czb_context_destroy(c);
    delete m;
}
extern "C" int czb_decode_batch_multi(czb_multi* m, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n, uint32_t flags,
                                      czb_shard_stat* stats) {
    if (!m || (n && (!descs || !results))) return CZS_BAD_ARGUMENT;
    const uint32_t S = (uint32_t)m->ctxs.size();
    std::vector<uint64_t> cost(n);
    for (uint64_t i = 0; i < n; i++) cost[i] = descs[i].src_len + descs[i].dst_cap;
    std::vector<uint32_t> shard_of(n);
    int rc = czb_partition_frames(cost.data(), n, S, shard_of.data(), nullptr);
    if (rc != CZS_OK) return rc;
    std::vector<std::vector<uint64_t>> idx(S);
    for (uint64_t i = 0; i < n; i++) idx[shard_of[i]].push_back(i);
    std::vector<int> rcs(S, CZS_OK);
    std::vector<double> ms(S, 0.0);
    std::vector<std::thread> th;
    auto now_ms = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    for (uint32_t sI = 0; sI < S; sI++) {
        th.emplace_back([&, sI]() {  // one host thread per device: a context is not shareable, different contexts are
            const double t0 = now_ms();
            const std::vector<uint64_t>& ix = idx[sI];
            std::vector<czb_frame_desc> d(ix.size());
            std::vector<czb_frame_result> r(ix.size());
            for (size_t k = 0; k < ix.size(); k++) d[k] = descs[ix[k]];
            rcs[sI] = czb_decode_batch_host(m->ctxs[sI], d.data(), r.data(), ix.size(), flags);
            if (rcs[sI] == CZS_OK) for (size_t k = 0; k < ix.size(); k++) results[ix[k]] = r[k];  // disjoint slots: the only "gather"
            ms[sI] = now_ms() - t0;
        });
    }
    for (auto& t : th) t.join();
    if (stats) {
        for (uint32_t sI = 0; sI < S; sI++) {
            czb_shard_stat& st = stats[sI];
            st.device = m->devices[sI]; st.pad = 0; st.frames = idx[sI].size(); st.bytes_in = 0; st.bytes_out = 0; st.ms = ms[sI];
            for (uint64_t i : idx[sI]) { st.bytes_in += descs[i].src_len; if (rcs[sI] == CZS_OK && results[i].status == CZS_OK) st.bytes_out += results[i].bytes_written; }
        }
    }
    for (uint32_t sI = 0; sI < S; sI++) if (rcs[sI] != CZS_OK) return rcs[sI];
    return CZS_OK;
}
extern "C" const char* czb_multi_last_error(const czb_multi* m, int shard) {
    return (m && shard >= 0 && (size_t)shard < m->ctxs.size()) ? czb_last_error(m->ctxs[shard]) : "bad shard";
}

// ---- dictionaries: the reference's parse, mirrored (row f4) ---------------------------------------
extern "C" int czb_dictionary_parse_host(czb_context* ctx, const uint8_t* dict, uint64_t len, czb_dictionary_info* out) {
    if (!ctx || !out || (!dict && len)) return CZS_BAD_ARGUMENT;
    memset(out, 0, sizeof *out);
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if ((rc = ensure(ctx, ctx->h_src[0], len + 64))) return rc;
    if ((rc = ensure(ctx, ctx->h_results, 4))) return rc;  // reused as the output slot (sizeof(czb_dictionary_info) <= 4 results)
    static_assert(sizeof(czb_dictionary_info) <= 4 * sizeof(czb_frame_result), "output slot");
    cudaStream_t st = ctx->compute;
    if (ctx->scratch_in_use) CZB_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_scratch_free, 0));
    if (!ctx->huf_big.p) {
        if ((rc = ensure(ctx, ctx->huf_big, huff_big_scratch_bytes()))) return rc;
        CZB_CUDA(ctx, cudaMemsetAsync(ctx->huf_big.p, 0, 64, st));
    }
    if (len) CZB_CUDA(ctx, cudaMemcpyAsync(ctx->h_src[0].p, dict, len, cudaMemcpyHostToDevice, st));
    LaunchCtx lc{st, &ctx->launches};
    launch_dict_parse(lc, ctx->h_src[0].p, len, reinterpret_cast<czb_dictionary_info*>(ctx->h_results.p), ctx->huf_big.p);
    CZB_CUDA(ctx, cudaMemcpyAsync(out, ctx->h_results.p, sizeof *out, cudaMemcpyDeviceToHost, st));
    CZB_CUDA(ctx, cudaStreamSynchronize(st));
    return out->status;
}

// ---- header pre-pass (CPU only) ---------------------------------------------------------------
extern "C" int czb_frame_header_info_host(const uint8_t* src, uint64_t src_len, czb_frame_header_info* out) {
    if (!out || (!src && src_len)) return CZS_BAD_ARGUMENT;
    memset(out, 0, sizeof *out);
    FrameHeader fh{};
    int32_t st = parse_frame_header(src, src_len, fh);
    uint64_t ws = 0;
    if (st == CZS_OK) st = frame_window_size(fh, false, ws);
    out->status = st;
    if (st != CZS_OK) return st;
    out->header_len = fh.hdr_len; out->content_size = fh.fcs; out->window_size = ws;
    out->fcs_present = fh.fcs_bytes != 0; out->has_checksum_flag = (fh.descriptor >> 2) & 1;
    out->single_segment = (fh.descriptor >> 5) & 1; out->dict_id = fh.dict_id;
    return CZS_OK;
}

extern "C" int czb_find_frame_end_host(const uint8_t* src, uint64_t src_len, uint64_t* frame_len) {
    if (!frame_len || (!src && src_len)) return CZS_BAD_ARGUMENT;
    *frame_len = 0;
    FrameHeader fh{};
    int32_t st = parse_frame_header(src, src_len, fh);
    if (st != CZS_OK) return st;
    uint64_t pos = fh.hdr_len;
    for (;;) {
        ParsedBlock pb;
        parse_block_at(src, src_len, pos, pb);
        if (pb.hdr_status != CZS_OK) return pb.hdr_status;
        pos += 3 + pb.content;
        if (pb.last) break;
    }
    if ((fh.descriptor >> 2) & 1) { if (src_len - pos < 4) return CZS_PANIC_TRUNCATED; pos += 4; }
    *frame_len = pos;
    return CZS_OK;
}

// ---- debug taps ---------------------------------------------------------------------------------
extern "C" int czb_debug_guard_faults(czb_context* ctx, uint64_t* faults) {  // CZB_GUARD=1: guard bytes found overwritten so far
    if (!ctx || !faults) return CZS_BAD_ARGUMENT;
    *faults = 0;
    if (!ctx->guard || !ctx->guard_faults.p) return CZS_OK;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    CZB_CUDA(ctx, cudaDeviceSynchronize());
    unsigned long long v = 0;
    CZB_CUDA(ctx, cudaMemcpy(&v, ctx->guard_faults.p, sizeof v, cudaMemcpyDeviceToHost));
    *faults = v;
    return CZS_OK;
}
static_assert(sizeof(czb_debug_wave_totals) == sizeof(WaveTotals) && offsetof(czb_debug_wave_totals, src_bytes) == offsetof(WaveTotals, src_bytes) &&
              offsetof(czb_debug_wave_totals, frame_cls) == offsetof(WaveTotals, frame_cls) &&
              offsetof(czb_debug_wave_totals, fse_cls) == offsetof(WaveTotals, fse_cls), "czb_debug_wave_totals mirrors WaveTotals");
extern "C" int czb_debug_plan_waves(const czb_batch_plan* plan, uint64_t* wave_frames, uint64_t* n_waves, czb_debug_wave_totals* out,
                                    uint64_t cap) {
    if (!plan || (cap && !out)) return CZS_BAD_ARGUMENT;
    if (wave_frames) *wave_frames = plan->W;
    if (n_waves) *n_waves = plan->n_waves;
    const uint64_t k = std::min<uint64_t>(cap, plan->totals.size());
    if (k) memcpy(out, plan->totals.data(), k * sizeof(WaveTotals));
    return CZS_OK;
}
extern "C" int czb_debug_last_wave_counts(czb_context* ctx, uint64_t* n_blocks, uint64_t* lit_bytes, uint64_t* n_seq) {
    if (!ctx) return CZS_BAD_ARGUMENT;
    if (n_blocks) *n_blocks = ctx->last_wave.n_blocks;
    if (lit_bytes) *lit_bytes = ctx->last_wave.lit_bytes;
    if (n_seq) *n_seq = ctx->last_wave.n_seq;
    return CZS_OK;
}
extern "C" int czb_debug_copy_blocks(czb_context* ctx, czb_debug_block* out, uint64_t cap) {
    if (!ctx || !out) return CZS_BAD_ARGUMENT;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    CZB_CUDA(ctx, cudaDeviceSynchronize());
    const uint64_t nb = std::min<uint64_t>(cap, ctx->last_wave.n_blocks);
    std::vector<BlockDesc> h(nb);
    if (nb) CZB_CUDA(ctx, cudaMemcpy(h.data(), ctx->blocks[ctx->last_set].p, nb * sizeof(BlockDesc), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < nb; i++) {
        const BlockDesc& d = h[i];
        czb_debug_block& o = out[i];
        o.frame = d.frame; o.block_type = d.type; o.lit_type = d.lit_type; o.n_streams = d.n_streams; o.modes = d.modes;
        o.regen_size = d.regen; o.n_seq = d.n_seq; o.lit_off = d.lit_off; o.seq_off = d.seq_off;
        int32_t st = d.pre_status;
        if (st == CZS_OK && d.type == BT_COMPRESSED) {
            if (d.lit_type >= LT_COMPRESSED && d.huf_status != CZS_OK) st = d.huf_status;
            else if (d.seqhdr_status != CZS_OK) st = d.seqhdr_status;
            else if (d.n_seq && d.fse_status != CZS_OK) st = d.fse_status;
        }
        o.status = st;
    }
    return CZS_OK;
}
extern "C" int czb_debug_copy_literals(czb_context* ctx, uint8_t* out, uint64_t cap) {
    if (!ctx || !out) return CZS_BAD_ARGUMENT;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    CZB_CUDA(ctx, cudaDeviceSynchronize());
    const uint64_t nbytes = std::min<uint64_t>(cap, ctx->last_wave.lit_bytes);
    if (nbytes) CZB_CUDA(ctx, cudaMemcpy(out, ctx->lit[ctx->last_set].p, nbytes, cudaMemcpyDeviceToHost));
    return CZS_OK;
}
extern "C" int czb_debug_copy_sequences(czb_context* ctx, uint32_t* out, uint64_t cap_seqs) {
    if (!ctx || !out) return CZS_BAD_ARGUMENT;
    CZB_CUDA(ctx, cudaSetDevice(ctx->device));
    CZB_CUDA(ctx, cudaDeviceSynchronize());
    const uint64_t ns = std::min<uint64_t>(cap_seqs, ctx->last_wave.n_seq);
    std::vector<Seq> h(ns);
    if (ns) CZB_CUDA(ctx, cudaMemcpy(h.data(), ctx->seq[ctx->last_set].p, ns * sizeof(Seq), cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < ns; i++) {
        out[3 * i] = seq_ll(h[i]); out[3 * i + 1] = seq_ml(h[i]);
        const uint32_t f = seq_off29(h[i]);
        out[3 * i + 2] = (f >> 28) ? (0xF0000000u | (f & 0x0FFFFFFFu)) : f;  // symbolic references keep the high nibble set
    }
    return CZS_OK;
}

extern "C" const char* czs_status_name(int s) {
    switch (s) {
#define N(x) case x: return #x;
        N(CZS_OK) N(CZS_MAGIC_NUMBER_READ_ERROR) N(CZS_FRAME_DESCRIPTOR_READ_ERROR) N(CZS_DICTIONARY_ID_READ_ERROR)
        N(CZS_WINDOW_DESCRIPTOR_READ_ERROR) N(CZS_BAD_MAGIC_NUMBER) N(CZS_SKIP_FRAME) N(CZS_WINDOW_TOO_BIG) N(CZS_WINDOW_TOO_SMALL)
        N(CZS_WINDOW_SIZE_TOO_BIG) N(CZS_FOUND_RESERVED_BLOCK) N(CZS_BLOCK_SIZE_TOO_LARGE) N(CZS_MALFORMED_SECTION_HEADER)
        N(CZS_LIT_GET_BITS_ERROR) N(CZS_LIT_NOT_ENOUGH_BYTES) N(CZS_SEQ_HDR_NOT_ENOUGH_BYTES) N(CZS_MISSING_BYTES_FOR_JUMP_HEADER)
        N(CZS_MISSING_BYTES_FOR_LITERALS) N(CZS_LIT_EXTRA_PADDING) N(CZS_BITSTREAM_READ_MISMATCH) N(CZS_DECODED_LITERAL_COUNT_MISMATCH)
        N(CZS_UNINITIALIZED_HUFFMAN_TABLE) N(CZS_HUF_SOURCE_IS_EMPTY) N(CZS_HUF_NOT_ENOUGH_BYTES_FOR_WEIGHTS) N(CZS_HUF_EXTRA_PADDING)
        N(CZS_HUF_TOO_MANY_WEIGHTS) N(CZS_HUF_MISSING_WEIGHTS) N(CZS_HUF_LEFTOVER_NOT_POWER_OF_2)
        N(CZS_HUF_NOT_ENOUGH_BYTES_TO_DECOMPRESS_WEIGHTS) N(CZS_HUF_FSE_TABLE_USED_TOO_MANY_BYTES) N(CZS_HUF_NOT_ENOUGH_BYTES_IN_SOURCE)
        N(CZS_HUF_WEIGHT_BIGGER_THAN_MAX_NUM_BITS) N(CZS_HUF_MAX_BITS_TOO_HIGH) N(CZS_FSE_ACC_LOG_IS_ZERO) N(CZS_FSE_ACC_LOG_TOO_BIG)
        N(CZS_FSE_PROBABILITY_COUNTER_MISMATCH) N(CZS_FSE_TOO_MANY_SYMBOLS) N(CZS_FSE_GET_BITS_ERROR) N(CZS_FSE_TABLE_IS_UNINITIALIZED)
        N(CZS_SEQ_EXTRA_PADDING) N(CZS_SEQ_UNSUPPORTED_OFFSET) N(CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES) N(CZS_SEQ_EXTRA_BITS)
        N(CZS_SEQ_GET_BITS_ERROR) N(CZS_MISSING_BYTE_FOR_RLE_LL_TABLE) N(CZS_MISSING_BYTE_FOR_RLE_OF_TABLE)
        N(CZS_MISSING_BYTE_FOR_RLE_ML_TABLE) N(CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE) N(CZS_EXEC_ZERO_OFFSET)
        N(CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY) N(CZS_OFFSET_TOO_BIG) N(CZS_DICT_BAD_MAGIC) N(CZS_PANIC_TRUNCATED) N(CZS_PANIC_INTERNAL) N(CZS_DST_TOO_SMALL)
        N(CZS_UNSUPPORTED) N(CZS_CUDA_ERROR) N(CZS_BAD_ARGUMENT) N(CZS_NOT_DECODED)
#undef N
    }
    return "CZS_UNKNOWN";
}
