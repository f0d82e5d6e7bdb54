// k_exec_flow_impl.cuh -- body of the data-flow ordered CTA-per-frame executor (see k_exec_flow.cu), compiled once per shape.
// Parameters (macros, set by the including file): FLOW_NS (namespace of this instance), FLOW_P_WARPS, FLOW_P_MIN_CTAS,
// FLOW_P_WIN_LOG, FLOW_P_SLICE.  No include guard on purpose.
namespace czb {
namespace FLOW_NS {

constexpr int FLOW_WARPS = FLOW_P_WARPS;
constexpr uint32_t FLOW_WIN = 1u << FLOW_P_WIN_LOG, FLOW_WIN_MASK = FLOW_WIN - 1;
constexpr uint32_t FLOW_SLICE = FLOW_P_SLICE;                              // largest chunk span built in the window
constexpr uint32_t FLOW_REACH = FLOW_WIN / 2 + FLOW_SLICE;                   // the window is trusted this far below a chunk's start
constexpr uint32_t FLOW_INFLIGHT = FLOW_WIN - FLOW_REACH - FLOW_SLICE - 64;  // unretired chunks lie within this span above the retired mark
static_assert(FLOW_INFLIGHT < FLOW_REACH, "what is read from dst must be retired");
static_assert(FLOW_INFLIGHT >= 2 * FLOW_SLICE, "at least two chunks in flight");
constexpr uint32_t FLOW_BATCH = 1024;   // chunks per batch (prefix tables)
constexpr uint32_t FLOW_NSLOT = 256;    // completion flags of the chunks between the retired head and the newest claim
constexpr uint32_t FLOW_BITWORDS = 2 * FLOW_WIN / 32;

struct FlowSmem {
    uint32_t chunk_lit[FLOW_BATCH + 4];   // exclusive prefix of literal bytes per chunk of the batch, [n] = batch total
    uint32_t chunk_out[FLOW_BATCH + 4];   // exclusive prefix of output bytes per chunk of the batch
    uint16_t prev_long[FLOW_BATCH];       // index of the last long chunk before this one (0xFFFF: none)
    __align__(16) uint8_t win[FLOW_WIN];
    uint32_t ready[FLOW_BITWORDS];
    uint32_t done[FLOW_NSLOT];            // chunk c + 1 once chunk c is complete and flushed
    uint32_t retired_out;                 // frame position below which everything is in dst and visible to the CTA
    uint32_t win_lo;                      // the window holds positions >= win_lo only (batch start / end of the last long chunk)
    uint32_t next_chunk, head;            // claim counter; first chunk not retired yet
    uint32_t err_chunk;                   // smallest failing chunk number of the batch, NONE32 if none
    int32_t err_status;
    uint32_t abort;                       // a wait loop gave up (flow_abort): everybody leaves, the frame fails
    __align__(16) uint8_t long_tile[EXEC_TILE + 48];
};

__device__ __forceinline__ void flow_fence() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }
__device__ __forceinline__ uint32_t vld(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }

// ready bits of positions [p, p + n), n >= 1.  The bitmap is indexed by position mod 2 * FLOW_WIN.
__device__ __forceinline__ bool flow_bits_ready(const uint32_t* bm, uint32_t p, uint32_t n) {
    uint32_t k = p >> 5;
    const uint32_t kl = (p + n - 1) >> 5;
    uint32_t lo = p & 31u;
    bool ok = true;
    for (; k <= kl; k++) {
        const uint32_t hi = k == kl ? ((p + n - 1) & 31u) : 31u;
        const uint32_t mask = (0xFFFFFFFFu >> (31u - hi)) & (0xFFFFFFFFu << lo);
        ok = ok && ((vld(bm + (k & (FLOW_BITWORDS - 1))) & mask) == mask);
        lo = 0;
    }
    return ok;
}
__device__ __forceinline__ void flow_bits_set(uint32_t* bm, uint32_t p, uint32_t n) {
    uint32_t k = p >> 5;
    const uint32_t kl = (p + n - 1) >> 5;
    uint32_t lo = p & 31u;
    for (; k <= kl; k++) {
        const uint32_t hi = k == kl ? ((p + n - 1) & 31u) : 31u;
        atomicOr(bm + (k & (FLOW_BITWORDS - 1)), (0xFFFFFFFFu >> (31u - hi)) & (0xFFFFFFFFu << lo));
        lo = 0;
    }
}
// fast forms for n <= 32 (at most two words)
__device__ __forceinline__ bool flow_bits_ready32(const uint32_t* bm, uint32_t p, uint32_t n) {
    const uint32_t k = p >> 5;
    const uint32_t w0 = vld(bm + (k & (FLOW_BITWORDS - 1))), w1 = vld(bm + ((k + 1) & (FLOW_BITWORDS - 1)));
    const uint32_t x = __funnelshift_r(w0, w1, p & 31u), mask = 0xFFFFFFFFu >> (32u - n);
    return (x & mask) == mask;
}
__device__ __forceinline__ void flow_bits_set32(uint32_t* bm, uint32_t p, uint32_t n) {
    const uint32_t k = p >> 5;
    const unsigned long long m = (unsigned long long)(0xFFFFFFFFu >> (32u - n)) << (p & 31u);
    atomicOr(bm + (k & (FLOW_BITWORDS - 1)), (uint32_t)m);
    if (m >> 32) atomicOr(bm + ((k + 1) & (FLOW_BITWORDS - 1)), (uint32_t)(m >> 32));
}
// the same for a long range, by the whole warp
__device__ __forceinline__ void flow_bits_set_warp(uint32_t* bm, uint32_t p, uint32_t n, unsigned lane) {
    const uint32_t k0 = p >> 5, kl = (p + n - 1) >> 5;
    for (uint32_t k = k0 + lane; k <= kl; k += 32) {
        const uint32_t lo = k == k0 ? (p & 31u) : 0u, hi = k == kl ? ((p + n - 1) & 31u) : 31u;
        atomicOr(bm + (k & (FLOW_BITWORDS - 1)), (0xFFFFFFFFu >> (31u - hi)) & (0xFFFFFFFFu << lo));
    }
}
// whole words covering [p, p + n) of the NEXT generation: done by a chunk that has completed (see the file comment)
__device__ __forceinline__ void flow_bits_clear_next(uint32_t* bm, uint32_t p, uint32_t n, unsigned lane) {
    if (n >= 2 * FLOW_WIN) { for (uint32_t k = lane; k < FLOW_BITWORDS; k += 32) bm[k] = 0u; return; }
    const uint32_t q = p + FLOW_WIN;
    const uint32_t k0 = q >> 5, kl = (q + n - 1) >> 5;
    for (uint32_t k = k0 + lane; k <= kl; k += 32) bm[k & (FLOW_BITWORDS - 1)] = 0u;
}

// advance the retired head over every chunk that is complete (any warp may call it; lane 0 works)
__device__ __forceinline__ void flow_try_retire(FlowSmem& sm, uint32_t nb, uint32_t batch_out0) {
    for (;;) {
        const uint32_t h = vld(&sm.head);
        if (h >= nb) break;
        if (vld(&sm.done[h % FLOW_NSLOT]) != h + 1u) break;
        flow_fence();
        if (atomicCAS(&sm.head, h, h + 1u) == h) atomicMax(&sm.retired_out, batch_out0 + sm.chunk_out[h + 1]);
    }
}

// Measurement aid (-DCZB_FLOW_CLOCK): cycles per phase, accumulated by lane 0 of warp 0 of CTA 0 and printed per launch.
#ifdef CZB_FLOW_CLOCK
__device__ unsigned long long czb_flow_clk[24];
#define FCLK(k) do { if (dbg) { const long long t_ = clock64(); atomicAdd(&czb_flow_clk[k], (unsigned long long)(t_ - *dbg)); *dbg = t_; } } while (0)
#define FCNT(k, v) do { if (dbg) atomicAdd(&czb_flow_clk[k], (unsigned long long)(v)); } while (0)
#else
#define FCLK(k) do { } while (0)
#define FCNT(k, v) do { } while (0)
#endif

// Safety net: the wait loops below cannot spin for ever.  A loop that has spun FLOW_SPIN_LIMIT times (tens of milliseconds; a healthy
// wait is microseconds) records what it was waiting for in czb_flow_wd (czb_debug_flow_watchdog), raises the CTA's abort flag -- every
// wait loop of the CTA leaves when it sees it -- and the frame fails with CZS_PANIC_INTERNAL instead of hanging the GPU.
__device__ unsigned int czb_flow_wd[16];
constexpr uint32_t FLOW_SPIN_LIMIT = 1u << 21;
__device__ __forceinline__ void flow_abort(uint32_t* abort_flag, unsigned code, uint32_t a, uint32_t b, uint32_t c2, uint32_t d2, uint32_t e, uint32_t f2,
                                           uint32_t g, uint32_t h) {
    if (atomicCAS(&czb_flow_wd[0], 0u, code) == 0u) {
        czb_flow_wd[1] = blockIdx.x; czb_flow_wd[2] = threadIdx.x >> 5; czb_flow_wd[3] = a; czb_flow_wd[4] = b; czb_flow_wd[5] = c2;
        czb_flow_wd[6] = d2; czb_flow_wd[7] = e; czb_flow_wd[8] = f2; czb_flow_wd[9] = g; czb_flow_wd[10] = h;
    }
    atomicExch(abort_flag, 1u);
}

struct FlowWin {
    uint8_t* win;
    __device__ __forceinline__ uint8_t rd(uint32_t p) const { return win[p & FLOW_WIN_MASK]; }
    __device__ __forceinline__ void wr(uint32_t p, uint8_t v) const { win[p & FLOW_WIN_MASK] = v; }
    __device__ __forceinline__ Vec16 load16(uint32_t p, uint32_t n) const { return win_load16<FLOW_WIN>(win, p, n); }
    __device__ __forceinline__ void store16(uint32_t p, const Vec16& v, uint32_t n) const { win_store16<FLOW_WIN>(win, p, v, n); }
};

__global__ void __launch_bounds__(FLOW_WARPS * 32, FLOW_P_MIN_CTAS) k_exec_flow(const czb_frame_desc* __restrict__ descs, const FrameInfo* __restrict__ infos,
                                                           BigRule rule,
                                                           const uint32_t* __restrict__ exec_order, BlockDesc* __restrict__ blocks,
                                                           const uint8_t* __restrict__ lit_scratch, const Seq* __restrict__ seq_scratch,
                                                           czb_frame_result* __restrict__ results, const FrameResume* __restrict__ resume) {
    extern __shared__ __align__(16) uint8_t flow_raw[];
    FlowSmem& sm = *reinterpret_cast<FlowSmem*>(flow_raw);
    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    const uint64_t f = exec_order[blockIdx.x];
    const FrameInfo fi = infos[f];
    if (fi.status != CZS_OK) return;      // k_header_results already reported it
    if (!frame_is_big(fi, rule)) return;  // k_exec's
    const czb_frame_desc fd = descs[f];
    const uint8_t* src = fd.src;
    uint8_t* dst = fd.dst;
    const uint64_t cap = fd.dst_cap < MAX_FRAME_OUT ? fd.dst_cap : MAX_FRAME_OUT;
    const int32_t cap_status = fd.dst_cap < MAX_FRAME_OUT ? CZS_DST_TOO_SMALL : CZS_UNSUPPORTED;
    const FlowWin W{sm.win};

    // every thread tracks the frame-level state identically (all of it is uniform)
    uint64_t out = 0;
    uint32_t h0 = 1, h1 = 4, h2 = 8;  // scratch.cairo:35
    int32_t status = CZS_OK;
    uint32_t n_done = 0;
    uint64_t bytes_read = fi.hdr_len;
    bool finished = false;
    if (resume) { const FrameResume r = resume[f]; out = r.out0; h0 = r.h0; h1 = r.h1; h2 = r.h2; n_done = r.start_block; bytes_read = r.bytes_read0; }

#ifdef CZB_FLOW_CLOCK
    long long dbg_t0 = clock64();
    long long* dbg = (blockIdx.x == 0 && threadIdx.x == 0) ? &dbg_t0 : nullptr;
#endif
    for (uint32_t k = n_done; k < fi.n_blocks && status == CZS_OK; k++) {
        const BlockDesc d = blocks[fi.block_base + k];
        const uint64_t out_before = out;
        if (d.type == BT_ERROR) { status = d.pre_status; break; }
        if (d.type == BT_RAW) {
            if (out + d.size > cap) { status = cap_status; break; }
            const uint64_t per = ((d.size + FLOW_WARPS - 1) / FLOW_WARPS + 15) & ~15ull, lo = (uint64_t)warp * per;
            if (lo < d.size) warp_copy(dst + out + lo, src + d.src_off + lo, (uint32_t)(d.size - lo < per ? d.size - lo : per));
            out += d.size; bytes_read += 3ull + d.size;
        } else if (d.type == BT_RLE) {
            if (out + d.size > cap) { status = cap_status; break; }
            const uint64_t per = ((d.size + FLOW_WARPS - 1) / FLOW_WARPS + 15) & ~15ull, lo = (uint64_t)warp * per;
            if (lo < d.size) warp_fill(dst + out + lo, src[d.src_off], (uint32_t)(d.size - lo < per ? d.size - lo : per));
            out += d.size; bytes_read += 4;
        } else {
            // error order of decompress_block (:139-235): literals header, literals, sequences header, sequences, execution
            if (d.pre_status != CZS_OK) { status = d.pre_status; break; }
            if (d.lit_type >= LT_COMPRESSED && d.huf_status != CZS_OK) { status = d.huf_status; break; }
            if (d.seqhdr_status != CZS_OK) { status = d.seqhdr_status; break; }
            if (d.n_seq && d.fse_status != CZS_OK) { status = d.fse_status; break; }
            const uint8_t* lits = d.lit_type >= LT_COMPRESSED ? lit_scratch + d.lit_off : src + d.lit_src_off;
            const bool lit_rle = d.lit_type == LT_RLE;
            const uint32_t rle_byte = lit_rle ? src[d.lit_src_off] : 0;
            const uint32_t n_lit = d.regen;
            const Seq* seqs = seq_scratch + d.seq_off;
            const uint32_t n_chunks = (d.n_seq + 31) / 32;
            uint32_t lit_total = 0, out_total = 0;  // literal / output bytes of the batches done so far
            bool failed = false;
            FCLK(0);
            for (uint32_t cb = 0; cb < n_chunks && !failed; cb += FLOW_BATCH) {
                const uint32_t nb = n_chunks - cb < FLOW_BATCH ? n_chunks - cb : FLOW_BATCH;
                // ---- pre-pass: literal and output bytes of every chunk of the batch, then one exclusive scan ----
                for (uint32_t q0 = warp * 4; q0 < nb; q0 += FLOW_WARPS * 4) {
                    Seq rec[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) { const uint32_t i = (cb + q0 + q) * 32 + lane; rec[q] = i < d.n_seq ? seqs[i] : 0ull; }
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        uint32_t ls = seq_ll(rec[q]), os = ls + seq_ml(rec[q]);
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) { ls += __shfl_xor_sync(0xFFFFFFFFu, ls, o); os += __shfl_xor_sync(0xFFFFFFFFu, os, o); }
                        if (lane == 0 && q0 + q < nb) { sm.chunk_lit[q0 + q] = ls; sm.chunk_out[q0 + q] = os; }
                    }
                }
                // (re)start the window: nothing of it is valid, no chunk is in flight
                for (uint32_t i = threadIdx.x; i < FLOW_BITWORDS; i += FLOW_WARPS * 32) sm.ready[i] = 0u;
                for (uint32_t i = threadIdx.x; i < FLOW_NSLOT; i += FLOW_WARPS * 32) sm.done[i] = 0u;
                __syncthreads();
                const uint32_t batch_out0 = (uint32_t)(out + out_total);  // frame position of the batch's first byte (<= cap < 2^31)
                if (warp == 0) {
                    // 64-bit running totals, stored saturated: a malformed block whose lengths add up to more than 2^31 must
                    // fail its capacity / literal checks, not wrap around them.  Output offsets saturate where the frame position
                    // reaches 2^31 (> cap), so that position + chunk span (< 2^25) stays below 2^32 in the chunks' u32 sums.
                    unsigned long long cl = 0, co = 0;
                    uint32_t last_long = 0xFFFFu;
                    auto sat = [](unsigned long long v) -> uint32_t { return v < 0x7FFFFFFFull ? (uint32_t)v : 0x7FFFFFFFu; };
                    const unsigned long long out_lim = 0x80000000ull - batch_out0;
                    auto sat_out = [out_lim](unsigned long long v) -> uint32_t { return (uint32_t)(v < out_lim ? v : out_lim); };
                    for (uint32_t b = 0; b < nb; b += 32) {
                        const uint32_t c = b + lane;
                        const uint32_t vl = c < nb ? sm.chunk_lit[c] : 0u, vo = c < nb ? sm.chunk_out[c] : 0u;
                        const unsigned lm = __ballot_sync(0xFFFFFFFFu, vo > FLOW_SLICE);  // chunks that do not fit a window slice
                        const unsigned below = lm & lanemask_lt();
                        if (c < nb) sm.prev_long[c] = (uint16_t)(below ? b + (31u - (uint32_t)__clz(below)) : last_long);
                        if (lm) last_long = b + (31u - (uint32_t)__clz(lm));
                        uint32_t il = vl, io = vo;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) {
                            const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, il, o), b2 = __shfl_up_sync(0xFFFFFFFFu, io, o);
                            if ((int)lane >= o) { il += a; io += b2; }
                        }
                        if (c < nb) { sm.chunk_lit[c] = sat(cl + il - vl); sm.chunk_out[c] = sat_out(co + io - vo); }
                        cl += __shfl_sync(0xFFFFFFFFu, il, 31); co += __shfl_sync(0xFFFFFFFFu, io, 31);
                    }
                    if (lane == 0) {
                        sm.chunk_lit[nb] = sat(cl); sm.chunk_out[nb] = sat_out(co);
                        sm.next_chunk = 0; sm.head = 0; sm.retired_out = batch_out0; sm.win_lo = batch_out0;
                        sm.err_chunk = NONE32; sm.err_status = CZS_OK; sm.abort = 0u;
                    }
                }
                __syncthreads();
                const uint32_t lit_batch = sm.chunk_lit[nb], out_batch = sm.chunk_out[nb];
                FCLK(1);

                // ---- chunks, claimed in order, completed in data-flow order ----
                // (Measured and dropped: claiming the next chunk and requesting its record while the current one is executed, and
                // raising a chunk's completion flag lazily at the warp's next wait -- 33 -> 22 GB/s on the long-window frames: a
                // claimed chunk cannot start before its warp is free, and every start that is late delays its dependants.)
                for (;;) {
                    uint32_t c = 0;
                    if (lane == 0) c = atomicAdd(&sm.next_chunk, 1u);
                    c = __shfl_sync(0xFFFFFFFFu, c, 0);
                    if (c >= nb) break;
                    const uint32_t i = (cb + c) * 32 + lane;
                    const bool have = i < d.n_seq;
                    const Seq rec = have ? __ldcs(seqs + i) : 0ull;
                    uint32_t ll = 0, ml = 0, off = 1;
                    if (have) { ll = seq_ll(rec); ml = seq_ml(rec); off = off29_resolve(seq_off29(rec), h0, h1, h2); }
                    uint32_t lsum = ll, osum = ll + ml;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, lsum, o), b = __shfl_up_sync(0xFFFFFFFFu, osum, o);
                        if ((int)lane >= o) { lsum += a; osum += b; }
                    }
                    const uint32_t O = batch_out0 + sm.chunk_out[c];          // frame position of the chunk's first byte
                    const uint32_t my_lit = lit_total + sm.chunk_lit[c] + lsum - ll;
                    const uint32_t segA = O + osum - ll - ml, segM = segA + ll;  // frame positions of the literal run and of the match
                    const uint32_t span = __shfl_sync(0xFFFFFFFFu, osum, 31);
                    // the reference's checks in its order (see k_exec); a failing chunk writes nothing but still completes
                    int32_t err = CZS_OK;
                    if (have) {
                        if (ll > 0 && (uint64_t)my_lit + ll > n_lit) err = CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE;  // :29-37
                        else if (off == 0) err = CZS_EXEC_ZERO_OFFSET;                                            // :47-49
                        else if (ml > 0 && off == OFF29_CLAMP && off29_far(seq_off29(rec), segM))                // the raw field, not the resolved offset
                            err = CZS_UNSUPPORTED;
                        else if (ml > 0 && off > segM)                                                              // decode_buffer.cairo:65-93
                            err = ((uint64_t)segM <= fi.window) ? CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY : CZS_OFFSET_TOO_BIG;
                        else if ((uint64_t)segM + ml > cap) err = cap_status;
                    }
                    const unsigned errm = __ballot_sync(0xFFFFFFFFu, err != CZS_OK);
                    const bool is_long = span > FLOW_SLICE;
                    FCLK(2); FCNT(16, 1);

                    if (errm || is_long) {
                        // ---- alone: everything before this chunk has retired ----
                        if (lane == 0) {
                            uint32_t spins = 0;
                            while (vld(&sm.head) != c && !vld(&sm.abort)) {
                                flow_try_retire(sm, nb, batch_out0); __nanosleep(64);
                                if (++spins > FLOW_SPIN_LIMIT) flow_abort(&sm.abort, 1u, c, vld(&sm.head), vld(&sm.next_chunk), vld(&sm.retired_out), vld(&sm.done[vld(&sm.head) % FLOW_NSLOT]), nb, 0u, 0u);
                            }
                        }
                        __syncwarp();
                        flow_fence();
                        FCLK(3); FCNT(17, 1);
                        if (errm) {  // chunks reach this point in order (head == c), so the first failing chunk wins
                            const int32_t e = __shfl_sync(0xFFFFFFFFu, err, __ffs(errm) - 1);
                            if (lane == 0 && c < sm.err_chunk) { sm.err_chunk = c; sm.err_status = e; }
                        } else {
                            // cut at sequence boundaries into pieces that fit a tile (each executed like a chunk of its own); a single
                            // sequence that does not fit is copied straight into dst (overlapping matches as a repeated pattern,
                            // decode_buffer.cairo:101-120)
                            uint8_t* obase = dst + O;
                            const uint32_t rel = segA - O;  // chunk-relative start of this lane's literal run
                            for (uint32_t start = 0; start < 32;) {
                                const uint32_t base_o = __shfl_sync(0xFFFFFFFFu, rel, start);
                                const unsigned fit = __ballot_sync(0xFFFFFFFFu, lane >= start && rel + ll + ml - base_o <= EXEC_TILE);
                                if (!((fit >> start) & 1u)) {
                                    const int j = (int)start;
                                    const uint32_t jl = __shfl_sync(0xFFFFFFFFu, ll, j), jm = __shfl_sync(0xFFFFFFFFu, ml, j), jo = __shfl_sync(0xFFFFFFFFu, off, j);
                                    const uint32_t jlit = __shfl_sync(0xFFFFFFFFu, my_lit, j);
                                    uint8_t* o = obase + base_o;
                                    if (jl) { if (lit_rle) warp_fill(o, (uint8_t)rle_byte, jl); else warp_copy(o, lits + jlit, jl); }
                                    o += jl;
                                    if (jm) {
                                        __syncwarp();
                                        flow_fence();
                                        if (jo >= jm) warp_copy(o, o - jo, jm);
                                        else for (uint32_t t = lane; t < jm; t += 32) o[t] = __ldcg(o - jo + (t % jo));
                                    }
                                    start++;
                                } else {
                                    const uint32_t last = 31u - (uint32_t)__clz(fit);  // fit is a run of lanes from `start` (offsets only grow)
                                    const bool in = lane >= start && lane <= last;
                                    const uint32_t span_p = __shfl_sync(0xFFFFFFFFu, rel + ll + ml, last) - base_o;
                                    exec_chunk_tile<true>(sm.long_tile, obase + base_o, lits, lit_rle, rle_byte, lane, in ? ll : 0u, in ? ml : 0u, off, my_lit,
                                                          in ? rel - base_o : 0u, span_p);
                                    start = last + 1;
                                }
                                __syncwarp();
                                flow_fence();  // the next piece reads this one's bytes from dst
                            }
                        }
                        flow_bits_clear_next(sm.ready, O, span, lane);  // these slots' next occupants must not see the bits of two generations ago
                        __syncwarp();
                        flow_fence();
                        if (lane == 0) {
                            atomicMax(&sm.win_lo, O + span);  // the window holds nothing of this chunk
                            flow_fence();
                            sm.done[c % FLOW_NSLOT] = c + 1u;
                            flow_fence();
                            flow_try_retire(sm, nb, batch_out0);
                        }
                        __syncwarp();
                        FCLK(4);
                        continue;
                    }

                    // ---- window path ----
                    // wait for room: the span must lie within FLOW_INFLIGHT of the retired mark, the completion flags must not wrap,
                    // and a long chunk before this one must have retired (it moves win_lo)
                    if (lane == 0) {
                        const uint32_t pl = sm.prev_long[c];
                        uint32_t spins = 0;
                        for (;;) {
                            const uint32_t hd = vld(&sm.head);
                            if (O + span <= vld(&sm.retired_out) + FLOW_INFLIGHT && c - hd < FLOW_NSLOT && (pl == 0xFFFFu || hd > pl)) break;
                            if (vld(&sm.abort)) break;
                            flow_try_retire(sm, nb, batch_out0);
                            __nanosleep(32);
                            if (++spins > FLOW_SPIN_LIMIT) flow_abort(&sm.abort, 2u, c, hd, vld(&sm.next_chunk), vld(&sm.retired_out), vld(&sm.done[hd % FLOW_NSLOT]), nb, O, span);
                        }
                    }
                    __syncwarp();
                    flow_fence();
                    FCLK(5);
                    const uint32_t wl = vld(&sm.win_lo);
                    const uint32_t lo_abs = max(O > FLOW_REACH ? O - FLOW_REACH : 0u, wl);  // positions >= lo_abs live in the window
                    // literal runs: first 16 bytes per lane, tails by the whole warp
                    {
                        const uint32_t nl = lit_rle ? 0u : (ll < 16u ? ll : 16u);
                        W.store16(segA, load16_unaligned(lits + my_lit, nl), nl);
                    }
                    for (unsigned m = __ballot_sync(0xFFFFFFFFu, !lit_rle && ll > 16u); m; m &= m - 1) {
                        const int j = __ffs(m) - 1;
                        const uint32_t dp = __shfl_sync(0xFFFFFFFFu, segA, j) + 16u, cnt = __shfl_sync(0xFFFFFFFFu, ll, j) - 16u, lp = __shfl_sync(0xFFFFFFFFu, my_lit, j) + 16u;
                        for (uint32_t t = lane; t < cnt; t += 32) W.wr(dp + t, lits[lp + t]);
                    }
                    if (lit_rle) for (uint32_t t = 0; __any_sync(0xFFFFFFFFu, t < ll); t++) if (t < ll) W.wr(segA + t, (uint8_t)rle_byte);
                    __syncwarp();
                    flow_fence();
                    if (ll) { if (ll <= 32u) flow_bits_set32(sm.ready, segA, ll); else if (ll <= 64u) flow_bits_set(sm.ready, segA, ll); }
                    for (unsigned m = __ballot_sync(0xFFFFFFFFu, ll > 64u); m; m &= m - 1) {
                        const int j = __ffs(m) - 1;
                        flow_bits_set_warp(sm.ready, __shfl_sync(0xFFFFFFFFu, segA, j), __shfl_sync(0xFFFFFFFFu, ll, j), lane);
                    }
                    FCLK(6);
                    // matches, in rounds: a match is copied once its own source bytes are ready.  Everything below lo_abs is retired
                    // (in dst, visible); a source at or above it is in the window and has ready bits.  A source may straddle lo_abs.
                    const uint32_t s_lo = segM - off;                        // frame position of the source (err == OK: off <= segM)
                    const uint32_t s_need = off < ml ? off : ml;             // a self-overlapping match needs its first period only
                    const uint32_t s_end = s_lo + s_need;                    // <= segM
                    const uint32_t chk_lo = s_lo > lo_abs ? s_lo : lo_abs;   // the part that needs ready bits starts here
                    const uint32_t head_n = ml < 16u ? ml : 16u;
                    const bool all_win = s_lo >= lo_abs, all_dst = s_lo + head_n <= lo_abs;
                    auto RD = [&](uint32_t p) -> uint8_t { return p >= lo_abs ? W.rd(p) : __ldcg(dst + p); };
                    // Rounds (multi-round resolution of back-references): in every round each lane whose source bytes are ready copies
                    // its match -- the first 16 bytes per lane, tails by the whole warp -- and then publishes its bits.  Matches that
                    // wait for other matches (of this chunk or of chunks in flight) take the next round.  With CZB_FLOW_SEQ_AFTER=k the
                    // matches still pending after k rounds are taken in sequence order by the whole warp instead (measured slower:
                    // an in-order pass makes every later match of the chunk wait behind the first one that is not ready).
                    bool pending = ml > 0;
                    uint32_t idle_spins = 0;
                    for (uint32_t round = 0; __any_sync(0xFFFFFFFFu, pending); round++) {
                        uint32_t r_now = 0, ab = 0;
                        if (lane == 0) { r_now = vld(&sm.retired_out); ab = vld(&sm.abort) | (vld(&sm.err_chunk) < c ? 1u : 0u); }
                        r_now = __shfl_sync(0xFFFFFFFFu, r_now, 0);
                        // somebody gave up, or an earlier chunk failed -- it writes nothing, so a source that reaches into its span never
                        // gets its ready bits: the frame fails with that chunk's status, nothing here matters any more
                        if (__shfl_sync(0xFFFFFFFFu, ab, 0)) break;
                        bool ready = false;
                        if (pending) {
                            if (s_end <= lo_abs || s_end <= r_now) ready = true;
                            else if (s_end - chk_lo <= 32u) ready = flow_bits_ready32(sm.ready, chk_lo, s_end - chk_lo);
                            else ready = flow_bits_ready(sm.ready, chk_lo, s_end - chk_lo);
                        }
                        const unsigned rm = __ballot_sync(0xFFFFFFFFu, ready);
                        if (!rm) {
                            if (lane == 0) {
                                flow_try_retire(sm, nb, batch_out0); __nanosleep(32);
                                if (++idle_spins > FLOW_SPIN_LIMIT) flow_abort(&sm.abort, 3u, c, vld(&sm.head), vld(&sm.next_chunk), r_now, O, span, lo_abs, 0u);
                            }
                            __syncwarp();
                            FCLK(7); FCNT(18, 1);
                            continue;
                        }
                        flow_fence();  // acquire: the bytes behind the bits / the retired mark
                        FCLK(8); FCNT(19, 1);
                        // first 16 bytes of every ready match that does not overlap itself and whose head lies on one side of lo_abs
                        const bool simple = ready && off >= ml && (all_win || all_dst);
                        {
                            const uint32_t nm = simple ? head_n : 0u;
                            const Vec16 xw = W.load16(s_lo, all_win ? nm : 0u);
                            const Vec16 xg = load16_unaligned<true>(dst + s_lo, all_win ? 0u : nm);
                            Vec16 x;
#pragma unroll
                            for (int q = 0; q < 4; q++) x.v[q] = all_win ? xw.v[q] : xg.v[q];
                            W.store16(segM, x, nm);
                        }
                        FCLK(9);
                        // tails, self-overlapping matches and straddling heads: the whole warp on one match at a time
                        for (unsigned m = __ballot_sync(0xFFFFFFFFu, ready && (ml > 16u || !simple)); m; m &= m - 1) {
                            const int j = __ffs(m) - 1;
                            const uint32_t dM = __shfl_sync(0xFFFFFFFFu, segM, j), n = __shfl_sync(0xFFFFFFFFu, ml, j), o = __shfl_sync(0xFFFFFFFFu, off, j);
                            const uint32_t t0 = __shfl_sync(0xFFFFFFFFu, simple ? 16u : 0u, j);
                            const uint32_t s0 = dM - o;
                            if (o >= n) for (uint32_t t = t0 + lane; t < n; t += 32) W.wr(dM + t, RD(s0 + t));
                            else for (uint32_t t = t0 + lane; t < n; t += 32) W.wr(dM + t, RD(s0 + (t % o)));
                        }
                        __syncwarp();
                        flow_fence();  // release: the bytes before their bits
                        FCLK(10);
                        if (ready) { if (ml <= 32u) flow_bits_set32(sm.ready, segM, ml); else if (ml <= 64u) flow_bits_set(sm.ready, segM, ml); }
                        for (unsigned m = __ballot_sync(0xFFFFFFFFu, ready && ml > 64u); m; m &= m - 1) {
                            const int j = __ffs(m) - 1;
                            flow_bits_set_warp(sm.ready, __shfl_sync(0xFFFFFFFFu, segM, j), __shfl_sync(0xFFFFFFFFu, ml, j), lane);
                        }
                        pending = pending && !ready;
                        __syncwarp();
                        FCLK(11);
                    }
                    // complete: copy the slice to dst (aligned 16-byte stores; window index and dst address agree modulo 16 when dst is
                    // 16-byte aligned; otherwise byte-wise)
                    {
                        uint8_t* obase = dst + O;
                        const uint32_t a0 = (uint32_t)(reinterpret_cast<uintptr_t>(obase) & 15u);
                        if (((reinterpret_cast<uintptr_t>(dst) & 15u) == 0)) {
                            const uint32_t head = span < ((16 - a0) & 15) ? span : ((16 - a0) & 15);
                            if (lane < head) obase[lane] = W.rd(O + lane);
                            const uint32_t body = span - head, nv = body >> 4, tail = body & 15;
                            uint4* g4 = reinterpret_cast<uint4*>(obase + head);
                            for (uint32_t v = lane; v < nv; v += 32) g4[v] = *reinterpret_cast<const uint4*>(sm.win + ((O + head + (v << 4)) & FLOW_WIN_MASK));
                            if (lane < tail) obase[head + (nv << 4) + lane] = W.rd(O + head + (nv << 4) + lane);
                        } else {
                            for (uint32_t t = lane; t < span; t += 32) obase[t] = W.rd(O + t);
                        }
                    }
                    FCLK(12);
                    flow_bits_clear_next(sm.ready, O, span, lane);
                    __syncwarp();
                    flow_fence();  // the flushed bytes before the flag
                    if (lane == 0) {
                        sm.done[c % FLOW_NSLOT] = c + 1u;  // an advance of the head missed here (store / load order) is made by the next poller
                        flow_try_retire(sm, nb, batch_out0);
                    }
                    __syncwarp();
                    FCLK(13);
                }
                FCLK(14);
                __syncthreads();  // everything of the batch is complete in dst and visible to the whole CTA
                FCLK(15);
                if (sm.err_chunk != NONE32) { status = sm.err_status; failed = true; }
                if (sm.abort) { status = CZS_PANIC_INTERNAL; failed = true; }  // a wait loop gave up (flow_abort): never seen; a bug, not an input error
                lit_total += lit_batch; out_total += out_batch;
                __syncthreads();
            }  // batch loop
            if (failed) break;
            out += out_total;
            if (d.n_seq) {  // history after this block (resolved against the history it started from)
                const uint32_t n0 = sym_is(d.hist_out[0]) ? sym_resolve(d.hist_out[0], h0, h1, h2) : d.hist_out[0];
                const uint32_t n1 = sym_is(d.hist_out[1]) ? sym_resolve(d.hist_out[1], h0, h1, h2) : d.hist_out[1];
                const uint32_t n2 = sym_is(d.hist_out[2]) ? sym_resolve(d.hist_out[2], h0, h1, h2) : d.hist_out[2];
                h0 = n0; h1 = n1; h2 = n2;
            }
            // rest literals (:72-78), or all literals when there are no sequences (block_decoder.cairo:229-232)
            const uint32_t rest = n_lit - lit_total;
            if (rest) {
                if (out + rest > cap) { status = cap_status; break; }
                const uint64_t per = ((rest + FLOW_WARPS - 1) / FLOW_WARPS + 15) & ~15ull, lo = (uint64_t)warp * per;
                if (lo < rest) {
                    const uint32_t cnt = (uint32_t)(rest - lo < per ? rest - lo : per);
                    if (lit_rle) warp_fill(dst + out + lo, (uint8_t)rle_byte, cnt);
                    else warp_copy(dst + out + lo, lits + lit_total + lo, cnt);
                }
                out += rest;
            }
            bytes_read += 3ull + d.size;
        }
        n_done++;
        if (threadIdx.x == 0) {
            BlockDesc& bd = blocks[fi.block_base + k];
            bd.out_bytes = (uint32_t)(out - out_before); bd.hist_out[0] = h0; bd.hist_out[1] = h1; bd.hist_out[2] = h2;
        }
        if (d.last) {
            finished = true;
            if ((fi.descriptor >> 2) & 1) bytes_read += 4;
        }
        __syncthreads();  // the block's output (incl. raw/rle/rest copies by all warps) is complete in dst
    }
#ifdef CZB_FLOW_CLOCK
    if (dbg) {
        const double nc = (double)czb_flow_clk[16] > 0 ? (double)czb_flow_clk[16] : 1.0;
        printf("flow clk (warp 0 of CTA 0, %llu chunks, %llu solo, %llu idle rounds, %llu work rounds), cycles per chunk of this warp:\n"
               "  block setup %.0f | batch prepass+scan %.0f | claim+records+prefix+checks %.0f | solo wait %.0f | solo work %.0f | wait room %.0f |\n"
               "  literals+bits %.0f | idle rounds %.0f | ready check %.0f | heads %.0f | tails %.0f | bits set %.0f | flush %.0f | done+retire %.0f | loop exit %.0f | batch barrier %.0f | seq-phase copies %.0f (%llu matches)\n",
               czb_flow_clk[16], czb_flow_clk[17], czb_flow_clk[18], czb_flow_clk[19],
               czb_flow_clk[0] / nc, czb_flow_clk[1] / nc, czb_flow_clk[2] / nc, czb_flow_clk[3] / nc, czb_flow_clk[4] / nc, czb_flow_clk[5] / nc,
               czb_flow_clk[6] / nc, czb_flow_clk[7] / nc, czb_flow_clk[8] / nc, czb_flow_clk[9] / nc, (czb_flow_clk[10]) / nc, czb_flow_clk[11] / nc,
               czb_flow_clk[12] / nc, czb_flow_clk[13] / nc, czb_flow_clk[14] / nc, czb_flow_clk[15] / nc, czb_flow_clk[20] / nc, czb_flow_clk[21]);
        for (int q = 0; q < 24; q++) czb_flow_clk[q] = 0;
    }
#endif
    if (threadIdx.x == 0) {
        czb_frame_result r;
        r.status = status;
        r.blocks_decoded = n_done;
        r.bytes_read = bytes_read;
        r.bytes_written = status == CZS_OK ? out : 0;
        r.content_size = fi.fcs;
        r.window_size = fi.window;
        r.checksum_from_data = fi.checksum;
        r.checksum_calculated = 0;
        r.has_checksum = fi.has_checksum;
        r.finished = (status == CZS_OK && finished && (!((fi.descriptor >> 2) & 1) || fi.has_checksum)) ? 1 : 0;
        results[f] = r;
    }
}

void launch_exec_flow(const LaunchCtx& lc, unsigned n_ctas, const czb_frame_desc* descs, const FrameInfo* infos, BigRule rule, const uint32_t* exec_order,
                      BlockDesc* blocks, const uint8_t* lit_scratch, const Seq* seq_scratch, czb_frame_result* results, const FrameResume* resume) {
    k_exec_flow<<<n_ctas, FLOW_WARPS * 32, sizeof(FlowSmem), lc.stream>>>(descs, infos, rule, exec_order, blocks, lit_scratch, seq_scratch, results, resume);
    ++*lc.launches;
}

int read_watchdog(unsigned int* out16) {
    if (cudaMemcpyFromSymbol(out16, czb_flow_wd, sizeof(czb_flow_wd)) != cudaSuccess) return CZS_CUDA_ERROR;
    unsigned int zero[16] = {0};
    cudaMemcpyToSymbol(czb_flow_wd, zero, sizeof(zero));
    return CZS_OK;
}

int setup_exec_flow_attributes() {
    return (int)cudaFuncSetAttribute(k_exec_flow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FlowSmem));
}

}  // namespace FLOW_NS
}  // namespace czb
