// k_exec.cu -- block loop and sequence execution: one warp per frame, blocks in order.
//
// Reference path: the block loop of FrameDecoder::decode_blocks (src/frame_decoder.cairo:156-222),
// decode_block_content (src/decoding/block_decoder.cairo:77-137; Raw :97-103, RLE :104-123),
// the tail of decompress_block (:216-232), execute_sequences (src/decoding/sequence_execution.cairo:12-83),
// DecodeBuffer::push / repeat (src/decoding/decode_buffer.cairo:57-133) and collect() (:224-231):
// the append-only RingBuffer (ring_buffer.cairo:6) is simply the caller's dst span.
//
// Mapping: sequences are taken 32 at a time (lane = sequence).  A warp prefix sum over literal/match lengths gives
// every sequence its literal source and output offsets.
//   * Tile path (the chunk's output span fits 1 KiB, the common case): the first 16 bytes of every literal run and of
//     every match whose source precedes the chunk go into a shared-memory tile with per-lane unaligned 16-byte copies;
//     everything sparse -- tails beyond 16 bytes, matches that read the chunk's own output (in sequence order,
//     overlapping ones as a repeated pattern, decode_buffer.cairo:101-120) -- is done by the whole warp, one item at
//     a time; the tile is flushed with aligned 16-byte stores.
//   * Row path (longer spans): each of the 64 segments publishes its start and a source delta in shared memory; output
//     is produced in rows of 128 bytes, lane l owns the aligned word at row + 4l; segment ownership of every row byte
//     comes from one warp max-scan over "segment id at its start byte" marks; each byte is one gather; bytes whose
//     source lies inside the row being built, overlapping matches and RLE literals chase the source back through
//     the row's segment map.
// HBM traffic per frame: literals + 8 B/sequence in, decoded bytes out; match sources are recent output (L1/L2 when the
// in-flight working set allows, DRAM otherwise: profiles/r01_final_ncu_summary.md).
#include <cstdio>

#include "czb_exec.cuh"
#include "czb_internal.cuh"

namespace czb {

// ---- k_exec_big's chunk executor: the frame's recent output lives in a shared-memory window ----
// k_exec_big commits the chunks of a frame in order, so whatever a chunk does between "everything before me is
// complete" and "I am complete" is a serial chain that every other warp of the CTA waits for.  With the chunk built in
// a private tile and handed over through dst, that chain held two global round trips (clock64, 17 MiB long-window
// frames, cycles per chunk: late-source loads from L2 1190, in-chunk dependent matches 830, flush 340, and 2050 for the
// fence that makes the flushed bytes visible before the commit counter moves).  Here every chunk is built in place in
// a CTA-wide window indexed by the low bits of its dst address: later chunks read recent output from the window, the
// chunk commits as soon as its slice is complete, and the copy to dst happens after the commit, off the chain.
//
// Validity: the window holds the output of the current run of window chunks (a run starts at a block, at a batch of
// chunks, or after a chunk that was too long for a slice) from `lo_rel` (chunk-relative, <= 0) on: the start of the run,
// or BIG_WIN_REACH bytes back.  Older bytes are read from dst: bytes before the run were published by a CTA barrier;
// bytes more than BIG_WIN_REACH (> 7 slices) back were flushed at least eight chunks ago by a warp that has since passed
// a fence and a commit, which this warp observed when it committed its own previous chunk.  All slices in flight lie
// within BIG_WARPS consecutive slices of at most EXEC_TILE bytes, so they never alias in the window.
constexpr uint32_t BIG_WIN = 16384, BIG_WIN_MASK = BIG_WIN - 1;
// How far below a chunk's start the window is trusted.  Upper bound: the other warps may be building the next
// BIG_WARPS - 1 chunks, whose slices must not alias what this one reads.  Lower bound: what is read from dst instead must
// be visible, i.e. lie at least 2 * BIG_WARPS - 1 slices back (the warp that flushed it has committed its next chunk, and
// this warp has seen that commit, before this warp's previous chunk committed; 2 * BIG_WARPS back it is this warp's own).
constexpr int BIG_WARPS_MAX = 4;
constexpr int BIG_WIN_REACH = 8128;
static_assert(BIG_WIN_REACH <= (int)BIG_WIN - 64 - BIG_WARPS_MAX * (int)EXEC_TILE, "slices in flight must not alias the trusted part of the window");
static_assert(BIG_WIN_REACH >= (2 * BIG_WARPS_MAX - 1) * (int)EXEC_TILE, "bytes read from dst must have been flushed before a commit this warp has seen");

struct WinView {
    uint8_t* win;     // BIG_WIN bytes of shared memory, 16-byte aligned
    uint8_t* obase;   // dst address of chunk-relative position 0
    uint32_t gb;      // low 32 bits of obase: window index of position x is (gb + x) & BIG_WIN_MASK (exact across a wrap of
                      // the 32-bit sum, BIG_WIN divides 2^32; x is chunk-relative and the frame position does not enter it)
    int lo_rel;       // positions >= lo_rel are in the window, older ones only in dst
    __device__ __forceinline__ uint32_t idx(int x) const { return (gb + (uint32_t)x) & BIG_WIN_MASK; }
    __device__ __forceinline__ uint8_t rd(int x) const { return x >= lo_rel ? win[idx(x)] : __ldcg(obase + x); }
    // first n (<= 16) bytes from position x, which lie in the window
    __device__ __forceinline__ Vec16 load16(int x, uint32_t n) const { return win_load16<BIG_WIN>(win, gb + (uint32_t)x, n); }
    __device__ __forceinline__ void store16(int x, const Vec16& v, uint32_t n) const { win_store16<BIG_WIN>(win, gb + (uint32_t)x, v, n); }
};

// Same contract as exec_chunk_tile (lane = sequence, chunk span <= EXEC_TILE), except that only output below obase + avail_rel
// (avail_rel <= 0) is complete in dst when the call starts; wait_prev() returns once everything below obase is, and publish()
// commits the chunk.
template <typename WaitPrev, typename Publish>
__device__ __forceinline__ void exec_chunk_win(uint8_t* win, uint8_t* obase, int lo_rel, const uint8_t* __restrict__ lits, bool lit_rle,
                                               uint32_t rle_byte, unsigned lane, uint32_t ll, uint32_t ml, uint32_t off,
                                               uint32_t my_lit, uint32_t segA, uint32_t span, int avail_rel, WaitPrev wait_prev, Publish publish,
                                               long long* dbg) {
    WinView W{win, obase, (uint32_t)reinterpret_cast<uintptr_t>(obase), lo_rel};
    const uint32_t segM = segA + ll;
    const int s_lo = (int)segM - (int)off;       // chunk-relative source start of the match
    const int s_end = s_lo + (int)ml;            // the match is complete below the chunk iff s_end <= 0 (then off >= ml)
    const uint8_t* msrc = obase + s_lo;
    // literal runs: first 16 bytes per lane, tails by the whole warp
    {
        const uint32_t nl = lit_rle ? 0u : (ll < 16u ? ll : 16u);
        W.store16((int)segA, load16_unaligned(lits + my_lit, nl), nl);
    }
    for (unsigned m = __ballot_sync(0xFFFFFFFFu, !lit_rle && ll > 16u); m; m &= m - 1) {
        const int j = __ffs(m) - 1;
        const uint32_t d = __shfl_sync(0xFFFFFFFFu, segA, j) + 16u, cnt = __shfl_sync(0xFFFFFFFFu, ll, j) - 16u, lp = __shfl_sync(0xFFFFFFFFu, my_lit, j) + 16u;
        for (uint32_t i = lane; i < cnt; i += 32) win[W.idx((int)(d + i))] = lits[lp + i];
    }
    if (lit_rle) for (uint32_t k = 0; __any_sync(0xFFFFFFFFu, k < ll); k++) if (k < ll) win[W.idx((int)(segA + k))] = (uint8_t)rle_byte;
    // matches whose whole source lies below the chunk and is complete: `pred` selects them (those available when the chunk
    // starts, then, after the wait, the rest).  Source in the window or in dst per lane; a source that straddles the
    // window's lower edge goes byte by byte.
    auto copy_far = [&](bool pred) {
        const bool in_win = pred && s_lo >= lo_rel, in_dst = pred && s_end <= lo_rel;
        const uint32_t nm = (in_win || in_dst) ? (ml < 16u ? ml : 16u) : 0u;
        const Vec16 xw = W.load16(in_win ? s_lo : 0, in_win ? nm : 0u), xg = load16_unaligned<true>(msrc, in_dst ? nm : 0u);
        Vec16 x;
#pragma unroll
        for (int k = 0; k < 4; k++) x.v[k] = in_win ? xw.v[k] : xg.v[k];
        W.store16((int)segM, x, nm);
        // tails and straddling sources: the whole warp on one match at a time
        for (unsigned m = __ballot_sync(0xFFFFFFFFu, pred && (ml > 16u || nm == 0u)); m; m &= m - 1) {
            const int j = __ffs(m) - 1;
            const uint32_t dM = __shfl_sync(0xFFFFFFFFu, segM, j), n = __shfl_sync(0xFFFFFFFFu, ml, j), skip = __shfl_sync(0xFFFFFFFFu, nm, j);
            const int s0 = __shfl_sync(0xFFFFFFFFu, s_lo, j);
            for (uint32_t i = skip + lane; i < n; i += 32) win[W.idx((int)(dM + i))] = W.rd(s0 + (int)i);
        }
    };
    const bool indep = ml > 0 && s_end <= avail_rel;
    copy_far(indep);
    __syncwarp();
    CLK_MARK(2);
    wait_prev();
    CLK_MARK(3);
    const bool late = ml > 0 && !indep && s_end <= 0;
    if (__any_sync(0xFFFFFFFFu, late)) { copy_far(late); __syncwarp(); }
    CLK_MARK(4);
    // Matches that read this chunk's own output: in sequence order, the whole warp on each one, so every source byte is
    // final when it is read.  A match that overlaps itself (offset < length, decode_buffer.cairo:101-120) repeats its
    // first `offset` source bytes, which lie before its destination.
    for (unsigned U = __ballot_sync(0xFFFFFFFFu, ml > 0 && s_end > 0); U; U &= U - 1) {
        const int j = __ffs(U) - 1;
        const uint32_t dM = __shfl_sync(0xFFFFFFFFu, segM, j), n = __shfl_sync(0xFFFFFFFFu, ml, j), o = __shfl_sync(0xFFFFFFFFu, off, j);
        const int s0 = (int)dM - (int)o;
        if (o >= n && s0 >= 0) {  // the usual case: source inside the chunk, no self-overlap
            for (uint32_t i = lane; i < n; i += 32) win[W.idx((int)(dM + i))] = win[W.idx(s0 + (int)i)];
        } else if (o >= n) {
            for (uint32_t i = lane; i < n; i += 32) win[W.idx((int)(dM + i))] = W.rd(s0 + (int)i);
        } else {
            for (uint32_t i = lane; i < n; i += 32) win[W.idx((int)(dM + i))] = W.rd(s0 + (int)(i % o));
        }
        __syncwarp();
    }
    CLK_MARK(5);
    publish();  // the slice is complete: later chunks may read it from the window
    CLK_MARK(7);
    // copy to dst, off the commit chain: aligned 16-byte stores (window index and dst address agree modulo 16)
    const uint32_t a0 = W.gb & 15u;
    const uint32_t head = span < ((16 - a0) & 15) ? span : ((16 - a0) & 15);
    if (lane < head) obase[lane] = win[W.idx((int)lane)];
    const uint32_t body = span - head, nv = body >> 4, tail = body & 15;
    uint4* g4 = reinterpret_cast<uint4*>(obase + head);
    for (uint32_t v = lane; v < nv; v += 32) g4[v] = *reinterpret_cast<const uint4*>(win + W.idx((int)(head + (v << 4))));
    if (lane < tail) obase[head + (nv << 4) + lane] = win[W.idx((int)(head + (nv << 4) + lane))];
    __syncwarp();
    CLK_MARK(6);
}

__global__ void __launch_bounds__(EXEC_WARPS * 32, EXEC_MIN_CTAS) k_exec(const czb_frame_desc* __restrict__ descs, const FrameInfo* __restrict__ infos,
                                                           BigRule rule, uint32_t n_exec, WaveCounters* __restrict__ counters, const uint32_t* __restrict__ exec_order,
                                                           BlockDesc* __restrict__ blocks,
                                                           const uint8_t* __restrict__ lit_scratch, const Seq* __restrict__ seq_scratch,
                                                           czb_frame_result* __restrict__ results, const FrameResume* __restrict__ resume) {
    __shared__ ExecWarpSmem smem[EXEC_WARPS];
    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    ExecWarpSmem& sm = smem[warp];
    // Persistent warps pulling frames from a queue: frames differ in size by orders of magnitude
    // (1 KiB .. tens of MiB), so a static frame -> warp map would leave most warps idle at the tail.
    for (;;) {
    unsigned int fq = 0;
    if (lane == 0) fq = atomicAdd(&counters->exec_next, 1u);
    const uint64_t qpos = __shfl_sync(0xFFFFFFFFu, fq, 0);
    if (qpos >= n_exec) break;
    const uint64_t f = exec_order[qpos];  // largest frames first
    const FrameInfo fi = infos[f];
    if (fi.status != CZS_OK) continue;  // k_header_results already reported it
    if (frame_is_big(fi, rule)) continue;  // k_exec_big's
    const czb_frame_desc fd = descs[f];
    const uint8_t* src = fd.src;
    uint8_t* dst = fd.dst;
    // (telling the compiler that src / dst are global memory -- __builtin_assume(__isGlobal(..)): LDG / STG instead of generic LD / ST --
    // was measured: k_exec 43.2 -> 44.9 ms per three waves)
    const uint64_t cap = fd.dst_cap < MAX_FRAME_OUT ? fd.dst_cap : MAX_FRAME_OUT;
    const int32_t cap_status = fd.dst_cap < MAX_FRAME_OUT ? CZS_DST_TOO_SMALL : CZS_UNSUPPORTED;

    uint64_t out = 0;  // bytes appended so far == DecodeBuffer.len() == total_output_counter
    uint32_t h0 = 1, h1 = 4, h2 = 8;  // scratch.cairo:35
    int32_t status = CZS_OK;
    uint32_t n_done = 0;
    uint64_t bytes_read = fi.hdr_len;
    bool finished = false;
    if (resume) { const FrameResume r = resume[f]; out = r.out0; h0 = r.h0; h1 = r.h1; h2 = r.h2; n_done = r.start_block; bytes_read = r.bytes_read0; }

    for (uint32_t k = n_done; k < fi.n_blocks && status == CZS_OK; k++) {
        const BlockDesc d = blocks[fi.block_base + k];
        const uint64_t out_before = out;
        if (d.type == BT_ERROR) { status = d.pre_status; break; }
        if (d.type == BT_RAW) {
            if (out + d.size > cap) { status = cap_status; break; }
            warp_copy(dst + out, src + d.src_off, d.size);
            out += d.size; bytes_read += 3ull + d.size;
        } else if (d.type == BT_RLE) {
            if (out + d.size > cap) { status = cap_status; break; }
            warp_fill(dst + out, src[d.src_off], d.size);
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
            uint32_t lit_pos = 0;
            __syncwarp();
            const Seq* seqs = seq_scratch + d.seq_off;
            // records are read exactly once: stream them (evict-first) so that L2 keeps the frame's recent output instead
            Seq rec_next = lane < d.n_seq ? __ldcs(seqs + lane) : 0ull;
            for (uint32_t s0 = 0; s0 < d.n_seq; s0 += 32) {
                const uint32_t i = s0 + lane;
                const bool have = i < d.n_seq;
                const Seq rec = rec_next;
                if (i + 32 < d.n_seq) rec_next = __ldcs(seqs + i + 32);  // next chunk's record is in flight while this chunk executes
                uint32_t ll = 0, ml = 0, off = 1;
                if (have) { ll = seq_ll(rec); ml = seq_ml(rec); off = off29_resolve(seq_off29(rec), h0, h1, h2); }
                // warp prefix sums: literal offsets and output offsets (u32 cannot wrap: 32 * (131071 + 131074) < 2^32)
                uint32_t lsum = ll, osum = ll + ml;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {  // (shfl.up's own "source lane exists" predicate on the adds, 22 instead of 35 instructions: measured, no gain)
                    const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, lsum, o), b = __shfl_up_sync(0xFFFFFFFFu, osum, o);
                    if ((int)lane >= o) { lsum += a; osum += b; }
                }
                const uint32_t my_lit = lit_pos + lsum - ll;      // literals_copy_counter before this sequence
                const uint32_t my_out = osum - ll - ml;           // output offset of the literal run, relative to chunk base
                const uint32_t span = __shfl_sync(0xFFFFFFFFu, osum, 31);
                const uint32_t lit_used = __shfl_sync(0xFFFFFFFFu, lsum, 31);
                // Errors are rare: one cheap test that is exact for "some lane fails" (totals for the literal and
                // capacity checks, one unsigned compare per lane for offset 0 / offset beyond the output so far;
                // out <= cap < 2^31 and a chunk spans < 2^25, so 32 bits suffice; one more for a possibly far offset,
                // see off29_far), then the reference's checks in its order only if it fires.
                const uint32_t before_match32 = (uint32_t)out + my_out + ll;
                const bool suspicious = (uint64_t)lit_pos + lit_used > n_lit || out + span > cap || (have && (off - 1u >= before_match32 || off == OFF29_CLAMP));
                if (__any_sync(0xFFFFFFFFu, suspicious)) {
                    const uint64_t before_match = out + my_out + ll;  // DecodeBuffer.len() when repeat() is called
                    int32_t err = CZS_OK;
                    if (have) {
                        if (ll > 0 && (uint64_t)my_lit + ll > n_lit) err = CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE;  // :29-37
                        else if (off == 0) err = CZS_EXEC_ZERO_OFFSET;                                            // :47-49
                        else if (ml > 0 && off == OFF29_CLAMP && off29_far(seq_off29(seqs[i]), before_match))     // the raw field, not the resolved offset
                            err = CZS_UNSUPPORTED;
                        else if (ml > 0 && off > before_match)                                                      // decode_buffer.cairo:65-93
                            err = (before_match <= fi.window) ? CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY : CZS_OFFSET_TOO_BIG;
                        else if (before_match + ml > cap) err = cap_status;
                    }
                    const unsigned errm = __ballot_sync(0xFFFFFFFFu, err != CZS_OK);
                    if (errm) { status = __shfl_sync(0xFFFFFFFFu, err, __ffs(errm) - 1); break; }
                }
                if (span <= EXEC_TILE) {  // the common case: short segments, span of a few hundred bytes
                    exec_chunk_tile<false>(sm.tile, dst + out, lits, lit_rle, rle_byte, lane, ll, ml, off, my_lit, my_out, span);
                    out += span; lit_pos += lit_used;
                    continue;
                }
                // general path (long segments): publish the 64 segments of this chunk.  The checks passed, so
                // off <= before_match <= cap < 2^31 and positions are chunk-relative (< 2^25): the int casts below hold.
                const uint32_t segA = my_out, segM = my_out + ll;
                sm.bound[2 * lane] = segA; sm.bound[2 * lane + 1] = segM;
                sm.segdelta[2 * lane] = (int)my_lit - (int)segA;
                sm.segdelta[2 * lane + 1] = -(int)off;
                uint8_t* obase = dst + out;
                // gather tables, indexed by id = segment index + 1 (0 = before the chunk, 65 = past the end):
                // source address of output position p is segbase[id] + p; the byte may be fetched directly iff
                // (p - rlo) < segthr[id]: always for literals, only while the source precedes the row for matches,
                // never for overlapping matches and RLE literals (those take the per-byte path).
                sm.segbase[2 * lane + 1] = (unsigned long long)(lits + my_lit) - segA;
                sm.segbase[2 * lane + 2] = (unsigned long long)obase - off;
                sm.segthr[2 * lane + 1] = lit_rle ? 0u : 0xFFFFFFFFu;
                sm.segthr[2 * lane + 2] = off < ml ? 0u : off;
                if (lane == 0) {
                    sm.bound[64] = span;
                    sm.segbase[0] = sm.segbase[65] = (unsigned long long)obase; sm.segthr[0] = sm.segthr[65] = 0u;
                }
                const uint32_t wrapmask = __ballot_sync(0xFFFFFFFFu, have && off < ml);  // overlapping matches
                const int a = (int)(reinterpret_cast<uintptr_t>(obase) & 3);
                uint32_t carry = 0;
                for (int r = -a; r < (int)span; r += (int)EXEC_ROW) {
                    // ---- which segment owns each byte of the row ----
                    *reinterpret_cast<uint32_t*>(&sm.rowmap[4 * lane]) = 0u;
                    __syncwarp();
                    if (ll && (uint32_t)((int)segA - r) < EXEC_ROW) sm.rowmap[(int)segA - r] = (uint8_t)(2 * lane + 1);
                    if (ml && (uint32_t)((int)segM - r) < EXEC_ROW) sm.rowmap[(int)segM - r] = (uint8_t)(2 * lane + 2);
                    if (lane == 0 && (uint32_t)((int)span - r) < EXEC_ROW) sm.rowmap[(int)span - r] = 65;  // pseudo segment: past the end
                    __syncwarp();
                    uint32_t x = *reinterpret_cast<const uint32_t*>(&sm.rowmap[4 * lane]);
                    x = __vmaxu4(x, x << 8);
                    x = __vmaxu4(x, x << 16);  // running maximum inside the word (ids grow with position)
                    uint32_t tot = x >> 24;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, tot, o); if ((int)lane >= o) tot = max(tot, t); }
                    uint32_t excl = __shfl_up_sync(0xFFFFFFFFu, tot, 1);
                    if (lane == 0) excl = 0;
                    x = __vmaxu4(x, max(excl, carry) * 0x01010101u);
                    carry = __shfl_sync(0xFFFFFFFFu, x >> 24, 31);
                    *reinterpret_cast<uint32_t*>(&sm.krow[4 * lane]) = x;
                    __syncwarp();
                    // ---- gather the four bytes of this lane's word ----
                    const int p0 = r + 4 * (int)lane;
                    const int rlo = r > 0 ? r : 0;  // match sources at or beyond this position are being built in this row
                    const uint32_t pr0 = (uint32_t)(p0 - rlo);
                    uint32_t word = 0, slow_mask = 0;
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint32_t kj = (x >> (8 * j)) & 0xFFu;
                        const unsigned long long bs = sm.segbase[kj];
                        const uint32_t thr = sm.segthr[kj];
                        const uint32_t pj = (uint32_t)(p0 + j);
                        const bool valid = pj < span;
                        const bool fast = (pr0 + (uint32_t)j) < thr;
                        uint32_t b = 0;
                        if (valid && fast) b = *reinterpret_cast<const uint8_t*>(bs + pj);
                        word |= b << (8 * j);
                        if (valid && !fast) slow_mask |= 1u << j;
                    }
                    if (__any_sync(0xFFFFFFFFu, slow_mask != 0)) {
                        for (int j = 0; j < 4; j++) {
                            if (!((slow_mask >> j) & 1)) continue;
                            int p = p0 + j;
                            uint32_t kq = ((x >> (8 * j)) & 0xFFu) - 1u, byte;
                            for (;;) {
                                const int dlt = sm.segdelta[kq];
                                if (!(kq & 1u)) { byte = lit_rle ? rle_byte : lits[p + dlt]; break; }
                                int q = p + dlt;  // p - offset
                                if ((wrapmask >> (kq >> 1)) & 1u) {  // overlapping match = periodic pattern (decode_buffer.cairo:101-120)
                                    const uint32_t o = (uint32_t)(-dlt), seg0 = sm.bound[kq];
                                    q = (int)seg0 + (int)(((uint32_t)p - seg0) % o) - (int)o;
                                }
                                if (q < rlo) { byte = obase[q]; break; }  // earlier rows / chunks are already in dst
                                kq = (uint32_t)sm.krow[q - r] - 1u;        // same row, strictly earlier byte: chase
                                p = q;
                            }
                            word |= byte << (8 * j);
                        }
                    }
                    if (p0 >= 0 && (uint32_t)(p0 + 3) < span) *reinterpret_cast<uint32_t*>(obase + p0) = word;
                    else {
#pragma unroll
                        for (int j = 0; j < 4; j++) if ((uint32_t)(p0 + j) < span) obase[p0 + j] = (uint8_t)(word >> (8 * j));
                    }
                    __syncwarp();
                }
                out += span; lit_pos += lit_used;
            }
            if (status != CZS_OK) break;
            if (d.n_seq) {  // history after this block (resolved against the history it started from)
                const uint32_t n0 = sym_is(d.hist_out[0]) ? sym_resolve(d.hist_out[0], h0, h1, h2) : d.hist_out[0];
                const uint32_t n1 = sym_is(d.hist_out[1]) ? sym_resolve(d.hist_out[1], h0, h1, h2) : d.hist_out[1];
                const uint32_t n2 = sym_is(d.hist_out[2]) ? sym_resolve(d.hist_out[2], h0, h1, h2) : d.hist_out[2];
                h0 = n0; h1 = n1; h2 = n2;
            }
            // rest literals (:72-78), or all literals when there are no sequences (block_decoder.cairo:229-232)
            const uint32_t rest = n_lit - lit_pos;
            if (rest) {
                if (out + rest > cap) { status = cap_status; break; }
                if (lit_rle) warp_fill(dst + out, (uint8_t)rle_byte, rest);
                else warp_copy(dst + out, lits + lit_pos, rest);
                out += rest;
            }
            bytes_read += 3ull + d.size;
        }
        n_done++;
        if (lane == 0) {  // what the FrameDecoder handle needs to continue after this block (FrameResume)
            BlockDesc& bd = blocks[fi.block_base + k];
            bd.out_bytes = (uint32_t)(out - out_before); bd.hist_out[0] = h0; bd.hist_out[1] = h1; bd.hist_out[2] = h2;
        }
        if (d.last) {
            finished = true;
            if ((fi.descriptor >> 2) & 1) bytes_read += 4;  // the trailer was verified present by the scan (else a pseudo block follows)
        }
        __syncwarp();
    }
    if (lane == 0) {
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
    __syncwarp();
    }  // frame loop
}


// ---------------------------------------------------------------------------------------
// k_exec_big: one CTA per large frame.  A frame's blocks and sequences are one sequential stream, so the
// one-warp-per-frame kernel leaves a 17 MiB frame to a single warp.  Here BIG_WARPS warps take consecutive
// 32-sequence chunks of a block round-robin.  A per-block pre-pass (chunk totals, one scan) gives every chunk its
// literal and output offsets up front.  Chunks commit in order through two shared counters:
//   * when a chunk starts, everything below `committed_out` is complete in dst, so matches whose source ends
//     below it are copied right away (the common case for long-window data);
//   * the rest (sources in chunks still in flight, or in this chunk) wait until all earlier chunks have
//     committed and are then done in sequence order by the whole warp, exactly as in k_exec.
// Same checks, same statuses, same results as k_exec; the first failing chunk in sequence order wins.
// ---------------------------------------------------------------------------------------
#ifndef CZB_BIG_POLL_NS
#define CZB_BIG_POLL_NS 32
#endif
constexpr unsigned BIG_POLL_NS = CZB_BIG_POLL_NS;
#ifndef CZB_BIG_WARPS
#define CZB_BIG_WARPS 4  // at most BIG_WARPS_MAX (window reach); swept 4/8/16 before the window: literal-heavy 1 MiB frames 398/367/346 GB/s, 17 MiB long-window frames 15.9/16.5/15.4 GB/s
#endif
constexpr int BIG_WARPS = CZB_BIG_WARPS;
#ifndef CZB_BIG_MIN_CTAS
#define CZB_BIG_MIN_CTAS 7  // 72 registers, no spills; ~25 KB of shared memory per CTA
#endif
constexpr int BIG_MIN_CTAS = CZB_BIG_MIN_CTAS;
static_assert(BIG_WARPS <= BIG_WARPS_MAX, "the window reach assumes at most BIG_WARPS_MAX warps");
constexpr uint32_t BIG_BATCH = 1024;  // chunks per batch (n_seq <= 0x7F00 + 0xFFFF, sequence_section.cairo: at most 3065 chunks per block)

struct BigSmem {
    uint32_t chunk_lit[BIG_BATCH + 4];  // exclusive prefix of literal bytes per chunk of the batch, [n] = batch total
    uint32_t chunk_out[BIG_BATCH + 4];  // exclusive prefix of output bytes per chunk of the batch
    __align__(16) uint8_t win[BIG_WIN];      // recent output of the current block (exec_chunk_win); warp 0's tile for a chunk longer than a slice
    unsigned long long committed_out;        // every output byte below this offset is complete (in the window or in dst)
    uint32_t n_long;                         // chunks of the current batch that are longer than a window slice
    uint16_t long_idx[BIG_BATCH];            // their indices, ascending
    uint32_t committed_chunks;               // chunks (numbered through the whole frame) committed so far
    uint32_t err_chunk;                      // smallest failing chunk number, NONE32 if none
    int32_t err_status;
};

// __threadfence_block() is membar.cta = fence.sc.cta, a sequentially consistent fence: several hundred cycles each, and
// k_exec_big has four of them on every chunk.  Acquire/release ordering is all the commit protocol needs.
__device__ __forceinline__ void fence_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }

__device__ __forceinline__ void cta_copy(uint8_t* dst, const uint8_t* src, uint64_t n, unsigned warp) {
    const uint64_t per = ((n + BIG_WARPS - 1) / BIG_WARPS + 15) & ~15ull;
    const uint64_t lo = (uint64_t)warp * per;
    if (lo < n) warp_copy(dst + lo, src + lo, (uint32_t)(n - lo < per ? n - lo : per));
}
__device__ __forceinline__ void cta_fill(uint8_t* dst, uint8_t byte, uint64_t n, unsigned warp) {
    const uint64_t per = ((n + BIG_WARPS - 1) / BIG_WARPS + 15) & ~15ull;
    const uint64_t lo = (uint64_t)warp * per;
    if (lo < n) warp_fill(dst + lo, byte, (uint32_t)(n - lo < per ? n - lo : per));
}

__global__ void __launch_bounds__(BIG_WARPS * 32, BIG_MIN_CTAS) k_exec_big(const czb_frame_desc* __restrict__ descs, const FrameInfo* __restrict__ infos,
                                                           BigRule rule,
                                                           const uint32_t* __restrict__ exec_order, BlockDesc* __restrict__ blocks,
                                                           const uint8_t* __restrict__ lit_scratch, const Seq* __restrict__ seq_scratch,
                                                           czb_frame_result* __restrict__ results, const FrameResume* __restrict__ resume) {
    extern __shared__ __align__(16) uint8_t big_raw[];
    BigSmem& sm = *reinterpret_cast<BigSmem*>(big_raw);
    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    const uint64_t f = exec_order[blockIdx.x];
    const FrameInfo fi = infos[f];
    if (fi.status != CZS_OK) return;  // k_header_results already reported it
    if (!frame_is_big(fi, rule)) return;  // k_exec's
    const czb_frame_desc fd = descs[f];
    const uint8_t* src = fd.src;
    uint8_t* dst = fd.dst;
    const uint64_t cap = fd.dst_cap < MAX_FRAME_OUT ? fd.dst_cap : MAX_FRAME_OUT;
    const int32_t cap_status = fd.dst_cap < MAX_FRAME_OUT ? CZS_DST_TOO_SMALL : CZS_UNSUPPORTED;
    volatile unsigned long long* v_out = &sm.committed_out;
    volatile uint32_t* v_chunks = &sm.committed_chunks;
    if (threadIdx.x == 0) { sm.committed_out = 0; sm.committed_chunks = 0; sm.err_chunk = NONE32; sm.err_status = CZS_OK; }
    __syncthreads();

    // every thread tracks the frame-level state identically (all of it is uniform)
    uint64_t out = 0;
    uint32_t h0 = 1, h1 = 4, h2 = 8;  // scratch.cairo:35
    int32_t status = CZS_OK;
    uint32_t n_done = 0, gc_base = 0;
    uint64_t bytes_read = fi.hdr_len;
    bool finished = false;
    if (resume) { const FrameResume r = resume[f]; out = r.out0; h0 = r.h0; h1 = r.h1; h2 = r.h2; n_done = r.start_block; bytes_read = r.bytes_read0; }
    if (threadIdx.x == 0) sm.committed_out = out;
    __syncthreads();

#ifdef CZB_BIG_CLOCK
    long long dbg_t0 = clock64();
    long long* dbg = (blockIdx.x == 0 && threadIdx.x == 0) ? &dbg_t0 : nullptr;
#else
    long long* dbg = nullptr;
#endif
    for (uint32_t k = n_done; k < fi.n_blocks && status == CZS_OK; k++) {
        CLK_MARK(9);
        const BlockDesc d = blocks[fi.block_base + k];
        const uint64_t out_before = out;
        if (d.type == BT_ERROR) { status = d.pre_status; break; }
        if (d.type == BT_RAW) {
            if (out + d.size > cap) { status = cap_status; break; }
            cta_copy(dst + out, src + d.src_off, d.size, warp);
            out += d.size; bytes_read += 3ull + d.size;
        } else if (d.type == BT_RLE) {
            if (out + d.size > cap) { status = cap_status; break; }
            cta_fill(dst + out, src[d.src_off], d.size, warp);
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
            // A block's chunks are taken in batches of BIG_BATCH (the two prefix tables stay small, so that seven CTAs fit an
            // SM; a block of text has ~250 chunks, i.e. one batch).
            uint32_t lit_total = 0, out_total = 0;  // literal / output bytes of the batches done so far
            for (uint32_t cb = 0; cb < n_chunks && sm.err_chunk == NONE32; cb += BIG_BATCH) {
            const uint32_t nb = n_chunks - cb < BIG_BATCH ? n_chunks - cb : BIG_BATCH;
            // ---- pre-pass: literal and output bytes of every chunk of the batch, then one exclusive scan ----
            // (four chunks per iteration so that four record loads are in flight: the loop is a chain of global round trips)
            for (uint32_t q0 = warp * 4; q0 < nb; q0 += BIG_WARPS * 4) {
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
            __syncthreads();
            if (warp == 0) {
                uint32_t cl = 0, co = 0, n_long = 0;
                for (uint32_t b = 0; b < nb; b += 32) {
                    const uint32_t c = b + lane;
                    const uint32_t vl = c < nb ? sm.chunk_lit[c] : 0u, vo = c < nb ? sm.chunk_out[c] : 0u;
                    const unsigned lm = __ballot_sync(0xFFFFFFFFu, vo > EXEC_TILE);  // chunks that do not fit a window slice
                    if (vo > EXEC_TILE) sm.long_idx[n_long + __popc(lm & lanemask_lt())] = (uint16_t)c;
                    n_long += __popc(lm);
                    uint32_t il = vl, io = vo;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, il, o), b2 = __shfl_up_sync(0xFFFFFFFFu, io, o);
                        if ((int)lane >= o) { il += a; io += b2; }
                    }
                    if (c < nb) { sm.chunk_lit[c] = cl + il - vl; sm.chunk_out[c] = co + io - vo; }
                    cl += __shfl_sync(0xFFFFFFFFu, il, 31); co += __shfl_sync(0xFFFFFFFFu, io, 31);
                }
                if (lane == 0) { sm.chunk_lit[nb] = cl; sm.chunk_out[nb] = co; sm.n_long = n_long; }
            }
            __syncthreads();
            const uint32_t lit_batch = sm.chunk_lit[nb], out_batch = sm.chunk_out[nb];
            const uint32_t n_long = sm.n_long;
            CLK_MARK(0);
            // ---- chunks, committed in order.  A chunk that fits a window slice (the usual case) goes round-robin over the
            // warps; a long one is done by warp 0 alone between two CTA barriers, straight into dst, and the window starts
            // afresh after it: so all slices in flight at any time lie within BIG_WARPS * EXEC_TILE bytes and never alias,
            // and what the window does not hold was made visible by a barrier. ----
            uint32_t seg = 0;  // first chunk of the current run of window chunks
            for (uint32_t kl = 0; kl <= n_long && seg < nb; kl++) {
            const uint32_t L = kl < n_long ? sm.long_idx[kl] : nb;  // the long chunk that ends the run (nb: none)
            const uint32_t seg_out0 = sm.chunk_out[seg];
            for (int pass = 0; pass < 2; pass++) {
            const uint32_t q_lo = pass == 0 ? seg + warp : (warp == 0 ? L : nb), q_hi = pass == 0 ? L : (L < nb ? L + 1 : L);
            for (uint32_t q = q_lo; q < q_hi; q += BIG_WARPS) {
                const uint32_t c = cb + q;
                const uint32_t gc = gc_base + c;
                const uint32_t i = c * 32 + lane;
                const bool have = i < d.n_seq;
                uint32_t ll = 0, ml = 0, off = 1;
                CLK_MARK(10);
                if (have) { const Seq rec = __ldcs(seqs + i); ll = seq_ll(rec); ml = seq_ml(rec); off = off29_resolve(seq_off29(rec), h0, h1, h2); }
#ifdef CZB_BIG_CLOCK
                if (dbg && ll == 0xFFFFFFFFu) printf("x");  // consume the record before the mark: the load's latency belongs to this phase
#endif
                CLK_MARK(11);
                uint32_t lsum = ll, osum = ll + ml;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, lsum, o), b = __shfl_up_sync(0xFFFFFFFFu, osum, o);
                    if ((int)lane >= o) { lsum += a; osum += b; }
                }
#ifdef CZB_BIG_CLOCK
                if (dbg && osum == 0xFFFFFFFFu) printf("y");  // likewise for the prefix sums
#endif
                CLK_MARK(12);
                const uint32_t lit_pos = lit_total + sm.chunk_lit[q];
                const uint64_t out_c = out + out_total + sm.chunk_out[q];
                const uint32_t my_lit = lit_pos + lsum - ll, my_out = osum - ll - ml;
                const uint32_t span = __shfl_sync(0xFFFFFFFFu, osum, 31);
                // the reference's checks in its order (see k_exec); a failing chunk writes nothing but still commits
                const uint64_t before_match = out_c + my_out + ll;
                int32_t err = CZS_OK;
                if (have) {
                    if (ll > 0 && (uint64_t)my_lit + ll > n_lit) err = CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE;  // :29-37
                    else if (off == 0) err = CZS_EXEC_ZERO_OFFSET;                                            // :47-49
                    else if (ml > 0 && off == OFF29_CLAMP && off29_far(seq_off29(seqs[i]), before_match))     // the raw field, not the resolved offset
                        err = CZS_UNSUPPORTED;
                    else if (ml > 0 && off > before_match)                                                      // decode_buffer.cairo:65-93
                        err = (before_match <= fi.window) ? CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY : CZS_OFFSET_TOO_BIG;
                    else if (before_match + ml > cap) err = cap_status;
                }
                const unsigned errm = __ballot_sync(0xFFFFFFFFu, err != CZS_OK);
                CLK_MARK(1);
                auto wait_prev = [&]() {
                    while (*v_chunks != gc) __nanosleep(BIG_POLL_NS);
                    fence_cta();
                };
                auto publish = [&]() {
                    __syncwarp();
                    if (lane == 0) { fence_cta(); *v_out = out_c + span; fence_cta(); *v_chunks = gc + 1; }
                };
                if (errm) {
                    const int32_t e = __shfl_sync(0xFFFFFFFFu, err, __ffs(errm) - 1);
                    wait_prev();  // every earlier chunk has committed: if one of them failed, its number is already there
                    if (lane == 0 && gc < sm.err_chunk) { sm.err_chunk = gc; sm.err_status = e; }
                    publish();
                } else if (span <= EXEC_TILE) {
                    const unsigned long long avail = *v_out;  // a lower bound is fine: it only grows
                    fence_cta();
                    const uint64_t behind = out_c - (avail < out_c ? avail : out_c);
                    const int avail_rel = -(int)(behind < 0x40000000ull ? behind : 0x40000000ull);
                    const uint32_t in_run = sm.chunk_out[q] - seg_out0;  // bytes of this run before the chunk: all of them went through the window
                    const int lo_rel = -(int)(in_run < (uint32_t)BIG_WIN_REACH ? in_run : (uint32_t)BIG_WIN_REACH);
                    exec_chunk_win(sm.win, dst + out_c, lo_rel, lits, lit_rle, rle_byte, lane, ll, ml, off, my_lit, my_out, span, avail_rel, wait_prev, publish, dbg);
                } else {
                    // A chunk that does not fit a slice: once everything before it is in dst, it is cut at sequence boundaries
                    // into pieces that do fit (each executed like a chunk of its own, through a tile, with the lanes outside
                    // the piece idle); a single sequence that does not fit is copied straight into dst by the whole warp
                    // (overlapping matches as a repeated pattern, decode_buffer.cairo:101-120).
                    wait_prev();
                    for (uint32_t start = 0; start < 32;) {
                        const uint32_t base_o = __shfl_sync(0xFFFFFFFFu, my_out, start);
                        const unsigned fit = __ballot_sync(0xFFFFFFFFu, lane >= start && my_out + ll + ml - base_o <= EXEC_TILE);
                        if (!((fit >> start) & 1u)) {
                            const int j = (int)start;
                            const uint32_t jl = __shfl_sync(0xFFFFFFFFu, ll, j), jm = __shfl_sync(0xFFFFFFFFu, ml, j), jo = __shfl_sync(0xFFFFFFFFu, off, j);
                            const uint32_t jlit = __shfl_sync(0xFFFFFFFFu, my_lit, j);
                            uint8_t* o = dst + out_c + base_o;
                            if (jl) { if (lit_rle) warp_fill(o, (uint8_t)rle_byte, jl); else warp_copy(o, lits + jlit, jl); }
                            o += jl;
                            if (jm) {
                                __syncwarp();
                                fence_cta();
                                if (jo >= jm) warp_copy(o, o - jo, jm);
                                else for (uint32_t t = lane; t < jm; t += 32) o[t] = __ldcg(o - jo + (t % jo));
                            }
                            start++;
                        } else {
                            const uint32_t last = 31u - (uint32_t)__clz(fit);  // fit is a run of lanes from `start` (offsets only grow)
                            const bool in = lane >= start && lane <= last;
                            const uint32_t span_p = __shfl_sync(0xFFFFFFFFu, my_out + ll + ml, last) - base_o;
                            exec_chunk_tile<true>(sm.win, dst + out_c + base_o, lits, lit_rle, rle_byte, lane, in ? ll : 0u, in ? ml : 0u, off, my_lit,
                                                  in ? my_out - base_o : 0u, span_p);
                            start = last + 1;
                        }
                        __syncwarp();
                        fence_cta();  // the next piece reads this one's bytes from dst
                    }
                    __syncwarp();
                    fence_cta();
                    publish();
                }
            }
            __syncthreads();  // everything up to here is complete in dst and visible to the whole CTA
            }  // pass
            seg = L + 1;
            }  // runs of window chunks
            CLK_MARK(8);
            lit_total += lit_batch; out_total += out_batch;
            }  // batch loop
            if (sm.err_chunk != NONE32) { status = sm.err_status; break; }
            gc_base += n_chunks;
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
                if (lit_rle) cta_fill(dst + out, (uint8_t)rle_byte, rest, warp);
                else cta_copy(dst + out, lits + lit_total, rest, warp);
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
        if (threadIdx.x == 0) { *v_out = out; }
        __syncthreads();
    }
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
#ifdef CZB_BIG_CLOCK
    if (dbg) {
        CLK_MARK(9);
        printf("big clk: prepass %llu | checks %llu | first pass %llu | wait %llu | late %llu | in-chunk %llu | flush %llu | publish %llu | block end %llu | block start/raw/rest %llu\n",
               czb_dbg_clk[0], czb_dbg_clk[1], czb_dbg_clk[2], czb_dbg_clk[3], czb_dbg_clk[4], czb_dbg_clk[5], czb_dbg_clk[6], czb_dbg_clk[7], czb_dbg_clk[8], czb_dbg_clk[9]);
        printf("   loop top + long chunks %llu | rec load %llu | prefix %llu\n", czb_dbg_clk[10], czb_dbg_clk[11], czb_dbg_clk[12]);
        for (int q = 0; q < 16; q++) czb_dbg_clk[q] = 0;
    }
#endif
}

void launch_exec(const LaunchCtx& lc, const ExecSide& side, int sm_count, const czb_frame_desc* descs, const FrameInfo* infos, uint64_t first, uint64_t count, uint32_t n_big_cls,
                 uint32_t n_exec, BigRule rule, WaveCounters* counters,
                 const uint32_t* exec_order, BlockDesc* blocks, const uint8_t* lit_scratch, const Seq* seq_scratch,
                 czb_frame_result* results) {
    if (!count || !n_exec) return;
    // exec_order lists the wave's frames largest size class first.  k_exec_big gets one CTA for each of the first
    // n_big_cls entries (the frames of at least 2^min(big_cls, share_cls) bytes) and takes those that pass frame_is_big;
    // k_exec walks the whole list and skips exactly those.  The two kernels run side by side: k_exec_big on its own
    // (higher priority) stream, forked from and joined to the caller's.
    if (n_big_cls) {
        cudaEventRecord(side.fork, lc.stream);
        cudaStreamWaitEvent(side.stream, side.fork, 0);
        if (side.flow) {
            LaunchCtx ls{side.stream, lc.launches};
            launch_exec_flow(ls, n_big_cls, descs + first, infos + first, rule, exec_order, blocks, lit_scratch, seq_scratch, results + first, side.resume ? side.resume + first : nullptr, side.flow_wide);
        } else {
            k_exec_big<<<n_big_cls, BIG_WARPS * 32, sizeof(BigSmem), side.stream>>>(descs + first, infos + first, rule, exec_order, blocks, lit_scratch, seq_scratch, results + first, side.resume ? side.resume + first : nullptr);
            ++*lc.launches;
        }
        cudaEventRecord(side.join, side.stream);
    }
    const uint64_t want = ((uint64_t)n_exec + EXEC_WARPS - 1) / EXEC_WARPS;
    const uint64_t persistent = (uint64_t)sm_count * EXEC_CTAS_PER_SM;  // per device: the context carries its own SM count
    const unsigned grid = (unsigned)(want < persistent ? want : persistent);
    k_exec<<<grid, EXEC_WARPS * 32, 0, lc.stream>>>(descs + first, infos + first, rule, n_exec, counters, exec_order, blocks, lit_scratch, seq_scratch, results + first, side.resume ? side.resume + first : nullptr);
    ++*lc.launches;
    if (n_big_cls) cudaStreamWaitEvent(lc.stream, side.join, 0);
}

int setup_exec_attributes() {
    return (int)cudaFuncSetAttribute(k_exec_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BigSmem));
}

}  // namespace czb
