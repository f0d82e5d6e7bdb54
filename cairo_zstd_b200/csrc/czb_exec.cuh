// czb_exec.cuh -- helpers shared by the sequence-execution kernels (k_exec, k_exec_big in k_exec.cu; k_exec_flow in
// k_exec_flow.cu): warp-wide copies, unaligned 16-byte loads, the shared-memory tile executor of one 32-sequence chunk,
// and the rule that decides which frames get a whole CTA.
#pragma once
#include "czb_internal.cuh"

namespace czb {

constexpr int EXEC_WARPS = 4;
#ifndef EXEC_MIN_CTAS
#define EXEC_MIN_CTAS 7
#endif
#ifndef EXEC_CTAS_PER_SM
#define EXEC_CTAS_PER_SM 7
#endif
constexpr uint32_t EXEC_ROW = 128;
constexpr uint32_t EXEC_TILE = 1024;

struct ExecWarpSmem {
    uint32_t bound[66];      // bound[2i] = first output byte of sequence i's literal run, [2i+1] = of its match, [64] = span
    int segdelta[66];        // per segment: source index = output position + delta (literal buffer for even ids, dst for odd);
                             // [64] is the "past the end" pseudo segment
    unsigned long long segbase[66];  // indexed by id = segment index + 1: address of the source byte for output position 0
    uint32_t segthr[66];     // indexed by id: a byte at row-relative... see gather: fast iff (p - rlo) < segthr[id]
    __align__(16) uint8_t tile[EXEC_TILE + 48];  // a chunk's whole output span (sequence-centric path)
    __align__(4) uint8_t rowmap[EXEC_ROW];  // (segment id + 1) at each non-empty segment's start byte inside the row
    __align__(4) uint8_t krow[EXEC_ROW];    // (segment id + 1) owning each row byte
};

// dst[0..n) = src[0..n): 16-byte stores to aligned dst; src may have any alignment (aligned
// 32-bit loads + funnel shifts).  Only aligned words containing at least one source byte are read.
__device__ __forceinline__ void warp_copy(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, uint32_t n) {
    const unsigned lane = lane_id();
    if (n >= 64) {
        const uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15);
        if (lane < head) dst[lane] = src[lane];
        dst += head; src += head; n -= head;
        const uint32_t nv = n >> 4;
        const uintptr_t sa = reinterpret_cast<uintptr_t>(src);
        const uint32_t sh = (uint32_t)(sa & 3) * 8;
        const uint32_t* sw = reinterpret_cast<const uint32_t*>(sa & ~uintptr_t(3));
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (uint32_t i = lane; i < nv; i += 32) {
            const uint32_t* w = sw + 4 * i;
            const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
            const uint32_t w4 = sh ? w[4] : 0u;
            uint4 v;
            v.x = __funnelshift_r(w0, w1, sh); v.y = __funnelshift_r(w1, w2, sh);
            v.z = __funnelshift_r(w2, w3, sh); v.w = __funnelshift_r(w3, w4, sh);
            d4[i] = v;
        }
        dst += nv << 4; src += nv << 4; n &= 15;
    }
    for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i];
}

__device__ __forceinline__ void warp_fill(uint8_t* dst, uint8_t byte, uint32_t n) {
    const unsigned lane = lane_id();
    if (n >= 64) {
        const uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15);
        if (lane < head) dst[lane] = byte;
        dst += head; n -= head;
        const uint32_t w = byte * 0x01010101u;
        const uint4 v = make_uint4(w, w, w, w);
        const uint32_t nv = n >> 4;
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (uint32_t i = lane; i < nv; i += 32) d4[i] = v;
        dst += nv << 4; n &= 15;
    }
    for (uint32_t i = lane; i < n; i += 32) dst[i] = byte;
}

// 16 source bytes starting at src (any alignment, GLOBAL memory) as four little-endian words.  Only the
// aligned 32-bit words that hold one of the first n bytes are read.
// The loads stay plain C: ptxas turns the "needed?" chain into branches that skip a word altogether when no lane needs it
// (literal runs average three bytes: words 2..4 are almost never read), which measured faster than one predicated ld.global
// per word (k_exec 43.2 against 44.4 ms per three waves).
struct Vec16 { uint32_t v[4]; };
template <bool CG = false>  // CG: read through L2 (data another warp of the CTA has just written)
__device__ __forceinline__ Vec16 load16_unaligned(const uint8_t* __restrict__ src, uint32_t n) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(src);
    const uint32_t mis = (uint32_t)(a & 3), sh = mis * 8, need = n + mis;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    auto ld = [&](int k) -> uint32_t { return CG ? __ldcg(w + k) : w[k]; };
    const uint32_t w0 = n ? ld(0) : 0u;
    const uint32_t w1 = need > 4 ? ld(1) : 0u, w2 = need > 8 ? ld(2) : 0u, w3 = need > 12 ? ld(3) : 0u, w4 = need > 16 ? ld(4) : 0u;
    Vec16 r;
    r.v[0] = __funnelshift_r(w0, w1, sh); r.v[1] = __funnelshift_r(w1, w2, sh);
    r.v[2] = __funnelshift_r(w2, w3, sh); r.v[3] = __funnelshift_r(w3, w4, sh);
    return r;
}
// t[0..n) = the first n bytes of x (byte stores into the shared-memory tile).  Groups of four bytes are skipped
// warp-uniformly when no lane needs them, so short segments do not pay for sixteen predicated stores.
// The stores go through inline asm on ONE address register with immediate offsets: left to itself ptxas re-forms
// "tile base + alignment + segment start" under every store's predicate (a three-input add per byte, to save a register under the
// 72-register cap): 4 instructions per byte instead of 3 on the integer pipe that issues one instruction per two cycles.
// No "memory" clobber on the stores (the loads of the next vector may move across them); tile_stores_done() orders them
// before anything that reads the tile.
__device__ __forceinline__ uint32_t tile_addr(const uint8_t* t) {
    uint32_t a = (uint32_t)__cvta_generic_to_shared(t);
    asm volatile("" : "+r"(a));  // opaque: one register, not a sum to re-form
    return a;
}
// byte K of the segment, if the segment has one: the predicate lives inside the asm (an `if` around it becomes a divergent branch per byte)
template <int K>
__device__ __forceinline__ void sts_u8_if(uint32_t a, uint32_t v, uint32_t n) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.gt.u32 p, %3, %2;\n\t@p st.shared.u8 [%0+%2], %1;\n\t}" ::"r"(a), "r"(v), "n"(K), "r"(n));
}
__device__ __forceinline__ void tile_stores_done() { asm volatile("" ::: "memory"); }
template <int G>
__device__ __forceinline__ void store4_to_tile(uint32_t a, uint32_t w, uint32_t n) {
    sts_u8_if<4 * G>(a, w, n); sts_u8_if<4 * G + 1>(a, w >> 8, n); sts_u8_if<4 * G + 2>(a, w >> 16, n); sts_u8_if<4 * G + 3>(a, w >> 24, n);
}
__device__ __forceinline__ void store16_to_tile(uint8_t* t, const Vec16& x, uint32_t n) {
    const uint32_t a = tile_addr(t);
    store4_to_tile<0>(a, x.v[0], n);
    if (__any_sync(0xFFFFFFFFu, n > 4u)) store4_to_tile<1>(a, x.v[1], n);
    if (__any_sync(0xFFFFFFFFu, n > 8u)) store4_to_tile<2>(a, x.v[2], n);
    if (__any_sync(0xFFFFFFFFu, n > 12u)) store4_to_tile<3>(a, x.v[3], n);
}

// All lanes copy n bytes src -> tile + dst_off for the lane `j` that owns the job (arguments are taken from lane j).
template <bool CG = false>
__device__ __forceinline__ void coop_copy_to_tile(uint8_t* tile, unsigned lane, int j, uint32_t dst_off, const uint8_t* src, uint32_t n) {
    const uint32_t d = __shfl_sync(0xFFFFFFFFu, dst_off, j), cnt = __shfl_sync(0xFFFFFFFFu, n, j);
    const unsigned long long sp = __shfl_sync(0xFFFFFFFFu, (unsigned long long)reinterpret_cast<uintptr_t>(src), j);
    const uint8_t* s = reinterpret_cast<const uint8_t*>((uintptr_t)sp);
    for (uint32_t i = lane; i < cnt; i += 32) tile[d + i] = CG ? __ldcg(s + i) : s[i];
}

// the same without the votes
__device__ __forceinline__ void store16_to_tile_all(uint8_t* t, const Vec16& x, uint32_t n) {
    const uint32_t a = tile_addr(t);
    store4_to_tile<0>(a, x.v[0], n); store4_to_tile<1>(a, x.v[1], n); store4_to_tile<2>(a, x.v[2], n); store4_to_tile<3>(a, x.v[3], n);
}

// Wrapping windows (k_exec_big, k_exec_flow): WIN bytes of shared memory (a power of two, 16-byte aligned) that hold
// position p at win[p % WIN].  The first n (<= 16) bytes from position p: aligned words and funnel shifts, word indices wrapped.
template <uint32_t WIN>
__device__ __forceinline__ Vec16 win_load16(const uint8_t* win, uint32_t p, uint32_t n) {
    const uint32_t mis = p & 3u, sh = mis * 8u, need = n + mis;
    const uint32_t* w32 = reinterpret_cast<const uint32_t*>(win);
    const uint32_t wi = p >> 2;
    auto ld = [&](uint32_t k) -> uint32_t { return w32[(wi + k) & (WIN / 4 - 1)]; };
    const uint32_t w0 = n ? ld(0) : 0u;
    const uint32_t w1 = need > 4 ? ld(1) : 0u, w2 = need > 8 ? ld(2) : 0u, w3 = need > 12 ? ld(3) : 0u, w4 = need > 16 ? ld(4) : 0u;
    Vec16 r;
    r.v[0] = __funnelshift_r(w0, w1, sh); r.v[1] = __funnelshift_r(w1, w2, sh);
    r.v[2] = __funnelshift_r(w2, w3, sh); r.v[3] = __funnelshift_r(w3, w4, sh);
    return r;
}
// Positions [p, p + n) = the first n (<= 16) bytes of v.  When no lane's sixteen bytes wrap around the window's end (all but one
// vector in WIN / 16): one address per lane and immediate offsets, as in store16_to_tile; otherwise byte stores at wrapped indices.
template <uint32_t WIN>
__device__ __forceinline__ void win_store16(uint8_t* win, uint32_t p, const Vec16& v, uint32_t n) {
    if (__all_sync(0xFFFFFFFFu, (p & (WIN - 1)) <= WIN - 16u)) {
        const uint32_t a = tile_addr(win) + (p & (WIN - 1));
        store4_to_tile<0>(a, v.v[0], n);
        if (__any_sync(0xFFFFFFFFu, n > 4u)) store4_to_tile<1>(a, v.v[1], n);
        if (__any_sync(0xFFFFFFFFu, n > 8u)) store4_to_tile<2>(a, v.v[2], n);
        if (__any_sync(0xFFFFFFFFu, n > 12u)) store4_to_tile<3>(a, v.v[3], n);
        tile_stores_done();
        return;
    }
#pragma unroll
    for (int g = 0; g < 4; g++) {
        if (g == 0 || __any_sync(0xFFFFFFFFu, n > 4u * g)) {
#pragma unroll
            for (int k = 4 * g; k < 4 * g + 4; k++) if ((uint32_t)k < n) win[(p + k) & (WIN - 1)] = (uint8_t)(v.v[g] >> (8 * (k & 3)));
        }
    }
}

// Which frames get a whole CTA (k_exec_big) instead of one warp (k_exec):
//  * large ones (>= 2^big_cls compressed bytes) with sparse sequences (>= big_seq_bytes compressed bytes per sequence:
//    literal-heavy data, long matches), whose warps rarely wait for each other (1 MiB literal-heavy frames 253 -> 400 GB/s);
//  * from 2^share_cls bytes on, frames that hold at least 1/big_share of the wave's compressed bytes.  A frame is one
//    sequential stream; on one warp among ~4000 it moves at ~1/4000 of the machine's rate, so a frame with more than
//    about 1/8000 of the wave's bytes is still running when everything else has finished.  A CTA moves it two to three
//    times faster (the in-order commit chain of k_exec_big is the limit) and runs beside k_exec on its own stream.
//    (mixed 1 KiB..4 MiB frames: 118 -> 150 GB/s; a batch of equal frames never qualifies.)
__device__ __forceinline__ bool frame_is_big(const FrameInfo& fi, const BigRule& r) {
    return (fi.size_cls >= r.big_cls && fi.n_seq * r.big_seq_bytes <= fi.src_end) || (fi.size_cls >= r.share_cls && fi.src_end >= r.share_bytes);
}

// Measurement aid (-DCZB_BIG_CLOCK): cycles per phase of k_exec_big, accumulated by thread 0 of CTA 0 and printed per launch.
#ifdef CZB_BIG_CLOCK
__device__ unsigned long long czb_dbg_clk[16];
#define CLK_MARK(k) do { if (dbg) { const long long t_ = clock64(); atomicAdd(&czb_dbg_clk[k], (unsigned long long)(t_ - *dbg)); *dbg = t_; } } while (0)
#else
#define CLK_MARK(k) do { } while (0)
#endif
// Sequence-centric execution of one chunk whose output span fits the tile: lane = sequence.  Everything below obase is
// complete in dst when the call starts.  The first 16 bytes of every literal run and of every match whose source is
// already in dst are copied by their own lane (all lanes in parallel, uniform control flow); tails and the matches that
// read this chunk's own output are done by the whole warp, one at a time, in sequence order.  The tile is flushed with
// aligned 16-byte stores.  CG_LOADS: match sources are read through L2 (another warp of the CTA may have just written them).
template <bool CG_LOADS>
__device__ __forceinline__ void exec_chunk_tile(uint8_t* tile_base, uint8_t* obase, const uint8_t* __restrict__ lits, bool lit_rle,
                                                uint32_t rle_byte, unsigned lane, uint32_t ll, uint32_t ml, uint32_t off,
                                                uint32_t my_lit, uint32_t segA, uint32_t span) {
    const uint32_t a0 = (uint32_t)(reinterpret_cast<uintptr_t>(obase) & 15);
    uint8_t* tile = tile_base + a0;  // tile[p] = output byte at chunk-relative position p
    const uint32_t segM = segA + ll;
    const bool indep = ml > 0 && (int)(segM + ml) - (int)off <= 0;  // the whole source ends at or below the chunk start: already in dst
    const uint8_t* msrc = obase + ((int64_t)segM - (int64_t)off);
    // first 16 bytes of every literal run and independent match: all loads are issued before the stores
    {
        const uint32_t nl = lit_rle ? 0u : (ll < 16u ? ll : 16u), nm = indep ? (ml < 16u ? ml : 16u) : 0u;
        const Vec16 xl = load16_unaligned(lits + my_lit, nl), xm = load16_unaligned<CG_LOADS>(msrc, nm);
        store16_to_tile(tile + segA, xl, nl);      // literal runs average under three bytes: later groups are usually skipped
        store16_to_tile_all(tile + segM, xm, nm);  // matches average nine: some lane always needs every group, votes only cost
        tile_stores_done();
    }
    // Tails beyond the first 16 bytes are rare (a few per cent of the segments) and may be long: the whole warp
    // copies each one instead of every lane looping in lockstep for the longest.
    for (unsigned m = __ballot_sync(0xFFFFFFFFu, !lit_rle && ll > 16u); m; m &= m - 1)
        coop_copy_to_tile(tile, lane, __ffs(m) - 1, segA + 16u, lits + my_lit + 16, ll - 16u);
    if (lit_rle) for (uint32_t k = 0; __any_sync(0xFFFFFFFFu, k < ll); k++) if (k < ll) tile[segA + k] = (uint8_t)rle_byte;
    for (unsigned m = __ballot_sync(0xFFFFFFFFu, indep && ml > 16u); m; m &= m - 1)
        coop_copy_to_tile<CG_LOADS>(tile, lane, __ffs(m) - 1, segM + 16u, msrc + 16, ml - 16u);
    __syncwarp();
    bool done = indep || ml == 0;
    if (CG_LOADS) {
        // A match whose source ends below obase but which the signed test above did not take (an offset of 2^31 or more,
        // which the callers' checks rule out) is copied from dst in one more per-lane pass.
        const bool late = !done && segM + ml <= off;
        const uint32_t nm = late ? (ml < 16u ? ml : 16u) : 0u;
        if (__any_sync(0xFFFFFFFFu, late)) {
            store16_to_tile(tile + segM, load16_unaligned<true>(msrc, nm), nm);
            tile_stores_done();
            for (unsigned m = __ballot_sync(0xFFFFFFFFu, late && ml > 16u); m; m &= m - 1)
                coop_copy_to_tile<true>(tile, lane, __ffs(m) - 1, segM + 16u, msrc + 16, ml - 16u);
            __syncwarp();
        }
        done = done || late;
    }
    // Matches that read this chunk's own output (a few per chunk): in sequence order, the whole warp on each one, so
    // every source byte is final when it is read.  A match that overlaps itself (offset < length,
    // decode_buffer.cairo:101-120) repeats its first `offset` source bytes, which lie before its destination.
    for (unsigned U = __ballot_sync(0xFFFFFFFFu, !done); U; U &= U - 1) {
        const int j = __ffs(U) - 1;
        const uint32_t dM = __shfl_sync(0xFFFFFFFFu, segM, j), n = __shfl_sync(0xFFFFFFFFu, ml, j), o = __shfl_sync(0xFFFFFFFFu, off, j);
        const int s0 = (int)dM - (int)o;  // chunk-relative source start, may lie before the chunk (already in dst)
        if (o >= n && s0 >= 0) {  // the usual case: source inside the tile, no self-overlap
            for (uint32_t i = lane; i < n; i += 32) tile[dM + i] = tile[(uint32_t)s0 + i];
        } else if (o >= n) {
            for (uint32_t i = lane; i < n; i += 32) { const int q = s0 + (int)i; tile[dM + i] = q < 0 ? (CG_LOADS ? __ldcg(obase + q) : obase[q]) : tile[q]; }
        } else {
            for (uint32_t i = lane; i < n; i += 32) { const int q = s0 + (int)(i % o); tile[dM + i] = q < 0 ? (CG_LOADS ? __ldcg(obase + q) : obase[q]) : tile[q]; }
        }
        __syncwarp();
    }
    // flush: aligned 16-byte stores (tile index and dst address agree modulo 16)
    const uint32_t head = span < ((16 - a0) & 15) ? span : ((16 - a0) & 15);
    if (lane < head) obase[lane] = tile[lane];
    const uint32_t body = span - head, nv = body >> 4, tail = body & 15;
    const uint4* t4 = reinterpret_cast<const uint4*>(tile + head);
    uint4* g4 = reinterpret_cast<uint4*>(obase + head);
    for (uint32_t v = lane; v < nv; v += 32) g4[v] = t4[v];
    if (lane < tail) obase[head + (nv << 4) + lane] = tile[head + (nv << 4) + lane];
    __syncwarp();
}

}  // namespace czb
