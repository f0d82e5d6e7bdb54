// k_xxh.cu -- XXH64 content checksum of each decoded frame (SURVEY.md section 8 row f1).
//
// Reference: XxHash64 (src/utils/xxhash64.cairo:32-163), fed by DecodeBuffer::drain
// (src/decoding/decode_buffer.cairo:157-166) and compared with the frame trailer in
// _test_decode (src/tests/decoding.cairo:16-19); get_calculated_checksum keeps the low 32 bits
// (src/frame_decoder.cairo:133-138).
//
// XXH64 has exactly four independent accumulators per 32-byte stripe, so a frame gets four
// lanes (lane k owns accumulator v_{k+1}); a warp hashes 8 frames at once and every load
// instruction reads whole 32-byte sectors.  HBM-bound streaming read of the decoded bytes.  Lengths and stripe indices are
// 64-bit: any frame size.  A frame of MAX_FRAME_OUT bytes is 2^26 stripes on four lanes.
#include "czb_internal.cuh"

namespace czb {

constexpr uint64_t XP1 = 0x9E3779B185EBCA87ull, XP2 = 0xC2B2AE3D27D4EB4Full, XP3 = 0x165667B19E3779F9ull,
                   XP4 = 0x85EBCA77C2B2AE63ull, XP5 = 0x27D4EB2F165667C5ull;

__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ uint64_t xxh_round(uint64_t acc, uint64_t in) { return rotl64(acc + in * XP2, 31) * XP1; }
__device__ __forceinline__ uint64_t xxh_merge(uint64_t acc, uint64_t v) { acc ^= xxh_round(0, v); return acc * XP1 + XP4; }
__device__ __forceinline__ uint64_t load64(const uint8_t* p, bool aligned) {
    if (aligned) return *reinterpret_cast<const uint64_t*>(p);
    uint64_t v = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) v |= (uint64_t)p[k] << (8 * k);
    return v;
}

// The stripes of one frame for accumulator k: the 8 bytes at 32 s + 8 k of every stripe s.  The loop is issue bound
// (two 64-bit multiplies, an add and a rotate per 8 bytes: ~13 SASS instructions), so the alignment case is decided
// once, outside it (with the byte-wise unaligned load predicated into the loop it was 42 instructions per round), and
// four loads are in flight per lane.  An unaligned frame reads aligned words and funnel-shifts; both words of a value
// hold bytes of it, so nothing beyond the granules of the frame's own bytes is touched.
template <bool ALIGNED>
__device__ __forceinline__ uint64_t xxh_stripes(const uint8_t* __restrict__ p, uint64_t stripes, unsigned k, uint64_t v) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p) + 8u * k;
    const uint64_t* q = reinterpret_cast<const uint64_t*>(a & ~uintptr_t(7));
    const unsigned sh = (unsigned)(a & 7) * 8u;  // != 0 iff !ALIGNED
    auto get = [&](uint64_t s) -> uint64_t {
        if (ALIGNED) return q[4 * s];
        return (q[4 * s] >> sh) | (q[4 * s + 1] << (64u - sh));
    };
    uint64_t s = 0;
    for (; s + 4 <= stripes; s += 4) {
        const uint64_t x0 = get(s), x1 = get(s + 1), x2 = get(s + 2), x3 = get(s + 3);
        v = xxh_round(v, x0); v = xxh_round(v, x1); v = xxh_round(v, x2); v = xxh_round(v, x3);
    }
    for (; s < stripes; s++) v = xxh_round(v, get(s));
    return v;
}

__global__ void __launch_bounds__(128) k_xxh64(const czb_frame_desc* __restrict__ descs, czb_frame_result* __restrict__ results,
                                                uint64_t count) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t f = t >> 2;
    const unsigned k = (unsigned)(t & 3);
    const bool live = f < count && results[f < count ? f : 0].status == CZS_OK;
    const uint8_t* p = live ? descs[f].dst : nullptr;
    const uint64_t len = live ? results[f].bytes_written : 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(p) & 7) == 0;
    uint64_t v = k == 0 ? XP1 + XP2 : (k == 1 ? XP2 : (k == 2 ? 0ull : 0ull - XP1));  // xxhash64.cairo:32-42, seed 0
    const uint64_t stripes = len >> 5;
    v = aligned ? xxh_stripes<true>(p, stripes, k, v) : xxh_stripes<false>(p, stripes, k, v);
    const unsigned base = lane_id() & ~3u;
    const uint64_t v1 = __shfl_sync(0xFFFFFFFFu, v, base), v2 = __shfl_sync(0xFFFFFFFFu, v, base + 1),
                   v3 = __shfl_sync(0xFFFFFFFFu, v, base + 2), v4 = __shfl_sync(0xFFFFFFFFu, v, base + 3);
    if (!live || k != 0) return;
    uint64_t h;
    if (len >= 32) {  // digest :94-113
        h = rotl64(v1, 1) + rotl64(v2, 7) + rotl64(v3, 12) + rotl64(v4, 18);
        h = xxh_merge(h, v1); h = xxh_merge(h, v2); h = xxh_merge(h, v3); h = xxh_merge(h, v4);
    } else {
        h = v3 + XP5;
    }
    h += len;
    const uint8_t* q = p + (stripes << 5);
    uint64_t n = len & 31;
    while (n >= 8) { h ^= xxh_round(0, load64(q, aligned)); h = rotl64(h, 27) * XP1 + XP4; q += 8; n -= 8; }  // finalize :136-163
    if (n >= 4) { uint32_t w = q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24); h ^= (uint64_t)w * XP1; h = rotl64(h, 23) * XP2 + XP3; q += 4; n -= 4; }
    while (n) { h ^= (uint64_t)(*q) * XP5; h = rotl64(h, 11) * XP1; q++; n--; }
    h ^= h >> 33; h *= XP2; h ^= h >> 29; h *= XP3; h ^= h >> 32;  // avalanche :126-134
    results[f].checksum_calculated = (uint32_t)h;
}

void launch_xxh64(const LaunchCtx& lc, const czb_frame_desc* descs, czb_frame_result* results, uint64_t first, uint64_t count) {
    if (!count) return;
    const uint64_t threads = count * 4;
    k_xxh64<<<(unsigned)((threads + 127) / 128), 128, 0, lc.stream>>>(descs + first, results + first, count);
    ++*lc.launches;
}

}  // namespace czb
