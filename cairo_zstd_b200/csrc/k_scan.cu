// k_scan.cu -- frame/block header scan and work-list construction (thread per frame).
//
// Reference path: read_frame_header (src/frame.cairo:152-284), FrameDecoderStateTrait::new
// (src/frame_decoder.cairo:54-76), the block loop of decode_blocks (:156-222) as far as the
// headers go, read_block_header (src/decoding/block_decoder.cairo:237-278) and the section
// headers (src/blocks/literals_section.cairo:81-175, src/blocks/sequence_section.cairo:77-114).
//
// Roofline: negligible traffic (a few bytes per block); latency-bound pointer chasing, one
// dependent load per block.  Frames are independent, so one thread per frame.
#include "czb_internal.cuh"
#include "czb_parse.cuh"

namespace czb {

__device__ __forceinline__ unsigned long long warp_sum_ull(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    return v;
}

// Reserve `n` units for this lane from a shared counter: one atomic per warp.
template <typename T>
__device__ __forceinline__ T warp_reserve(T* counter, T n) {
    const unsigned lane = lane_id();
    T incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    T total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    T base = 0;
    if (lane == 0 && total) base = atomicAdd(counter, total);
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    return base + incl - n;
}

struct Walk {
    uint32_t n_blocks, n_huf, n_fse;
    uint64_t lit_bytes, n_seq, src_end;
    uint32_t checksum;
    uint8_t has_checksum;
};

__device__ __forceinline__ uint64_t align16(uint64_t v) { return (v + 15) & ~15ull; }

__global__ void __launch_bounds__(128) k_scan_frames(const czb_frame_desc* __restrict__ descs, FrameInfo* __restrict__ infos,
                                                      uint64_t n, uint64_t wave_frames, WaveTotals* __restrict__ totals,
                                                      const FrameResume* __restrict__ resume) {
    __shared__ unsigned int hist[2][32];
    if (threadIdx.x < 64) hist[threadIdx.x >> 5][threadIdx.x & 31] = 0;
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    FrameInfo fi;
    memset(&fi, 0, sizeof fi);
    uint64_t src_bytes = 0;
    if (i < n) {
        const uint8_t* src = descs[i].src;
        uint64_t len = descs[i].src_len;
        if (len > 0xFFFFFFF0ull) len = 0xFFFFFFF0ull;
        FrameHeader fh;
        int32_t st = parse_frame_header(src, len, fh);
        uint64_t ws = 0;
        if (st == CZS_OK) st = frame_window_size(fh, false, ws);
        fi.status = st;
        if (st == CZS_OK) {
            fi.hdr_len = fh.hdr_len; fi.fcs = fh.fcs; fi.window = ws; fi.descriptor = fh.descriptor;
            uint64_t pos = fh.hdr_len;
            const uint32_t start_block = resume ? resume[i].start_block : 0u;  // earlier blocks need no entropy work (FrameResume)
            for (;;) {
                ParsedBlock pb;
                parse_block_at(src, len, pos, pb);
                fi.n_blocks++;
                if (pb.hdr_status != CZS_OK) break;
                if (pb.type == BT_COMPRESSED && pb.pre_status == CZS_OK && fi.n_blocks > start_block) {
                    if (pb.lit_type >= LT_COMPRESSED) { fi.n_huf++; fi.lit_bytes += align16((uint64_t)pb.regen + 16); }
                    if (pb.seqhdr_status == CZS_OK && pb.n_seq) { fi.n_fse++; fi.n_seq += seq_slots(pb.n_seq); fi.n_seq_true += pb.n_seq; }
                }
                pos += 3 + pb.content;
                if (pb.last) {
                    if ((fh.descriptor >> 2) & 1) {
                        if (len - pos < 4) { fi.n_blocks++; break; }  // pseudo block: source.slice(0,4) traps, frame_decoder.cairo:190
                        fi.checksum = (uint32_t)src[pos] | ((uint32_t)src[pos + 1] << 8) | ((uint32_t)src[pos + 2] << 16) | ((uint32_t)src[pos + 3] << 24);
                        fi.has_checksum = 1;
                        pos += 4;
                    }
                    fi.src_end = pos;
                    break;
                }
            }
            src_bytes = pos;
            fi.size_cls = size_class(pos);
            fi.fse_cls = fi.n_fse ? size_class(fi.n_seq_true / fi.n_fse) : 0u;
            atomicAdd(&hist[0][fi.size_cls], 1u);
            if (fi.n_fse) atomicAdd(&hist[1][fi.fse_cls], fi.n_fse);
        }
        infos[i] = fi;
    }
    // per-wave totals: a warp never straddles waves (wave_frames is a multiple of 128)
    unsigned long long nb = warp_sum_ull(fi.n_blocks), lb = warp_sum_ull(fi.lit_bytes), ns = warp_sum_ull(fi.n_seq);
    unsigned long long nh = warp_sum_ull(fi.n_huf), nf = warp_sum_ull(fi.n_fse), sb = warp_sum_ull(src_bytes);
    if (lane_id() == 0 && i < n) {
        WaveTotals* t = totals + i / wave_frames;
        if (nb) atomicAdd(&t->n_blocks, nb);
        if (lb) atomicAdd(&t->lit_bytes, lb);
        if (ns) atomicAdd(&t->n_seq, ns);
        if (nh) atomicAdd(&t->n_huf, nh);
        if (nf) atomicAdd(&t->n_fse, nf);
        if (sb) atomicAdd(&t->src_bytes, sb);
    }
    // size-class histograms: one global atomic per class per CTA (a CTA never straddles waves)
    __syncthreads();
    if (threadIdx.x < 64 && (uint64_t)blockIdx.x * blockDim.x < n) {
        const unsigned int c = hist[threadIdx.x >> 5][threadIdx.x & 31];
        WaveTotals* t = totals + ((uint64_t)blockIdx.x * blockDim.x) / wave_frames;
        if (c) atomicAdd((threadIdx.x >> 5) ? &t->fse_cls[threadIdx.x & 31] : &t->frame_cls[threadIdx.x & 31], c);
    }
}

// Reserve n units in the per-class counter of class `cls` for this lane; lanes of a warp that share a class get
// one atomic and consecutive ranges in lane order, so neighbouring frames stay neighbours in the work lists
// (k_fse's 27 lanes then read neighbouring bitstreams: same DRAM pages, same TLB entries).
__device__ __forceinline__ unsigned int warp_reserve_by_class(unsigned int* counters, uint32_t cls, unsigned int n) {
    const unsigned lane = lane_id();
    unsigned int before = 0, total = 0;
    int leader = -1;
#pragma unroll 8
    for (int j = 0; j < 32; j++) {
        const uint32_t cj = __shfl_sync(0xFFFFFFFFu, cls, j);
        const unsigned int nj = __shfl_sync(0xFFFFFFFFu, n, j);
        if (cj == cls) { if (leader < 0) leader = j; total += nj; if (j < (int)lane) before += nj; }
    }
    unsigned int base = 0;
    if ((int)lane == leader && total) base = atomicAdd(&counters[cls & 31u], total);
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    return base + before;
}

// Second walk: write one BlockDesc per block, resolve the table-reuse chains
// (Treeless literals: literals_section_decoder.cairo:82-86; Repeat modes:
// sequence_section_decoder.cairo:483, :551, :643) and append the entropy work items.
__global__ void __launch_bounds__(128) k_fill_blocks(const czb_frame_desc* __restrict__ descs, FrameInfo* __restrict__ infos,
                                                      uint64_t first, uint64_t count, BlockDesc* __restrict__ blocks,
                                                      uint32_t* __restrict__ huf_items, uint32_t* __restrict__ fse_items,
                                                      WaveCounters* __restrict__ ctr, const WaveTotals* __restrict__ wt,
                                                      uint32_t* __restrict__ exec_order, const FrameResume* __restrict__ resume) {
    // start of every size class in the work lists, largest class first
    __shared__ unsigned int frame_start[32], fse_start[32];
    if (threadIdx.x == 0) {
        unsigned int a = 0, b = 0;
        for (int c = 31; c >= 0; c--) { frame_start[c] = a; a += wt->frame_cls[c]; fse_start[c] = b; b += wt->fse_cls[c]; }
    }
    __syncthreads();
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = t < count;
    const uint64_t i = first + (active ? t : 0);
    FrameInfo fi;
    if (active) fi = infos[i]; else memset(&fi, 0, sizeof fi);
    const bool walk = active && fi.status == CZS_OK;
    unsigned long long blk_base = warp_reserve<unsigned long long>(&ctr->n_blocks, walk ? fi.n_blocks : 0);
    unsigned long long lit_base = warp_reserve<unsigned long long>(&ctr->lit_bytes, walk ? fi.lit_bytes : 0);
    unsigned long long seq_base = warp_reserve<unsigned long long>(&ctr->n_seq, walk ? fi.n_seq : 0);
    unsigned int huf_base = warp_reserve<unsigned int>(&ctr->n_huf, walk ? fi.n_huf : 0);
    unsigned int fse_base = warp_reserve<unsigned int>(&ctr->n_fse, walk ? fi.n_fse : 0);
    (void)fse_base;
    // positions in the size-ordered work lists (inactive lanes get private dummy classes with nothing to reserve)
    const uint32_t fcls = walk ? (fi.size_cls & 31u) : 64u + lane_id(), scls = (walk && fi.n_fse) ? (fi.fse_cls & 31u) : 64u + lane_id();
    const unsigned int frame_pos = warp_reserve_by_class(ctr->frame_fill, fcls, walk ? 1u : 0u);
    unsigned int fse_pos = warp_reserve_by_class(ctr->fse_fill, scls, (walk && fi.n_fse) ? fi.n_fse : 0u);
    if (!active) return;
    infos[i].block_base = (uint32_t)blk_base;
    if (!walk) return;
    exec_order[frame_start[fi.size_cls & 31u] + frame_pos] = (uint32_t)(i - first);  // k_exec takes the biggest size class first
    fse_pos += fse_start[fi.fse_cls & 31u];

    const uint8_t* src = descs[i].src;
    uint64_t len = descs[i].src_len;
    if (len > 0xFFFFFFF0ull) len = 0xFFFFFFF0ull;
    uint64_t pos = fi.hdr_len;
    uint32_t bidx = (uint32_t)blk_base;
    uint32_t last_huf = NONE32, last_tbl[3] = {NONE32, NONE32, NONE32};
    bool seen_seq = false;
    const uint32_t start_block = resume ? resume[i].start_block : 0u;  // earlier blocks: descriptors (for the reuse chains) but no work items
    for (uint32_t k = 0; k < fi.n_blocks; k++, bidx++) {
        BlockDesc d;
        memset(&d, 0, sizeof d);
        d.frame = (uint32_t)(i - first);
        d.huf_src_blk = NONE32; d.tbl_src_blk[0] = d.tbl_src_blk[1] = d.tbl_src_blk[2] = NONE32;
        d.huf_status = CZS_OK; d.fse_status = CZS_OK;
        if (pos == ~0ull) {  // pseudo block for the missing checksum trailer
            d.type = BT_ERROR; d.pre_status = CZS_PANIC_TRUNCATED;
            blocks[bidx] = d;
            break;
        }
        ParsedBlock pb;
        parse_block_at(src, len, pos, pb);
        d.src_off = (uint32_t)(pos + 3);
        d.size = pb.size; d.type = pb.type; d.last = pb.last;
        if (pb.hdr_status != CZS_OK) {
            d.type = BT_ERROR; d.pre_status = pb.hdr_status;
            blocks[bidx] = d;
            break;
        }
        if (pb.type == BT_COMPRESSED) {
            d.pre_status = pb.pre_status; d.seqhdr_status = pb.seqhdr_status;
            d.lit_type = pb.lit_type; d.n_streams = pb.n_streams; d.regen = pb.regen;
            d.lit_src_off = d.src_off + pb.lit_hdr; d.lit_comp = pb.lit_payload;
            if (pb.pre_status == CZS_OK) {
                if (pb.lit_type >= LT_COMPRESSED) {
                    if (pb.lit_type == LT_COMPRESSED) last_huf = bidx;
                    d.huf_src_blk = last_huf;
                    if (k >= start_block) {
                        d.lit_off = lit_base; lit_base += align16((uint64_t)pb.regen + 16);
                        huf_items[huf_base++] = bidx;
                    }
                }
                if (pb.seqhdr_status == CZS_OK) {
                    d.n_seq = pb.n_seq; d.modes = pb.modes;
                    d.seq_src_off = d.lit_src_off + pb.lit_payload + pb.seq_hdr;
                    d.seq_src_len = d.src_off + pb.size - d.seq_src_off;
                    if (pb.n_seq) {
                        const uint32_t m[3] = {(uint32_t)pb.modes >> 6, ((uint32_t)pb.modes >> 4) & 3u, ((uint32_t)pb.modes >> 2) & 3u};
#pragma unroll
                        for (int s = 0; s < 3; s++) {
                            if (m[s] != MODE_REPEAT) last_tbl[s] = bidx;
                            d.tbl_src_blk[s] = last_tbl[s];
                        }
                        d.first_in_frame = seen_seq ? 0 : 1;
                        seen_seq = true;
                        if (k >= start_block) {
                            d.seq_off = seq_base; seq_base += seq_slots(pb.n_seq);
                            fse_items[fse_pos++] = bidx;
                        }
                    }
                }
            }
        }
        blocks[bidx] = d;
        pos += 3 + pb.content;
        if (pb.last) pos = ~0ull;  // only reached again if the scan counted a trailer pseudo block
    }
}

// Frames whose header failed never reach k_exec's block loop; give every frame its
// header-level result first (k_exec overwrites the rest).
__global__ void __launch_bounds__(256) k_header_results(const FrameInfo* __restrict__ infos, czb_frame_result* __restrict__ results, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const FrameInfo fi = infos[i];
    czb_frame_result r;
    memset(&r, 0, sizeof r);
    r.status = fi.status;
    r.content_size = fi.fcs; r.window_size = fi.window;
    results[i] = r;
}

// Copies the per-wave totals into host-mapped memory with plain stores (no copy engine involved).
__global__ void k_publish_totals(const WaveTotals* __restrict__ src, WaveTotals* __restrict__ dst_host, uint64_t n_waves) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t n_words = n_waves * (sizeof(WaveTotals) / sizeof(unsigned long long));
    if (i < n_words) reinterpret_cast<volatile unsigned long long*>(dst_host)[i] = reinterpret_cast<const unsigned long long*>(src)[i];
    __threadfence_system();
}

// Exact decoded size of every frame without executing it (SURVEY.md section 8 row f2: 51 of the 100 corpus frames carry
// no Frame_Content_Size).  After the scan, the block walk and k_fse: a Raw/RLE block regenerates Block_Size bytes
// (block_decoder.cairo:97-123), a Compressed block all of its literals plus every match: regen + sum(ml)
// (sequence_execution.cairo:72-81).  Errors the literal decode or the execution would raise are not seen here.
__global__ void __launch_bounds__(128) k_frame_sizes(const FrameInfo* __restrict__ infos, uint64_t first, uint64_t count,
                                                      const BlockDesc* __restrict__ blocks, czb_frame_result* __restrict__ results) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const FrameInfo fi = infos[first + t];
    if (fi.status != CZS_OK) return;  // k_header_results already reported it
    uint64_t out = 0, bytes_read = fi.hdr_len;
    int32_t status = CZS_OK;
    uint32_t n_done = 0;
    bool finished = false;
    for (uint32_t k = 0; k < fi.n_blocks && status == CZS_OK; k++) {
        const BlockDesc d = blocks[fi.block_base + k];
        if (d.type == BT_ERROR) { status = d.pre_status; break; }
        if (d.type == BT_RAW) { out += d.size; bytes_read += 3ull + d.size; }
        else if (d.type == BT_RLE) { out += d.size; bytes_read += 4; }
        else {
            if (d.pre_status != CZS_OK) { status = d.pre_status; break; }
            if (d.seqhdr_status != CZS_OK) { status = d.seqhdr_status; break; }
            if (d.n_seq && d.fse_status != CZS_OK) { status = d.fse_status; break; }
            out += (uint64_t)d.regen + (d.n_seq ? d.ml_sum : 0u);
            bytes_read += 3ull + d.size;
        }
        n_done++;
        if (d.last) { finished = true; if ((fi.descriptor >> 2) & 1) bytes_read += 4; }
    }
    czb_frame_result r;
    r.status = status; r.blocks_decoded = n_done; r.bytes_read = bytes_read;
    r.bytes_written = status == CZS_OK ? out : 0;
    r.content_size = fi.fcs; r.window_size = fi.window; r.checksum_from_data = fi.checksum; r.checksum_calculated = 0;
    r.has_checksum = fi.has_checksum;
    r.finished = (status == CZS_OK && finished && (!((fi.descriptor >> 2) & 1) || fi.has_checksum)) ? 1 : 0;
    results[first + t] = r;
}
void launch_frame_sizes(const LaunchCtx& lc, const FrameInfo* infos, uint64_t first, uint64_t count, const BlockDesc* blocks,
                        czb_frame_result* results) {
    if (!count) return;
    k_frame_sizes<<<(unsigned)((count + 127) / 128), 128, 0, lc.stream>>>(infos, first, count, blocks, results);
    ++*lc.launches;
}

// Frame-boundary walk over a concatenated buffer, one thread (each frame starts where the previous one ends, so the walk
// is one chain of dependent loads): skippable frames are stepped over (frame.cairo:160-166), every zstd frame's end is
// found from its block headers (block_decoder.cairo:237-278) without decoding.  counts = {frames, skipped, consumed, status}.
__global__ void k_split_frames(const uint8_t* __restrict__ buf, uint64_t len, czb_frame_span* __restrict__ spans, uint64_t cap,
                               unsigned long long* __restrict__ counts) {
    if (blockIdx.x || threadIdx.x) return;
    uint64_t n = 0, skipped = 0, pos = 0;
    const int32_t st = split_frames_walk(buf, len, spans, cap, n, skipped, pos);
    counts[0] = n; counts[1] = skipped; counts[2] = pos; counts[3] = (unsigned long long)(long long)st;
}
void launch_split_frames(const LaunchCtx& lc, const uint8_t* buf, uint64_t len, czb_frame_span* spans, uint64_t cap, unsigned long long* counts) {
    k_split_frames<<<1, 32, 0, lc.stream>>>(buf, len, spans, cap, counts);
    ++*lc.launches;
}

void launch_publish_totals(const LaunchCtx& lc, const WaveTotals* totals_d, WaveTotals* totals_host_mapped, uint64_t n_waves) {
    const uint64_t n_words = n_waves * (sizeof(WaveTotals) / sizeof(unsigned long long));
    k_publish_totals<<<(unsigned)((n_words + 127) / 128), 128, 0, lc.stream>>>(totals_d, totals_host_mapped, n_waves);
    ++*lc.launches;
}

void launch_scan_frames(const LaunchCtx& lc, const czb_frame_desc* descs, FrameInfo* infos, uint64_t n, uint64_t wave_frames,
                        WaveTotals* totals, const FrameResume* resume) {
    if (!n) return;
    k_scan_frames<<<(unsigned)((n + 127) / 128), 128, 0, lc.stream>>>(descs, infos, n, wave_frames, totals, resume);
    ++*lc.launches;
}
void launch_fill_blocks(const LaunchCtx& lc, const czb_frame_desc* descs, FrameInfo* infos, uint64_t first, uint64_t count,
                        BlockDesc* blocks, uint32_t* huf_items, uint32_t* fse_items, WaveCounters* counters,
                        const WaveTotals* wave_totals, uint32_t* exec_order, const FrameResume* resume) {
    if (!count) return;
    k_fill_blocks<<<(unsigned)((count + 127) / 128), 128, 0, lc.stream>>>(descs, infos, first, count, blocks, huf_items, fse_items, counters,
                                                                          wave_totals, exec_order, resume);
    ++*lc.launches;
}
void launch_header_results(const LaunchCtx& lc, const FrameInfo* infos, czb_frame_result* results, uint64_t n) {
    if (!n) return;
    k_header_results<<<(unsigned)((n + 255) / 256), 256, 0, lc.stream>>>(infos, results, n);
    ++*lc.launches;
}

}  // namespace czb
