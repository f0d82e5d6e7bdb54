// czb_handle.cu -- FrameDecoderState / FrameDecoder mirror (src/frame_decoder.cairo:54-335) on top
// of the batch path.  The handle keeps the reference's observable state (block_counter,
// bytes_read_counter, frame_finished, check_sum, DecodeBuffer len/head/window) on the host and
// lets the GPU do all decoding: whenever blocks beyond what has been decoded are asked for, the
// blocks that have become available since the last run are decoded on the device -- the run
// RESUMES after the blocks already executed (FrameResume: their output stays in the handle's
// device buffer, offset history and counters are carried over, table-reuse chains are re-derived
// from the source), so a frame fed in small pieces costs O(frame), not O(frame^2) -- and the
// per-block byte counts written by k_exec drive the incremental strategies (UptoBlocks / UptoBytes :202-214,
// decode_from_to :245-326) and the window-limited draining (decode_buffer.cairo:135-203),
// including RingBuffer::len ignoring `head` (ring_buffer.cairo:20-22).
#include <algorithm>
#include <cstring>
#include <vector>

#include "czb_host.h"
#include "czb_internal.cuh"
#include "czb_parse.cuh"

using namespace czb;

namespace {
struct BlockRec {
    int32_t status;      // CZS_OK, or the error this block raises
    uint8_t header_err;  // error is raised by read_block_header (no bytes counted)
    uint8_t last;
    uint32_t body_bytes; // bytes of block content in the source
    uint32_t out_bytes;
};
}  // namespace

struct czb_frame_decoder {
    czb_context* ctx = nullptr;
    FrameHeader hdr{};
    uint64_t window = 0;
    std::vector<uint8_t> acc;       // frame bytes seen so far, from the magic number on
    std::vector<BlockRec> blocks;   // outcome of the last device run over acc
    uint64_t decoded_acc_len = 0;   // acc.size() at the last device run
    bool run_complete = false;      // that run reached the last block or a hard error
    std::vector<uint8_t> out_all;   // decoded bytes of the executed blocks
    uint8_t* d_src = nullptr; uint64_t d_src_cap = 0;
    uint64_t uploaded = 0;          // acc[0 .. uploaded) is already in d_src
    uint8_t* d_dst = nullptr; uint64_t d_dst_cap = 0;
    czb_frame_desc* d_desc = nullptr;
    czb_frame_result* d_res = nullptr;
    FrameResume* d_resume = nullptr;
    // resume point: blocks [0, exec_blocks) were executed by earlier runs
    uint32_t exec_blocks = 0;
    uint32_t hist[3] = {1, 4, 8};
    uint64_t exec_out = 0, exec_bytes_read = 0;
    uint64_t device_runs = 0, device_blocks = 0;  // bookkeeping for the tests: blocks executed on the device, all runs
    // reference state (frame_decoder.cairo:21-30, decode_buffer.cairo:9-15)
    bool frame_finished = false;
    uint32_t block_counter = 0;
    uint64_t bytes_read_counter = 0;
    bool has_check_sum = false;
    uint32_t check_sum = 0;
    uint64_t buf_len = 0;   // RingBuffer elements.len()
    uint64_t head = 0;      // RingBuffer.head
    uint64_t abs_base = 0;  // position in the frame's output of element 0 (moves on clear())
};

#define FD_CUDA(fd, call)                                                                         \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            (fd)->ctx->last_error = std::string(#call) + ": " + cudaGetErrorString(e__);          \
            return CZS_CUDA_ERROR;                                                                \
        }                                                                                         \
    } while (0)

static bool checksum_flag(const czb_frame_decoder* fd) { return (fd->hdr.descriptor >> 2) & 1; }
static bool is_finished(const czb_frame_decoder* fd) {  // :144-150
    return checksum_flag(fd) ? (fd->frame_finished && fd->has_check_sum) : fd->frame_finished;
}

static int fd_setup(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint64_t* consumed, bool is_reset) {
    FrameHeader fh{};
    int32_t st = parse_frame_header(src, src_len, fh);
    if (st != CZS_OK) return st;
    uint64_t ws = 0;
    if ((st = frame_window_size(fh, is_reset, ws)) != CZS_OK) return st;
    fd->hdr = fh; fd->window = ws;
    fd->acc.assign(src, src + fh.hdr_len);
    fd->blocks.clear(); fd->decoded_acc_len = 0; fd->run_complete = false; fd->out_all.clear();
    fd->uploaded = 0; fd->exec_blocks = 0; fd->hist[0] = 1; fd->hist[1] = 4; fd->hist[2] = 8; fd->exec_out = 0; fd->exec_bytes_read = fh.hdr_len;
    fd->frame_finished = false; fd->block_counter = 0; fd->bytes_read_counter = fh.hdr_len;
    fd->has_check_sum = false; fd->check_sum = 0; fd->buf_len = 0; fd->head = 0; fd->abs_base = 0;
    if (consumed) *consumed = fh.hdr_len;
    return CZS_OK;
}

extern "C" int czb_fd_new(czb_context* ctx, const uint8_t* src, uint64_t src_len, uint64_t* consumed, czb_frame_decoder** out) {
    if (!ctx || !out || (!src && src_len)) return CZS_BAD_ARGUMENT;
    *out = nullptr;
    czb_frame_decoder* fd = new czb_frame_decoder();
    fd->ctx = ctx;
    int st = fd_setup(fd, src, src_len, consumed, false);
    if (st != CZS_OK) { delete fd; return st; }
    *out = fd;
    return CZS_OK;
}

extern "C" int czb_fd_reset(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint64_t* consumed) {
    if (!fd || (!src && src_len)) return CZS_BAD_ARGUMENT;
    return fd_setup(fd, src, src_len, consumed, true);
}

extern "C" void czb_fd_free(czb_frame_decoder* fd) {
    if (!fd) return;
    cudaSetDevice(fd->ctx->device);
    cudaFree(fd->d_src); cudaFree(fd->d_dst); cudaFree(fd->d_desc); cudaFree(fd->d_res); cudaFree(fd->d_resume);
    delete fd;
}

// Decode the blocks of fd->acc that earlier runs have not executed yet and append to fd->blocks / fd->out_all.
static int fd_run_device(czb_frame_decoder* fd) {
    czb_context* ctx = fd->ctx;
    FD_CUDA(fd, cudaSetDevice(ctx->device));
    const uint64_t n = fd->acc.size();
    cudaStream_t st = ctx->compute;
    // host walk over the blocks not executed yet: an output bound for them
    uint64_t bound = fd->exec_out, pos = fd->exec_bytes_read;
    for (;;) {
        ParsedBlock pb;
        parse_block_at(fd->acc.data(), n, pos, pb);
        if (pb.hdr_status != CZS_OK) break;
        bound += pb.type == BT_COMPRESSED ? MAX_BLOCK_SIZE : pb.size;
        pos += 3 + pb.content;
        if (pb.last) break;
    }
    if (fd->hdr.fcs_bytes && fd->hdr.fcs > bound && fd->hdr.fcs <= MAX_FRAME_OUT) bound = fd->hdr.fcs;
    uint64_t cap = bound + 64;
    // source: only the bytes that arrived since the last run travel to the device
    if (n + 64 > fd->d_src_cap) {
        uint8_t* nsrc = nullptr;
        const uint64_t ncap = n + 64 + n / 2;
        FD_CUDA(fd, cudaMalloc(reinterpret_cast<void**>(&nsrc), ncap));
        if (fd->d_src && fd->uploaded) FD_CUDA(fd, cudaMemcpyAsync(nsrc, fd->d_src, fd->uploaded, cudaMemcpyDeviceToDevice, st));
        FD_CUDA(fd, cudaStreamSynchronize(st));
        cudaFree(fd->d_src);
        fd->d_src = nsrc; fd->d_src_cap = ncap;
    }
    if (n > fd->uploaded) FD_CUDA(fd, cudaMemcpyAsync(fd->d_src + fd->uploaded, fd->acc.data() + fd->uploaded, n - fd->uploaded, cudaMemcpyHostToDevice, st));
    fd->uploaded = n;
    if (!fd->d_desc) FD_CUDA(fd, cudaMalloc(reinterpret_cast<void**>(&fd->d_desc), sizeof(czb_frame_desc)));
    if (!fd->d_res) FD_CUDA(fd, cudaMalloc(reinterpret_cast<void**>(&fd->d_res), sizeof(czb_frame_result)));
    if (!fd->d_resume) FD_CUDA(fd, cudaMalloc(reinterpret_cast<void**>(&fd->d_resume), sizeof(FrameResume)));
    const FrameResume rs{fd->exec_blocks, fd->hist[0], fd->hist[1], fd->hist[2], fd->exec_out, fd->exec_bytes_read};
    FD_CUDA(fd, cudaMemcpyAsync(fd->d_resume, &rs, sizeof rs, cudaMemcpyHostToDevice, st));
    czb_frame_result res{};
    for (;;) {
        if (cap > fd->d_dst_cap) {  // grow, keeping the output of the executed blocks (later matches read it)
            uint8_t* ndst = nullptr;
            const uint64_t ncap = cap + cap / 2;
            FD_CUDA(fd, cudaMalloc(reinterpret_cast<void**>(&ndst), ncap));
            if (fd->d_dst && fd->exec_out) FD_CUDA(fd, cudaMemcpyAsync(ndst, fd->d_dst, fd->exec_out, cudaMemcpyDeviceToDevice, st));
            FD_CUDA(fd, cudaStreamSynchronize(st));
            cudaFree(fd->d_dst);
            fd->d_dst = ndst; fd->d_dst_cap = ncap;
        }
        czb_frame_desc d{fd->d_src, n, fd->d_dst, fd->d_dst_cap};
        FD_CUDA(fd, cudaMemcpyAsync(fd->d_desc, &d, sizeof d, cudaMemcpyHostToDevice, st));
        int rc = czb_decode_batch_device_resume(ctx, fd->d_desc, fd->d_res, 1, 0, st, fd->d_resume);
        if (rc != CZS_OK) return rc;
        FD_CUDA(fd, cudaMemcpyAsync(&res, fd->d_res, sizeof res, cudaMemcpyDeviceToHost, st));
        FD_CUDA(fd, cudaStreamSynchronize(st));
        if (res.status != CZS_DST_TOO_SMALL || cap >= MAX_FRAME_OUT) break;
        cap = std::min<uint64_t>(cap * 4, MAX_FRAME_OUT);  // a block may legally exceed 128 KiB in the reference
    }
    fd->device_runs++;
    // per-block records of the blocks from the resume point on
    const uint64_t nb = ctx->last_wave.n_blocks;
    std::vector<BlockDesc> bd(nb);
    if (nb) FD_CUDA(fd, cudaMemcpy(bd.data(), ctx->blocks[ctx->last_set].p, nb * sizeof(BlockDesc), cudaMemcpyDeviceToHost));
    fd->blocks.resize(fd->exec_blocks);  // drop the record of a block that could not be read last time: it is re-examined
    uint64_t produced = fd->exec_out;
    bool complete = false;
    for (uint64_t k = fd->exec_blocks; k < nb; k++) {
        const BlockDesc& b = bd[k];
        BlockRec r{};
        if (b.type == BT_ERROR) {
            r.status = b.pre_status; r.header_err = 1;
            fd->blocks.push_back(r);
            complete = b.pre_status != CZS_PANIC_TRUNCATED;
            break;
        }
        r.last = b.last;
        r.body_bytes = b.type == BT_RLE ? 1u : b.size;
        if (k < res.blocks_decoded) {
            r.status = CZS_OK; r.out_bytes = b.out_bytes; produced += b.out_bytes;
            fd->blocks.push_back(r);
            fd->exec_blocks = (uint32_t)(k + 1);
            fd->hist[0] = b.hist_out[0]; fd->hist[1] = b.hist_out[1]; fd->hist[2] = b.hist_out[2];
            fd->exec_bytes_read += 3ull + r.body_bytes;
            fd->device_blocks++;
        } else { r.status = res.status; fd->blocks.push_back(r); complete = true; break; }
        if (b.last) { complete = true; break; }
    }
    fd->run_complete = complete;
    fd->decoded_acc_len = n;
    fd->out_all.resize(produced);
    if (produced > fd->exec_out) FD_CUDA(fd, cudaMemcpy(fd->out_all.data() + fd->exec_out, fd->d_dst + fd->exec_out, produced - fd->exec_out, cudaMemcpyDeviceToHost));
    fd->exec_out = produced;
    return CZS_OK;
}

static int fd_ensure_block(czb_frame_decoder* fd, uint32_t j) {
    const bool have = j < fd->blocks.size() && !(fd->blocks[j].header_err && fd->blocks[j].status == CZS_PANIC_TRUNCATED && fd->acc.size() > fd->decoded_acc_len);
    if (have) return CZS_OK;
    if (fd->run_complete && fd->acc.size() == fd->decoded_acc_len) return CZS_OK;
    return fd_run_device(fd);
}

// One iteration of the block loop.  Returns CZS_OK and advances, or the block's error.
static int fd_step_block(czb_frame_decoder* fd, bool* was_last) {
    int rc = fd_ensure_block(fd, fd->block_counter);
    if (rc != CZS_OK) return rc;
    if (fd->block_counter >= fd->blocks.size()) return CZS_PANIC_INTERNAL;
    const BlockRec& r = fd->blocks[fd->block_counter];
    if (r.header_err) return r.status;     // FailedToReadBlockHeader: counters untouched (:166-171)
    fd->bytes_read_counter += 3;           // :173
    if (r.status != CZS_OK) return r.status;  // FailedToReadBlockBody (:175-184)
    fd->bytes_read_counter += r.body_bytes;
    fd->buf_len += r.out_bytes;
    fd->block_counter++;
    *was_last = r.last;
    return CZS_OK;
}

static void fd_append_source(czb_frame_decoder* fd, const uint8_t* src, uint64_t len) {
    // the caller's span starts at the first byte not yet consumed
    if (fd->acc.size() > fd->bytes_read_counter) fd->acc.resize(fd->bytes_read_counter);
    if (fd->uploaded > fd->acc.size()) fd->uploaded = fd->acc.size();  // the unconsumed tail is replaced by the caller's new span
    fd->acc.insert(fd->acc.end(), src, src + len);
}

extern "C" int czb_fd_decode_blocks(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint64_t* consumed, int strategy,
                                    uint32_t n, int32_t* finished) {
    if (!fd || (!src && src_len)) return CZS_BAD_ARGUMENT;
    const uint64_t start = fd->bytes_read_counter;
    const uint64_t prev_acc = fd->acc.size();
    fd_append_source(fd, src, src_len);
    if (fd->acc.size() != prev_acc || fd->acc.size() != fd->decoded_acc_len) { /* new bytes: a later run may see more blocks */ }
    const uint64_t size_before = fd->buf_len;
    const uint32_t blocks_before = fd->block_counter;
    int rc = CZS_OK;
    for (;;) {
        bool last = false;
        if ((rc = fd_step_block(fd, &last)) != CZS_OK) break;
        if (last) {
            fd->frame_finished = true;
            if (checksum_flag(fd)) {  // :189-199
                const uint64_t pos = fd->bytes_read_counter;
                if (fd->acc.size() < pos + 4) { rc = CZS_PANIC_TRUNCATED; break; }
                const uint8_t* p = fd->acc.data() + pos;
                fd->check_sum = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
                fd->has_check_sum = true;
                fd->bytes_read_counter += 4;
            }
            break;
        }
        if (strategy == CZB_STRATEGY_UPTO_BLOCKS) { if (fd->block_counter - blocks_before >= n) break; }
        else if (strategy == CZB_STRATEGY_UPTO_BYTES) { if (fd->buf_len - size_before >= n) break; }
    }
    if (consumed) *consumed = fd->bytes_read_counter - start;
    if (finished) *finished = fd->frame_finished ? 1 : 0;
    return rc;
}

// drain_to (decode_buffer.cairo:168-186)
static uint64_t fd_drain_to(czb_frame_decoder* fd, uint64_t amount, uint8_t* dst, uint64_t cap, bool* overflow) {
    if (amount == 0) return 0;
    const uint64_t avail = fd->buf_len - fd->head;
    const uint64_t n = std::min(avail, amount);
    if (n > cap) { *overflow = true; return 0; }
    if (n) memcpy(dst, fd->out_all.data() + fd->abs_base + fd->head, n);
    fd->head += n;
    return n;
}

extern "C" uint64_t czb_fd_can_collect(const czb_frame_decoder* fd) {
    if (!fd) return 0;
    if (is_finished(fd)) return fd->buf_len;
    return fd->buf_len > fd->window ? fd->buf_len - fd->window : 0;
}

extern "C" int czb_fd_collect(czb_frame_decoder* fd, uint8_t* dst, uint64_t dst_cap, uint64_t* written) {
    if (!fd || !written) return -CZS_BAD_ARGUMENT;
    *written = 0;
    if (is_finished(fd)) {  // drain(): everything from head, then clear (decode_buffer.cairo:157-166)
        const uint64_t n = fd->buf_len - fd->head;
        if (n > dst_cap) return -CZS_DST_TOO_SMALL;
        if (n) memcpy(dst, fd->out_all.data() + fd->abs_base + fd->head, n);
        fd->abs_base += fd->buf_len; fd->buf_len = 0; fd->head = 0;
        *written = n;
        return 1;
    }
    if (fd->buf_len > fd->window) {
        bool ovf = false;
        const uint64_t n = fd_drain_to(fd, fd->buf_len - fd->window, dst, dst_cap, &ovf);
        if (ovf) return -CZS_DST_TOO_SMALL;
        *written = n;
        return 1;
    }
    return 0;
}

extern "C" int64_t czb_fd_read(czb_frame_decoder* fd, uint8_t* dst, uint64_t dst_cap) {  // :328-334
    if (!fd) return -CZS_BAD_ARGUMENT;
    const uint64_t amount = fd->frame_finished ? fd->buf_len : (fd->buf_len > fd->window ? fd->buf_len - fd->window : 0);
    bool ovf = false;
    (void)fd_drain_to(fd, amount, dst, dst_cap, &ovf);
    if (ovf) return -CZS_DST_TOO_SMALL;
    return (int64_t)amount;  // the reference returns `amount`, not the bytes actually drained
}

extern "C" int czb_fd_decode_from_to(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint8_t* dst, uint64_t dst_cap,
                                     uint64_t* read_len, uint64_t* written) {
    if (!fd || !read_len || !written || (!src && src_len)) return CZS_BAD_ARGUMENT;
    const uint64_t start = fd->bytes_read_counter;
    if (!is_finished(fd)) {
        fd_append_source(fd, src, src_len);
        if (checksum_flag(fd) && fd->frame_finished && !fd->has_check_sum) {  // :256-267
            if (src_len >= 4) {
                fd->check_sum = (uint32_t)src[0] | ((uint32_t)src[1] << 8) | ((uint32_t)src[2] << 16) | ((uint32_t)src[3] << 24);
                fd->has_check_sum = true; fd->bytes_read_counter += 4;
            }
            *read_len = 4; *written = 0;
            return CZS_OK;
        }
        for (;;) {
            const uint64_t pos = fd->bytes_read_counter;
            if (fd->acc.size() - pos < 3) break;  // :270-272
            ParsedBlock pb;
            // header errors surface through fd_step_block; here only the "enough bytes?" test of :282-284
            const uint8_t* a = fd->acc.data();
            const uint32_t t = (a[pos] >> 1) & 3;
            const uint32_t size = (a[pos] >> 3) | ((uint32_t)a[pos + 1] << 5) | ((uint32_t)a[pos + 2] << 13);
            if (t != 3 && size <= MAX_BLOCK_SIZE) {
                const uint32_t content = t == BT_RLE ? 1u : size;
                if (fd->acc.size() - pos - 3 < content) break;
            }
            (void)pb;
            bool last = false;
            int rc = fd_step_block(fd, &last);
            if (rc != CZS_OK) return rc;
            if (last) {
                fd->frame_finished = true;
                if (checksum_flag(fd) && fd->acc.size() >= fd->bytes_read_counter + 4) {  // :307-316
                    const uint8_t* p = fd->acc.data() + fd->bytes_read_counter;
                    fd->check_sum = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
                    fd->has_check_sum = true; fd->bytes_read_counter += 4;
                }
                break;
            }
        }
    }
    const int64_t got = czb_fd_read(fd, dst, dst_cap);
    if (got < 0) return (int)-got;
    *written = (uint64_t)got;
    *read_len = fd->bytes_read_counter - start;
    return CZS_OK;
}

// tests only: how much device work the handle has caused so far (runs, blocks executed over all runs)
extern "C" int czb_debug_fd_device_work(const czb_frame_decoder* fd, uint64_t* runs, uint64_t* blocks) {
    if (!fd) return CZS_BAD_ARGUMENT;
    if (runs) *runs = fd->device_runs;
    if (blocks) *blocks = fd->device_blocks;
    return CZS_OK;
}

extern "C" uint64_t czb_fd_content_size(const czb_frame_decoder* fd) { return fd ? fd->hdr.fcs : 0; }
extern "C" int czb_fd_get_checksum_from_data(const czb_frame_decoder* fd, uint32_t* out) {
    if (!fd || !out) return 0;
    *out = fd->check_sum;
    return fd->has_check_sum ? 1 : 0;
}
extern "C" uint64_t czb_fd_bytes_read_from_source(const czb_frame_decoder* fd) { return fd ? fd->bytes_read_counter : 0; }
extern "C" int czb_fd_is_finished(const czb_frame_decoder* fd) { return fd && is_finished(fd) ? 1 : 0; }
extern "C" uint32_t czb_fd_blocks_decoded(const czb_frame_decoder* fd) { return fd ? fd->block_counter : 0; }

// get_calculated_checksum (:133-138): XXH64 of everything drained so far.  Drained bytes are always
// a prefix of the frame's output, which still sits in the handle's device buffer: hash it there.
extern "C" int czb_fd_get_calculated_checksum(const czb_frame_decoder* fdc, uint32_t* out) {
    czb_frame_decoder* fd = const_cast<czb_frame_decoder*>(fdc);
    if (!fd || !out) return 0;
    czb_context* ctx = fd->ctx;
    const uint64_t hashed = fd->abs_base + fd->head;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return 0;
    if (!fd->d_desc && cudaMalloc(reinterpret_cast<void**>(&fd->d_desc), sizeof(czb_frame_desc)) != cudaSuccess) return 0;
    if (!fd->d_res && cudaMalloc(reinterpret_cast<void**>(&fd->d_res), sizeof(czb_frame_result)) != cudaSuccess) return 0;
    if (!fd->d_dst) { if (cudaMalloc(reinterpret_cast<void**>(&fd->d_dst), 64) != cudaSuccess) return 0; fd->d_dst_cap = 64; }
    czb_frame_desc d{nullptr, 0, fd->d_dst, fd->d_dst_cap};
    czb_frame_result r{};
    r.status = CZS_OK; r.bytes_written = hashed;
    cudaStream_t st = ctx->compute;
    LaunchCtx lc{st, &ctx->launches};
    if (cudaMemcpyAsync(fd->d_desc, &d, sizeof d, cudaMemcpyHostToDevice, st) != cudaSuccess) return 0;
    if (cudaMemcpyAsync(fd->d_res, &r, sizeof r, cudaMemcpyHostToDevice, st) != cudaSuccess) return 0;
    launch_xxh64(lc, fd->d_desc, fd->d_res, 0, 1);
    if (cudaMemcpyAsync(&r, fd->d_res, sizeof r, cudaMemcpyDeviceToHost, st) != cudaSuccess) return 0;
    if (cudaStreamSynchronize(st) != cudaSuccess) return 0;
    *out = r.checksum_calculated;
    return 1;
}
