/*
 * cairo_zstd_b200.h -- C ABI of the B200-native zstd decoder (libcairo_zstd_b200.so).
 *
 * Drop-in boundary for the decode path of NethermindEth/cairo_zstd.  Cairo has no
 * FFI; the reference's "operator API" is the FrameDecoder trait surface over borrowed
 * byte spans (SURVEY.md section 8b).  Each entry point below names the reference item it
 * replaces (paths relative to the reference repo).  Plain pointers and sizes only:
 * no torch / C++ types cross this boundary.  Nothing here unwinds; every failure is a
 * czs_status (czstd_status.h), reported per frame.
 *
 * Two families:
 *   1. czb_decode_batch*   -- the hot path: many independent frames per call.
 *   2. czb_fd_*            -- a handle mirroring FrameDecoderState/FrameDecoder 1:1 for
 *                             one frame at a time (runs the same GPU path underneath).
 *
 * Threading: a context / handle is not shareable between threads (the reference is
 * single-threaded too, SURVEY section 8b).  Different contexts may be used concurrently.
 * Calls on one context may use different streams: every batch call first waits (on its stream)
 * for the previous call's kernels, because the context's scratch is reused.
 *
 * Deliberate differences from the reference (all visible as statuses, see also czstd_status.h):
 *   1. Direct 4-bit Huffman weights are read in RFC 8878 order (even index = high nibble).
 *      src/huff0/huff0_decoder.cairo:302 reads `idx | 1 == 1`, i.e. (idx|1)==1; the reference's
 *      own fixtures pin only the RFC behaviour (DESIGN.md section 2).
 *   2. CZS_UNSUPPORTED marks input this build does not decode:
 *      a. frames whose output exceeds CZB_MAX_FRAME_OUTPUT (2^31 - 1) bytes, when dst_cap is at least that
 *         (with a smaller dst_cap the frame fails with CZS_DST_TOO_SMALL, as any frame that overflows dst);
 *      b. a sequence with a directly coded offset of 2^28 - 1 or more whose match starts at output position
 *         2^28 - 1 or later: the decoded sequence keeps 28 bits of such an offset.  The status replaces the
 *         reference's offset check (CZS_OFFSET_TOO_BIG / CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY) in its order,
 *         after the literal-length check and before the capacity check, so the frame may also be malformed.
 *         A repeat code that takes such an offset from an earlier block's history resolves it exactly, and
 *         a far offset whose match starts below 2^28 - 1 exceeds the output so far: the reference's status.
 *      (Huffman-weight FSE tables with an accuracy log above 9 -- the reference passes a limit of
 *      100, huff0_decoder.cairo:176 -- are decoded: tests/test_gpu_fuzz.py.)
 */
#ifndef CAIRO_ZSTD_B200_H
#define CAIRO_ZSTD_B200_H

#include <stddef.h>
#include <stdint.h>
#include "czstd_status.h"

#ifdef __cplusplus
extern "C" {
#endif

#define CZB_ABI_VERSION 1

/* Largest decoded size of one frame this build decodes (bytes).  Size dst spans and route larger frames elsewhere:
 * a frame with more output gets CZS_UNSUPPORTED (or CZS_DST_TOO_SMALL when dst_cap is below this). */
#define CZB_MAX_FRAME_OUTPUT 0x7FFFFFFFull

/* One frame of a batch: the reference's `ref source: @ByteArraySlice` (borrowed, immutable,
 * src/utils/byte_array.cairo:9-13) plus the caller-owned span that receives what
 * `collect()` would return (src/frame_decoder.cairo:224-231). */
typedef struct czb_frame_desc {
    const uint8_t* src;  /* first byte of the frame (magic number)           */
    uint64_t src_len;    /* bytes available at src (may extend past the frame) */
    uint8_t* dst;        /* where the decoded bytes go                       */
    uint64_t dst_cap;    /* capacity at dst                                  */
} czb_frame_desc;

/* Per-frame outcome: the FrameDecoder getters after decode_blocks(All) + collect()
 * (src/frame_decoder.cairo:125-154), flattened. */
typedef struct czb_frame_result {
    int32_t status;               /* czs_status; CZS_OK iff decode_blocks returned Ok        */
    uint32_t blocks_decoded;      /* blocks_decoded()            :152                         */
    uint64_t bytes_read;          /* bytes_read_from_source()    :140                         */
    uint64_t bytes_written;       /* length of collect()'s ByteArray :224                     */
    uint64_t content_size;        /* content_size()              :125 (0 when the field is absent) */
    uint64_t window_size;         /* FrameHeader::window_size    src/frame.cairo:106-129      */
    uint32_t checksum_from_data;  /* get_checksum_from_data()    :129                         */
    uint32_t checksum_calculated; /* get_calculated_checksum()   :133, 0 unless CZB_FLAG_VERIFY_CHECKSUM */
    int32_t has_checksum;         /* Option::is_some of checksum_from_data                    */
    int32_t finished;             /* is_finished()               :144                         */
} czb_frame_result;

/* Frame header facts without decoding: read_frame_header (src/frame.cairo:152-284) and
 * content_size (src/frame_decoder.cairo:125-127).  fcs_present = 0 means the field is
 * absent (51 of the 100 corpus frames). */
typedef struct czb_frame_header_info {
    int32_t status;
    uint32_t header_len;
    uint64_t content_size;
    uint64_t window_size;
    int32_t fcs_present;
    int32_t has_checksum_flag;
    int32_t single_segment;
    uint32_t dict_id; /* 0 = none; parsed and ignored downstream, as in the reference */
} czb_frame_header_info;

typedef struct czb_context czb_context;

/* flags for czb_decode_batch* */
#define CZB_FLAG_VERIFY_CHECKSUM 1u /* also compute XXH64 low-32 of each output on the device
                                       (reference: DecodeBuffer.hash, decode_buffer.cairo:162) */

/* ---- context ---------------------------------------------------------------------- */
/* device: CUDA ordinal.  workspace_budget_bytes: soft cap for per-wave scratch (0 = default). */
int czb_context_create(int device, uint64_t workspace_budget_bytes, czb_context** out);
void czb_context_destroy(czb_context* ctx);
const char* czb_last_error(const czb_context* ctx);
int czb_abi_version(void);

/* ---- batch decode: the hot path ------------------------------------------------------ */
/* Device-resident form.  `descs` and `results` are DEVICE pointers to arrays of n
 * entries; every src/dst inside descs is a DEVICE pointer.  Work is enqueued on
 * `stream` (a cudaStream_t passed as void*; NULL = default stream).  The call itself
 * synchronises `stream` internally once (a small planning read-back) and returns after
 * the last kernel is enqueued, not after it finished.  Some kernels run on streams owned by
 * the context, forked from and joined back to `stream` with events: work enqueued on
 * `stream` after the call sees every result; a context must not be used from two host
 * threads at once (as the reference's FrameDecoder, it is not shareable).
 * Replaces: one FrameDecoderStateTrait::new + FrameDecoderTrait::new + decode_blocks(All) +
 * collect() per frame (src/tests/decoding.cairo:4-21). */
int czb_decode_batch_device(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results,
                            uint64_t n_frames, uint32_t flags, void* stream);

/* The same without the planning read-back.  czb_plan_batch_device scans the frames once, synchronises `stream`, sizes the
 * context's scratch and keeps the wave split; czb_decode_batch_device_planned then decodes the SAME frames (same count, same
 * compressed bytes at the same or other addresses) without any host synchronisation: every kernel is only enqueued, so the
 * call can be pipelined behind other work or captured into a CUDA graph (inside a capture the call takes no part in the
 * cross-stream ordering of ordinary calls: replay the graph only while no other call uses the context). */
typedef struct czb_batch_plan czb_batch_plan;
int czb_plan_batch_device(czb_context* ctx, const czb_frame_desc* descs, uint64_t n_frames, void* stream, czb_batch_plan** out);
void czb_plan_destroy(czb_batch_plan* plan);
int czb_decode_batch_device_planned(czb_context* ctx, const czb_batch_plan* plan, const czb_frame_desc* descs,
                                    czb_frame_result* results, uint64_t n_frames, uint32_t flags, void* stream);

/* Host form: descs/results and every src/dst are HOST pointers.  Copies inputs to the
 * device, decodes, copies outputs back, and returns when results are valid. */
int czb_decode_batch_host(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results,
                          uint64_t n_frames, uint32_t flags);

/* Packed host form for large batches: frame i is src_base[src_off[i] .. src_off[i+1]) and
 * its output goes to dst_base[dst_off[i] .. dst_off[i+1]).  Both bases are HOST pointers
 * (pinned memory gives full PCIe rate); offsets arrays have n_frames+1 entries.  Transfers
 * are chunked and overlapped with decoding. */
int czb_decode_batch_host_packed(czb_context* ctx, const uint8_t* src_base, const uint64_t* src_off,
                                 uint8_t* dst_base, const uint64_t* dst_off, czb_frame_result* results,
                                 uint64_t n_frames, uint32_t flags);

/* Header pre-pass so callers can size outputs (host pointers, CPU only, no GPU work). */
int czb_frame_header_info_host(const uint8_t* src, uint64_t src_len, czb_frame_header_info* out);
/* Walk block headers to find where the frame ends without decoding (next row f2). Host, CPU only.
 * *frame_len = header + blocks + checksum bytes. */
int czb_find_frame_end_host(const uint8_t* src, uint64_t src_len, uint64_t* frame_len);

/* ---- batch splitter and output sizing (SURVEY.md section 8 row f2) ------------------------ */
/* One zstd frame found inside a buffer of concatenated frames. */
typedef struct czb_frame_span {
    uint64_t offset;         /* of the frame's magic number inside the buffer                    */
    uint64_t length;         /* header + blocks + checksum trailer                               */
    uint64_t content_size;   /* Frame_Content_Size (valid iff fcs_present), content_size() :125  */
    uint64_t window_size;    /* FrameHeader::window_size, src/frame.cairo:106-129                */
    int32_t fcs_present;
    int32_t has_checksum_flag;
} czb_frame_span;
/* Walk `buf`: skippable frames (src/frame.cairo:160-166 reports them as SkipFrame) are stepped over and counted, every
 * zstd frame is delimited from its block headers (src/decoding/block_decoder.cairo:237-278) without decoding and
 * appended to spans[0..cap).  *consumed = offset where the walk stopped: the end of the buffer, the frame that did
 * not fit spans[], or the first frame that cannot be delimited (then its czs_status is returned).
 * Host form: CPU only, no GPU work.  Device form: buf/spans/counts are DEVICE pointers, counts = uint64[4] =
 * {frames, skipped, consumed, status}; one thread walks (frame k+1 starts where frame k ends). */
int czb_split_frames_host(const uint8_t* buf, uint64_t len, czb_frame_span* spans, uint64_t cap, uint64_t* n_frames,
                          uint64_t* n_skipped, uint64_t* consumed);
int czb_split_frames_device(czb_context* ctx, const uint8_t* buf, uint64_t len, czb_frame_span* spans, uint64_t cap,
                            uint64_t* counts, void* stream);
/* Exact decoded size of every frame WITHOUT executing it, for frames that carry no Frame_Content_Size: header scan,
 * block walk and the sequence-section decode only (a Raw/RLE block regenerates Block_Size bytes, a Compressed block
 * regenerated_size + sum of match lengths: src/decoding/sequence_execution.cairo:72-81).  descs[i].dst/dst_cap are
 * ignored.  results[i].bytes_written = the size, .bytes_read = the frame's length, .status = the first header /
 * sequence-section error (errors that only literal decoding or execution would raise are not seen here). */
int czb_frame_sizes_device(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n_frames,
                           void* stream);
int czb_frame_sizes_host(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n_frames);

/* ---- one host batch over several GPUs (SURVEY.md section 8e) ------------------------------- */
/* Frames are independent (DecoderScratch::reset clears everything, src/decoding/scratch.cairo:42-58), so a batch
 * shards with no data-path collective and a frame is never split.  czb_partition_frames: greedy largest-first
 * assignment of frames to n_shards by cost[i] (use compressed + decoded bytes), deterministic; shard_of[i] receives the
 * shard, shard_load[s] (optional) the summed cost. */
int czb_partition_frames(const uint64_t* cost, uint64_t n_frames, uint32_t n_shards, uint32_t* shard_of, uint64_t* shard_load);
typedef struct czb_multi czb_multi;
typedef struct czb_shard_stat {
    int32_t device;
    uint32_t pad;
    uint64_t frames, bytes_in, bytes_out; /* this shard's frames, compressed and decoded bytes */
    double ms;                            /* host wall clock of this device's part of the call   */
} czb_shard_stat;
/* One context per listed device; czb_decode_batch_multi partitions the HOST batch (same meaning of descs/results as
 * czb_decode_batch_host) by src_len + dst_cap, runs every shard on its device from its own host thread and writes
 * results[] in the caller's order.  stats (optional) receives n_devices entries. */
int czb_multi_create(const int* devices, int n_devices, uint64_t workspace_budget_bytes, czb_multi** out);
void czb_multi_destroy(czb_multi* m);
int czb_decode_batch_multi(czb_multi* m, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n_frames,
                           uint32_t flags, czb_shard_stat* stats);
const char* czb_multi_last_error(const czb_multi* m, int shard);

/* ---- dictionaries (SURVEY.md section 8 row f4) -------------------------------------------------- */
/* Dictionary::decode_dict (src/decoding/dictionary.cairo:35-90): the reference PARSES a dictionary -- magic 0xEC30A437, id, a
 * Huffman table, the OF / ML / LL FSE tables (max logs 8 / 9 / 9), three repeat offsets, the content -- and never applies it
 * (frame_decoder.cairo:73 passes an empty dictionary; README: "Dictionary support" is not done).  This entry point mirrors the
 * parse on the device with the kernels' own table builders and reports what the reference's Dictionary struct would hold.
 * table_hash = FNV-1a (32 bit) over the four decoding tables' entries in index order: Huffman `symbol | num_bits << 8`, then OF, ML,
 * LL `symbol | num_bits << 8 | base_line << 12` (FSE symbols above 63 -- invalid codes for every stream -- count as 63).
 * Errors: CZS_DICT_BAD_MAGIC, the HuffmanTableError / FSETableError leaf codes, CZS_PANIC_TRUNCATED where the reference's
 * `.expect()` would trap.  dict is a HOST pointer. */
typedef struct czb_dictionary_info {
    int32_t status;
    uint32_t id;
    uint32_t huf_bytes, of_bytes, ml_bytes, ll_bytes; /* bytes each table description occupies */
    uint32_t huf_max_bits, n_weights;
    uint32_t of_log, ml_log, ll_log;
    uint32_t offset_hist[3];
    uint32_t table_hash;
    uint64_t content_off, content_len;                /* dict_content = dict[content_off .. content_off + content_len) */
} czb_dictionary_info;
int czb_dictionary_parse_host(czb_context* ctx, const uint8_t* dict, uint64_t len, czb_dictionary_info* out);

/* ---- FrameDecoder handle (1:1 mirror of src/frame_decoder.cairo) --------------------- */
typedef struct czb_frame_decoder czb_frame_decoder;

/* BlockDecodingStrategy, src/frame_decoder.cairo:33-37 */
#define CZB_STRATEGY_ALL 0
#define CZB_STRATEGY_UPTO_BLOCKS 1
#define CZB_STRATEGY_UPTO_BYTES 2

/* FrameDecoderStateTrait::new (:54-76) + FrameDecoderTrait::new (:109-111).
 * Parses the frame header from [src, src+src_len); *consumed = header bytes (the callee
 * "re-points" the span, src/frame.cairo:282).  Host pointers. */
int czb_fd_new(czb_context* ctx, const uint8_t* src, uint64_t src_len, uint64_t* consumed, czb_frame_decoder** out);
/* FrameDecoderStateTrait::reset (:78-105) + FrameDecoderTrait::reset/init (:113-123):
 * same as new on an existing handle, plus the 100 MiB window check (:92-94). */
int czb_fd_reset(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint64_t* consumed);
void czb_fd_free(czb_frame_decoder* fd);
/* decode_blocks (:156-222).  src = the span right after what previous calls consumed.
 * *consumed = bytes used by this call; *finished = the Ok(bool). */
int czb_fd_decode_blocks(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint64_t* consumed,
                         int strategy, uint32_t n, int32_t* finished);
/* collect (:224-231): returns 1 = Some (bytes in dst, *written set), 0 = None, <0 = -czs_status. */
int czb_fd_collect(czb_frame_decoder* fd, uint8_t* dst, uint64_t dst_cap, uint64_t* written);
uint64_t czb_fd_can_collect(const czb_frame_decoder* fd);                 /* :233-243 */
/* decode_from_to (:245-326) and read (:328-334) */
int czb_fd_decode_from_to(czb_frame_decoder* fd, const uint8_t* src, uint64_t src_len, uint8_t* dst,
                          uint64_t dst_cap, uint64_t* read_len, uint64_t* written);
int64_t czb_fd_read(czb_frame_decoder* fd, uint8_t* dst, uint64_t dst_cap);
uint64_t czb_fd_content_size(const czb_frame_decoder* fd);                /* :125 */
int czb_fd_get_checksum_from_data(const czb_frame_decoder* fd, uint32_t* out);   /* :129; returns 1 if Some */
int czb_fd_get_calculated_checksum(const czb_frame_decoder* fd, uint32_t* out);  /* :133; always Some */
uint64_t czb_fd_bytes_read_from_source(const czb_frame_decoder* fd);      /* :140 */
int czb_fd_is_finished(const czb_frame_decoder* fd);                      /* :144 */
uint32_t czb_fd_blocks_decoded(const czb_frame_decoder* fd);              /* :152 */

/* ---- debug / parity taps (tests only): intermediate products of the last batch ------- */
typedef struct czb_debug_block {
    uint32_t frame;
    uint8_t block_type, lit_type, n_streams, modes;
    uint32_t regen_size, n_seq;
    int32_t status;
    uint64_t lit_off; /* offset into the literal scratch (Huffman-coded sections only) */
    uint64_t seq_off; /* index into the sequence scratch */
} czb_debug_block;
/* Enable keeping the last wave's scratch readable (disables nothing else). */
int czb_debug_last_wave_counts(czb_context* ctx, uint64_t* n_blocks, uint64_t* lit_bytes, uint64_t* n_seq);
int czb_debug_copy_blocks(czb_context* ctx, czb_debug_block* out, uint64_t cap);
int czb_debug_copy_literals(czb_context* ctx, uint8_t* out, uint64_t cap);
int czb_debug_copy_sequences(czb_context* ctx, uint32_t* out /* 3 u32 per seq: ll, ml, offset */, uint64_t cap_seqs);

/* Device work a handle has caused so far: runs, and blocks executed summed over all runs (an incremental decode of a
 * frame executes every block once however small the feeds are). */
int czb_debug_fd_device_work(const czb_frame_decoder* fd, uint64_t* runs, uint64_t* blocks);
/* CZB_GUARD=1 (environment, read at context creation): guard zones behind the used part of the literal / sequence / block
 * scratch, checked after every wave; returns how many guard bytes were found overwritten so far (0 = clean). */
int czb_debug_guard_faults(czb_context* ctx, uint64_t* faults);
int czb_debug_flow_watchdog(unsigned int* out16); /* -DCZB_FLOW_WATCHDOG builds: what a stuck wait loop of k_exec_flow recorded */
/* The wave split a plan holds: frames per wave, number of waves, and per wave what the scan counted (blocks, bytes of Huffman
 * literal scratch, sequence slots, Huffman and sequence sections, the compressed bytes the block walk covered in frames whose
 * header parsed (the whole frame when it is valid), and the histograms of frames by compressed-size class and of sequence sections by sequence-count class, class = floor(log2)).
 * Copies min(cap, n_waves) entries into out (out may be NULL when cap is 0). */
typedef struct czb_debug_wave_totals {
    uint64_t n_blocks, lit_bytes, n_seq, n_huf, n_fse, src_bytes;
    uint32_t frame_cls[32], fse_cls[32];
} czb_debug_wave_totals;
int czb_debug_plan_waves(const czb_batch_plan* plan, uint64_t* wave_frames, uint64_t* n_waves, czb_debug_wave_totals* out, uint64_t cap);

/* Number of kernel launches issued by this context since creation (bench bookkeeping). */
uint64_t czb_kernel_launches(const czb_context* ctx);

/* Per-kernel device timing (CUDA events recorded on the launching stream around every kernel).
 * Classes: 0 scan, 1 fill, 2 huff, 3 fse, 4 exec, 5 xxh64, 6 header-results, 7 frame-sizes.
 * czb_profile_collect synchronises on the recorded events, adds their elapsed times (ms) and
 * launch counts per class into the arrays (8 entries each) and clears the recording. */
#define CZB_PROFILE_CLASSES 8
int czb_profile_enable(czb_context* ctx, int on);
int czb_profile_collect(czb_context* ctx, double* ms, uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* CAIRO_ZSTD_B200_H */
