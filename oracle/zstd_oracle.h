/*
 * zstd_oracle.h -- CPU restatement of the NethermindEth/cairo_zstd decode path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product (cairo_zstd_b200/, include/,
 * the C-ABI library) may include, link or call this.  Allowed users: tests/,
 * __graft_entry__.smoke(), and bench.py's cpu_baseline / --impl reference legs.
 *
 * Parity pin: every public function here is checked in tests/test_oracle.py
 * against the reference's own golden data -- the 100 data/decode_corpus pairs
 * (output bytes + XXH64 trailer), the LL predefined-table entries
 * (sequence_section_decoder.cairo:707-737), both bit-reader vectors
 * (tests/bit_reader.cairo:13-16, :55-58) and the 14 XXH64 vectors
 * (tests/utils.cairo:134-150).  The Cairo itself cannot run in this image
 * (no scarb / cairo-run; SURVEY.md section 8c), so those vectors are the pin.
 */
#ifndef ZSTD_ORACLE_H
#define ZSTD_ORACLE_H

#include <stddef.h>
#include <stdint.h>
#include "../include/czstd_status.h"

#ifdef __cplusplus
extern "C" {
#endif

/* flags */
#define ORACLE_FLAG_NIBBLE_AS_WRITTEN 1u /* huff0_decoder.cairo:302 `idx | 1 == 1` taken literally */
#define ORACLE_FLAG_RESET_LIMIT 2u       /* apply the 100 MiB window check of reset() (frame_decoder.cairo:92-94) */

typedef struct oracle_result {
    int32_t status;              /* czs_status */
    uint32_t blocks_decoded;     /* FrameDecoder::blocks_decoded  frame_decoder.cairo:152 */
    uint64_t bytes_read;         /* bytes_read_from_source        :140 */
    uint64_t bytes_written;      /* length of what collect() returns after decode_blocks(All) */
    uint64_t content_size;       /* content_size()                :125 */
    uint64_t window_size;        /* FrameHeader::window_size      frame.cairo:106-129 */
    uint32_t checksum_from_data; /* get_checksum_from_data()      :129 */
    uint32_t checksum_calculated;/* get_calculated_checksum()     :133 (XXH64 low 32 of the output) */
    int32_t has_checksum;        /* Option::is_some of the above  */
    int32_t finished;            /* is_finished()                 :144 */
} oracle_result;

/* Intermediate products, so each GPU stage can be diffed in isolation. */
typedef struct oracle_block_trace {
    uint8_t block_type;   /* 0 Raw 1 RLE 2 Compressed */
    uint8_t lit_type;     /* 0 Raw 1 RLE 2 Compressed 3 Treeless (Compressed blocks only) */
    uint8_t n_streams;
    uint8_t modes;        /* sequences mode byte */
    uint32_t regen_size;
    uint32_t n_seq;
    uint32_t out_bytes;   /* bytes this block appended to the decode buffer */
    uint64_t lit_off;     /* offset of this block's literals in oracle_trace.lits */
    uint64_t seq_off;     /* index of this block's first sequence in oracle_trace.seqs (units of 4 u32) */
} oracle_block_trace;

typedef struct oracle_trace {
    oracle_block_trace* blocks;
    size_t n_blocks, cap_blocks;
    uint8_t* lits;
    size_t n_lits, cap_lits;
    uint32_t* seqs;       /* 4 u32 per sequence: literals_length, match_length, raw offset value, actual offset */
    size_t n_seqs, cap_seqs;
} oracle_trace;

void oracle_trace_free(oracle_trace* t);

/* _test_decode equivalent (src/tests/decoding.cairo:4-21): FrameDecoderState::new,
 * decode_blocks(All), collect().  Writes the collected bytes to dst. */
int oracle_decode_frame(const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                        uint32_t flags, oracle_result* res, oracle_trace* trace /* may be NULL */);

/* Decode n frames with up to n_threads host threads (one frame per task).
 * srcs/dsts are arrays of pointers.  Returns number of frames with status != OK. */
int oracle_decode_batch(size_t n, const uint8_t* const* srcs, const size_t* src_lens,
                        uint8_t* const* dsts, const size_t* dst_caps, uint32_t flags,
                        oracle_result* results, int n_threads);

/* ---- incremental FrameDecoder surface (frame_decoder.cairo:54-335) ---- */
typedef struct oracle_fd oracle_fd;
/* FrameDecoderStateTrait::new + FrameDecoderTrait::new; *consumed = header bytes. */
oracle_fd* oracle_fd_new(const uint8_t* src, size_t src_len, size_t* consumed, uint32_t flags, int32_t* status);
/* FrameDecoderStateTrait::reset + FrameDecoderTrait::reset */
int32_t oracle_fd_reset(oracle_fd* fd, const uint8_t* src, size_t src_len, size_t* consumed);
void oracle_fd_free(oracle_fd* fd);
/* strategy: 0 All, 1 UptoBlocks(n), 2 UptoBytes(n).  *consumed = bytes of src used by this call.
 * *finished = Result::Ok(value).  Returns status. */
int32_t oracle_fd_decode_blocks(oracle_fd* fd, const uint8_t* src, size_t src_len, size_t* consumed,
                                int strategy, uint32_t n, int32_t* finished);
/* collect(): returns 1 if Some, 0 if None; bytes to dst (cap checked -> -1). */
int oracle_fd_collect(oracle_fd* fd, uint8_t* dst, size_t dst_cap, size_t* written);
size_t oracle_fd_can_collect(const oracle_fd* fd);
/* decode_from_to (:245-326): returns status; *read_len, *written as in the tuple */
int32_t oracle_fd_decode_from_to(oracle_fd* fd, const uint8_t* src, size_t src_len,
                                 uint8_t* dst, size_t dst_cap, size_t* read_len, size_t* written);
/* read (:328-334) */
size_t oracle_fd_read(oracle_fd* fd, uint8_t* dst, size_t dst_cap);
void oracle_fd_getters(const oracle_fd* fd, oracle_result* res);
/* the decode buffer's RingBuffer len and head: `read` reports an amount, len - head bounds what it drained */
void oracle_fd_buffer_state(const oracle_fd* fd, size_t* len, size_t* head);

/* ---- unit-level entry points used to pin the oracle against reference vectors ---- */
uint64_t oracle_xxh64(const uint8_t* p, size_t len, uint64_t seed);
/* Streaming XXH64 over chunked updates (xxhash64.cairo:32-113): chunk sizes from `chunks`. */
uint64_t oracle_xxh64_chunked(const uint8_t* p, size_t len, const size_t* chunks, size_t n_chunks);
/* Reverse / forward bit readers: read `n_reads` fields of widths[i] bits; values out. Returns status. */
int oracle_bitreader_reverse(const uint8_t* p, size_t len, const uint8_t* widths, size_t n_reads,
                             uint64_t* values, int64_t* bits_remaining_after);
int oracle_bitreader_forward(const uint8_t* p, size_t len, const uint8_t* widths, size_t n_reads,
                             uint64_t* values);
/* FSE table from probabilities (fse_decoder.cairo:143-256); entries out as (base_line,num_bits,symbol). */
int oracle_fse_build_from_probs(uint8_t acc_log, const int32_t* probs, size_t n_probs,
                                uint32_t* base_line, uint8_t* num_bits, uint8_t* symbol);
/* which = 0 LL, 1 OF, 2 ML predefined (sequence_section_decoder.cairo:417-617) */
int oracle_fse_predefined(int which, uint32_t* base_line, uint8_t* num_bits, uint8_t* symbol, uint32_t* table_size);
/* FSE table from a normalized-count description (fse_decoder.cairo:132-141, :258-368). */
int oracle_fse_build_decoder(const uint8_t* p, size_t len, uint8_t max_log, uint32_t* base_line,
                             uint8_t* num_bits, uint8_t* symbol, uint32_t* table_size, size_t* bytes_read);
/* Huffman table from a tree description (huff0_decoder.cairo:149-470). symbol/num_bits sized 2048. */
int oracle_huf_build_decoder(const uint8_t* p, size_t len, uint32_t flags, uint8_t* symbol,
                             uint8_t* num_bits, uint32_t* max_num_bits, size_t* bytes_read,
                             uint8_t* weights_out /*>=258*/, uint32_t* n_weights);
/* Dictionary::decode_dict (src/decoding/dictionary.cairo:35-90).  table_hash: FNV-1a over the four decoding tables' entries in
 * index order (Huffman: symbol | num_bits << 8; FSE OF, ML, LL: symbol | num_bits << 8 | base_line << 12). */
typedef struct {
    uint32_t id;
    uint32_t huf_bytes, of_bytes, ml_bytes, ll_bytes;
    uint32_t huf_max_bits, n_weights;
    uint32_t of_log, ml_log, ll_log;
    uint32_t offset_hist[3];
    uint32_t table_hash;
    uint64_t content_off, content_len;
} oracle_dict_info;
int oracle_dict_decode(const uint8_t* raw, size_t len, oracle_dict_info* out);
/* do_offset_history (sequence_execution.cairo:85-129) */
uint32_t oracle_offset_history(uint32_t offset_value, uint32_t lit_len, uint32_t hist[3]);

#ifdef __cplusplus
}
#endif
#endif
