/*
 * czstd_status.h -- flat integer status codes shared by the C-ABI library, the
 * CUDA kernels and the CPU oracle.
 *
 * The reference reports failures as nested Cairo `Result` enums and *panics*
 * on truncated input / internal invariant failures (SURVEY.md section 5 row 3,
 * section 8b "Error convention").  A C ABI cannot carry nested enums or unwind, so
 * every LEAF variant gets one code here (cited below) and the two panic
 * families get CZS_PANIC_*.  Codes >= 100 have no counterpart in the
 * reference: they are produced only by the C-ABI boundary itself.
 */
#ifndef CZSTD_STATUS_H
#define CZSTD_STATUS_H

#ifdef __cplusplus
extern "C" {
#endif

typedef enum czs_status {
    CZS_OK = 0,

    /* ReadFrameHeaderError -- src/frame.cairo:141-150 */
    CZS_MAGIC_NUMBER_READ_ERROR = 1,       /* :155-158 */
    CZS_FRAME_DESCRIPTOR_READ_ERROR = 2,   /* :161-164, :172-175 */
    CZS_DICTIONARY_ID_READ_ERROR = 3,      /* :204-226; FCS read failures reuse it :245-270 */
    CZS_WINDOW_DESCRIPTOR_READ_ERROR = 4,  /* :187-192 */
    CZS_BAD_MAGIC_NUMBER = 7,              /* :168-170 */
    CZS_SKIP_FRAME = 8,                    /* :160-166 */

    /* FrameHeaderError -- src/frame.cairo:94-103 */
    CZS_WINDOW_TOO_BIG = 9,                /* :122-124 */
    CZS_WINDOW_TOO_SMALL = 10,             /* :125-127 */
    /* FrameDecoderError::WindowSizeTooBig -- src/frame_decoder.cairo:92-94 (reset only) */
    CZS_WINDOW_SIZE_TOO_BIG = 11,

    /* BlockHeaderReadError -- src/decoding/block_decoder.cairo:33-47 */
    CZS_FOUND_RESERVED_BLOCK = 12,         /* :248-250 */
    CZS_BLOCK_SIZE_TOO_LARGE = 13,         /* :306-313 */

    /* DecompressBlockError -- src/decoding/block_decoder.cairo:49-57 */
    CZS_MALFORMED_SECTION_HEADER = 14,     /* :172-176 */

    /* LiteralsSectionParseError -- src/blocks/literals_section.cairo:24-30 */
    CZS_LIT_GET_BITS_ERROR = 16,           /* :85-90 (empty block content) */
    CZS_LIT_NOT_ENOUGH_BYTES = 17,         /* :99-102 */

    /* SequencesHeaderParseError -- src/blocks/sequence_section.cairo:66-69 */
    CZS_SEQ_HDR_NOT_ENOUGH_BYTES = 18,     /* :81-103 */

    /* DecompressLiteralsError -- src/decoding/literals_section_decoder.cairo:18-30 */
    CZS_MISSING_BYTES_FOR_JUMP_HEADER = 19, /* :92-94 */
    CZS_MISSING_BYTES_FOR_LITERALS = 20,    /* :101-105 */
    CZS_LIT_EXTRA_PADDING = 21,             /* :139-141, :209-211 */
    CZS_BITSTREAM_READ_MISMATCH = 22,       /* :234-240 */
    CZS_DECODED_LITERAL_COUNT_MISMATCH = 23,/* :172-178 */
    CZS_UNINITIALIZED_HUFFMAN_TABLE = 24,   /* :82-86 */

    /* HuffmanTableError -- src/huff0/huff0_decoder.cairo:27-43 */
    CZS_HUF_SOURCE_IS_EMPTY = 25,                    /* :162-164 */
    CZS_HUF_NOT_ENOUGH_BYTES_FOR_WEIGHTS = 26,       /* :171-175 */
    CZS_HUF_EXTRA_PADDING = 27,                      /* :223-225 */
    CZS_HUF_TOO_MANY_WEIGHTS = 28,                   /* :271-273 */
    CZS_HUF_MISSING_WEIGHTS = 29,                    /* :349-351 */
    CZS_HUF_LEFTOVER_NOT_POWER_OF_2 = 30,            /* :357-359 */
    CZS_HUF_NOT_ENOUGH_BYTES_TO_DECOMPRESS_WEIGHTS = 31, /* :194-200 */
    CZS_HUF_FSE_TABLE_USED_TOO_MANY_BYTES = 32,      /* :181-185 */
    CZS_HUF_NOT_ENOUGH_BYTES_IN_SOURCE = 33,         /* :289-293 */
    CZS_HUF_WEIGHT_BIGGER_THAN_MAX_NUM_BITS = 34,    /* :335-337 */
    CZS_HUF_MAX_BITS_TOO_HIGH = 35,                  /* :385-387 */

    /* FSETableError -- src/fse/fse_decoder.cairo:29-35 */
    CZS_FSE_ACC_LOG_IS_ZERO = 36,                    /* :147-149, :275-277 */
    CZS_FSE_ACC_LOG_TOO_BIG = 37,                    /* :272-274 */
    CZS_FSE_PROBABILITY_COUNTER_MISMATCH = 38,       /* :349-353 */
    CZS_FSE_TOO_MANY_SYMBOLS = 39,                   /* :354-356 */
    CZS_FSE_GET_BITS_ERROR = 40,                     /* :266-268, :345-347 */

    /* FSEDecoderError -- src/fse/fse_decoder.cairo:42-46 */
    CZS_FSE_TABLE_IS_UNINITIALIZED = 41,             /* :82-84 */

    /* DecodeSequenceError -- src/decoding/sequence_section_decoder.cairo:19-33 */
    CZS_SEQ_EXTRA_PADDING = 42,                      /* :62-64 */
    CZS_SEQ_UNSUPPORTED_OFFSET = 43,                 /* :125-127, :235-237 */
    CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES = 45, /* :179-181 */
    CZS_SEQ_EXTRA_BITS = 46,                         /* :190-194, :292-296 */
    CZS_SEQ_GET_BITS_ERROR = 47,                     /* TooManyBits via lookup_*_code (0,255) :343, :393 */
    CZS_MISSING_BYTE_FOR_RLE_LL_TABLE = 48,          /* :462-464 */
    CZS_MISSING_BYTE_FOR_RLE_OF_TABLE = 49,          /* :530-532 */
    CZS_MISSING_BYTE_FOR_RLE_ML_TABLE = 50,          /* :622-624 */

    /* ExecuteSequencesError -- src/decoding/sequence_execution.cairo:5-10 */
    CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE = 51,     /* :29-37 */
    CZS_EXEC_ZERO_OFFSET = 52,                       /* :47-49 */
    /* DecodeBufferError -- src/decoding/decode_buffer.cairo:17-21 */
    CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY = 53,         /* :69-75 */
    CZS_OFFSET_TOO_BIG = 54,                         /* :91-93 */

    /* DictionaryDecodeError -- src/decoding/dictionary.cairo:21-25 (FSETableError / HuffmanTableError reuse the codes above) */
    CZS_DICT_BAD_MAGIC = 55,                         /* :47-49 */

    /* Reference PANICS flattened (process abort in Cairo; SURVEY.md section 5) */
    CZS_PANIC_TRUNCATED = 100, /* slice/index past the end of the source span:
                                  src/utils/byte_array.cairo:20-21 reached from
                                  block_decoder.cairo:240, :98, :105, :146 and
                                  frame_decoder.cairo:192 */
    CZS_PANIC_INTERNAL = 101,  /* any other assert/unwrap, e.g. block_decoder.cairo:194,
                                  :208-214; sequence_section_decoder.cairo:279;
                                  huff0_decoder.cairo:431, :455 */

    /* Boundary-only codes (no reference counterpart) */
    CZS_DST_TOO_SMALL = 102,   /* caller's output span cannot hold the frame */
    CZS_UNSUPPORTED = 103,     /* outside this build's limits (DESIGN.md "Limits"): a frame whose
                                  output exceeds CZB_MAX_FRAME_OUTPUT (2^31 - 1) bytes, or a direct
                                  offset of 2^28 - 1 or more whose match starts at output position
                                  2^28 - 1 or later (sequence records keep 28 bits of such an offset).
                                  The second case is reported where the reference checks the offset,
                                  whether the offset is valid or not: the frame may be malformed too */
    CZS_CUDA_ERROR = 104,      /* CUDA runtime failure; see czb_last_error() */
    CZS_BAD_ARGUMENT = 105,
    CZS_NOT_DECODED = 106      /* result slot never written (internal) */
} czs_status;

const char* czs_status_name(int status);

#ifdef __cplusplus
}
#endif
#endif /* CZSTD_STATUS_H */
