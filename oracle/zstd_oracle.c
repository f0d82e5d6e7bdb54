/*
 * zstd_oracle.c -- CPU restatement of the NethermindEth/cairo_zstd decode path.
 *
 * TEST INFRASTRUCTURE ONLY (see zstd_oracle.h).  Each function cites the
 * reference file:line it restates (paths relative to /root/reference/).
 * This is a restatement in C of what the Cairo computes, not a translation of
 * its data structures: Cairo's dict-backed vectors become flat arrays, the
 * append-only RingBuffer becomes the caller's output span, Result/panic become
 * czs_status codes.
 *
 * Known divergence kept switchable: direct Huffman weights are read in RFC 8878
 * nibble order by default; ORACLE_FLAG_NIBBLE_AS_WRITTEN reproduces
 * huff0_decoder.cairo:302 literally (SURVEY.md section 0).
 */
#include "zstd_oracle.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------- */
/* small helpers (src/utils/math.cairo:239-284)                               */
/* ------------------------------------------------------------------------- */
static inline unsigned highest_bit_set_u32(uint32_t v) { /* math.cairo:266-272: BITS - leading_zeros */
    return v ? 32u - (unsigned)__builtin_clz(v) : 0u;
}
static inline int is_power_of_two_u32(uint32_t v) { return v != 0 && (v & (v - 1)) == 0; } /* :278-284 */

typedef struct { const uint8_t* p; size_t len; } slice_t;

/* ------------------------------------------------------------------------- */
/* XXH64 (src/utils/xxhash64.cairo)                                           */
/* ------------------------------------------------------------------------- */
#define XP1 0x9E3779B185EBCA87ULL
#define XP2 0xC2B2AE3D27D4EB4FULL
#define XP3 0x165667B19E3779F9ULL
#define XP4 0x85EBCA77C2B2AE63ULL
#define XP5 0x27D4EB2F165667C5ULL

typedef struct { uint64_t v1, v2, v3, v4; uint8_t mem[32]; uint32_t memsize; uint64_t total_len; } xxh64_t;

static inline uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
static inline uint64_t rd64le(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }
static inline uint32_t rd32le(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static inline uint64_t xxh_round(uint64_t acc, uint64_t in) { /* xxhash64.cairo:115-118 */
    return rotl64(acc + in * XP2, 31) * XP1;
}
static inline uint64_t xxh_merge(uint64_t acc, uint64_t v) { /* :120-124 */
    acc ^= xxh_round(0, v);
    return acc * XP1 + XP4;
}
static void xxh64_init(xxh64_t* s, uint64_t seed) { /* :32-42 */
    s->v1 = seed + XP1 + XP2; s->v2 = seed + XP2; s->v3 = seed; s->v4 = seed - XP1;
    s->memsize = 0; s->total_len = 0;
}
static void xxh64_update(xxh64_t* s, const uint8_t* in, size_t len) { /* :44-92 */
    s->total_len += len;
    if (s->memsize + len < 32) { memcpy(s->mem + s->memsize, in, len); s->memsize += (uint32_t)len; return; }
    size_t p = 0;
    if (s->memsize > 0) {
        size_t fill = 32 - s->memsize;
        memcpy(s->mem + s->memsize, in, fill);
        s->v1 = xxh_round(s->v1, rd64le(s->mem));      s->v2 = xxh_round(s->v2, rd64le(s->mem + 8));
        s->v3 = xxh_round(s->v3, rd64le(s->mem + 16)); s->v4 = xxh_round(s->v4, rd64le(s->mem + 24));
        p += fill; s->memsize = 0;
    }
    while (len - p >= 32) {
        s->v1 = xxh_round(s->v1, rd64le(in + p));      s->v2 = xxh_round(s->v2, rd64le(in + p + 8));
        s->v3 = xxh_round(s->v3, rd64le(in + p + 16)); s->v4 = xxh_round(s->v4, rd64le(in + p + 24));
        p += 32;
    }
    if (len - p > 0) { memcpy(s->mem, in + p, len - p); s->memsize = (uint32_t)(len - p); }
}
static uint64_t xxh64_digest(const xxh64_t* s) { /* :94-113, finalize :136-163, avalanche :126-134 */
    uint64_t h;
    if (s->total_len >= 32) {
        h = rotl64(s->v1, 1) + rotl64(s->v2, 7) + rotl64(s->v3, 12) + rotl64(s->v4, 18);
        h = xxh_merge(h, s->v1); h = xxh_merge(h, s->v2); h = xxh_merge(h, s->v3); h = xxh_merge(h, s->v4);
    } else {
        h = s->v3 + XP5;
    }
    h += s->total_len;
    const uint8_t* p = s->mem; size_t n = s->memsize;
    while (n >= 8) { h ^= xxh_round(0, rd64le(p)); h = rotl64(h, 27) * XP1 + XP4; p += 8; n -= 8; }
    if (n >= 4) { h ^= (uint64_t)rd32le(p) * XP1; h = rotl64(h, 23) * XP2 + XP3; p += 4; n -= 4; }
    while (n) { h ^= (uint64_t)(*p) * XP5; h = rotl64(h, 11) * XP1; p++; n--; }
    h ^= h >> 33; h *= XP2; h ^= h >> 29; h *= XP3; h ^= h >> 32;
    return h;
}
uint64_t oracle_xxh64(const uint8_t* p, size_t len, uint64_t seed) {
    xxh64_t s; xxh64_init(&s, seed); xxh64_update(&s, p, len); return xxh64_digest(&s);
}
uint64_t oracle_xxh64_chunked(const uint8_t* p, size_t len, const size_t* chunks, size_t n_chunks) {
    xxh64_t s; xxh64_init(&s, 0); size_t off = 0;
    for (size_t i = 0; i < n_chunks && off < len; i++) {
        size_t c = chunks[i]; if (c > len - off) c = len - off;
        xxh64_update(&s, p + off, c); off += c;
    }
    if (off < len) xxh64_update(&s, p + off, len - off);
    return xxh64_digest(&s);
}

/* ------------------------------------------------------------------------- */
/* forward bit reader (src/decoding/bit_reader.cairo:18-110)                  */
/* ------------------------------------------------------------------------- */
typedef struct { slice_t s; size_t idx; } fbr_t;

/* get_bits :38-104.  Returns 0 ok, 1 NotEnoughRemainingBits, 2 TooManyBits. */
static int fbr_get_bits(fbr_t* r, unsigned n, uint64_t* out) {
    if (n > 64) return 2;
    if (r->s.len * 8 - r->idx < n) return 1;
    uint64_t v = 0;
    for (unsigned got = 0; got < n;) { /* LSB-first: bit idx of the source is bit `got` of the value */
        size_t byte = r->idx >> 3; unsigned sh = (unsigned)(r->idx & 7);
        unsigned take = 8 - sh; if (take > n - got) take = n - got;
        v |= (uint64_t)((r->s.p[byte] >> sh) & ((1u << take) - 1u)) << got;
        got += take; r->idx += take;
    }
    *out = v;
    return 0;
}
static void fbr_return_bits(fbr_t* r, size_t n) { r->idx -= n; } /* :31-36 */

int oracle_bitreader_forward(const uint8_t* p, size_t len, const uint8_t* widths, size_t n_reads, uint64_t* values) {
    fbr_t r = {{p, len}, 0};
    for (size_t i = 0; i < n_reads; i++) { int e = fbr_get_bits(&r, widths[i], &values[i]); if (e) return e; }
    return 0;
}

/* ------------------------------------------------------------------------- */
/* reverse bit reader (src/decoding/bit_reader_reverse.cairo:44-275)          */
/* ------------------------------------------------------------------------- */
/*
 * The Cairo keeps a 64-bit container refilled from the tail (:52-123).  Seen
 * from outside it behaves as: X = the stream as a little-endian integer,
 * rem = bits not yet consumed (bits_remaining(), :45-50).  get_bits(n):
 *   n == 0            -> 0                                   (:130-132)
 *   rem <= 0          -> 0, rem -= n                         (:147-150)
 *   0 < rem < n       -> low rem bits << (n-rem), rem -= n   (:152-159)
 *   otherwise         -> bits [rem-n, rem) of X, rem -= n
 * n > 56 on the cold path -> TooManyBits (:141-143).  On this decode path n is
 * 0..31, or 255 from lookup_*_code's out-of-range arm, so "n > 56 -> error" is
 * exact (a 64-bit container never holds 255 bits).
 */
typedef struct { const uint8_t* p; size_t len; int64_t rem; } rbr_t;

static inline void rbr_init(rbr_t* r, slice_t s) { r->p = s.p; r->len = s.len; r->rem = (int64_t)s.len * 8; }

static inline uint64_t rbr_extract(const rbr_t* r, int64_t pos, unsigned n) { /* bits [pos,pos+n), n<=56 */
    size_t byte = (size_t)(pos >> 3); unsigned sh = (unsigned)(pos & 7);
    uint64_t w;
    if (byte + 8 <= r->len) w = rd64le(r->p + byte);
    else { w = 0; for (size_t i = 0; byte + i < r->len && i < 8; i++) w |= (uint64_t)r->p[byte + i] << (8 * i); }
    return (w >> sh) & ((n >= 64) ? ~0ULL : ((1ULL << n) - 1ULL));
}
/* returns 0 ok, 1 TooManyBits */
static inline int rbr_get_bits(rbr_t* r, unsigned n, uint64_t* out) {
    if (n == 0) { *out = 0; return 0; }
    if (n > 56) return 1;
    if (r->rem <= 0) { r->rem -= n; *out = 0; return 0; }
    if (r->rem < (int64_t)n) {
        unsigned have = (unsigned)r->rem;
        uint64_t v = rbr_extract(r, 0, have);
        *out = v << (n - have);
        r->rem -= n;
        return 0;
    }
    r->rem -= n;
    *out = rbr_extract(r, r->rem, n);
    return 0;
}
/* get_bits_triple :175-253: three reads in order; TooManyBits from the first offending field. */
static inline int rbr_get_bits_triple(rbr_t* r, unsigned n1, unsigned n2, unsigned n3, uint64_t* v1, uint64_t* v2, uint64_t* v3) {
    int e;
    if ((e = rbr_get_bits(r, n1, v1))) return e;
    if ((e = rbr_get_bits(r, n2, v2))) return e;
    return rbr_get_bits(r, n3, v3);
}

int oracle_bitreader_reverse(const uint8_t* p, size_t len, const uint8_t* widths, size_t n_reads,
                             uint64_t* values, int64_t* bits_remaining_after) {
    rbr_t r; slice_t s = {p, len}; rbr_init(&r, s);
    for (size_t i = 0; i < n_reads; i++) { int e = rbr_get_bits(&r, widths[i], &values[i]); if (e) return CZS_SEQ_GET_BITS_ERROR; }
    if (bits_remaining_after) *bits_remaining_after = r.rem;
    return 0;
}

/* skip padding: read single bits until a 1; more than 8 -> ExtraPadding
 * (literals_section_decoder.cairo:190-211, huff0_decoder.cairo:206-225,
 *  sequence_section_decoder.cairo:46-64).  Returns 0 ok, 1 extra padding. */
static int rbr_skip_padding(rbr_t* r) {
    int skipped = 0;
    for (;;) {
        uint64_t v = 0; rbr_get_bits(r, 1, &v);
        skipped++;
        if (v == 1 || skipped > 8) break;
    }
    return skipped > 8;
}

/* ------------------------------------------------------------------------- */
/* FSE (src/fse/fse_decoder.cairo)                                            */
/* ------------------------------------------------------------------------- */
typedef struct { uint32_t base_line; uint8_t num_bits; uint8_t symbol; } fse_entry_t; /* :48-53 */

#define FSE_MAX_PROBS 260
typedef struct {
    fse_entry_t* decode; uint32_t decode_len, decode_cap;
    uint8_t accuracy_log;
    int32_t probs[FSE_MAX_PROBS]; uint32_t n_probs; /* n_probs may exceed FSE_MAX_PROBS (count only) */
} fse_table_t;

static void fse_table_init(fse_table_t* t) { memset(t, 0, sizeof *t); }
static void fse_table_free(fse_table_t* t) { free(t->decode); t->decode = NULL; t->decode_cap = t->decode_len = 0; }
static void fse_table_reset(fse_table_t* t) { t->decode_len = 0; t->accuracy_log = 0; t->n_probs = 0; } /* :125-130 */

/* next_position :371-375 */
static inline uint32_t fse_next_position(uint32_t p, uint32_t size) { return (p + (size >> 1) + (size >> 3) + 3) & (size - 1); }

/* calc_baseline_and_numbits :377-400 */
static void fse_calc_baseline_and_numbits(uint32_t total, uint32_t n_sym, uint32_t k, uint32_t* bl, uint8_t* nb) {
    uint32_t mask = 1u << (highest_bit_set_u32(n_sym) - 1);
    uint32_t slices = (mask == n_sym) ? n_sym : mask * 2;
    uint32_t n_double = slices - n_sym;
    uint32_t n_single = n_sym - n_double;
    uint32_t width = total / slices;
    uint32_t bits = highest_bit_set_u32(width) - 1;
    if (k < n_double) { *bl = n_single * width + k * width * 2; *nb = (uint8_t)(bits + 1); }
    else { *bl = (k - n_double) * width; *nb = (uint8_t)bits; }
}

/* build_decoding_table :156-256.  Returns 0, or CZS_PANIC_INTERNAL where the Cairo would trap. */
static int fse_build_decoding_table(fse_table_t* t) {
    uint32_t size = 1u << t->accuracy_log;
    if (t->decode_cap < size) {
        fse_entry_t* nd = (fse_entry_t*)realloc(t->decode, (size_t)size * sizeof(fse_entry_t));
        if (!nd) return CZS_PANIC_INTERNAL;
        t->decode = nd; t->decode_cap = size;
    }
    memset(t->decode, 0, (size_t)size * sizeof(fse_entry_t));
    t->decode_len = size;
    uint32_t n = t->n_probs; if (n > FSE_MAX_PROBS) n = FSE_MAX_PROBS;
    uint32_t negative_idx = size;
    for (uint32_t i = 0; i < n; i++) { /* :169-189 "less than one" symbols from the top */
        if (t->probs[i] == -1) {
            if (negative_idx == 0) return CZS_PANIC_INTERNAL;
            negative_idx--;
            t->decode[negative_idx].symbol = (uint8_t)i;
            t->decode[negative_idx].base_line = 0;
            t->decode[negative_idx].num_bits = t->accuracy_log;
        }
    }
    uint32_t pos = 0;
    for (uint32_t i = 0; i < n; i++) { /* :191-226 spread */
        int32_t prob = t->probs[i];
        for (int32_t j = 0; j < prob; j++) {
            t->decode[pos].symbol = (uint8_t)i;
            pos = fse_next_position(pos, size);
            while (pos >= negative_idx) pos = fse_next_position(pos, size);
        }
    }
    uint32_t counter[FSE_MAX_PROBS]; memset(counter, 0, sizeof counter);
    for (uint32_t i = 0; i < negative_idx; i++) { /* :231-255 */
        uint8_t s = t->decode[i].symbol;
        int32_t prob = t->probs[s];
        if (prob <= 0) return CZS_PANIC_INTERNAL; /* prob.try_into::<u32>().unwrap() / NonZero */
        uint32_t bl; uint8_t nb;
        fse_calc_baseline_and_numbits(size, (uint32_t)prob, counter[s], &bl, &nb);
        counter[s]++;
        t->decode[i].base_line = bl; t->decode[i].num_bits = nb;
    }
    return 0;
}

/* read_probabilities :258-368 */
static int fse_read_probabilities(fse_table_t* t, slice_t src, uint8_t max_log, size_t* bytes_read) {
    t->n_probs = 0;
    fbr_t br = {src, 0};
    uint64_t v;
    if (fbr_get_bits(&br, 4, &v)) return CZS_FSE_GET_BITS_ERROR;
    t->accuracy_log = (uint8_t)(5 + v);
    if (t->accuracy_log > max_log) return CZS_FSE_ACC_LOG_TOO_BIG;
    uint32_t sum = 1u << t->accuracy_log, counter = 0;
    while (counter < sum) {
        uint32_t max_remaining = sum - counter + 1;
        unsigned bits = highest_bit_set_u32(max_remaining);
        uint64_t unchecked;
        if (fbr_get_bits(&br, bits, &unchecked)) return CZS_FSE_GET_BITS_ERROR;
        uint64_t low_threshold = ((1ULL << bits) - 1) - max_remaining;
        uint64_t mask = (1ULL << (bits - 1)) - 1;
        uint64_t small = unchecked & mask;
        uint64_t value;
        if (small < low_threshold) { fbr_return_bits(&br, 1); value = small; }
        else if (unchecked > mask) value = unchecked - low_threshold;
        else value = unchecked;
        int32_t prob = (int32_t)value - 1;
        if (t->n_probs < FSE_MAX_PROBS) t->probs[t->n_probs] = prob;
        t->n_probs++;
        if (prob != 0) {
            counter += (prob > 0) ? (uint32_t)prob : 1u;
        } else {
            for (;;) { /* :322-340 zero-run flags */
                uint64_t skip;
                if (fbr_get_bits(&br, 2, &skip)) return CZS_FSE_GET_BITS_ERROR;
                for (uint64_t k = 0; k < skip; k++) { if (t->n_probs < FSE_MAX_PROBS) t->probs[t->n_probs] = 0; t->n_probs++; }
                if (skip != 3) break;
            }
        }
    }
    if (counter != sum) return CZS_FSE_PROBABILITY_COUNTER_MISMATCH;
    if (t->n_probs > 256) return CZS_FSE_TOO_MANY_SYMBOLS;
    *bytes_read = (br.idx + 7) / 8;
    return 0;
}

/* build_decoder :132-141 */
static int fse_build_decoder(fse_table_t* t, slice_t src, uint8_t max_log, size_t* bytes_read) {
    t->accuracy_log = 0;
    int e = fse_read_probabilities(t, src, max_log, bytes_read);
    if (e) return e;
    return fse_build_decoding_table(t);
}
/* build_from_probabilities :143-154 */
static int fse_build_from_probabilities(fse_table_t* t, uint8_t acc_log, const int32_t* probs, uint32_t n) {
    if (acc_log == 0) return CZS_FSE_ACC_LOG_IS_ZERO;
    memcpy(t->probs, probs, n * sizeof(int32_t)); t->n_probs = n;
    t->accuracy_log = acc_log;
    return fse_build_decoding_table(t);
}

/* FSEDecoder :64-104 */
typedef struct { fse_entry_t state; } fse_dec_t;
static void fse_dec_new(fse_dec_t* d, const fse_table_t* t) { /* :65-72 */
    if (t->decode_len > 0) d->state = t->decode[0]; else memset(&d->state, 0, sizeof d->state);
}
static int fse_dec_init_state(fse_dec_t* d, const fse_table_t* t, rbr_t* br) { /* :78-91 */
    if (t->accuracy_log == 0) return CZS_FSE_TABLE_IS_UNINITIALIZED;
    uint64_t v;
    if (rbr_get_bits(br, t->accuracy_log, &v)) return CZS_PANIC_INTERNAL; /* .unwrap() */
    if (v >= t->decode_len) return CZS_PANIC_INTERNAL;
    d->state = t->decode[v];
    return 0;
}
static int fse_dec_update_state(fse_dec_t* d, const fse_table_t* t, rbr_t* br) { /* :93-103 */
    uint64_t add;
    if (rbr_get_bits(br, d->state.num_bits, &add)) return CZS_PANIC_INTERNAL;
    uint64_t ns = (uint64_t)d->state.base_line + add;
    if (ns >= t->decode_len) return CZS_PANIC_INTERNAL; /* decode.at() out of range */
    d->state = t->decode[ns];
    return 0;
}

/* predefined distributions (sequence_section_decoder.cairo:417-456, :493-525, :561-617) */
static const int32_t LL_DEFAULT[36] = {4, 3, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 2, 1, 1, 1, 1, 1, -1, -1, -1, -1};
static const int32_t OF_DEFAULT[29] = {1, 1, 1, 1, 1, 1, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1};
static const int32_t ML_DEFAULT[53] = {1, 4, 3, 2, 2, 2, 2, 2, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, -1, -1, -1, -1, -1, -1, -1};

static void fse_export(const fse_table_t* t, uint32_t* bl, uint8_t* nb, uint8_t* sym) {
    for (uint32_t i = 0; i < t->decode_len; i++) { bl[i] = t->decode[i].base_line; nb[i] = t->decode[i].num_bits; sym[i] = t->decode[i].symbol; }
}
int oracle_fse_build_from_probs(uint8_t acc_log, const int32_t* probs, size_t n_probs, uint32_t* bl, uint8_t* nb, uint8_t* sym) {
    if (n_probs > 256) return CZS_FSE_TOO_MANY_SYMBOLS;
    fse_table_t t; fse_table_init(&t);
    int e = fse_build_from_probabilities(&t, acc_log, probs, (uint32_t)n_probs);
    if (!e) fse_export(&t, bl, nb, sym);
    fse_table_free(&t);
    return e;
}
int oracle_fse_predefined(int which, uint32_t* bl, uint8_t* nb, uint8_t* sym, uint32_t* table_size) {
    fse_table_t t; fse_table_init(&t);
    int e;
    if (which == 0) e = fse_build_from_probabilities(&t, 6, LL_DEFAULT, 36);
    else if (which == 1) e = fse_build_from_probabilities(&t, 5, OF_DEFAULT, 29);
    else e = fse_build_from_probabilities(&t, 6, ML_DEFAULT, 53);
    if (!e) { fse_export(&t, bl, nb, sym); *table_size = t.decode_len; }
    fse_table_free(&t);
    return e;
}
int oracle_fse_build_decoder(const uint8_t* p, size_t len, uint8_t max_log, uint32_t* bl, uint8_t* nb, uint8_t* sym,
                             uint32_t* table_size, size_t* bytes_read) {
    fse_table_t t; fse_table_init(&t);
    slice_t s = {p, len};
    int e = fse_build_decoder(&t, s, max_log, bytes_read);
    if (!e) { fse_export(&t, bl, nb, sym); *table_size = t.decode_len; }
    fse_table_free(&t);
    return e;
}

/* ------------------------------------------------------------------------- */
/* Huffman (src/huff0/huff0_decoder.cairo)                                    */
/* ------------------------------------------------------------------------- */
typedef struct { uint8_t symbol, num_bits; } huf_entry_t; /* :57-61 */
typedef struct {
    huf_entry_t decode[2048]; uint32_t decode_len;
    uint8_t weights[260]; uint32_t n_weights;
    uint8_t bits[260];
    uint8_t max_num_bits;
    fse_table_t fse;
} huf_table_t;

static void huf_table_init(huf_table_t* h) { memset(h, 0, sizeof *h); fse_table_init(&h->fse); }
static void huf_table_reset(huf_table_t* h) { h->decode_len = 0; h->n_weights = 0; h->max_num_bits = 0; fse_table_reset(&h->fse); } /* :136-144 */

#define HUF_PUSH_WEIGHT(h, w) do { if ((h)->n_weights < 260) (h)->weights[(h)->n_weights] = (w); (h)->n_weights++; } while (0)

/* read_weights :159-319 */
static int huf_read_weights(huf_table_t* h, slice_t src, uint32_t flags, size_t* bytes_read) {
    if (src.len == 0) return CZS_HUF_SOURCE_IS_EMPTY;
    uint8_t header = src.p[0];
    size_t bits_read = 8;
    if (header <= 127) {
        slice_t fse_stream = {src.p + 1, src.len - 1};
        if ((size_t)header > fse_stream.len) return CZS_HUF_NOT_ENOUGH_BYTES_FOR_WEIGHTS;
        size_t used;
        int e = fse_build_decoder(&h->fse, fse_stream, 100, &used); /* :176 limit passed as 100 */
        if (e) return e;
        if (used > header) return CZS_HUF_FSE_TABLE_USED_TOO_MANY_BYTES;
        fse_dec_t d1, d2; fse_dec_new(&d1, &h->fse); fse_dec_new(&d2, &h->fse);
        size_t clen = header - used;
        slice_t cw = {fse_stream.p + used, fse_stream.len - used};
        if (cw.len < clen) return CZS_HUF_NOT_ENOUGH_BYTES_TO_DECOMPRESS_WEIGHTS;
        cw.len = clen;
        rbr_t br; rbr_init(&br, cw);
        bits_read += (used + clen) * 8;
        if (rbr_skip_padding(&br)) return CZS_HUF_EXTRA_PADDING;
        if ((e = fse_dec_init_state(&d1, &h->fse, &br))) return e;
        if ((e = fse_dec_init_state(&d2, &h->fse, &br))) return e;
        h->n_weights = 0;
        for (;;) { /* :242-274 two interleaved states */
            HUF_PUSH_WEIGHT(h, d1.state.symbol);
            if ((e = fse_dec_update_state(&d1, &h->fse, &br))) return e;
            if (br.rem <= -1) { HUF_PUSH_WEIGHT(h, d2.state.symbol); break; }
            HUF_PUSH_WEIGHT(h, d2.state.symbol);
            if ((e = fse_dec_update_state(&d2, &h->fse, &br))) return e;
            if (br.rem <= -1) { HUF_PUSH_WEIGHT(h, d1.state.symbol); break; }
            if (h->n_weights > 255) return CZS_HUF_TOO_MANY_WEIGHTS;
        }
    } else {
        slice_t raw = {src.p + 1, src.len - 1};
        uint32_t nw = (uint32_t)header - 127;
        size_t need = (nw + 1) / 2;
        if (raw.len < need) return CZS_HUF_NOT_ENOUGH_BYTES_IN_SOURCE;
        h->n_weights = nw;
        for (uint32_t i = 0; i < nw; i++) { /* :296-311 */
            int low_nibble = (flags & ORACLE_FLAG_NIBBLE_AS_WRITTEN) ? ((i | 1u) == 1u) /* :302 literally */
                                                                     : ((i & 1u) == 1u); /* RFC 8878 4.2.1.1 */
            h->weights[i] = low_nibble ? (raw.p[i / 2] & 0xF) : (raw.p[i / 2] >> 4);
            bits_read += 4;
        }
    }
    *bytes_read = (bits_read + 7) / 8;
    return 0;
}

/* build_table_from_weights :321-470 */
static int huf_build_table_from_weights(huf_table_t* h) {
    uint32_t nw = h->n_weights;
    uint32_t sum = 0;
    for (uint32_t i = 0; i < nw; i++) {
        uint8_t w = h->weights[i];
        if (w > 11) return CZS_HUF_WEIGHT_BIGGER_THAN_MAX_NUM_BITS;
        sum += w > 0 ? (1u << (w - 1)) : 0;
    }
    if (sum == 0) return CZS_HUF_MISSING_WEIGHTS;
    uint32_t max_bits = highest_bit_set_u32(sum);
    uint32_t left_over = (1u << max_bits) - sum;
    if (!is_power_of_two_u32(left_over)) return CZS_HUF_LEFTOVER_NOT_POWER_OF_2;
    uint32_t last_weight = highest_bit_set_u32(left_over);
    for (uint32_t s = 0; s < nw; s++) h->bits[s] = h->weights[s] > 0 ? (uint8_t)(max_bits + 1 - h->weights[s]) : 0;
    h->bits[nw] = (uint8_t)(max_bits + 1 - last_weight);
    h->max_num_bits = (uint8_t)max_bits;
    if (max_bits > 11) return CZS_HUF_MAX_BITS_TOO_HIGH;
    uint32_t bit_ranks[13]; memset(bit_ranks, 0, sizeof bit_ranks);
    for (uint32_t i = 0; i <= nw; i++) bit_ranks[h->bits[i]]++;
    uint32_t size = 1u << max_bits;
    memset(h->decode, 0, size * sizeof(huf_entry_t));
    h->decode_len = size;
    uint32_t rank_idx[13]; memset(rank_idx, 0, sizeof rank_idx);
    rank_idx[max_bits] = 0;
    for (uint32_t b = max_bits; b >= 1; b--) rank_idx[b - 1] = rank_idx[b] + bit_ranks[b] * (1u << (max_bits - b)); /* :413-429 */
    if (rank_idx[0] != size) return CZS_PANIC_INTERNAL; /* :431 */
    for (uint32_t s = 0; s <= nw; s++) { /* :433-467 */
        uint8_t b = h->bits[s];
        if (b != 0) {
            if (s > 255) return CZS_PANIC_INTERNAL; /* symbol.try_into::<u8>().unwrap() :455 */
            uint32_t base = rank_idx[b], len = 1u << (max_bits - b);
            rank_idx[b] += len;
            for (uint32_t i = 0; i < len; i++) { h->decode[base + i].symbol = (uint8_t)s; h->decode[base + i].num_bits = b; }
        }
    }
    return 0;
}

/* build_decoder :149-157 */
static int huf_build_decoder(huf_table_t* h, slice_t src, uint32_t flags, size_t* bytes_read) {
    h->decode_len = 0;
    int e = huf_read_weights(h, src, flags, bytes_read);
    if (e) return e;
    if (h->n_weights >= 260) return CZS_PANIC_INTERNAL;
    return huf_build_table_from_weights(h);
}

int oracle_huf_build_decoder(const uint8_t* p, size_t len, uint32_t flags, uint8_t* symbol, uint8_t* num_bits,
                             uint32_t* max_num_bits, size_t* bytes_read, uint8_t* weights_out, uint32_t* n_weights) {
    huf_table_t* h = (huf_table_t*)malloc(sizeof *h); huf_table_init(h);
    slice_t s = {p, len};
    int e = huf_build_decoder(h, s, flags, bytes_read);
    if (!e) {
        for (uint32_t i = 0; i < h->decode_len; i++) { symbol[i] = h->decode[i].symbol; num_bits[i] = h->decode[i].num_bits; }
        *max_num_bits = h->max_num_bits;
    }
    if (weights_out) { uint32_t n = h->n_weights < 258 ? h->n_weights : 258; memcpy(weights_out, h->weights, n); }
    if (n_weights) *n_weights = h->n_weights;
    fse_table_free(&h->fse); free(h);
    return e;
}

/* one Huffman stream: literals_section_decoder.cairo:183-243 (check_end=1) and :121-170 (check_end=0).
 * HuffmanDecoder init_state/decode_symbol/next_state: huff0_decoder.cairo:75-106. */
static int huf_decode_stream(const huf_table_t* h, slice_t stream, uint8_t* target, size_t* tlen, size_t tcap, int check_end) {
    rbr_t br; rbr_init(&br, stream);
    if (rbr_skip_padding(&br)) return CZS_LIT_EXTRA_PADDING;
    uint64_t state = 0;
    rbr_get_bits(&br, h->max_num_bits, &state);
    const int64_t lim = -(int64_t)h->max_num_bits;
    const uint64_t mask = (uint64_t)h->decode_len - 1;
    size_t n = *tlen;
    while (br.rem > lim) {
        huf_entry_t e = h->decode[state];
        if (n < tcap) target[n] = e.symbol;
        n++;
        uint64_t nb = 0; rbr_get_bits(&br, e.num_bits, &nb);
        state = ((state << e.num_bits) & mask) | nb;
    }
    *tlen = n;
    if (check_end && br.rem != lim) return CZS_BITSTREAM_READ_MISMATCH;
    return 0;
}

/* ------------------------------------------------------------------------- */
/* block-level structures                                                     */
/* ------------------------------------------------------------------------- */
typedef struct { uint32_t regen; int has_comp; uint32_t comp; int n_streams; int ls_type; } lit_section_t; /* literals_section.cairo:9-14 */

/* parse_from_header :81-175 */
static int lit_parse_header(lit_section_t* s, slice_t raw, unsigned* hdr_bytes) {
    if (raw.len == 0) return CZS_LIT_GET_BITS_ERROR; /* br.get_bits(2) on an empty span :85-90 */
    uint8_t b0 = raw.p[0];
    s->ls_type = b0 & 3;
    unsigned sf = (b0 >> 2) & 3;
    unsigned need;
    if (s->ls_type <= 1) need = (sf == 0 || sf == 2) ? 1 : (sf == 1 ? 2 : 3);
    else need = (sf <= 1) ? 3 : (sf == 2 ? 4 : 5);
    if (raw.len < need) return CZS_LIT_NOT_ENOUGH_BYTES;
    const uint8_t* r = raw.p;
    s->has_comp = 0; s->comp = 0; s->n_streams = 0;
    if (s->ls_type <= 1) {
        if (sf == 0 || sf == 2) s->regen = b0 >> 3;
        else if (sf == 1) s->regen = (b0 >> 4) + ((uint32_t)r[1] << 4);
        else s->regen = (b0 >> 4) + ((uint32_t)r[1] << 4) + ((uint32_t)r[2] << 12);
    } else {
        s->n_streams = sf == 0 ? 1 : 4;
        s->has_comp = 1;
        if (sf <= 1) { s->regen = (b0 >> 4) + (((uint32_t)r[1] & 0x3f) << 4); s->comp = (r[1] >> 6) + ((uint32_t)r[2] << 2); }
        else if (sf == 2) { s->regen = (b0 >> 4) + ((uint32_t)r[1] << 4) + (((uint32_t)r[2] & 3) << 12); s->comp = (r[2] >> 2) + ((uint32_t)r[3] << 6); }
        else { s->regen = (b0 >> 4) + ((uint32_t)r[1] << 4) + (((uint32_t)r[2] & 0x3f) << 12); s->comp = (r[2] >> 6) + ((uint32_t)r[3] << 2) + ((uint32_t)r[4] << 10); }
    }
    *hdr_bytes = need;
    return 0;
}

typedef struct { uint32_t n_seq; int has_modes; uint8_t modes; } seq_header_t; /* sequence_section.cairo:5-9 */
/* parse_from_header :77-114 */
static int seq_parse_header(seq_header_t* h, slice_t src, unsigned* hdr_bytes) {
    h->has_modes = 0; h->n_seq = 0; h->modes = 0;
    if (src.len == 0) return CZS_SEQ_HDR_NOT_ENOUGH_BYTES;
    uint8_t b0 = src.p[0]; unsigned br = 0;
    if (b0 == 0) { *hdr_bytes = 1; return 0; }
    else if (b0 <= 127) { if (src.len < 2) return CZS_SEQ_HDR_NOT_ENOUGH_BYTES; h->n_seq = b0; br = 1; }
    else if (b0 <= 254) { if (src.len < 3) return CZS_SEQ_HDR_NOT_ENOUGH_BYTES; h->n_seq = (((uint32_t)b0 - 128) << 8) + src.p[1]; br = 2; }
    else { if (src.len < 4) return CZS_SEQ_HDR_NOT_ENOUGH_BYTES; h->n_seq = (uint32_t)src.p[1] + ((uint32_t)src.p[2] << 8) + 0x7F00; br = 3; }
    h->modes = src.p[br]; h->has_modes = 1;
    *hdr_bytes = br + 1;
    return 0;
}

typedef struct { uint32_t ll, ml, of; } sequence_t; /* sequence_section.cairo:11-16 */

/* DecodeBuffer + RingBuffer (decode_buffer.cairo, ring_buffer.cairo): append-only bytes + head. */
typedef struct {
    uint8_t* data; size_t len, cap; int owned;
    size_t head;               /* RingBuffer.head (ring_buffer.cairo:54-59) */
    size_t window_size;
    uint64_t total_output_counter;
    xxh64_t hash;
} decode_buffer_t;

typedef struct { /* DecoderScratch scratch.cairo:10-19 */
    huf_table_t huf;
    fse_table_t ll, of, ml;
    int ll_rle, of_rle, ml_rle;  /* -1 = None */
    decode_buffer_t buffer;
    uint32_t offset_hist[3];
    uint8_t* literals; size_t n_literals, cap_literals;
    sequence_t* sequences; size_t n_sequences, cap_sequences;
    uint32_t flags;
} scratch_t;

static int buf_reserve(decode_buffer_t* b, size_t extra) {
    if (b->len + extra <= b->cap) return 0;
    if (!b->owned) return CZS_DST_TOO_SMALL;
    size_t nc = b->cap ? b->cap : 4096; while (nc < b->len + extra) nc *= 2;
    uint8_t* nd = (uint8_t*)realloc(b->data, nc); if (!nd) return CZS_PANIC_INTERNAL;
    b->data = nd; b->cap = nc; return 0;
}
/* RingBuffer::len ignores head (ring_buffer.cairo:20-22) */
static inline size_t buf_len(const decode_buffer_t* b) { return b->len; }
static int buf_push(decode_buffer_t* b, const uint8_t* p, size_t n) { /* decode_buffer.cairo:57-60 */
    int e = buf_reserve(b, n); if (e) return e;
    memcpy(b->data + b->len, p, n); b->len += n; b->total_output_counter += n; return 0;
}
static int buf_fill(decode_buffer_t* b, uint8_t byte, size_t n) { /* append_byte x n :52-55 */
    int e = buf_reserve(b, n); if (e) return e;
    memset(b->data + b->len, byte, n); b->len += n; b->total_output_counter += n; return 0;
}
/* repeat :62-133 (dict_content is always empty: frame_decoder.cairo:73) */
static int buf_repeat(decode_buffer_t* b, size_t offset, size_t match_length) {
    if (offset > b->len) {
        if (b->total_output_counter <= b->window_size) return CZS_NOT_ENOUGH_BYTES_IN_DICTIONARY;
        return CZS_OFFSET_TOO_BIG;
    }
    int e = buf_reserve(b, match_length); if (e) return e;
    size_t start = b->len - offset;
    if (offset >= match_length) memcpy(b->data + b->len, b->data + start, match_length);
    else { uint8_t* d = b->data + b->len; const uint8_t* s = b->data + start; for (size_t i = 0; i < match_length; i++) d[i] = s[i]; } /* :101-120 */
    b->len += match_length; b->total_output_counter += match_length;
    return 0;
}

static int scratch_init(scratch_t* s, size_t window, uint32_t flags) { /* scratch.cairo:23-40 */
    memset(s, 0, sizeof *s);
    huf_table_init(&s->huf); fse_table_init(&s->ll); fse_table_init(&s->of); fse_table_init(&s->ml);
    s->ll_rle = s->of_rle = s->ml_rle = -1;
    s->offset_hist[0] = 1; s->offset_hist[1] = 4; s->offset_hist[2] = 8;
    s->buffer.window_size = window; xxh64_init(&s->buffer.hash, 0);
    s->cap_literals = (1u << 20) + 16; s->literals = (uint8_t*)malloc(s->cap_literals);
    s->cap_sequences = 0x7F00 + 0x10000 + 8; s->sequences = (sequence_t*)malloc(s->cap_sequences * sizeof(sequence_t));
    s->flags = flags;
    return (s->literals && s->sequences) ? 0 : CZS_PANIC_INTERNAL;
}
static void scratch_reset(scratch_t* s, size_t window) { /* scratch.cairo:42-58 */
    s->offset_hist[0] = 1; s->offset_hist[1] = 4; s->offset_hist[2] = 8;
    s->n_literals = 0; s->n_sequences = 0;
    s->buffer.window_size = window; s->buffer.len = 0; s->buffer.head = 0; s->buffer.total_output_counter = 0;
    xxh64_init(&s->buffer.hash, 0);
    fse_table_reset(&s->ll); fse_table_reset(&s->ml); fse_table_reset(&s->of);
    s->ll_rle = s->ml_rle = s->of_rle = -1;
    huf_table_reset(&s->huf);
}
static void scratch_free(scratch_t* s) {
    fse_table_free(&s->huf.fse); fse_table_free(&s->ll); fse_table_free(&s->of); fse_table_free(&s->ml);
    free(s->literals); free(s->sequences);
    if (s->buffer.owned) free(s->buffer.data);
}

/* ------------------------------------------------------------------------- */
/* literals (src/decoding/literals_section_decoder.cairo)                     */
/* ------------------------------------------------------------------------- */
/* decompress_literals :58-181 */
static int decompress_literals(const lit_section_t* sec, scratch_t* sc, slice_t source, uint32_t* bytes_read_out) {
    slice_t src = {source.p, sec->comp};
    size_t bytes_read = 0;
    if (sec->ls_type == 2) {
        int e = huf_build_decoder(&sc->huf, src, sc->flags, &bytes_read);
        if (e) return e;
    } else {
        if (sc->huf.max_num_bits == 0) return CZS_UNINITIALIZED_HUFFMAN_TABLE;
    }
    src.p += bytes_read; src.len -= bytes_read;
    size_t n = 0;
    if (sec->n_streams == 4) {
        if (src.len < 6) return CZS_MISSING_BYTES_FOR_JUMP_HEADER;
        size_t j1 = src.p[0] + ((size_t)src.p[1] << 8);
        size_t j2 = j1 + src.p[2] + ((size_t)src.p[3] << 8);
        size_t j3 = j2 + src.p[4] + ((size_t)src.p[5] << 8);
        bytes_read += 6; src.p += 6; src.len -= 6;
        if (src.len < j3) return CZS_MISSING_BYTES_FOR_LITERALS;
        slice_t s1 = {src.p, j1}, s2 = {src.p + j1, j2 - j1}, s3 = {src.p + j2, j3 - j2}, s4 = {src.p + j3, src.len - j3};
        int e;
        if ((e = huf_decode_stream(&sc->huf, s1, sc->literals, &n, sc->cap_literals, 1))) return e;
        if ((e = huf_decode_stream(&sc->huf, s2, sc->literals, &n, sc->cap_literals, 1))) return e;
        if ((e = huf_decode_stream(&sc->huf, s3, sc->literals, &n, sc->cap_literals, 1))) return e;
        if ((e = huf_decode_stream(&sc->huf, s4, sc->literals, &n, sc->cap_literals, 1))) return e;
        bytes_read += src.len;
    } else {
        int e = huf_decode_stream(&sc->huf, src, sc->literals, &n, sc->cap_literals, 0); /* no end check :118-170 */
        if (e) return e;
        bytes_read += src.len;
    }
    if (n != sec->regen) return CZS_DECODED_LITERAL_COUNT_MISMATCH;
    sc->n_literals = n;
    *bytes_read_out = (uint32_t)bytes_read;
    return 0;
}

/* decode_literals :32-56 */
static int decode_literals(const lit_section_t* sec, scratch_t* sc, slice_t source, uint32_t* bytes_read) {
    switch (sec->ls_type) {
    case 0:
        if (source.len < sec->regen) return CZS_PANIC_TRUNCATED; /* unreachable: caller sliced to regen */
        memcpy(sc->literals, source.p, sec->regen); sc->n_literals = sec->regen; *bytes_read = sec->regen; return 0;
    case 1:
        if (source.len < 1) return CZS_PANIC_TRUNCATED;
        memset(sc->literals, source.p[0], sec->regen); sc->n_literals = sec->regen; *bytes_read = 1; return 0;
    default:
        return decompress_literals(sec, sc, source, bytes_read);
    }
}

/* ------------------------------------------------------------------------- */
/* sequences (src/decoding/sequence_section_decoder.cairo)                    */
/* ------------------------------------------------------------------------- */
static inline void lookup_ll_code(uint8_t c, uint32_t* base, unsigned* bits) { /* :299-345 */
    static const uint32_t B[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
    static const uint8_t N[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
    if (c <= 35) { *base = B[c]; *bits = N[c]; } else { *base = 0; *bits = 255; }
}
static inline void lookup_ml_code(uint8_t c, uint32_t* base, unsigned* bits) { /* :347-395 */
    static const uint32_t B[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539};
    static const uint8_t N[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
    if (c <= 52) { *base = B[c]; *bits = N[c]; } else { *base = 0; *bits = 255; }
}

/* maybe_update_fse_tables :405-647 */
static int maybe_update_fse_tables(const seq_header_t* sec, slice_t source, scratch_t* sc, size_t* bytes_read_out) {
    uint8_t modes = sec->modes;
    size_t br = 0; int e; size_t used;
    unsigned m = modes >> 6;
    if (m == 0) { if ((e = fse_build_from_probabilities(&sc->ll, 6, LL_DEFAULT, 36))) return e; sc->ll_rle = -1; }
    else if (m == 1) { if (source.len == 0) return CZS_MISSING_BYTE_FOR_RLE_LL_TABLE; br += 1; sc->ll_rle = source.p[0]; }
    else if (m == 2) { if ((e = fse_build_decoder(&sc->ll, source, 9, &used))) return e; br += used; sc->ll_rle = -1; }
    slice_t ofs = {source.p + br, source.len - br};
    m = (modes >> 4) & 3;
    if (m == 0) { if ((e = fse_build_from_probabilities(&sc->of, 5, OF_DEFAULT, 29))) return e; sc->of_rle = -1; }
    else if (m == 1) { if (ofs.len == 0) return CZS_MISSING_BYTE_FOR_RLE_OF_TABLE; br += 1; sc->of_rle = ofs.p[0]; }
    else if (m == 2) { if ((e = fse_build_decoder(&sc->of, ofs, 8, &used))) return e; br += used; sc->of_rle = -1; }
    slice_t mls = {source.p + br, source.len - br};
    m = (modes >> 2) & 3;
    if (m == 0) { if ((e = fse_build_from_probabilities(&sc->ml, 6, ML_DEFAULT, 53))) return e; sc->ml_rle = -1; }
    else if (m == 1) { if (mls.len == 0) return CZS_MISSING_BYTE_FOR_RLE_ML_TABLE; br += 1; sc->ml_rle = mls.p[0]; }
    else if (m == 2) { if ((e = fse_build_decoder(&sc->ml, mls, 9, &used))) return e; br += used; sc->ml_rle = -1; }
    *bytes_read_out = br;
    return 0;
}

/* decode_sequences :35-71 with both loop variants :73-195 / :197-297 */
static int decode_sequences(const seq_header_t* sec, slice_t source, scratch_t* sc) {
    size_t used; int e;
    if ((e = maybe_update_fse_tables(sec, source, sc, &used))) return e;
    slice_t bs = {source.p + used, source.len - used};
    rbr_t br; rbr_init(&br, bs);
    if (rbr_skip_padding(&br)) return CZS_SEQ_EXTRA_PADDING;
    const int with_rle = sc->ll_rle >= 0 || sc->ml_rle >= 0 || sc->of_rle >= 0;
    fse_dec_t ll, ml, of;
    fse_dec_new(&ll, &sc->ll); fse_dec_new(&ml, &sc->ml); fse_dec_new(&of, &sc->of);
    /* init order LL, OF, ML (:83-100, :207-218) */
    if (sc->ll_rle < 0 && (e = fse_dec_init_state(&ll, &sc->ll, &br))) return e;
    if (sc->of_rle < 0 && (e = fse_dec_init_state(&of, &sc->of, &br))) return e;
    if (sc->ml_rle < 0 && (e = fse_dec_init_state(&ml, &sc->ml, &br))) return e;
    sc->n_sequences = 0;
    for (uint32_t i = 0; i < sec->n_seq; i++) {
        uint8_t ll_code = sc->ll_rle >= 0 ? (uint8_t)sc->ll_rle : ll.state.symbol;
        uint8_t ml_code = sc->ml_rle >= 0 ? (uint8_t)sc->ml_rle : ml.state.symbol;
        uint8_t of_code = sc->of_rle >= 0 ? (uint8_t)sc->of_rle : of.state.symbol;
        uint32_t ll_val, ml_val; unsigned ll_bits, ml_bits;
        lookup_ll_code(ll_code, &ll_val, &ll_bits);
        lookup_ml_code(ml_code, &ml_val, &ml_bits);
        if (of_code >= 32) return CZS_SEQ_UNSUPPORTED_OFFSET;
        uint64_t obits, ml_add, ll_add;
        if (rbr_get_bits_triple(&br, of_code, ml_bits, ll_bits, &obits, &ml_add, &ll_add)) return CZS_SEQ_GET_BITS_ERROR;
        sequence_t s; s.of = (uint32_t)obits + (1u << of_code); s.ml = ml_val + (uint32_t)ml_add; s.ll = ll_val + (uint32_t)ll_add;
        sc->sequences[sc->n_sequences++] = s;
        if (sc->n_sequences < sec->n_seq) { /* update order LL, ML, OF (:153-176, :258-276) */
            if (sc->ll_rle < 0 && (e = fse_dec_update_state(&ll, &sc->ll, &br))) return e;
            if (sc->ml_rle < 0 && (e = fse_dec_update_state(&ml, &sc->ml, &br))) return e;
            if (sc->of_rle < 0 && (e = fse_dec_update_state(&of, &sc->of, &br))) return e;
        }
        if (br.rem < 0) {
            /* without_rle variant traps on `bits_remaining().try_into::<u64>().unwrap()` :279 */
            return with_rle ? CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES : CZS_PANIC_INTERNAL;
        }
    }
    if (br.rem > 0) return CZS_SEQ_EXTRA_BITS;
    return 0;
}

/* do_offset_history (sequence_execution.cairo:85-129) */
uint32_t oracle_offset_history(uint32_t v, uint32_t lit_len, uint32_t h[3]) {
    uint32_t actual;
    if (lit_len > 0) actual = v == 1 ? h[0] : v == 2 ? h[1] : v == 3 ? h[2] : v - 3;
    else actual = v == 1 ? h[1] : v == 2 ? h[2] : v == 3 ? h[0] - 1 : v - 3;
    uint32_t h0 = h[0], h1 = h[1];
    if (lit_len > 0) {
        if (v == 1) { /* unchanged */ }
        else if (v == 2) { h[0] = actual; h[1] = h0; }
        else { h[0] = actual; h[1] = h0; h[2] = h1; }
    } else {
        if (v == 1) { h[0] = actual; h[1] = h0; }
        else { h[0] = actual; h[1] = h0; h[2] = h1; }
    }
    return actual;
}

/* execute_sequences (sequence_execution.cairo:12-83) */
static int execute_sequences(scratch_t* sc, oracle_trace* tr) {
    size_t lit_pos = 0;
    for (size_t i = 0; i < sc->n_sequences; i++) {
        sequence_t s = sc->sequences[i];
        if (s.ll > 0) {
            size_t high = lit_pos + s.ll;
            if (high > sc->n_literals) return CZS_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE;
            int e = buf_push(&sc->buffer, sc->literals + lit_pos, s.ll); if (e) return e;
            lit_pos = high;
        }
        uint32_t nh[3] = {sc->offset_hist[0], sc->offset_hist[1], sc->offset_hist[2]};
        uint32_t actual = oracle_offset_history(s.of, s.ll, nh);
        if (actual == 0) return CZS_EXEC_ZERO_OFFSET;
        memcpy(sc->offset_hist, nh, sizeof nh);
        if (tr) tr->seqs[(tr->n_seqs - sc->n_sequences + i) * 4 + 3] = actual;
        if (s.ml > 0) { int e = buf_repeat(&sc->buffer, actual, s.ml); if (e) return e; }
    }
    if (lit_pos < sc->n_literals) { int e = buf_push(&sc->buffer, sc->literals + lit_pos, sc->n_literals - lit_pos); if (e) return e; }
    return 0;
}

/* ------------------------------------------------------------------------- */
/* trace helpers                                                              */
/* ------------------------------------------------------------------------- */
static oracle_block_trace* trace_new_block(oracle_trace* t) {
    if (t->n_blocks == t->cap_blocks) {
        t->cap_blocks = t->cap_blocks ? t->cap_blocks * 2 : 64;
        t->blocks = (oracle_block_trace*)realloc(t->blocks, t->cap_blocks * sizeof *t->blocks);
    }
    oracle_block_trace* b = &t->blocks[t->n_blocks++]; memset(b, 0, sizeof *b);
    b->lit_off = t->n_lits; b->seq_off = t->n_seqs;
    return b;
}
static void trace_add_lits(oracle_trace* t, const uint8_t* p, size_t n) {
    if (t->n_lits + n > t->cap_lits) { while (t->n_lits + n > t->cap_lits) t->cap_lits = t->cap_lits ? t->cap_lits * 2 : (1 << 16); t->lits = (uint8_t*)realloc(t->lits, t->cap_lits); }
    memcpy(t->lits + t->n_lits, p, n); t->n_lits += n;
}
static void trace_add_seqs(oracle_trace* t, const sequence_t* s, size_t n) {
    if (t->n_seqs + n > t->cap_seqs) { while (t->n_seqs + n > t->cap_seqs) t->cap_seqs = t->cap_seqs ? t->cap_seqs * 2 : (1 << 12); t->seqs = (uint32_t*)realloc(t->seqs, t->cap_seqs * 16); }
    for (size_t i = 0; i < n; i++) { uint32_t* o = t->seqs + (t->n_seqs + i) * 4; o[0] = s[i].ll; o[1] = s[i].ml; o[2] = s[i].of; o[3] = 0; }
    t->n_seqs += n;
}
void oracle_trace_free(oracle_trace* t) { free(t->blocks); free(t->lits); free(t->seqs); memset(t, 0, sizeof *t); }

/* ------------------------------------------------------------------------- */
/* block decoder (src/decoding/block_decoder.cairo)                           */
/* ------------------------------------------------------------------------- */
typedef struct { int last; int type; uint32_t decompressed_size, content_size; } block_header_t; /* block.cairo:10-15 */

/* read_block_header :237-278, :284-321; advances *src by 3 */
static int read_block_header(slice_t* src, block_header_t* h) {
    if (src->len < 3) return CZS_PANIC_TRUNCATED; /* r.slice(0,3) asserts */
    uint8_t a = src->p[0], b = src->p[1], c = src->p[2];
    src->p += 3; src->len -= 3;
    h->type = (a >> 1) & 3;
    if (h->type == 3) return CZS_FOUND_RESERVED_BLOCK;
    uint32_t size = (a >> 3) | ((uint32_t)b << 5) | ((uint32_t)c << 13);
    if (size > 128 * 1024) return CZS_BLOCK_SIZE_TOO_LARGE;
    h->decompressed_size = (h->type == 2) ? 0 : size;
    h->content_size = (h->type == 1) ? 1 : size;
    h->last = a & 1;
    return 0;
}

/* decompress_block :139-235 */
static int decompress_block(const block_header_t* h, scratch_t* sc, slice_t* src, oracle_trace* tr, oracle_block_trace* bt) {
    if (src->len < h->content_size) return CZS_PANIC_TRUNCATED;
    slice_t raw = {src->p, h->content_size};
    src->p += h->content_size; src->len -= h->content_size;
    lit_section_t sec; unsigned lit_hdr;
    int e = lit_parse_header(&sec, raw, &lit_hdr); if (e) return e;
    raw.p += lit_hdr; raw.len -= lit_hdr;
    size_t upper = sec.has_comp ? sec.comp : (sec.ls_type == 1 ? 1 : sec.regen);
    if (raw.len < upper) return CZS_MALFORMED_SECTION_HEADER;
    slice_t raw_lits = {raw.p, upper};
    uint32_t used_lits;
    if ((e = decode_literals(&sec, sc, raw_lits, &used_lits))) return e;
    if (used_lits != upper) return CZS_PANIC_INTERNAL; /* assert :194 */
    raw.p += upper; raw.len -= upper;
    seq_header_t sh; unsigned seq_hdr;
    if ((e = seq_parse_header(&sh, raw, &seq_hdr))) return e;
    raw.p += seq_hdr; raw.len -= seq_hdr;
    if (bt) { bt->lit_type = (uint8_t)sec.ls_type; bt->n_streams = (uint8_t)sec.n_streams; bt->regen_size = sec.regen; bt->n_seq = sh.n_seq; bt->modes = sh.modes; trace_add_lits(tr, sc->literals, sc->n_literals); }
    if (sh.n_seq != 0) {
        if ((e = decode_sequences(&sh, raw, sc))) return e;
        if (tr) trace_add_seqs(tr, sc->sequences, sc->n_sequences);
        if ((e = execute_sequences(sc, tr))) return e;
    } else {
        if ((e = buf_push(&sc->buffer, sc->literals, sc->n_literals))) return e;
        sc->n_sequences = 0;
    }
    return 0;
}

/* decode_block_content :77-137 */
static int decode_block_content(const block_header_t* h, scratch_t* sc, slice_t* src, uint64_t* body_bytes, oracle_trace* tr) {
    oracle_block_trace* bt = tr ? trace_new_block(tr) : NULL;
    size_t before = sc->buffer.len;
    int e = 0;
    if (bt) bt->block_type = (uint8_t)h->type;
    if (h->type == 0) {
        if (src->len < h->decompressed_size) return CZS_PANIC_TRUNCATED;
        if ((e = buf_push(&sc->buffer, src->p, h->decompressed_size))) return e;
        src->p += h->decompressed_size; src->len -= h->decompressed_size;
        *body_bytes = h->decompressed_size;
    } else if (h->type == 1) {
        if (src->len < 1) return CZS_PANIC_TRUNCATED;
        uint8_t byte = src->p[0]; src->p += 1; src->len -= 1;
        if ((e = buf_fill(&sc->buffer, byte, h->decompressed_size))) return e;
        *body_bytes = 1;
    } else {
        if ((e = decompress_block(h, sc, src, tr, bt))) return e;
        *body_bytes = h->content_size;
    }
    if (bt) bt->out_bytes = (uint32_t)(sc->buffer.len - before);
    return 0;
}

/* ------------------------------------------------------------------------- */
/* frame header (src/frame.cairo)                                             */
/* ------------------------------------------------------------------------- */
typedef struct { uint8_t descriptor, window_descriptor; int has_dict; uint32_t dict_id; uint64_t fcs; } frame_header_t;

/* read_frame_header :152-284 */
static int read_frame_header(slice_t* src, frame_header_t* fh, unsigned* hdr_len) {
    size_t i = 0; const uint8_t* p = src->p; size_t n = src->len;
    if (n < 4) return CZS_MAGIC_NUMBER_READ_ERROR;
    uint32_t magic = rd32le(p); i = 4;
    if (magic >= 0x184D2A50u && magic <= 0x184D2A5Fu) { if (n < 8) return CZS_FRAME_DESCRIPTOR_READ_ERROR; return CZS_SKIP_FRAME; }
    if (magic != 0xFD2FB528u) return CZS_BAD_MAGIC_NUMBER;
    if (n < i + 1) return CZS_FRAME_DESCRIPTOR_READ_ERROR;
    uint8_t d = p[i++];
    memset(fh, 0, sizeof *fh); fh->descriptor = d;
    int single = (d >> 5) & 1;
    if (!single) { if (n < i + 1) return CZS_WINDOW_DESCRIPTOR_READ_ERROR; fh->window_descriptor = p[i++]; }
    static const unsigned DL[4] = {0, 1, 2, 4};
    unsigned dl = DL[d & 3];
    if (dl) {
        if (n < i + dl) return CZS_DICTIONARY_ID_READ_ERROR;
        uint32_t id = 0; for (unsigned k = 0; k < dl; k++) id |= (uint32_t)p[i + k] << (8 * k);
        i += dl;
        if (id != 0) { fh->has_dict = 1; fh->dict_id = id; }
    }
    unsigned flag = d >> 6;
    unsigned fl = flag == 0 ? (single ? 1 : 0) : flag == 1 ? 2 : flag == 2 ? 4 : 8;
    if (fl) {
        if (n < i + fl) return CZS_DICTIONARY_ID_READ_ERROR; /* sic: :245-270 reuse this variant */
        uint64_t v = 0; for (unsigned k = 0; k < fl; k++) v |= (uint64_t)p[i + k] << (8 * k);
        i += fl;
        if (fl == 2) v += 256;
        fh->fcs = v;
    }
    src->p += i; src->len -= i;
    *hdr_len = (unsigned)i;
    return 0;
}

/* FrameHeader::window_size :106-129 */
static int frame_window_size(const frame_header_t* fh, uint64_t* ws) {
    if ((fh->descriptor >> 5) & 1) { *ws = fh->fcs; return 0; }
    uint64_t exp = fh->window_descriptor >> 3, mant = fh->window_descriptor & 7;
    uint64_t base = 1ULL << (10 + exp);
    uint64_t w = base + (base / 8) * mant;
    if (w >= 1024) { if (w < 4123168604160ULL) { *ws = w; return 0; } return CZS_WINDOW_TOO_BIG; }
    return CZS_WINDOW_TOO_SMALL;
}

/* ------------------------------------------------------------------------- */
/* FrameDecoder (src/frame_decoder.cairo)                                     */
/* ------------------------------------------------------------------------- */
struct oracle_fd {
    frame_header_t header;
    scratch_t scratch;
    int frame_finished;
    uint32_t block_counter;
    uint64_t bytes_read_counter;
    int has_check_sum; uint32_t check_sum;
    uint64_t window_size;
    uint32_t flags;
    int scratch_ready;
};

static int fd_is_finished(const oracle_fd* fd) { /* :144-150 */
    if ((fd->header.descriptor >> 2) & 1) return fd->frame_finished && fd->has_check_sum;
    return fd->frame_finished;
}

static int32_t fd_setup(oracle_fd* fd, const uint8_t* src, size_t src_len, size_t* consumed, int is_reset) { /* :54-105 */
    slice_t s = {src, src_len}; unsigned hl;
    int e = read_frame_header(&s, &fd->header, &hl); if (e) return e;
    uint64_t ws; if ((e = frame_window_size(&fd->header, &ws))) return e;
    if ((is_reset || (fd->flags & ORACLE_FLAG_RESET_LIMIT)) && ws > 100ULL * 1024 * 1024) return CZS_WINDOW_SIZE_TOO_BIG;
    if (ws > 0xFFFFFFFFULL) return CZS_PANIC_INTERNAL; /* window_size.try_into::<usize>().unwrap() :71, :99 */
    fd->window_size = ws;
    if (!fd->scratch_ready) { if ((e = scratch_init(&fd->scratch, (size_t)ws, fd->flags))) return e; fd->scratch_ready = 1; }
    else scratch_reset(&fd->scratch, (size_t)ws);
    fd->frame_finished = 0; fd->block_counter = 0; fd->bytes_read_counter = hl; fd->has_check_sum = 0; fd->check_sum = 0;
    if (consumed) *consumed = hl;
    return 0;
}

/* decode_blocks :156-222 */
static int32_t fd_decode_blocks(oracle_fd* fd, slice_t* src, int strategy, uint32_t n, oracle_trace* tr) {
    size_t size_before = buf_len(&fd->scratch.buffer);
    uint32_t blocks_before = fd->block_counter;
    for (;;) {
        block_header_t bh; int e = read_block_header(src, &bh); if (e) return e;
        fd->bytes_read_counter += 3;
        uint64_t body = 0;
        if ((e = decode_block_content(&bh, &fd->scratch, src, &body, tr))) return e;
        fd->bytes_read_counter += body;
        fd->block_counter++;
        if (bh.last) {
            fd->frame_finished = 1;
            if ((fd->header.descriptor >> 2) & 1) {
                if (src->len < 4) return CZS_PANIC_TRUNCATED; /* source.slice(0,4) :190 */
                fd->check_sum = rd32le(src->p); fd->has_check_sum = 1;
                src->p += 4; src->len -= 4; fd->bytes_read_counter += 4;
            }
            break;
        }
        if (strategy == 1) { if (fd->block_counter - blocks_before >= n) break; }
        else if (strategy == 2) { if (buf_len(&fd->scratch.buffer) - size_before >= n) break; }
    }
    return 0;
}

/* drain_to :168-186 (hash.update on the drained bytes) */
static size_t buf_drain_to(decode_buffer_t* b, size_t amount, uint8_t* dst, size_t cap, int* overflow) {
    if (amount == 0) return 0;
    size_t avail = b->len - b->head; /* as_slice(): elements[head..] ring_buffer.cairo:61-63 */
    size_t n = avail < amount ? avail : amount;
    xxh64_update(&b->hash, b->data + b->head, n);
    if (dst) { if (n > cap) { *overflow = 1; } else memcpy(dst, b->data + b->head, n); }
    b->head += n; /* drop_first_n :54-59 */
    return n;
}

static void fd_fill_result(const oracle_fd* fd, oracle_result* r) {
    r->blocks_decoded = fd->block_counter; r->bytes_read = fd->bytes_read_counter;
    r->content_size = fd->header.fcs; r->window_size = fd->window_size;
    r->checksum_from_data = fd->check_sum; r->has_checksum = fd->has_check_sum;
    r->checksum_calculated = (uint32_t)(xxh64_digest(&fd->scratch.buffer.hash) & 0xFFFFFFFFu); /* :133-138 */
    r->finished = fd_is_finished(fd);
}

int oracle_decode_frame(const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap, uint32_t flags,
                        oracle_result* res, oracle_trace* trace) {
    memset(res, 0, sizeof *res);
    oracle_fd* fd = (oracle_fd*)calloc(1, sizeof *fd);
    fd->flags = flags;
    size_t consumed = 0;
    int32_t st = fd_setup(fd, src, src_len, &consumed, 0);
    if (st) { res->status = st; if (fd->scratch_ready) scratch_free(&fd->scratch); free(fd); return st; }
    fd->scratch.buffer.data = dst; fd->scratch.buffer.cap = dst_cap; fd->scratch.buffer.owned = 0;
    slice_t s = {src + consumed, src_len - consumed};
    st = fd_decode_blocks(fd, &s, 0, 0, trace);
    /* collect(): drain() hashes everything then clears (decode_buffer.cairo:157-166) */
    if (!st) {
        xxh64_update(&fd->scratch.buffer.hash, fd->scratch.buffer.data, fd->scratch.buffer.len);
        res->bytes_written = fd->scratch.buffer.len;
    }
    fd_fill_result(fd, res);
    res->status = st;
    scratch_free(&fd->scratch); free(fd);
    return st;
}

/* ---- incremental surface ---- */
oracle_fd* oracle_fd_new(const uint8_t* src, size_t src_len, size_t* consumed, uint32_t flags, int32_t* status) {
    oracle_fd* fd = (oracle_fd*)calloc(1, sizeof *fd);
    fd->flags = flags;
    int32_t st = fd_setup(fd, src, src_len, consumed, 0);
    if (status) *status = st;
    if (st) { if (fd->scratch_ready) scratch_free(&fd->scratch); free(fd); return NULL; }
    fd->scratch.buffer.owned = 1;
    return fd;
}
int32_t oracle_fd_reset(oracle_fd* fd, const uint8_t* src, size_t src_len, size_t* consumed) {
    return fd_setup(fd, src, src_len, consumed, 1);
}
void oracle_fd_free(oracle_fd* fd) { if (!fd) return; if (fd->scratch_ready) scratch_free(&fd->scratch); free(fd); }
int32_t oracle_fd_decode_blocks(oracle_fd* fd, const uint8_t* src, size_t src_len, size_t* consumed, int strategy, uint32_t n, int32_t* finished) {
    slice_t s = {src, src_len};
    int32_t st = fd_decode_blocks(fd, &s, strategy, n, NULL);
    if (consumed) *consumed = src_len - s.len;
    if (finished) *finished = fd->frame_finished; /* Result::Ok(self.state.frame_finished) :221 */
    return st;
}
size_t oracle_fd_can_collect(const oracle_fd* fd) { /* :233-243 */
    const decode_buffer_t* b = &fd->scratch.buffer;
    if (fd_is_finished(fd)) return buf_len(b);
    return buf_len(b) > b->window_size ? buf_len(b) - b->window_size : 0;
}
int oracle_fd_collect(oracle_fd* fd, uint8_t* dst, size_t dst_cap, size_t* written) { /* :224-231 */
    decode_buffer_t* b = &fd->scratch.buffer;
    *written = 0;
    if (fd_is_finished(fd)) { /* drain(): as_slice() = elements[head..], hash, clear (decode_buffer.cairo:157-166) */
        size_t n = b->len - b->head;
        if (n > dst_cap) return -1;
        memcpy(dst, b->data + b->head, n);
        xxh64_update(&b->hash, b->data + b->head, n);
        b->len = 0; b->head = 0;
        *written = n; return 1;
    }
    if (buf_len(b) > b->window_size) { /* drain_to_window_size :146-155 */
        int ovf = 0;
        size_t n = buf_drain_to(b, buf_len(b) - b->window_size, dst, dst_cap, &ovf);
        if (ovf) return -1;
        *written = n; return 1;
    }
    return 0;
}
size_t oracle_fd_read(oracle_fd* fd, uint8_t* dst, size_t dst_cap) { /* :328-334; decode_buffer.cairo:188-203 */
    decode_buffer_t* b = &fd->scratch.buffer;
    size_t amount = fd->frame_finished ? buf_len(b) : (buf_len(b) > b->window_size ? buf_len(b) - b->window_size : 0);
    int ovf = 0;
    (void)buf_drain_to(b, amount, dst, dst_cap, &ovf);
    return ovf ? (size_t)-1 : amount; /* returns `amount`, not the bytes actually drained (quirk) */
}
int32_t oracle_fd_decode_from_to(oracle_fd* fd, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                                 size_t* read_len, size_t* written) { /* :245-326 */
    uint64_t start = fd->bytes_read_counter;
    if (!fd_is_finished(fd)) {
        slice_t s = {src, src_len};
        if (((fd->header.descriptor >> 2) & 1) && fd->frame_finished && !fd->has_check_sum) {
            if (s.len >= 4) { fd->check_sum = rd32le(s.p); fd->has_check_sum = 1; fd->bytes_read_counter += 4; }
            *read_len = 4; *written = 0; return 0; /* Ok((4,0)) :266 */
        }
        for (;;) {
            if (s.len < 3) break;
            block_header_t bh; int e = read_block_header(&s, &bh); if (e) return e;
            if (s.len < bh.content_size) break;
            fd->bytes_read_counter += 3;
            uint64_t body = 0;
            if ((e = decode_block_content(&bh, &fd->scratch, &s, &body, NULL))) return e;
            fd->bytes_read_counter += body; fd->block_counter++;
            if (bh.last) {
                fd->frame_finished = 1;
                if ((fd->header.descriptor >> 2) & 1) {
                    if (s.len >= 4) { fd->check_sum = rd32le(s.p); fd->has_check_sum = 1; s.p += 4; s.len -= 4; fd->bytes_read_counter += 4; }
                }
                break;
            }
        }
    }
    *written = oracle_fd_read(fd, dst, dst_cap);
    *read_len = (size_t)(fd->bytes_read_counter - start);
    return 0;
}
void oracle_fd_getters(const oracle_fd* fd, oracle_result* res) { memset(res, 0, sizeof *res); fd_fill_result(fd, res); }
void oracle_fd_buffer_state(const oracle_fd* fd, size_t* len, size_t* head) { *len = fd->scratch.buffer.len; *head = fd->scratch.buffer.head; }

/* ------------------------------------------------------------------------- */
/* Dictionary::decode_dict (src/decoding/dictionary.cairo:35-90): parsed, never applied by the reference  */
/* (frame_decoder.cairo:73 passes an empty dictionary).                                                   */
/* ------------------------------------------------------------------------- */
static uint32_t fnv_step(uint32_t h, uint32_t v) { return (h ^ v) * 16777619u; }
int oracle_dict_decode(const uint8_t* raw, size_t len, oracle_dict_info* out) {
    memset(out, 0, sizeof *out);
    out->offset_hist[0] = 2; out->offset_hist[1] = 4; out->offset_hist[2] = 8; /* :43 */
    if (len < 8) return CZS_PANIC_TRUNCATED;            /* word_u32_le(..).expect :46, :51 */
    uint32_t magic = rd32le(raw);
    if (magic != 0xEC30A437u) return CZS_DICT_BAD_MAGIC; /* :47-49 */
    out->id = rd32le(raw + 4);
    slice_t t = {raw + 8, len - 8};
    uint32_t h = 2166136261u;
    {   /* Huffman table :56-61 */
        huf_table_t* ht = (huf_table_t*)malloc(sizeof *ht); huf_table_init(ht);
        size_t used = 0;
        int e = huf_build_decoder(ht, t, 0, &used);
        if (!e) {
            out->huf_bytes = (uint32_t)used; out->huf_max_bits = ht->max_num_bits; out->n_weights = ht->n_weights;
            for (uint32_t i = 0; i < ht->decode_len; i++) h = fnv_step(h, (uint32_t)ht->decode[i].symbol | ((uint32_t)ht->decode[i].num_bits << 8));
        }
        fse_table_free(&ht->fse); free(ht);
        if (e) return e;
        t.p += used; t.len -= used;
    }
    const uint8_t max_log[3] = {8, 9, 9}; /* OF, ML, LL :63-79 */
    uint32_t* bytes_out[3] = {&out->of_bytes, &out->ml_bytes, &out->ll_bytes};
    uint32_t* log_out[3] = {&out->of_log, &out->ml_log, &out->ll_log};
    for (int k = 0; k < 3; k++) {
        fse_table_t ft; fse_table_init(&ft);
        size_t used = 0;
        int e = fse_build_decoder(&ft, t, max_log[k], &used);
        if (!e) {
            *bytes_out[k] = (uint32_t)used; *log_out[k] = ft.accuracy_log;
            for (uint32_t i = 0; i < ft.decode_len; i++)
                h = fnv_step(h, (uint32_t)(ft.decode[i].symbol > 63 ? 63 : ft.decode[i].symbol) | ((uint32_t)ft.decode[i].num_bits << 8) | (ft.decode[i].base_line << 12));
        }
        fse_table_free(&ft);
        if (e) return e;
        t.p += used; t.len -= used;
    }
    if (t.len < 12) return CZS_PANIC_TRUNCATED;          /* word_u32_le(..).expect :82-84 */
    out->offset_hist[0] = rd32le(t.p); out->offset_hist[1] = rd32le(t.p + 4); out->offset_hist[2] = rd32le(t.p + 8);
    out->content_off = (uint64_t)(t.p + 12 - raw); out->content_len = t.len - 12;
    out->table_hash = h;
    return 0;
}

/* ------------------------------------------------------------------------- */
/* multi-threaded batch (CPU baseline: one frame per task)                    */
/* ------------------------------------------------------------------------- */
typedef struct {
    size_t n; const uint8_t* const* srcs; const size_t* src_lens; uint8_t* const* dsts; const size_t* dst_caps;
    uint32_t flags; oracle_result* results; size_t next; pthread_mutex_t mu; int failures;
} batch_ctx_t;

static void* batch_worker(void* arg) {
    batch_ctx_t* c = (batch_ctx_t*)arg;
    int fails = 0;
    for (;;) {
        pthread_mutex_lock(&c->mu);
        size_t lo = c->next; size_t hi = lo + 16; if (hi > c->n) hi = c->n; c->next = hi;
        pthread_mutex_unlock(&c->mu);
        if (lo >= hi) break;
        for (size_t i = lo; i < hi; i++)
            if (oracle_decode_frame(c->srcs[i], c->src_lens[i], c->dsts[i], c->dst_caps[i], c->flags, &c->results[i], NULL)) fails++;
    }
    pthread_mutex_lock(&c->mu); c->failures += fails; pthread_mutex_unlock(&c->mu);
    return NULL;
}

int oracle_decode_batch(size_t n, const uint8_t* const* srcs, const size_t* src_lens, uint8_t* const* dsts,
                        const size_t* dst_caps, uint32_t flags, oracle_result* results, int n_threads) {
    batch_ctx_t c; memset(&c, 0, sizeof c);
    c.n = n; c.srcs = srcs; c.src_lens = src_lens; c.dsts = dsts; c.dst_caps = dst_caps; c.flags = flags; c.results = results;
    pthread_mutex_init(&c.mu, NULL);
    if (n_threads < 1) n_threads = 1;
    if (n_threads == 1) { batch_worker(&c); }
    else {
        pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
        for (int i = 0; i < n_threads; i++) pthread_create(&th[i], NULL, batch_worker, &c);
        for (int i = 0; i < n_threads; i++) pthread_join(th[i], NULL);
        free(th);
    }
    pthread_mutex_destroy(&c.mu);
    return c.failures;
}
