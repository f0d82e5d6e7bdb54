// k_fse.cu -- sequence section decode: FSE tables in shared memory, one lane per block.
//
// Reference path: decode_sequences, maybe_update_fse_tables, decode_sequences_{with,without}_rle,
// lookup_ll_code / lookup_ml_code (src/decoding/sequence_section_decoder.cairo:35-647),
// FSETable / FSEDecoder (src/fse/fse_decoder.cairo:64-400), BitReaderReversed
// (src/decoding/bit_reader_reverse.cairo), and do_offset_history
// (src/decoding/sequence_execution.cairo:85-129), which is folded in here because it is a serial
// chain over the same sequences.
//
// Mapping: the interleaved LL/OF/ML state machine is one dependency chain per block and cannot be
// split, so parallelism comes from blocks: a CTA owns 27 blocks, its 4 warps build the 81 tables
// cooperatively, then warp 0 decodes with lane = block.  Throughput is bounded by
// (blocks resident per SM) / (cycles per sequence step of a warp that is alone on its scheduler);
// 16-bit table entries (czb_fse_build.cuh) keep a block's three tables at <= 2.5 KiB so 81 blocks
// fit per SM (three CTAs).  HBM traffic: the bitstream in (a few bytes per sequence, through
// per-lane cp.async rings) and one packed 8-byte record per sequence out to scratch.
#include <type_traits>

#include "czb_fse_build.cuh"
#include "czb_internal.cuh"

namespace czb {

#ifndef CZB_FSE_WARPS
#define CZB_FSE_WARPS 4  // table-building warps per CTA (6 / 8 measured: see DESIGN.md)
#endif
constexpr int FSE_WARPS = CZB_FSE_WARPS;
#ifndef CZB_FSE_SLOTS
#define CZB_FSE_SLOTS 27
#endif
constexpr int FSE_SLOTS = CZB_FSE_SLOTS;  // 27 * 2560 B of tables + scratch = ~75 KB -> three CTAs (81 decode lanes) per SM
constexpr int FSE_SLOT_ENTRIES = 512 + 512 + 256;  // LL (log<=9), ML (log<=9), OF (log<=8)
constexpr int FSE_LL_OFS = 0, FSE_ML_OFS = 512, FSE_OF_OFS = 1024;

struct FseSlot {
    const uint8_t* bits;   // sequence bitstream
    Seq* out;
    uint32_t bits_len;
    uint32_t n_seq;
    uint32_t blk;
    int32_t status;
    uint16_t tbl[3];       // LL, OF, ML: entry index of the table inside FseSmem::entries (flat)
    uint16_t n_probs[3];   // phase 1a -> 1b: normalized counts parked in the table's region (0: nothing to build)
    int8_t log[3];         // accuracy log; 0 = RLE (one entry); -1 = never initialised
    uint8_t first_in_frame;
    uint8_t any_rle;
    uint8_t risky;         // some table holds a symbol beyond the code tables (LL > 35, OF > 31, ML > 52): the lean loop, which does not look, is skipped
};

struct alignas(16) FseWarpTmp {
    int16_t probs[FSE_MAX_SYMBOLS];
    uint8_t rank_sym[1 << FSE_MAX_LOG];
};
static_assert(sizeof(FseWarpTmp) * FSE_WARPS >= FSE_SLOTS * (RevBitsWin::RING + 16) + 16, "phase-2 rings (+ a 16-byte mirror per lane, one 16-byte dummy slot) reuse phase-1 scratch");

struct FseSmem {
    uint16_t entries[FSE_SLOTS * FSE_SLOT_ENTRIES + 64 + 32 + 64];  // per-slot tables, then predefined LL, OF, ML
    FseSlot slot[FSE_SLOTS];
    FseWarpTmp tmp[FSE_WARPS];
    uint32_t ll_code[64];  // base | bits << 27 (lookup_ll_code :299-345); bit 20 = code beyond the table -> (0,255)
    uint32_t ml_code[64];  // (lookup_ml_code :347-395)
};
constexpr int FSE_PREDEF_LL = FSE_SLOTS * FSE_SLOT_ENTRIES, FSE_PREDEF_OF = FSE_PREDEF_LL + 64, FSE_PREDEF_ML = FSE_PREDEF_OF + 32;

__device__ __constant__ uint32_t kLLBase[36] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 18, 20, 22, 24, 28, 32, 40, 48, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384, 32768, 65536};
__device__ __constant__ uint8_t kLLBits[36] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};
__device__ __constant__ uint32_t kMLBase[53] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34, 35, 37, 39, 41, 43, 47, 51, 59, 67, 83, 99, 131, 259, 515, 1027, 2051, 4099, 8195, 16387, 32771, 65539};
__device__ __constant__ uint8_t kMLBits[53] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16};

constexpr uint32_t FSE_BAD_CODE = 1u << 20;  // in ll_code / ml_code entries: a code beyond the table
__device__ __forceinline__ int stream_max_log(int s) { return s == 1 ? 8 : 9; }  // LL 9, OF 8, ML 9 (:397-399)

// Bytes a table description of `mode` occupies at p (for skipping to a later stream's description).
// One thread.  Returns false if the description cannot be parsed.
__device__ inline bool skip_description(int mode, int s, const uint8_t* p, int len, int& bytes) {
    bytes = 0;
    if (mode == MODE_RLE) { if (len < 1) return false; bytes = 1; return true; }
    if (mode == MODE_FSE) {
        int n_probs, log;
        return fse_read_probabilities(p, len, stream_max_log(s), nullptr, n_probs, log, bytes) == CZS_OK;
    }
    return true;
}

__global__ void __launch_bounds__(FSE_WARPS * 32, 3) k_fse(const czb_frame_desc* __restrict__ descs, BlockDesc* __restrict__ blocks,
                                                         const uint32_t* __restrict__ items,
                                                         const WaveCounters* __restrict__ counters, Seq* __restrict__ seq_scratch) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    FseSmem& sm = *reinterpret_cast<FseSmem*>(smem_raw);
    const uint32_t n_items = counters->n_fse;
    const unsigned warp = threadIdx.x >> 5, lane = lane_id();
    const uint32_t first = blockIdx.x * FSE_SLOTS;
    if (first >= n_items) return;  // whole CTA
    FseWarpTmp& tmp = sm.tmp[warp];

    // ---- predefined tables and code tables, once per CTA ----
    if (warp < 3) {
        const int n = warp == 0 ? 36 : (warp == 1 ? 29 : 53);
        const int8_t* src = warp == 0 ? kLLDefault : (warp == 1 ? kOFDefault : kMLDefault);
        for (int i = lane; i < n; i += 32) tmp.probs[i] = src[i];
        __syncwarp();
        fse_build_table_warp(tmp.probs, n, warp == 1 ? 5 : 6,
                             sm.entries + (warp == 0 ? FSE_PREDEF_LL : (warp == 1 ? FSE_PREDEF_OF : FSE_PREDEF_ML)), tmp.rank_sym);
    } else if (warp == 3) {
        for (int i = lane; i < 64; i += 32) sm.ll_code[i] = i < 36 ? (kLLBase[i] | ((uint32_t)kLLBits[i] << 27)) : FSE_BAD_CODE;
        for (int i = lane; i < 64; i += 32) sm.ml_code[i] = i < 53 ? (kMLBase[i] | ((uint32_t)kMLBits[i] << 27)) : FSE_BAD_CODE;
    }
    __syncwarp();

    __syncthreads();  // (the predefined tables' scratch is the build scratch below)

    // ---- phase 1a: maybe_update_fse_tables per block (:405-647): ONE THREAD per block walks the block's table descriptions ----
    // Reading normalized counts (read_probabilities) is a serial bit-by-bit walk; with one lane per warp doing it for one
    // block at a time it was half of this phase's instructions at 1/32 lane efficiency.  Here every block has its own
    // thread (spread over the warps so that few lanes diverge in each); the counts of a stream are parked in the stream's
    // own table region (256 x int16 fit into the smallest one) until phase 1b builds the table over them.
    {
        const int s = (int)lane * FSE_WARPS + (int)warp;
        if (s < FSE_SLOTS) {
            FseSlot& sl = sm.slot[s];
            const uint32_t item = first + s;
            sl.n_probs[0] = sl.n_probs[1] = sl.n_probs[2] = 0;
            if (item >= n_items) { sl.status = CZS_NOT_DECODED; sl.blk = NONE32; sl.n_seq = 0; }
            else {
                const uint32_t bi = items[item];
                const BlockDesc d = blocks[bi];
                const uint8_t* fsrc = descs[d.frame].src;
                uint32_t cursor = d.seq_src_off;
                const uint32_t end = d.seq_src_off + d.seq_src_len;
                int32_t st = CZS_OK;
                bool any_rle = false, risky = false;
                for (int k = 0; k < 3 && st == CZS_OK; k++) {
                    // lookup_ll_code / offset codes / lookup_ml_code (:235-237, :299-395); offset code 31 is legal but its value can pass
                    // REAL_OFF_CLAMP, which the lean loop does not apply: it goes to the exact loop as well
                    const uint32_t n_codes = k == 0 ? 36u : (k == 1 ? 31u : 53u);
                    const int region = s * FSE_SLOT_ENTRIES + (k == 0 ? FSE_LL_OFS : (k == 1 ? FSE_OF_OFS : FSE_ML_OFS));
                    uint32_t mode = ((uint32_t)d.modes >> (6 - 2 * k)) & 3u;
                    const uint8_t* p = fsrc + cursor;
                    int plen = (int)(end - cursor);
                    const bool own = mode != MODE_REPEAT;
                    sl.tbl[k] = (uint16_t)region; sl.log[k] = -1;  // until proven usable
                    if (!own) {  // Repeat: re-derive the table from the block that last set it
                        const uint32_t sb = d.tbl_src_blk[k];
                        if (sb == NONE32) continue;
                        const BlockDesc sd = blocks[sb];  // same frame
                        uint32_t scur = sd.seq_src_off;
                        const uint32_t send = sd.seq_src_off + sd.seq_src_len;
                        bool ok = true;
                        for (int q = 0; q < k && ok; q++) {
                            int bytes = 0;
                            ok = skip_description((int)(((uint32_t)sd.modes >> (6 - 2 * q)) & 3u), q, fsrc + scur, (int)(send - scur), bytes);
                            scur += (uint32_t)bytes;
                        }
                        if (!ok) continue;  // the source block failed the frame earlier
                        mode = ((uint32_t)sd.modes >> (6 - 2 * k)) & 3u;
                        p = fsrc + scur;
                        plen = (int)(send - scur);
                    }
                    if (mode == MODE_PREDEFINED) {
                        sl.tbl[k] = (uint16_t)(k == 0 ? FSE_PREDEF_LL : (k == 1 ? FSE_PREDEF_OF : FSE_PREDEF_ML)); sl.log[k] = (int8_t)(k == 1 ? 5 : 6);
                    } else if (mode == MODE_RLE) {
                        if (plen < 1) {
                            if (own) st = k == 0 ? CZS_MISSING_BYTE_FOR_RLE_LL_TABLE : (k == 1 ? CZS_MISSING_BYTE_FOR_RLE_OF_TABLE : CZS_MISSING_BYTE_FOR_RLE_ML_TABLE);
                        } else {
                            sm.entries[region] = fse_entry(p[0], 1u); sl.log[k] = 0;
                            any_rle = true;
                            risky = risky || p[0] >= n_codes;
                            if (own) cursor += 1;
                        }
                    } else {  // MODE_FSE
                        int n_probs = 0, log = 0, used = 0;
                        const int32_t pst = fse_read_probabilities(p, plen, stream_max_log(k), reinterpret_cast<int16_t*>(sm.entries + region), n_probs, log, used);
                        if (pst != CZS_OK) { if (own) st = pst; }
                        else {
                            sl.n_probs[k] = (uint16_t)n_probs; sl.log[k] = (int8_t)log;
                            risky = risky || (uint32_t)n_probs > n_codes;  // the last symbol of a description never has probability zero
                            if (own) cursor += (uint32_t)used;
                        }
                    }
                }
                sl.blk = bi; sl.n_seq = d.n_seq; sl.status = st;
                sl.bits = fsrc + cursor; sl.bits_len = end - cursor;
                sl.out = seq_scratch + d.seq_off;
                sl.first_in_frame = d.first_in_frame; sl.any_rle = any_rle ? 1 : 0; sl.risky = risky ? 1 : 0;
            }
        }
    }
    __syncthreads();
    // ---- phase 1b: build_decoding_table (fse_decoder.cairo:156-256), one table per warp at a time ----
    for (int s = warp; s < FSE_SLOTS; s += FSE_WARPS) {
        const FseSlot& sl = sm.slot[s];
        if (sl.blk == NONE32 || sl.status != CZS_OK) continue;
#pragma unroll 1
        for (int k = 0; k < 3; k++) {
            const int np = sl.n_probs[k];
            if (!np) continue;
            uint16_t* table = sm.entries + sl.tbl[k];
            for (int i = lane; i < np; i += 32) tmp.probs[i] = reinterpret_cast<const int16_t*>(table)[i];
            __syncwarp();
            fse_build_table_warp(tmp.probs, np, sl.log[k], table, tmp.rank_sym);
            __syncwarp();
        }
    }
    __syncthreads();
    if (warp != 0) return;  // (rotating the decode warp over the CTAs of an SM was measured: 28.3 -> 33.4 ms; the hardware already spreads them over the schedulers)

    // ---- phase 2: lane = block ----
    if (lane >= FSE_SLOTS) return;
    const FseSlot& sl = sm.slot[lane];
    if (sl.blk == NONE32) return;
    int32_t st = sl.status;
    uint32_t h0, h1, h2;
    if (sl.first_in_frame) { h0 = 1; h1 = 4; h2 = 8; }  // scratch.cairo:35
    else { h0 = sym_enc(0); h1 = sym_enc(1); h2 = sym_enc(2); }
    const uint32_t h_in0 = h0, h_in1 = h1, h_in2 = h2;
    uint32_t ml_total = 0;
    // The decode loop exists twice.  The fast form (decode_lean, below) only notes THAT something went wrong; a block for
    // which it did, or which it does not take, is decoded again by this exact form, which records WHICH error came first,
    // in the reference's order (two compares and selects per step: 8 % of the kernel when it was always on).
    auto decode = [&]() -> int32_t {
    int32_t st = CZS_OK;
    h0 = h_in0; h1 = h_in1; h2 = h_in2;
    ml_total = 0;
    {
        // phase 1's scratch is dead now (the other warps have left): it becomes the lanes' bitstream rings
        RevBitsWin br;
        const bool init_ok = br.init(sl.bits, (int)sl.bits_len, (uint32_t)__cvta_generic_to_shared(sm.tmp) + lane * (RevBitsWin::RING + 16) + 16u);
        if (!init_ok) st = CZS_SEQ_EXTRA_PADDING;  // :46-64
        else if (sl.log[0] < 0 || sl.log[1] < 0 || sl.log[2] < 0) st = CZS_FSE_TABLE_IS_UNINITIALIZED;  // fse_decoder.cairo:82-84
        else {
            const uint32_t logLL = (uint32_t)sl.log[0], logOF = (uint32_t)sl.log[1], logML = (uint32_t)sl.log[2];
            const uint32_t mLL = (1u << logLL) - 1u, mOF = (1u << logOF) - 1u, mML = (1u << logML) - 1u;
            const uint16_t* tLL = sm.entries + sl.tbl[0];
            const uint16_t* tOF = sm.entries + sl.tbl[1];
            const uint16_t* tML = sm.entries + sl.tbl[2];
            // init order LL, OF, ML (:207-218)
            uint32_t eLL = tLL[br.get((int)logLL)];
            uint32_t eOF = tOF[br.get((int)logOF)];
            uint32_t eML = tML[br.get((int)logML)];
            const uint32_t n_seq = sl.n_seq;
            Seq* out = sl.out;
            const int32_t short_status = sl.any_rle ? CZS_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES : CZS_PANIC_INTERNAL;
            // One sequence (:223-286).  MORE = false is the last sequence: states are not updated (:258).
            //
            // The lane runs alone on its scheduler most of the time, so a step costs the sum of its issue stalls.
            // Hence: (a) all lookups are software-pipelined -- the next states, their num_bits, their code words
            // (lookup_ll_code / lookup_ml_code) and the next 32 stream bits are requested as soon as their inputs
            // exist and consumed one step later; (b) no data-dependent branches -- errors are recorded (first one
            // wins) and the loop runs on, which is safe because table indices are masked, records stay inside
            // this block's slice of the scratch and ring reads wrap; the ring refill is a predicated cp.async.
            uint32_t lle = sm.ll_code[fse_entry_sym(eLL)], mle = sm.ml_code[fse_entry_sym(eML)];
            RevBitsWin::Raw64 win = br.window64_raw();
            const uint32_t dummy = (uint32_t)__cvta_generic_to_shared(sm.tmp) + FSE_SLOTS * (RevBitsWin::RING + 16);  // one slot for all lanes: only zeros are ever written
            uint32_t nbLL = fse_entry_nbits(eLL, logLL), nbML = fse_entry_nbits(eML, logML), nbOF = fse_entry_nbits(eOF, logOF);
            Seq quad[4];  // four records leave as two 16-byte stores: a block's slice of the scratch is 32-byte aligned (k_fill_blocks)
            auto step = [&](uint32_t i, auto more_tag, auto refill_tag, auto quad_tag) {
                constexpr bool MORE = decltype(more_tag)::value;
                constexpr int REFILLS = decltype(refill_tag)::value;  // ring slots to look after in this step
                constexpr int QUAD = decltype(quad_tag)::value;       // position inside the group of four (-1: store it alone)
                br.step_sync();
                const uint32_t ofc = fse_entry_sym(eOF);
                // :235-237; codes beyond the tables give (0,255) -> TooManyBits
                const bool bad_code = ((ofc >> 5) | (((lle | mle) >> 20) & 1u)) != 0;
                const int32_t code_status = ofc >= 32 ? CZS_SEQ_UNSUPPORTED_OFFSET : CZS_SEQ_GET_BITS_ERROR;
                st = (st == CZS_OK && bad_code) ? code_status : st;
                const uint32_t llb = lle >> 27, mlb = mle >> 27, ofb = ofc & 31u;
                const uint32_t extras = ofb + mlb + llb;  // <= 63 bits, read in the order OF, ML, LL (:239)
                // The three state updates (LL, ML, OF, <= 26 bits, :258-276) come from their own 32-bit window below the
                // extra bits, whose position is known from the start of the step: no "does it all fit in 32 bits" branch.
                RevBitsWin::Raw winB;
                if (MORE) winB = br.window_raw_at(br.P - (int)extras);
                const uint32_t xh = __funnelshift_r(win.w1, win.w2, win.sh), xl = __funnelshift_r(win.w0, win.w1, win.sh);
                const uint32_t ofv = shr_clamp(xh, 32u - ofb);
                const uint32_t y = __funnelshift_l(xl, xh, ofb);
                const uint32_t mlv = shr_clamp(y, 32u - mlb), llv = shr_clamp(y << mlb, 32u - llb);
                uint32_t aLL = 0, aML = 0, aOF = 0;
                if (MORE) {
                    const uint32_t z = RevBitsWin::window_of(winB);
                    aLL = shr_clamp(z, 32u - nbLL); aML = shr_clamp(z << nbLL, 32u - nbML); aOF = shr_clamp(z << (nbLL + nbML), 32u - nbOF);
                    br.P -= (int)(extras + nbLL + nbML + nbOF);
#pragma unroll
                    for (int r = 0; r < REFILLS; r++) br.refill_nobranch(dummy);
                    win = br.window64_raw();  // the next step's bits: three LDS issued next to the state lookups below
                } else {
                    br.P -= (int)extras;
                }
                const uint32_t ll = (lle & 0xFFFFFu) + llv, ml = (mle & 0xFFFFFu) + mlv;
                if (MORE) {  // issue the next-state lookups now; they complete under the history/pack/store work below
                    eLL = tLL[(fse_entry_base(eLL, nbLL, logLL) + aLL) & mLL];
                    eML = tML[(fse_entry_base(eML, nbML, logML) + aML) & mML];
                    eOF = tOF[(fse_entry_base(eOF, nbOF, logOF) + aOF) & mOF];
                }
                const uint32_t v = (1u << ofb) + ofv;  // :243
                // do_offset_history (sequence_execution.cairo:85-129) with selects only:
                // idx 0,1,2 = history slot, 3 = h0 - 1 (reachable only when ll == 0)
                const uint32_t idx = v - (ll != 0);
                const bool rep = v <= 3;
                uint32_t cand = h0 - 1u;
                cand = idx == 2 ? h2 : cand;
                cand = idx == 1 ? h1 : cand;
                cand = idx == 0 ? h0 : cand;
                const uint32_t nz = min(v - 3u, REAL_OFF_CLAMP);
                const uint32_t act = rep ? cand : nz;
                h2 = (rep & (idx <= 1)) ? h2 : h1;
                h1 = (rep & (idx == 0)) ? h1 : h0;
                h0 = act;
                ml_total += ml;  // the block's output size is regen + sum(ml): what czb_frame_sizes_* reports without executing
                const Seq rec = (Seq)ll | ((Seq)ml << 17) | ((Seq)off29_pack(act) << 35);
                if constexpr (QUAD < 0) __stcs(out + i, rec);  // written once, read by a later kernel: streaming store
                else quad[QUAD] = rec;
                if (MORE) {
                    lle = sm.ll_code[fse_entry_sym(eLL)]; mle = sm.ml_code[fse_entry_sym(eML)];
                    nbLL = fse_entry_nbits(eLL, logLL); nbML = fse_entry_nbits(eML, logML); nbOF = fse_entry_nbits(eOF, logOF);
                }
                // :281-283; the no-RLE variant traps on the unwrap at :279 instead
                st = (st == CZS_OK && br.rem() < 0) ? short_status : st;
            };
            // Four steps consume at most 356 bits, i.e. leave at most three 16-byte chunks behind: the ring is looked after
            // once per four steps (three always-issued cp.async) instead of once per step.
            using R0 = std::integral_constant<int, 0>; using R1 = std::integral_constant<int, 1>; using R3 = std::integral_constant<int, 3>;
            using Q0 = std::integral_constant<int, 0>; using Q1 = std::integral_constant<int, 1>; using Q2 = std::integral_constant<int, 2>;
            using Q3 = std::integral_constant<int, 3>; using QN = std::integral_constant<int, -1>;
            uint32_t i = 0;
            for (; i + 4 < n_seq; i += 4) {
                step(i, std::true_type{}, R0{}, Q0{}); step(i + 1, std::true_type{}, R0{}, Q1{});
                step(i + 2, std::true_type{}, R0{}, Q2{}); step(i + 3, std::true_type{}, R3{}, Q3{});
                uint4* o4 = reinterpret_cast<uint4*>(out + i);
                __stcs(o4, make_uint4((uint32_t)quad[0], (uint32_t)(quad[0] >> 32), (uint32_t)quad[1], (uint32_t)(quad[1] >> 32)));
                __stcs(o4 + 1, make_uint4((uint32_t)quad[2], (uint32_t)(quad[2] >> 32), (uint32_t)quad[3], (uint32_t)(quad[3] >> 32)));
            }
            for (; i + 1 < n_seq; i++) step(i, std::true_type{}, R1{}, QN{});
            step(i, std::false_type{}, R0{}, QN{});
            if (st == CZS_OK && br.rem() > 0) st = CZS_SEQ_EXTRA_BITS;  // :292-296
        }
    }
    return st;
    };
    // The fast form, one warp, written for instruction count.  ALU instructions issue at one per two cycles per scheduler
    // and the decode warp is alone on its scheduler, so a step costs ~1.6 cycles per instruction whatever the dependency
    // chain looks like (154 instructions and ~250 cycles in the round-1 form; splitting the step over two warps left the
    // chain warp with its stalls and nothing to fill them: same time, see DESIGN.md).  Savings: a 96-bit window read once
    // per step serves the extra bits and the state bits (no second, position-dependent ring read); the ring has a mirror of
    // its top below it, so the four words come from one address with immediate offsets; next state = one funnel shift
    // (state << nb | bits) and one mask; table addresses are byte addresses kept opaque (one add per lookup); refills
    // are one always-issued cp.async per four steps plus rare warp-uniform extras; the cp.async wait depth follows the
    // stream (three groups in flight when it moves slowly).  It only notes THAT something went wrong.
    auto decode_lean = [&]() -> int32_t {
        h0 = h_in0; h1 = h_in1; h2 = h_in2;
        ml_total = 0;
        constexpr uint32_t RING_STRIDE = RevBitsWin::RING + 16;
        RevBitsWin br;
        if (!br.init(sl.bits, (int)sl.bits_len, (uint32_t)__cvta_generic_to_shared(sm.tmp) + lane * RING_STRIDE + 16u)) return CZS_NOT_DECODED;
        if (sl.log[0] < 0 || sl.log[1] < 0 || sl.log[2] < 0 || sl.risky) return CZS_NOT_DECODED;  // risky: a code beyond the tables may turn up (:235-237), and this loop does not look
        const uint32_t dummy = (uint32_t)__cvta_generic_to_shared(sm.tmp) + FSE_SLOTS * RING_STRIDE;
        const uint32_t logLL = (uint32_t)sl.log[0], logOF = (uint32_t)sl.log[1], logML = (uint32_t)sl.log[2];
        const uint32_t mLL = (1u << logLL) - 1u, mOF = (1u << logOF) - 1u, mML = (1u << logML) - 1u;
        const uint32_t ent = (uint32_t)__cvta_generic_to_shared(sm.entries);
        uint32_t tLL = ent + 2u * sl.tbl[0], tOF = ent + 2u * sl.tbl[1], tML = ent + 2u * sl.tbl[2];  // byte addresses
        asm volatile("" : "+r"(tLL), "+r"(tOF), "+r"(tML));  // opaque: keeps "base + 2 * index" one add instead of (table + index) * 2 + smem base
        auto lds16 = [](uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; };
        // init order LL, OF, ML (:207-218)
        uint32_t eLL = lds16(tLL + 2u * br.get((int)logLL));
        uint32_t eOF = lds16(tOF + 2u * br.get((int)logOF));
        uint32_t eML = lds16(tML + 2u * br.get((int)logML));
        cp_async_commit();
        cp_async_wait<0>();
        {   // the mirror starts out equal to the ring's top chunk
            uint8_t* ring_gen = reinterpret_cast<uint8_t*>(sm.tmp) + lane * RING_STRIDE + 16;
            *reinterpret_cast<uint4*>(ring_gen - 16) = *reinterpret_cast<const uint4*>(ring_gen + RevBitsWin::RING - 16);
        }
        const uint32_t n = sl.n_seq;
        Seq* out = sl.out;
        uint32_t x0, x1, x2;   // 96 unread bits at P, x2 first: extra bits (<= 63) and state bits (<= 26) of one step all lie inside
        auto load_window = [&]() {
            const uint32_t a = br.ring + (((uint32_t)br.P >> 3) & (RevBitsWin::RING - 4)), sh = (uint32_t)br.P & 31u;
            uint32_t w0, w1, w2, w3;  // the word holding bit P and the three below it (mirror: no wrap)
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w3) : "r"(a) : "memory");
            asm volatile("ld.shared.u32 %0, [%1+-4];" : "=r"(w2) : "r"(a) : "memory");
            asm volatile("ld.shared.u32 %0, [%1+-8];" : "=r"(w1) : "r"(a) : "memory");
            asm volatile("ld.shared.u32 %0, [%1+-12];" : "=r"(w0) : "r"(a) : "memory");
            x2 = __funnelshift_r(w2, w3, sh); x1 = __funnelshift_r(w1, w2, sh); x0 = __funnelshift_r(w0, w1, sh);
        };
        auto refill = [&](unsigned act) {  // the ring's look-after with the mirror kept equal
            const int cn = (br.P - 1) >> 7;
            const bool left = cn < br.chunk, need = left && br.chunk >= RevBitsWin::RING / 16;
            const uint32_t slot = (uint32_t)br.chunk & (RevBitsWin::RING / 16 - 1);
            const uint8_t* src = br.c_lo + (need ? ((br.chunk - RevBitsWin::RING / 16) << 4) : 0);
            cp_async16_sz(need ? br.ring + (slot << 4) : dummy, src, need ? 16u : 0u);
            const bool top = need && slot == RevBitsWin::RING / 16 - 1;
            if (__any_sync(act, top)) cp_async16_sz(top ? br.ring - 16u : dummy, src, top ? 16u : 0u);  // one chunk in eight
            br.chunk -= left ? 1 : 0;
        };
        uint32_t lle, mle, nbLL, nbML, nbOF;
        uint32_t llc = (uint32_t)__cvta_generic_to_shared(sm.ll_code), mlc = (uint32_t)__cvta_generic_to_shared(sm.ml_code);
        asm volatile("" : "+r"(llc), "+r"(mlc));  // opaque, as above: one shift and one scaled add per code lookup
        const uint32_t kLL = logLL - 9u, kOF = logOF - 9u, kML = logML - 9u;
        auto prep = [&]() {  // what the next step needs from the entries just looked up
            // address = table + 4 * symbol as ONE multiply-add (the other pipe); ptxas otherwise makes (entry >> 8) & 0xfc and an add of it
            uint32_t al, am;
            asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(al) : "r"(fse_entry_sym(eLL)), "r"(llc));
            asm("mad.lo.u32 %0, %1, 4, %2;" : "=r"(am) : "r"(fse_entry_sym(eML)), "r"(mlc));
            lle = lds32(al); mle = lds32(am);
            // num_bits = log - floor(log2(next_state)), next_state in the entry's low 10 bits (the shift can go to the other pipe)
            nbLL = kLL + (uint32_t)__clz(eLL << 22); nbML = kML + (uint32_t)__clz(eML << 22); nbOF = kOF + (uint32_t)__clz(eOF << 22);
        };
        load_window(); prep();
        // One sequence (:223-286).  MORE = false is the last sequence: states are not updated (:258).
        auto step = [&](auto more_tag, auto sym_tag) -> Seq {  // sym_tag: some lane of the warp runs on symbolic history (a block that is not first in its frame)
            constexpr bool MORE = decltype(more_tag)::value;
            const uint32_t llb = lle >> 27, mlb = mle >> 27, ofb = fse_entry_sym(eOF) & 31u;
            const uint32_t extras = ofb + mlb + llb;  // read in the order OF, ML, LL (:239)
            // funnel shifts: (hi << n) | (lo >> (32 - n)) is "hi, then the top n bits of lo" -- also right for n = 0
            const uint32_t v = __funnelshift_l(x2, 1u, ofb);  // (1 << ofb) + the ofb extra bits (:243)
            const uint32_t y = __funnelshift_l(x1, x2, ofb);
            const uint32_t mlv = __funnelshift_l(y, 0u, mlb), llv = __funnelshift_l(y << mlb, 0u, llb);
            // literal-length baselines are multiples of 2^bits (16,18,20,22 | 24,28 | 32,40 | 48 | 64 ...): "|" is "+"; match-length ones are not (35,37,..)
            const uint32_t ll = (lle & 0xFFFFFu) | llv, ml = (mle & 0xFFFFFu) + mlv;
            if (MORE) {
                // state bits (LL, ML, OF, :258-276) start `extras` bits into the window
                const uint32_t za = __funnelshift_l(x1, x2, extras), zb = __funnelshift_l(x0, x1, extras);  // shift taken modulo 32
                const uint32_t z = (extras & 32u) ? zb : za;
                // next state = base_line + bits = ((next_state << nb) | top nb bits) without bit `log` and above
                const uint32_t iLL = __funnelshift_l(z, eLL, nbLL) & mLL;
                const uint32_t z1 = z << nbLL;
                const uint32_t iML = __funnelshift_l(z1, eML, nbML) & mML;
                const uint32_t z2 = z1 << nbML;
                const uint32_t iOF = __funnelshift_l(z2, eOF, nbOF) & mOF;
                br.P -= (int)(extras + nbLL + nbML + nbOF);
                eLL = lds16(tLL + 2u * iLL); eML = lds16(tML + 2u * iML); eOF = lds16(tOF + 2u * iOF);
                load_window();
            } else {
                br.P -= (int)extras;
            }
            // do_offset_history (sequence_execution.cairo:85-129) with selects only:
            // idx 0,1,2 = history slot, 3 = h0 - 1 (reachable only when ll == 0)
            const uint32_t idx = v - (ll != 0);
            const bool rep = v <= 3;
            uint32_t cand = h0 - 1u;
            cand = idx == 2 ? h2 : cand;
            cand = idx == 1 ? h1 : cand;
            cand = idx == 0 ? h0 : cand;
            const uint32_t nz = v - 3u;  // < 2^31: offset code 31 never gets here (risky), so no REAL_OFF_CLAMP
            const uint32_t act = rep ? cand : nz;
            h2 = (rep & (idx <= 1)) ? h2 : h1;
            h1 = (rep & (idx == 0)) ? h1 : h0;
            h0 = act;
            ml_total += ml;  // the block's output size is regen + sum(ml): what czb_frame_sizes_* reports without executing
            if (MORE) prep();
            uint32_t packed = min(act, OFF29_CLAMP);
            if (decltype(sym_tag)::value) {
                // off29_pack without its branches: symbolic v = SYM_BASE + (k << 24) + SYM_MID - c  ->  1 << 28 | k << 24 | c
                //   = v - 2 * (v & 0xFFFFFF) + (1 << 28) + 2 * SYM_MID - SYM_BASE - SYM_MID   (mod 2^32; c < SYM_MID)
                const uint32_t packed_sym = act - 2u * (act & 0x00FFFFFFu) + ((1u << 28) + SYM_MID - SYM_BASE);
                packed = act >= SYM_BASE ? packed_sym : packed;
            }
            return (Seq)ll | ((Seq)ml << 17) | ((Seq)packed << 35);
        };
        auto run = [&](auto sym_tag) {
        int p1 = 0x40000000, p2 = 0x40000000, p3 = 0x40000000;  // P at the start of the previous three groups of four ("far above": nothing may stay in flight yet)
        uint32_t i = 0;
        for (; i + 4 < n; i += 4) {
            // Ring: what these four steps read must have landed.  One commit group per four steps; the group of round j asked for
            // chunks up to (head chunk at the start of j) - 8, and this round reads no chunk below (head chunk now) - 4: a group
            // may stay in flight while the head has moved less than four chunks since its round began, which holds if it moved
            // at most 384 bits.  Always true for the previous round (<= 356 bits per round); typical streams (~25 bits per
            // sequence) leave three groups, i.e. a dozen steps, for a request to come back from DRAM.
            const unsigned act = __activemask();
            if (__all_sync(act, p3 - br.P <= 384)) cp_async_wait<3>();
            else if (__all_sync(act, p2 - br.P <= 384)) cp_async_wait<2>();
            else cp_async_wait<1>();
            p3 = p2; p2 = p1; p1 = br.P;
            // four records leave as two 16-byte stores: a block's slice of the scratch is 32-byte aligned (k_fill_blocks)
            const Seq r0 = step(std::true_type{}, sym_tag), r1 = step(std::true_type{}, sym_tag), r2 = step(std::true_type{}, sym_tag), r3 = step(std::true_type{}, sym_tag);
            uint4* o4 = reinterpret_cast<uint4*>(out + i);
            __stcs(o4, make_uint4((uint32_t)r0, (uint32_t)(r0 >> 32), (uint32_t)r1, (uint32_t)(r1 >> 32)));
            __stcs(o4 + 1, make_uint4((uint32_t)r2, (uint32_t)(r2 >> 32), (uint32_t)r3, (uint32_t)(r3 >> 32)));
            // four steps consume at most 356 bits, i.e. leave at most three 16-byte chunks behind; usually less than one
            refill(act);
            if (__any_sync(act, ((br.P - 1) >> 7) < br.chunk)) { refill(act); refill(act); }
            cp_async_commit();
        }
        for (; i < n; i++) {  // the block's last one to four sequences
            cp_async_wait<0>();
            const Seq r = i + 1 < n ? step(std::true_type{}, sym_tag) : step(std::false_type{}, sym_tag);
            __stcs(out + i, r);  // written once, read by a later kernel: streaming store
            refill(__activemask());
            cp_async_commit();
        }
        };
        if (__any_sync(__activemask(), !sl.first_in_frame)) run(std::true_type{}); else run(std::false_type{});
        cp_async_wait<0>();
        // rem only ever decreases: one look tells whether it went negative on the way (:281-283)
        if (br.rem() < 0) return CZS_NOT_DECODED;  // placeholder: the exact form decides
        return br.rem() > 0 ? CZS_SEQ_EXTRA_BITS : CZS_OK;  // :292-296
    };
    if (st == CZS_OK) {
        const unsigned decoders = __activemask();
        st = decode_lean();
        __syncwarp(decoders);  // the exact loop lays its rings over the same scratch
        if (st == CZS_NOT_DECODED) st = decode();
    }
    BlockDesc& d = blocks[sl.blk];
    d.fse_status = st;
    d.hist_out[0] = h0; d.hist_out[1] = h1; d.hist_out[2] = h2;
    d.ml_sum = ml_total;
}

void launch_fse(const LaunchCtx& lc, const czb_frame_desc* descs, BlockDesc* blocks, const uint32_t* items,
                const WaveCounters* counters, uint32_t max_items, Seq* seq_scratch) {
    if (!max_items) return;
    const unsigned grid = (max_items + FSE_SLOTS - 1) / FSE_SLOTS;
    k_fse<<<grid, FSE_WARPS * 32, sizeof(FseSmem), lc.stream>>>(descs, blocks, items, counters, seq_scratch);
    ++*lc.launches;
}

int setup_fse_attributes() {
    return (int)cudaFuncSetAttribute(k_fse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FseSmem));
}

}  // namespace czb
