// czb_host.h -- host-side context shared by czb_api.cu and czb_handle.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "czb_internal.cuh"

template <typename T>
struct DevBuf {
    T* p = nullptr;
    uint64_t cap = 0;  // elements
};

constexpr uint64_t kMaxWaves = 4096;

struct czb_context {
    int device = 0;
    uint64_t budget = 0;        // soft cap on per-wave scratch bytes
    uint64_t wave_frames = 0;   // upper bound on frames per wave
    uint64_t host_chunk_bytes = 3ull << 30;  // src+dst bytes per chunk of the packed host path
    std::string last_error;
    uint64_t launches = 0;

    // decode workspace (device)
    DevBuf<czb::FrameInfo> infos;
    DevBuf<czb::WaveTotals> totals_d;
    czb::WaveTotals* totals_h = nullptr;      // pinned + mapped
    czb::WaveTotals* totals_h_dev = nullptr;  // device alias of totals_h
    // per-wave scratch, double-buffered: the entropy stage of wave w+1 overlaps sequence execution of wave w
    DevBuf<czb::WaveCounters> counters[2];
    DevBuf<czb::BlockDesc> blocks[2];
    DevBuf<uint32_t> huf_items[2], fse_items[2], huf_cls0[2], huf_cls1[2], exec_order[2];
    DevBuf<czb::HufRec> huf_recs[2];
    DevBuf<uint8_t> huf_big;    // FseBigScratch: Huffman-weight FSE tables with accuracy log 10..20
    DevBuf<uint8_t> lit[2];
    DevBuf<czb::Seq> seq[2];
    // verify calls: the caller's descs with dst / dst_cap of the output scratch (k_place_outputs), the output scratch itself
    // (double-buffered like the rest), and the placement's per-frame sizes, per-CTA sums and used end
    DevBuf<czb_frame_desc> vdescs;
    DevBuf<uint8_t> out[2];
    DevBuf<unsigned long long> out_ctl[2], out_sizes, out_cta;
    cudaStream_t exec_stream = nullptr;
    cudaEvent_t ev_entropy[2] = {nullptr, nullptr}, ev_exec[2] = {nullptr, nullptr}, ev_fork = nullptr;
    cudaEvent_t ev_scratch_free = nullptr;  // recorded at the end of every batch call: the next call (any stream) waits on it
    bool scratch_in_use = false;
    int sm_count = 148;
    int last_set = 0;
    bool no_overlap = false;
    int big_cls = 19;           // frames of >= 2^big_cls compressed bytes are executed by one CTA each (k_exec_big); 32 = never
    int big_seq_bytes = 16;     // ... if they have at least this many compressed bytes per sequence (sparse sequences)
    int share_cls = 15;         // ... or, from 2^share_cls compressed bytes on, if they hold at least 1/big_share of their wave's
    int big_resident = 1036;    //     (with more frames than resident CTAs in the wave: and at least 1.5x the mean frame)
    int big_share = 8192;       //     compressed bytes: one warp would still be on such a frame when the others have finished
    bool guard = false;         // CZB_GUARD=1: guard zones behind the used part of the scratch buffers, checked after every wave
    bool guard_zeroed = false;
    DevBuf<unsigned long long> guard_faults;
    uint64_t flow_max = 296;    // k_exec_flow takes a wave's large frames only if there are at most this many (else k_exec_big)
    bool flow_wide_forced = false;  // with CZB_BIG_SEQ_BYTES=0 (tests): force the 32-warp shape of k_exec_flow
    bool big_flow = true;       // CTA-per-frame executor: k_exec_flow (data-flow order) or k_exec_big (in-order commit)
    cudaStream_t big_stream = nullptr;  // k_exec_big runs beside k_exec (its CTAs are latency bound and leave most issue slots free)
    cudaEvent_t ev_big_fork = nullptr, ev_big_join = nullptr;

    // staging for the host-pointer entry points
    static constexpr int kHostSlots = 3;  // staging slots of the packed host path
    DevBuf<uint8_t> h_src[kHostSlots], h_dst[kHostSlots];
    DevBuf<czb_frame_desc> h_descs;
    DevBuf<czb_frame_result> h_results;
    uint8_t* pin_a = nullptr; uint64_t pin_a_cap = 0;
    uint8_t* pin_b = nullptr; uint64_t pin_b_cap = 0;
    cudaStream_t copy_in = nullptr, copy_out = nullptr, compute = nullptr;
    cudaEvent_t ev_in[kHostSlots] = {}, ev_dec[kHostSlots] = {}, ev_out[kHostSlots] = {};  // packed host path pipeline

    // per-kernel profiling
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct ProfRec { int cls; size_t e0, e1; };
    std::vector<ProfRec> prof;

    // debug taps
    czb::WaveTotals last_wave{};
    uint64_t last_wave_first = 0, last_wave_count = 0;
};

// internal (czb_handle.cu): the batch entry point with per-frame resume points
int czb_decode_batch_device_resume(czb_context* ctx, const czb_frame_desc* descs, czb_frame_result* results, uint64_t n, uint32_t flags,
                                   void* stream, const czb::FrameResume* resume);
