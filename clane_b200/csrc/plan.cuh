// clane_plan: device-side schedule + scratch of one (graph shape, row range).  See clane_b200.h.
#pragma once
#include <vector>

#include "common.cuh"

struct clane_plan {
    int32_t n = 0, d = 0, ld = 0;
    int64_t e = 0;
    int32_t row_lo = 0, row_hi = 0;
    int64_t edge_lo = 0, edge_hi = 0;   // rowptr[row_lo], rowptr[row_hi]
    int32_t hub_threshold = 1024;
    bool has_schedule = false;
    int32_t G = 8;              // rows per group
    int32_t nslab = 1;
    int32_t fuse = 0;           // L1 change fused into the sweep (d in {32, 64, 128}, whole graph)
    int32_t n_groups = 0;       // groups covering [row_lo, row_hi)
    int32_t span_edges = 128;   // edge budget of a span
    int32_t n_spans = 0, n_fix_groups = 0, n_hub_rows = 0;
    int32_t n_long_hub_rows = 0;   // the first n_long_hub_rows hub rows (degree-descending) have >= kLongBlocks blocks
    // the sweep's schedule (sweep.cuh): tasks sorted by work descending (hub segments first)
    void* d_tasks = nullptr;           // SweepTask[n_tasks]
    int32_t n_tasks = 0;
    int32_t* d_fix_groups = nullptr;   // fused mode: groups whose chunk partial is recomputed from memory
    int32_t* d_hub_rows = nullptr;     // rows of degree > hub_threshold, degree-descending
    int32_t* d_long_rows = nullptr;    // rows of >= 64 neighbours (row softmax: one CTA each)
    int32_t n_long_rows = 0;
    void* d_hub_info = nullptr;        // int4 per hub row: {row, first edge, degree, first scratch block}
    int64_t hub_blocks = 0;            // 8-neighbour blocks of all hub rows
    int32_t limit = 0, ntail4 = 0, nslab32b = 0;   // 16*floor(d/16); float4 pieces beyond it; 32-column slabs below it
    void* d_hubS = nullptr;            // float4[hub_blocks][ld]  {z6, z4, X, Y}
    void* d_hubT = nullptr;            // float4[hub_blocks * 8][ntail4]  raw z, sequential-regime columns
    int32_t n_seg_tasks = 0;           // the first n_seg_tasks tasks are hub segments (launched on `side`)
    // plan-owned streams: hub segments + long-row chains | short-row chains | the exact-L1 tail of a sweep.  Forked from
    // and joined to the caller's stream with events of `evs` (a pool: a multi-sweep enqueue needs a few per sweep)
    cudaStream_t side = nullptr, side2 = nullptr, tail = nullptr;
    int prio_hi = 0, prio_lo = 0;      // kernel priorities: hub / tail work beside the span tasks goes first
    std::vector<cudaEvent_t> evs;
    // row-partitioned run: peer Znext buffers for the two Z ping-pong buffers (entry self = own buffer)
    int32_t n_peers = 0, self_rank = 0;
    float* peers[3][16] = {};            // per Z buffer (two, or three when the caller rotates three): every rank's address
    float* mc[3] = {nullptr, nullptr, nullptr};   // multicast (NVLS) addresses of the two buffers, or null
    int32_t* d_coloff = nullptr;       // col[e] * ld / 4 as uint32 bits, rebuilt when the caller's column array changes
    const int32_t* coloff_src = nullptr;
    // CUDA-graph cache of enqueued sweep batches (all streams, all kernels): a propagate() call cycles through a few
    // argument sets (Z buffer rotation), so a handful of entries suffice; anything else evicts the oldest.
    struct SweepGraph {
        const void* key[12] = {nullptr};
        float gamma = 0.0f;
        int log_cap = 0, n_sweeps = 0, nz = 0, c0 = 0, loop = 0;
        cudaGraphExec_t exec = nullptr;
        unsigned long long last_use = 0;
    } graphs[6];
    unsigned long long graph_clock = 0;
    bool use_graphs = true;
    bool while_ok = true;              // conditional-WHILE graphs available (cleared when their creation fails once)
    bool profile = false;              // record timing events around the kernels of each sweep
    cudaEvent_t ev_prof[8] = {};
    unsigned prof_mask = 0;            // which of them the last profiled sweep recorded
    unsigned long long* d_trace = nullptr;   // measurement aid: [kTraceSweeps][kTraceSlots][2] globaltimer stamps
    float* d_P0 = nullptr;      // [2][n_groups + 1][32]   (fused only; one copy per sweep parity)
    size_t p0_stride = 0;       // floats per copy
    // cascade scratch: level-1 slots and level-2 slots, sized for max(n*d x1, e*d x2)
    float* d_p1 = nullptr;
    float* d_p2 = nullptr;
    size_t p1_floats = 0, p2_floats = 0;
};

constexpr int kTraceSweeps = 64, kTraceSlots = 6;   // slots: segments, long chains, short chains, spans, L1 tail, -

extern "C" int clane_internal_prepare_kernels(void);
extern "C" int clane_internal_sweeps_direct(clane_plan* plan, const float* d_X, float* const* d_Z3, int32_t cur,
                                            const int32_t* d_rowptr, const int32_t* d_col, const float* d_w, float gamma,
                                            int32_t n_sweeps, clane_patience* d_state, float* d_amounts_log, int32_t log_cap,
                                            clane_stream_t s);
