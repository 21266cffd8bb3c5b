// The sweep's host-built program (clane_plan_create) and the constants k_sweep_rows decodes it with.
#pragma once
#include <stdint.h>

namespace clane {

// One warp's work: a span (consecutive ordinary rows of one row group) or a hub segment.  Two int4; a span only
// needs the first.
struct SweepTask {
    int32_t e_first;      // first edge of the task's contiguous edge stream
    int32_t e_total;      // edges in the stream
    int32_t r0;           // span: first row.  segment: its first 8-block within the hub row
    int32_t flags;        // rows in span (bits 0-7) | direct << 8 | segment << 9 | hub row index << 10 (segment)
    int32_t nb;           // segment: its 8-blocks
    int32_t blk_base;     // segment: first block of the hub row in the hub scratch
    int32_t nblk_row;     // segment: 8-blocks of the hub row
    int32_t reserved;
};
static_assert(sizeof(SweepTask) == 32, "two int4 per task");

constexpr int kTaskDirect = 1 << 8;
constexpr int kTaskSegment = 1 << 9;
constexpr int kTaskHubShift = 10;

constexpr int kMaxPeers = 15;                  // remote ranks of a row-partitioned run (one NVLink domain)
constexpr int kLongBlocks = 2048;              // hub rows of >= 16384 neighbours take the heavy chain kernel
constexpr int kSegEdges = 128;                 // neighbours per hub segment task (16 blocks)
constexpr int kMetaRing = 128;                 // (offset, w) pairs of a warp's window

}  // namespace clane
