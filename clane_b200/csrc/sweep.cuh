// Jacobi sweep of Embedder.propagate (/root/reference/clane/embedder.py:84-94) for sm_100a.
//
//   z_v <- fl(x_v + fl(gamma * (w_v[1,k] @ Zcur[nbrs(v)][k,d])))        for every row with k > 0
//
// with the [1,k]x[k,d] product in oneMKL sgemm's summation order (SURVEY 7.1 step 4 /
// Appendix A.1): per output column, neighbours in ascending column id;
//   k < 8 or column >= 16*floor(d/16): sequential fma chain;
//   else per block of 8 neighbours:  a = fma(w6,z6,a); a = fma(w4,z4,a);
//        a += fma(w5,z5, w7*z7);  a += fma(w0,z0, w2*z2) + fma(w1,z1, w3*z3);
//   then the k mod 8 leftovers sequentially.
// A row's neighbours are therefore never split across lanes: parallelism is over columns
// (one float4 of columns per lane) and rows, and memory-level parallelism comes from issuing
// the (address-independent) gathers ahead of the in-order chains.
//
// The graph is static, so the schedule of the sweep is made once per graph on the host (clane_plan_create):
//
//   task      : one warp per (task, 128-column slab).  A span task is a run of consecutive ordinary rows of one
//               row group (<= span_edges edges, or one longer row); a segment task is 128 neighbours (16 blocks)
//               of a hub row.  Tasks are sorted by work, descending ("degree-sorted row blocks").
//   span      : the warp stages the span's (offset, w) pairs in shared memory (one coalesced round trip), takes
//               the degrees from rowptr, and walks the rows in order: per row the X piece, the row's own Zcur
//               piece (fused L1) and <= 8 gathers are issued together as 128-bit loads straight into registers
//               -- lane L loads exactly the float4 it will reduce, so a gathered byte crosses the SM's L1 data
//               path once -- then reduced in the reference's order.  ~3 instructions per neighbour beside the
//               arithmetic; one batch of loads in flight per warp, 32 resident warps per SM (64 registers).
//   hub rows  : the reference's 8-neighbour block is  a = fma(w6,z6,a); a = fma(w4,z4,a); a += X; a += Y
//               with X = fma(w5,z5,w7*z7), Y = fma(w0,z0,w2*z2) + fma(w1,z1,w3*z3) independent of the
//               running sum.  Segment tasks (all SMs, inside k_sweep_rows) gather the neighbours and park
//               {z6, z4, X, Y} per (block, column); k_hub_chain then runs the 4-op chain per block over
//               that contiguous stream (one warp per (hub row, 32 columns), cp.async ring).  Columns in
//               the sequential regime (>= 16*floor(d/16)) are parked raw and chained by one more warp.
#pragma once
#include "common.cuh"
#include "program.cuh"

namespace clane {

struct SweepParams {
    const float* X;
    const float* Zc;
    float* Zn;
    int ld, d, n;
    const int32_t* rowptr;
    const int32_t* coloff;      // col[e] * ld / 4: float4 index of the neighbour's row, read as uint32 (n * ld <= 2^34)
    const float* w;
    float gamma;
    const SweepTask* tasks;     // sorted by work, descending (segments first)
    int n_tasks;
    int row_lo;
    int G;                      // rows per group (<= 32)
    int nslab;                  // 128-column slabs per row
    int fuse;                   // 1: direct spans write one 32-lane |delta| partial per group to P0
    float* P0;
    // hub rows
    const int4* hub_info;       // per hub row (degree-descending): {row, first edge, degree, first scratch block}
    int n_hub_rows;
    int limit;                  // 16 * floor(d / 16): columns below it use the 8-block order
    int ntail4;                 // (ld - limit) / 4: float4 pieces per row in the sequential regime (0..4)
    int nslab32b;               // 32-column slabs below `limit`
    int sld;                    // 32 * nslab32b: columns per block in hubS
    float4* hubS;               // per hub row [32-column slab][block][32] {z6, z4, X, Y}
    float4* hubT;               // per hub row [sequential-regime column][neighbour] raw z (floats)
    int hub_first;              // first hub row of this chain launch
    int task_lo;                // first task of this row-kernel launch (segments and spans are launched separately)
    const clane_patience* st;
    // row-partitioned run: the other ranks' Znext buffers (peer memory over NVLink); every finished row is
    // stored to all of them from inside the kernel, so the exchange overlaps the sweep row by row
    float* peer[kMaxPeers];
    int n_remote;
    float* mc;                  // multicast (NVLS) address of Znext: one store reaches every rank; replaces peer[]
    int bulk;                   // 1 (k_sweep_rows<true>): a span's finished rows are staged in shared memory and leave as one
                                //    bulk store per destination (own Znext + every peer) instead of a store per lane, row and peer
    unsigned long long* trace;  // measurement aid (clane_plan_trace): {first CTA start, last CTA end} in ns, or null
};

// timeline stamps of a kernel: earliest start / latest end over its CTAs (globaltimer, ns)
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void trace_begin(unsigned long long* tr) {
    if (tr != nullptr && threadIdx.x == 0) atomicMin(tr, globaltimer_ns());
}
__device__ __forceinline__ void trace_end(unsigned long long* tr) {
    if (tr != nullptr && threadIdx.x == 0) atomicMax(tr + 1, globaltimer_ns());
}
__global__ void k_trace_stamp(unsigned long long* tr, int end) {
    if (end) atomicMax(tr + 1, globaltimer_ns()); else atomicMin(tr, globaltimer_ns());
}

constexpr int kRowWarps = 2;                   // row kernel: warps (= tasks) per CTA
constexpr int kRowThreads = 32 * kRowWarps;
// resident warps per SM the row kernel is compiled for (register budget: 65536 / (32 * warps) per thread)
constexpr int kRowWarpsPerSM = 24;
// row kernel shared memory per warp: (offset, w) window | two 512-byte transpose buffers (fused L1) | the row's X and
// own Zcur pieces (cp.async) | stream position of a row longer than the window
constexpr size_t kRowWarpSmem = (size_t)kMetaRing * sizeof(int2) + 2 * 512 + 2 * 512 + 16;
constexpr size_t kRowSmemBytes = (size_t)kRowWarps * kRowWarpSmem;

// hub chain kernel: one warp per CTA
// Two variants.  Light (every hub row but the very longest): 8 blocks per cp.async group, 8 groups in flight (32 KB), no
// register double buffer, compiled for 64 registers -- a CTA of 64 x 64 registers is exactly what an SM full of span
// CTAs (12 x 64 threads x 80 registers) still has room for, so the chains run BESIDE the span tasks instead of waiting
// for the machine to drain.  Heavy (rows of >= kLongBlocks blocks, where the chain itself bounds the sweep): 16 blocks
// per group, register double buffer, and a ring of 26 groups = 216 KB: nothing else fits on the SM, which is the point --
// beside 24 span warps a chain warp wins an issue slot only every ~12 cycles instead of every 4 (measured: 9 ns per
// dependent operation), so the few chains that bound a sweep get an SM each to themselves.
constexpr int kHeavyGroup = 16, kHeavyStages = 26;
constexpr int kLightGroup = 8, kLightStages = 8;
__host__ __device__ constexpr size_t chain_smem_bytes(int stages, int group) {
    return (size_t)stages * group * 32 * sizeof(float4) + (size_t)stages * group * sizeof(float2);
}
constexpr size_t kHeavySmemBytes = chain_smem_bytes(kHeavyStages, kHeavyGroup);
constexpr size_t kLightSmemBytes = chain_smem_bytes(kLightStages, kLightGroup);
// sequential-regime chain: neighbours per ring stage (light / heavy) and floats per (stage, column): + 4, so that the
// columns' 128-bit loads spread over the banks.  The heavy chain pays its mbarrier round trip once per 128 neighbours.
constexpr int kLightTailGroup = 32, kHeavyTailGroup = 128;
constexpr int kMaxStages = 128;                // mbarrier pairs per chain CTA
constexpr int kChainThreads = 64;              // producer warp + chain warp
static_assert(kHeavyStages <= kMaxStages && kLightStages <= kMaxStages, "mbarriers");

__device__ __forceinline__ void fma4(float wv, const float4& z, float4& acc) {
    acc.x = ffma(wv, z.x, acc.x); acc.y = ffma(wv, z.y, acc.y);
    acc.z = ffma(wv, z.z, acc.z); acc.w = ffma(wv, z.w, acc.w);
}

__device__ __forceinline__ float blocked8(float a, const float* w, float z0, float z1, float z2, float z3,
                                          float z4, float z5, float z6, float z7) {
    a = ffma(w[6], z6, a);
    a = ffma(w[4], z4, a);
    a = fadd(a, ffma(w[5], z5, fmul(w[7], z7)));
    a = fadd(a, fadd(ffma(w[0], z0, fmul(w[2], z2)), ffma(w[1], z1, fmul(w[3], z3))));
    return a;
}

__device__ __forceinline__ void blocked8x4(float4& acc, const float* ww, const float4* z) {
    acc.x = blocked8(acc.x, ww, z[0].x, z[1].x, z[2].x, z[3].x, z[4].x, z[5].x, z[6].x, z[7].x);
    acc.y = blocked8(acc.y, ww, z[0].y, z[1].y, z[2].y, z[3].y, z[4].y, z[5].y, z[6].y, z[7].y);
    acc.z = blocked8(acc.z, ww, z[0].z, z[1].z, z[2].z, z[3].z, z[4].z, z[5].z, z[6].z, z[7].z);
    acc.w = blocked8(acc.w, ww, z[0].w, z[1].w, z[2].w, z[3].w, z[4].w, z[5].w, z[6].w, z[7].w);
}

// the two sub-trees of an 8-block that do not involve the running sum, parked with z6 and z4
__device__ __forceinline__ float4 park8(const float* w, float z0, float z1, float z2, float z3, float z4,
                                        float z5, float z6, float z7) {
    const float x = ffma(w[5], z5, fmul(w[7], z7));
    const float y = fadd(ffma(w[0], z0, fmul(w[2], z2)), ffma(w[1], z1, fmul(w[3], z3)));
    return make_float4(z6, z4, x, y);
}

__device__ __forceinline__ float4 finish_row(const float4& x, const float4& acc, float gamma) {
    float4 out;
    out.x = fadd(x.x, fmul(gamma, acc.x));
    out.y = fadd(x.y, fmul(gamma, acc.y));
    out.z = fadd(x.z, fmul(gamma, acc.z));
    out.w = fadd(x.w, fmul(gamma, acc.w));
    return out;
}

__device__ __forceinline__ float4 absdiff4(const float4& a, const float4& b) {
    return make_float4(fabsf(fsub(a.x, b.x)), fabsf(fsub(a.y, b.y)), fabsf(fsub(a.z, b.z)), fabsf(fsub(a.w, b.w)));
}

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async16_sa(unsigned smem_addr, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4_sa(unsigned smem_addr, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(gsrc) : "memory");
}
// one store, replicated by the NVSwitch into every rank's buffer (multicast mapping of symmetric memory)
__device__ __forceinline__ void multimem_st4(float* mc, const float4& v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
                 :: "l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void multimem_st1(float* mc, float v) {
    asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" :: "l"(mc), "f"(v) : "memory");
}

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// mbarriers of the hub chain's producer / consumer ring
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// arrive on `bar` once all cp.async issued so far by this thread have landed
__device__ __forceinline__ void cp_async_arrive(unsigned long long* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred done;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 done, [%0], %1;\n\t"
        "@!done bra WAIT_%=;\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Predicated loads in straight-line code (a load under a branch makes ptxas wait for it at the join).
__device__ __forceinline__ void ldg_i32_if(int& v, const int* p, bool pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.b32 %0, [%1];\n\t}"
                 : "+r"(v) : "l"(p), "r"((int)pred));
}
__device__ __forceinline__ void ldg_f32_if(float& v, const float* p, bool pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.f32 %0, [%1];\n\t}"
                 : "+f"(v) : "l"(p), "r"((int)pred));
}

// L2 cache-policy hints (evict_last on the Zcur gathers, evict_first on X / Znext) were measured in round 1: the
// sector hit rate stays at 44 % either way and the policy descriptors cost 8 % more instructions (R2UR / UMOV),
// so plain accesses are used; Znext is written with the streaming (.cs) qualifier.
// neighbour row piece of this lane: 16 bytes at float4 index `off16` of the lane's column base
// (an unsigned index: the address is a 32-bit unsigned multiply-add, IMAD.WIDE.U32)
__device__ __forceinline__ float4 gather4(const float4* __restrict__ zb, int off16) {
    return __ldg(zb + (unsigned)off16);
}
__device__ __forceinline__ float4 ldg_stream4(const float* p) {   // X: read once per sweep, keep it out of L1
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// the gathers of one batch: 128-bit loads straight into registers (lane L loads exactly the float4 of columns it
// will reduce)
template <int M>
__device__ __forceinline__ void load_batch(float4 (&buf)[8], const int2* __restrict__ mp, const float4* __restrict__ zb) {
#pragma unroll
    for (int i = 0; i < M; ++i) buf[i] = gather4(zb, mp[i].x);
}

// <= 7 neighbours in the sequential order (a row shorter than 8, or the k mod 8 leftovers of a longer one):
// (offset, w) pairs out of shared memory, M independent 128-bit gathers, then the fma chain
template <int M>
__device__ __forceinline__ void seq_batch(const int2* __restrict__ mp, const float4* __restrict__ zb, float4& acc) {
    int2 m[M];
    float4 z[M];
#pragma unroll
    for (int i = 0; i < M; ++i) m[i] = mp[i];
#pragma unroll
    for (int i = 0; i < M; ++i) z[i] = gather4(zb, m[i].x);
#pragma unroll
    for (int i = 0; i < M; ++i) fma4(__int_as_float(m[i].y), z[i], acc);
}

// one full 8-block of a row with k >= 8.  kUniform: every lane of the warp is in the 8-block regime (d % 16 == 0),
// so the choice is a uniform branch; otherwise lanes at or beyond `limit` run the sequential chain.
__device__ __forceinline__ void block_batch(const int2* __restrict__ mp, const float4* __restrict__ zb, float4& acc,
                                            bool all_blocked, bool col_blocked) {
    int2 m[8];
    float4 z[8];
    float w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) m[i] = mp[i];
#pragma unroll
    for (int i = 0; i < 8; ++i) z[i] = gather4(zb, m[i].x);
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = __int_as_float(m[i].y);
    if (all_blocked || col_blocked) {
        blocked8x4(acc, w, z);
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) fma4(w[i], z[i], acc);
    }
}

// ------------------------------------------------------------------------------------------
// row kernel: one warp per (task, 128-column slab)
// ------------------------------------------------------------------------------------------
// Row-partitioned runs with whole rows per warp (ld <= 128): the rows of a span are contiguous in every Znext copy, so the
// warp parks them in shared memory and one lane per destination hands [first row, last row] to the bulk-copy engine.
// The stores leave the SM as full 128-byte lines (a 400-byte row of the products shape starts on a 16-byte boundary:
// stored lane by lane, every row ends in partial sectors on NVLink) and cost one instruction per destination and span
// instead of one per destination and row.
constexpr int kStageRows = 8;                                   // rows of a span in a partitioned run (G = 8)
constexpr size_t kRowStageBytes = (size_t)kStageRows * 128 * sizeof(float);   // per warp, dynamic shared memory
__device__ __forceinline__ void bulk_store(float* dst, const float* src_smem, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// rows [ra, rb) of the span starting at row r0 are parked at stage + r * ld: lane 0 stores them to Znext, lane j to peer j - 1
__device__ __forceinline__ void flush_rows(const SweepParams& p, const float* stage, int r0, int ra, int rb, int lane) {
    fence_async_smem();                        // the lanes' generic-proxy writes, before the async proxy reads them
    __syncwarp();
    float* dst = p.Zn;
#pragma unroll
    for (int j = 0; j < kMaxPeers; ++j)
        if (lane == j + 1) dst = p.peer[j];
    if (lane <= p.n_remote) {
        bulk_store(dst + (size_t)(r0 + ra) * p.ld, stage + ra * p.ld, (unsigned)((rb - ra) * p.ld) * 4u);
        bulk_commit();
    }
}

// (offset, w) pairs of up to kMetaRing consecutive edges of the task's stream, starting at edge `e0` (cnt left)
// -> the warp's shared-memory window.  Four predicated, independent load pairs per lane: one round trip.
__device__ __forceinline__ void stage_meta(const SweepParams& p, int e0, int cnt, int lane, int2* meta) {
    const int* __restrict__ offp = p.coloff + e0;
    const float* __restrict__ wp = p.w + e0;
    int c[kMetaRing / 32];
    float w[kMetaRing / 32];
#pragma unroll
    for (int q = 0; q < kMetaRing / 32; ++q) {
        c[q] = 0; w[q] = 0.0f;
        const int i = q * 32 + lane;
        ldg_i32_if(c[q], offp + i, i < cnt);
        ldg_f32_if(w[q], wp + i, i < cnt);
    }
#pragma unroll
    for (int q = 0; q < kMetaRing / 32; ++q) meta[q * 32 + lane] = make_int2(c[q], __float_as_int(w[q]));
    __syncwarp();
}
// the next window of a row longer than kMetaRing (a span of its own): the stream position lives in shared memory,
// not in registers the common path would have to carry
__device__ __noinline__ void restage_meta(const SweepParams& p, int lane, int2* meta, int* state) {
    __syncwarp();                              // every lane has read the old window
    const int e0 = state[0] + kMetaRing, left = state[1] - kMetaRing;
    __syncwarp();
    if (lane == 0) { state[0] = e0; state[1] = left; }
    stage_meta(p, e0, left, lane, meta);
}

// Span task: a run of consecutive ordinary rows of one row group (a whole group when `direct`), one row at a time:
// the row's X piece, its own Zcur piece (fused L1) and <= 8 gathers are issued together and reduced in the
// reference's order -- one memory round trip per 8 neighbours.  No descriptors: the degrees come from rowptr (lane r
// holds the degree of row r0 + r, r < nrows <= 32), the edges from the staged window.  The gathers are 128-bit
// loads straight into registers; X and the own piece go through cp.async into 1 KB of the warp's shared memory, so
// that the 8 registers they would occupy while the gathers are in flight are free: the kernel fits 64 registers = 32
// resident warps per SM, each with one batch of loads in flight (tools/l1pf_probe.cu: resident warps beat deeper
// per-warp pipelines on this access pattern).
template <bool kBulk>
__device__ __forceinline__ void run_span(const SweepParams& p, const int4 t0, int slab, int lane, int2* meta, float* scratch,
                                         float4* rowbuf, int* state, float* stage) {
    const int r0 = t0.z, nrows = t0.w & 0xff;
    const bool direct = (t0.w & kTaskDirect) != 0 && p.fuse != 0;
    const int c0 = slab * 128 + lane * 4;
    const bool active = c0 < p.ld;
    const int cc = active ? c0 : 0;            // idle lanes shadow lane 0 (same sectors: no extra traffic)
    const bool col_blocked = cc < p.limit;
    const bool all_blocked = p.limit == p.ld;  // uniform
    // lane r: the degree of row r0 + r from its own pair of rowptr entries (same line).  A span has up to 32 rows, so
    // lane 31 has no lane 32 to take its row's end from; lanes past the span read rowptr[r0 + nrows] twice (degree 0)
    const int rp = __ldg(p.rowptr + r0 + min(lane, nrows));
    const int rp_next = __ldg(p.rowptr + r0 + min(lane + 1, nrows));
    if (lane == 0) { state[0] = t0.x; state[1] = t0.y; }
    stage_meta(p, t0.x, t0.y, lane, meta);
    const int deg = rp_next - rp;
    const float4* zb = reinterpret_cast<const float4*>(p.Zc + cc);
    const unsigned rowbuf_sa = smem_u32(rowbuf + lane);
    const int nseg = p.d >> 5;
    int mpos = 0;                              // position inside the window
    float chunk_acc = 0.0f;
    const int slab_bytes = min(128, p.ld - slab * 128) * 4;
    // the rows' X and own Zcur pieces, known in advance: request the span's lines now
    if (p.nslab == 1) {                        // consecutive rows are contiguous: one line per lane
        const int bytes = nrows * p.ld * 4, o = lane * 128;
        if (o < bytes) {
            prefetch_l2(reinterpret_cast<const char*>(p.X + (size_t)r0 * p.ld) + o);
            if (direct) prefetch_l2(reinterpret_cast<const char*>(p.Zc + (size_t)r0 * p.ld) + o);
        }
    } else if ((lane >> 2) < nrows && (lane & 3) * 128 < slab_bytes) {
        const size_t o = ((size_t)(r0 + (lane >> 2)) * p.ld + slab * 128) * 4 + (lane & 3) * 128;
        prefetch_l2(reinterpret_cast<const char*>(p.X) + o);
    }
    int run0 = -1;                             // bulk mode: first row of the run of finished rows parked in `stage`
    for (int r = 0; r < nrows; ++r) {
        int k = __shfl_sync(kFull, deg, r);
        if (k == 0) {                          // a sink inside the span: never updated (embedder.py:88-89), |delta| = +0
            if (kBulk && run0 >= 0) { flush_rows(p, stage, r0, run0, r, lane); run0 = -1; }
            continue;
        }
        // float4 index of the lane's piece of the row: 32 bits unsigned (n * ld <= 2^34, clane_plan_create), so the
        // addresses below are IMAD.WIDE.U32 of one 32-bit register, as the gathers'
        const unsigned row4 = (unsigned)(r0 + r) * (unsigned)(p.ld >> 2) + (unsigned)(cc >> 2);
        cp_async16_sa(rowbuf_sa, reinterpret_cast<const float4*>(p.X) + row4);
        if (direct) cp_async16_sa(rowbuf_sa + 512, reinterpret_cast<const float4*>(p.Zc) + row4);
        cp_async_commit();
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (; k >= 8; k -= 8) {
            if (mpos == kMetaRing) { restage_meta(p, lane, meta, state); mpos = 0; }
            block_batch(meta + mpos, zb, acc, all_blocked, col_blocked);
            mpos += 8;
        }
        if (k != 0) {
            if (mpos == kMetaRing) { restage_meta(p, lane, meta, state); mpos = 0; }
            const int2* mp = meta + mpos;
            switch (k) {
                case 1: seq_batch<1>(mp, zb, acc); break;
                case 2: seq_batch<2>(mp, zb, acc); break;
                case 3: seq_batch<3>(mp, zb, acc); break;
                case 4: seq_batch<4>(mp, zb, acc); break;
                case 5: seq_batch<5>(mp, zb, acc); break;
                case 6: seq_batch<6>(mp, zb, acc); break;
                default: seq_batch<7>(mp, zb, acc); break;
            }
            mpos += k;
        }
        cp_async_wait<0>();                    // each lane reads back the 16 bytes it copied itself: no barrier
        const float4 out = finish_row(rowbuf[lane], acc, p.gamma);
        if (kBulk) {
            if (active) *reinterpret_cast<float4*>(stage + r * p.ld + cc) = out;
            if (run0 < 0) run0 = r;
        } else if (active) {
            st_stream4(reinterpret_cast<float*>(reinterpret_cast<float4*>(p.Zn) + row4), out);
            if (p.mc != nullptr) multimem_st4(reinterpret_cast<float*>(reinterpret_cast<float4*>(p.mc) + row4), out);
            for (int j = 0; j < p.n_remote; ++j) reinterpret_cast<float4*>(p.peer[j])[row4] = out;
        }
        if (direct) {
            // the row is d / 32 consecutive cascade rows: transpose the float4-per-lane |delta| through 512 bytes of
            // shared memory (two buffers, alternating: the next row's barrier orders this row's reads before the
            // buffer's next use) and add them to the chunk accumulator in order
            const float4 dl = active ? absdiff4(out, rowbuf[32 + lane]) : make_float4(0.f, 0.f, 0.f, 0.f);
            float* sc = scratch + (r & 1) * 128;
            reinterpret_cast<float4*>(sc)[lane] = dl;
            __syncwarp();
#pragma unroll
            for (int seg = 0; seg < 4; ++seg)
                if (seg < nseg) chunk_acc = fadd(chunk_acc, sc[seg * 32 + lane]);
        }
    }
    // the span is one whole level-0 chunk: its rows were added in order, skipped rows count +0
    if (direct) p.P0[(size_t)((r0 - p.row_lo) / p.G) * 32 + lane] = chunk_acc;
    if (kBulk) {
        if (run0 >= 0) flush_rows(p, stage, r0, run0, nrows, lane);
        bulk_wait_read();                      // the copy engine has read the parked rows: the CTA may give up its shared memory
    }
}

// hub segment task: up to 16 full 8-blocks of one hub row; park {z6, z4, X, Y} per (block, column), or the
// raw z in the sequential regime, for k_hub_chain
__device__ __forceinline__ void run_segment(const SweepParams& p, const int4 t0, const int4 t1, int slab, int lane,
                                            int2* meta) {
    // t0 = {first edge, edges, first 8-block within the hub row, flags}; t1 = {blocks, first scratch block of the row,
    // 8-blocks of the row, -}
    const int c0 = slab * 128 + lane * 4;
    const bool active = c0 < p.ld, col_blocked = c0 < p.limit;
    const int cc = active ? c0 : 0;
    const float4* zb = reinterpret_cast<const float4*>(p.Zc + cc);
    const int nb = t1.x, b_first = t0.z, nblk_row = t1.z;
    const size_t B0 = (size_t)t1.y;
    // lane's four columns c0..c0+3 sit in 32-column slab c0 / 32 of the row's scratch: [slab][block][32]
    float4* sdst = p.hubS + B0 * p.sld + ((size_t)(cc >> 5) * nblk_row + b_first) * 32 + (cc & 31);
    // sequential-regime scratch of the row: [column][8 * nblk_row] floats; this lane's first column, this segment
    float* tdst = reinterpret_cast<float*>(p.hubT) + B0 * 32 * p.ntail4 +
                  (size_t)(col_blocked ? 0 : cc - p.limit) * nblk_row * 8 + (size_t)b_first * 8;
    const int* __restrict__ offp = p.coloff + t0.x;
    const float* __restrict__ wp = p.w + t0.x;
    // a segment is at most 128 edges: the whole (offset, w) stream fits the ring
    const int slab_bytes = min(128, p.ld - slab * 128) * 4;
    for (int i = lane; i < t0.y; i += 32) {
        const int off16 = __ldg(offp + i);
        meta[i] = make_int2(off16, __float_as_int(__ldg(wp + i)));
        if (i >= 16) {   // the first two blocks are loaded right away
            const char* a = reinterpret_cast<const char*>(reinterpret_cast<const float4*>(p.Zc + slab * 128) + (unsigned)off16);
            prefetch_l2(a);
            if (slab_bytes > 128) prefetch_l2(a + 128);
            if (slab_bytes > 256) prefetch_l2(a + 256);
            if (slab_bytes > 384) prefetch_l2(a + 384);
        }
    }
    __syncwarp();
    float4 A[8];
    for (int cb = 0; cb < nb; ++cb) {
        load_batch<8>(A, meta + cb * 8, zb);
        const int2* mp = meta + cb * 8;
        float w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = __int_as_float(mp[i].y);
        if (active) {
            if (col_blocked) {
                float4* o = sdst + (size_t)cb * 32;
                o[0] = park8(w, A[0].x, A[1].x, A[2].x, A[3].x, A[4].x, A[5].x, A[6].x, A[7].x);   // kept in L2 for the chain
                o[1] = park8(w, A[0].y, A[1].y, A[2].y, A[3].y, A[4].y, A[5].y, A[6].y, A[7].y);   // kept in L2 for the chain
                o[2] = park8(w, A[0].z, A[1].z, A[2].z, A[3].z, A[4].z, A[5].z, A[6].z, A[7].z);   // kept in L2 for the chain
                o[3] = park8(w, A[0].w, A[1].w, A[2].w, A[3].w, A[4].w, A[5].w, A[6].w, A[7].w);   // kept in L2 for the chain
            } else {
                // sequential regime: every column's values contiguous over the row's neighbours
                float* o = tdst + (size_t)cb * 8;
                const size_t cp = (size_t)nblk_row * 8;
                *reinterpret_cast<float4*>(o) = make_float4(A[0].x, A[1].x, A[2].x, A[3].x);
                *reinterpret_cast<float4*>(o + 4) = make_float4(A[4].x, A[5].x, A[6].x, A[7].x);
                *reinterpret_cast<float4*>(o + cp) = make_float4(A[0].y, A[1].y, A[2].y, A[3].y);
                *reinterpret_cast<float4*>(o + cp + 4) = make_float4(A[4].y, A[5].y, A[6].y, A[7].y);
                *reinterpret_cast<float4*>(o + 2 * cp) = make_float4(A[0].z, A[1].z, A[2].z, A[3].z);
                *reinterpret_cast<float4*>(o + 2 * cp + 4) = make_float4(A[4].z, A[5].z, A[6].z, A[7].z);
                *reinterpret_cast<float4*>(o + 3 * cp) = make_float4(A[0].w, A[1].w, A[2].w, A[3].w);
                *reinterpret_cast<float4*>(o + 3 * cp + 4) = make_float4(A[4].w, A[5].w, A[6].w, A[7].w);
            }
        }
    }
}

template <bool kBulk>
__global__ void __launch_bounds__(kRowThreads, kRowWarpsPerSM / kRowWarps) k_sweep_rows(SweepParams p) {
    __shared__ __align__(16) unsigned char smem[kRowSmemBytes];
    extern __shared__ __align__(128) unsigned char stage_smem[];     // kRowWarps * kRowStageBytes when p.bulk, else none
    if (p.st != nullptr && p.st->stop) return;
    trace_begin(p.trace);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* mine = smem + (size_t)warp * kRowWarpSmem;
    int2* meta = reinterpret_cast<int2*>(mine);
    float* scratch = reinterpret_cast<float*>(meta + kMetaRing);
    float4* rowbuf = reinterpret_cast<float4*>(scratch + 256);
    int* state = reinterpret_cast<int*>(rowbuf + 64);
    const int wtask = blockIdx.x * kRowWarps + warp;
    int ti = wtask, slab = 0;
    if (p.nslab > 1) { ti = wtask / p.nslab; slab = wtask - ti * p.nslab; }
    ti += p.task_lo;
    if (ti < p.n_tasks) {
        const int4 t0 = __ldg(reinterpret_cast<const int4*>(p.tasks + ti));
        if (t0.w & kTaskSegment) run_segment(p, t0, __ldg(reinterpret_cast<const int4*>(p.tasks + ti) + 1), slab, lane, meta);
        else run_span<kBulk>(p, t0, slab, lane, meta, scratch, rowbuf, state,
                      reinterpret_cast<float*>(stage_smem + (size_t)warp * kRowStageBytes));
    }
    if (p.trace != nullptr) { __syncthreads(); trace_end(p.trace); }
}

// ------------------------------------------------------------------------------------------
// hub chain: one warp per (hub row, 32 columns below `limit`), plus one warp per hub row for the
// sequential-regime columns.  Runs after k_sweep_rows (same stream).
// ------------------------------------------------------------------------------------------
// CTA = two warps: warp 1 copies the row's parked stream into a shared-memory ring (cp.async, completion
// signalled on "full" mbarriers), warp 0 runs the in-order chain out of the ring and hands the stages back
// ("empty" mbarriers) -- the chain warp issues nothing but the loads and the dependent operations of the chain.
//   slab s < nslab32b : 32 columns in the 8-block order, lane = column;  per block {z6, z4, X, Y} + {w4, w6}
//   slab s = nslab32b : the <= 16 sequential-regime columns, lane = column; per neighbour z (transposed by the
//                       segment warps: every column's values are contiguous) + w
// Launched on the plan's side stream right after the segment tasks (a launch of k_sweep_rows over the segment part
// of the task list, same stream): ordinary stream order, no flags, no waiting inside the kernel.  The span tasks
// run on the caller's stream at the same time, so the chains cost the sweep nothing unless a hub row is long
// enough to outlast all ordinary rows.
// kLight: short rows -- 4-stage ring, no register double buffer.  !kLight: long rows (>= kLongBlocks blocks) --
//         12 stages, the chain never waits for the ring.
template <bool kLight>
__global__ void __launch_bounds__(kChainThreads, kLight ? 16 : 1) k_hub_chain(SweepParams p) {
    constexpr int kStages = kLight ? kLightStages : kHeavyStages;
    constexpr int kChainGroup = kLight ? kLightGroup : kHeavyGroup;
    constexpr int kTailGroup = kLight ? kLightTailGroup : kHeavyTailGroup;
    constexpr int kTailPitch = kTailGroup + 4;
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ unsigned long long full[kMaxStages], empty[kMaxStages];
    __shared__ int stop;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int per = p.nslab32b + (p.ntail4 > 0 ? 1 : 0);
    const int hr = p.hub_first + blockIdx.x / per, s = blockIdx.x % per;
    const int4 info = __ldg(p.hub_info + hr);
    const int row = info.x, a = info.y, k = info.z;
    const int nblk = k >> 3;
    const size_t B0 = (size_t)info.w;
    const int nleft = k - nblk * 8;
    if (threadIdx.x == 0) {
        // one read of the flag for the whole CTA: the tail of the previous sweep may set it while this (speculative)
        // sweep runs, and a producer warp that returned while the chain warp went on would leave it waiting forever
        stop = p.st != nullptr && p.st->stop;
#pragma unroll
        for (int i = 0; i < kMaxStages; ++i) { mbar_init(full + i, 32); mbar_init(empty + i, 1); }   // (unrolled: ~0.3 us)
        fence_mbar_init();
    }
    __syncthreads();
    if (stop) return;
    trace_begin(p.trace);
    const bool blocked = s < p.nslab32b;
    const int nt = p.ntail4, ntc = p.ld - p.limit;                  // sequential-regime float4 pieces / columns
    const int nnb = nblk * 8;
    const int ngroups = blocked ? (nblk + kChainGroup - 1) / kChainGroup : (nnb + kTailGroup - 1) / kTailGroup;
    float4* ringS = reinterpret_cast<float4*>(smem);                                  // blocked: [stage][16][32]
    float2* wq = reinterpret_cast<float2*>(ringS + kStages * kChainGroup * 32);       //          [stage][16]
    // sequential regime: stage = [ntc columns][kTailPitch] z | [32] w; as many stages as the shared memory holds
    float* zr = reinterpret_cast<float*>(smem);
    const int tstride = ntc * kTailPitch + kTailGroup;
    const int tstages = min(kMaxStages, (int)(chain_smem_bytes(kStages, kChainGroup) / sizeof(float)) / max(tstride, 1));

    if (warp == 1) {
        // ---------------- producer ----------------
        if (blocked) {
            const float4* src = p.hubS + B0 * p.sld + (size_t)s * nblk * 32 + lane;   // contiguous 512 B per block
            // {w4, w6} of every block straight from w (constant during a sweep; no scratch copy that another SM's
            // segment warp could be rewriting while this SM's L1 holds a stale sector of it)
            const float* wsrc = p.w + a + 4;
            const unsigned ring_sa = smem_u32(ringS) + lane * 16;
            const unsigned wq_sa = smem_u32(wq) + (lane & 15) * 8;
            for (int g = 0; g < ngroups; ++g) {
                const int st = g % kStages;
                if (g >= kStages) mbar_wait(empty + st, (unsigned)(g / kStages - 1) & 1u);
                const int b0 = g * kChainGroup;
                const unsigned dst = ring_sa + (unsigned)st * (kChainGroup * 512);
#pragma unroll
                for (int j = 0; j < kChainGroup; ++j)
                    if (b0 + j < nblk) cp_async16_sa(dst + j * 512, src + (size_t)(b0 + j) * 32);
                if (lane < kChainGroup && b0 + lane < nblk) {
                    cp_async4_sa(wq_sa + (unsigned)st * (kChainGroup * 8), wsrc + (size_t)(b0 + lane) * 8);
                    cp_async4_sa(wq_sa + (unsigned)st * (kChainGroup * 8) + 4, wsrc + (size_t)(b0 + lane) * 8 + 2);
                }
                cp_async_arrive(full + st);
            }
        } else {
            const float* tsrc = reinterpret_cast<const float*>(p.hubT) + B0 * 32 * nt;   // [column][nnb]
            for (int g = 0; g < ngroups; ++g) {
                const int st = g % tstages;
                if (g >= tstages) mbar_wait(empty + st, (unsigned)(g / tstages - 1) & 1u);
                const int i0 = g * kTailGroup;
                const int cnt = min(kTailGroup, nnb - i0);            // multiple of 8
                // 16-byte pieces: column q / (kTailGroup / 4), neighbours 4 * (q % (kTailGroup / 4)) .. + 3
                constexpr int kPieces = kTailGroup / 4;
                for (int q = lane; q < ntc * kPieces; q += 32) {
                    const int c = q / kPieces, pc = (q % kPieces) * 4;
                    if (pc < cnt)
                        cp_async16_sa(smem_u32(zr + (size_t)st * tstride + c * kTailPitch + pc), tsrc + (size_t)c * nnb + i0 + pc);
                }
                for (int q = lane; q < cnt; q += 32)
                    cp_async4_sa(smem_u32(zr + (size_t)st * tstride + ntc * kTailPitch + q), p.w + a + i0 + q);
                cp_async_arrive(full + st);
            }
        }
        return;
    }

    // ---------------- consumer: the chain ----------------
    float acc = 0.0f;
    const int col = blocked ? s * 32 + lane : p.limit + lane;
    const bool act = blocked ? col < p.limit : col < p.ld;
    const int ccol = act ? col : (blocked ? 0 : p.limit);
    const float xv = __ldg(p.X + (size_t)row * p.ld + ccol);   // needed last, fetched first
    // the k mod 8 leftovers: gathered now, added after the blocks
    float lz[7], lw[7];
#pragma unroll
    for (int o = 0; o < 7; ++o) {
        lz[o] = 0.0f; lw[o] = 0.0f;
        if (o < nleft) {
            lw[o] = __ldg(p.w + a + nnb + o);
            lz[o] = __ldg(p.Zc + (size_t)(unsigned)__ldg(p.coloff + a + nnb + o) * 4 + ccol);
        }
    }
    if (blocked) {
        // ---- 8-block order: a = fma(w6,z6,a); a = fma(w4,z4,a); a += X; a += Y per block ----
        // Register double buffer: the shared-memory loads of stage g + 1 are issued before the 64 dependent
        // operations of stage g, so the chain itself never waits for the ring.
        float4 v[kChainGroup], vn[kChainGroup];
        float2 wv[kChainGroup], wn[kChainGroup];
        auto fetch = [&](int g, float4 (&dv)[kChainGroup], float2 (&dw)[kChainGroup]) {
            const bool live = g < ngroups;   // past the end: no wait, the loads below return stale data nobody uses
            const int st = g % kStages;      //   (they stay unconditional: loads under a branch would be waited for at its join)
            if (live) mbar_wait(full + st, (unsigned)(g / kStages) & 1u);
            const float4* rs = ringS + (size_t)st * kChainGroup * 32 + lane;
            const float2* ws = wq + st * kChainGroup;
#pragma unroll
            for (int j = 0; j < kChainGroup; ++j) { dv[j] = rs[j * 32]; dw[j] = ws[j]; }   // past the row's end: stale, unused
            __syncwarp();                    // every lane has read the stage
            if (live && lane == 0) mbar_arrive(empty + st);
        };
        auto chain = [&](int g, const float4 (&dv)[kChainGroup], const float2 (&dw)[kChainGroup]) {
            const int cnt = min(kChainGroup, nblk - g * kChainGroup);
            if (cnt == kChainGroup) {
#pragma unroll
                for (int j = 0; j < kChainGroup; ++j) {
                    acc = ffma(dw[j].y, dv[j].x, acc);
                    acc = ffma(dw[j].x, dv[j].y, acc);
                    acc = fadd(acc, dv[j].z);
                    acc = fadd(acc, dv[j].w);
                }
            } else {
#pragma unroll
                for (int j = 0; j < kChainGroup; ++j)
                    if (j < cnt) {
                        acc = ffma(dw[j].y, dv[j].x, acc);
                        acc = ffma(dw[j].x, dv[j].y, acc);
                        acc = fadd(acc, dv[j].z);
                        acc = fadd(acc, dv[j].w);
                    }
            }
        };
        if (kLight) {
            for (int g = 0; g < ngroups; ++g) { fetch(g, v, wv); chain(g, v, wv); }
        } else {
            fetch(0, v, wv);
            for (int g = 0; g < ngroups; g += 2) {
                fetch(g + 1, vn, wn);
                chain(g, v, wv);
                if (g + 1 >= ngroups) break;
                fetch(g + 2, v, wv);
                chain(g + 1, vn, wn);
            }
        }
    } else {
        // ---- sequential regime: a = fma(w_i, z_i, a) over all neighbours ----
        // One mbarrier round trip per stage; inside a stage, pieces of 32 neighbours go through a register double
        // buffer (the shared-memory loads of piece s + 1 are issued before the 32 dependent fmas of piece s).
        const int cl = min(lane, ntc - 1);
        constexpr int kPiece = 32;
        float4 zv[kPiece / 4], zn[kPiece / 4], wv[kPiece / 4], wn[kPiece / 4];
        auto load_piece = [&](const float* zs, const float* ws, int s0, float4 (&dz)[kPiece / 4], float4 (&dw)[kPiece / 4]) {
#pragma unroll
            for (int j = 0; j < kPiece / 4; ++j) {
                dz[j] = *reinterpret_cast<const float4*>(zs + s0 + 4 * j);     // past the stage's end: stale, unused
                dw[j] = *reinterpret_cast<const float4*>(ws + s0 + 4 * j);
            }
        };
        auto chain_piece = [&](int cnt, const float4 (&dz)[kPiece / 4], const float4 (&dw)[kPiece / 4]) {   // cnt: multiple of 8
#pragma unroll
            for (int j = 0; j < kPiece / 4; ++j)
                if (cnt >= kPiece || 4 * j < cnt) {
                    acc = ffma(dw[j].x, dz[j].x, acc);
                    acc = ffma(dw[j].y, dz[j].y, acc);
                    acc = ffma(dw[j].z, dz[j].z, acc);
                    acc = ffma(dw[j].w, dz[j].w, acc);
                }
        };
        for (int g = 0; g < ngroups; ++g) {
            const int st = g % tstages;
            mbar_wait(full + st, (unsigned)(g / tstages) & 1u);
            const float* zs = zr + (size_t)st * tstride + cl * kTailPitch;
            const float* ws = zr + (size_t)st * tstride + ntc * kTailPitch;
            const int cnt = min(kTailGroup, nnb - g * kTailGroup);           // multiple of 8
            load_piece(zs, ws, 0, zv, wv);
#pragma unroll 1
            for (int s0 = 0; s0 < cnt; s0 += 2 * kPiece) {
                if (kTailGroup > kPiece) load_piece(zs, ws, min(s0 + kPiece, kTailGroup - kPiece), zn, wn);
                chain_piece(cnt - s0, zv, wv);
                if (kTailGroup > kPiece) {
                    if (s0 + kPiece >= cnt) break;
                    load_piece(zs, ws, min(s0 + 2 * kPiece, kTailGroup - kPiece), zv, wv);
                    chain_piece(cnt - s0 - kPiece, zn, wn);
                }
            }
            __syncwarp();                    // every lane has read the stage
            if (lane == 0) mbar_arrive(empty + st);
        }
    }
#pragma unroll
    for (int o = 0; o < 7; ++o)
        if (o < nleft) acc = ffma(lw[o], lz[o], acc);
    if (act) {
        const size_t off = (size_t)row * p.ld + col;
        const float v = fadd(xv, fmul(p.gamma, acc));
        p.Zn[off] = v;
        if (p.mc != nullptr) multimem_st1(p.mc + off, v);
        for (int j = 0; j < p.n_remote; ++j) p.peer[j][off] = v;
    }
    trace_end(p.trace);
}

// Fused mode: the level-0 partial of every group that was not swept by a single warp (it holds
// a hub row or was cut into several spans), recomputed from memory.
__global__ void __launch_bounds__(256)
k_fix_chunks(const float* __restrict__ Zn, const float* __restrict__ Zc, int d, int n, int G,
             const int32_t* __restrict__ fix_groups, int n_fix_groups, float* __restrict__ P0,
             const clane_patience* __restrict__ st) {
    if (st != nullptr && st->stop) return;
    const int lane = threadIdx.x & 31;
    const int i = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (i >= n_fix_groups) return;
    const int g = __ldg(fix_groups + i);
    const int r0 = g * G, nrows = min(G, n - r0);
    const int ncr = nrows * (d >> 5);                   // cascade rows of the chunk (ld == d here)
    const size_t base = (size_t)r0 * d + lane;
    // a chunk is at most 32 cascade rows (G*d <= 1024): fetch them all, then add in order -- one round trip
    float v[32];
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        const size_t t = base + (size_t)r * 32;
        v[r] = (r < ncr) ? fabsf(fsub(__ldcg(Zn + t), __ldg(Zc + t))) : 0.0f;
    }
    float acc = 0.0f;
#pragma unroll
    for (int r = 0; r < 32; ++r)
        if (r < ncr) acc = fadd(acc, v[r]);
    P0[(size_t)g * 32 + lane] = acc;
}

}  // namespace clane
