// libclane_b200.so -- the AsymmertricSimilarity scorer (/root/reference/clane/similarity.py:40-57) as a fused path:
//
//     score(v -> u) = <Phi_src z_v, Phi_dst z_u>        (nn.Linear without bias: Phi z = W z, W = [out, in])
//
// The reference projects the GATHERED rows ([E, d] x [d, d], twice); here every node is projected once,
//     [P_src | P_dst] = Z [N, d] x [W_src ; W_dst]^T [d, 2d]
// -- the one true GEMM on this surface (SURVEY 8f-3) -- on the 5th-generation tensor cores: tcgen05.mma (kind::tf32, fp32
// accumulators in TMEM), operands staged in shared memory by TMA (cp.async.bulk.tensor, 128-byte swizzle), one
// elected thread issuing the MMAs, tcgen05.ld for the epilogue.  The per-edge dot of the projected rows and the row
// softmax are the kernels of the cosine path (k_dots over two matrices, the row softmax without the norm divisor).
//
// Two projection kernels:
//   k_asym_project (d in {32, 64, 96, 128}): the inputs of the MMA are read as TF32 (10-bit mantissa), the accumulation
//     is fp32: each projected value carries a relative error of ~2^-11 of |z| |W row|.  One CTA per 128 rows of Z; the
//     whole K = d <= 128 in shared memory in blocks of 32 floats (= one 128-byte swizzle row), N = 2d <= 256.
//   k_asym_project_fp32 (any d >= 1): 3xTF32, fp32-accurate; K through a ring of 32-float blocks, N in tiles of <= 256.
// This is a TRAINABLE scorer (the reference trains W with Adam), not part of the bit-exact cosine path; the tests state
// each kernel's tolerance.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "clane_b200.h"
#include "common.cuh"

namespace clane {
namespace asym {

constexpr int kTileM = 128;          // rows of Z per CTA = TMEM lanes
constexpr int kBlockK = 32;          // floats per K block: 128 bytes = the swizzle span
constexpr int kUmmaK = 8;            // tf32 elements per tcgen05.mma (32 bytes)
constexpr int kThreads = 128;        // 4 warps: each owns 32 TMEM lanes in the epilogue

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded wait: a wrong byte count or a faulting copy must not hang the device (returns false after ~1 s)
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t spins = 0; spins < (1u << 20); ++spins) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) return true;
    }
    return false;
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// shared-memory matrix descriptor, K-major, 128-byte swizzle: 8-row groups of 128-byte rows, 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    uint64_t desc = 0;
    desc |= (uint64_t)((smem_addr & 0x3ffff) >> 4);          // start address, bits [0, 14)
    desc |= (uint64_t)1 << 16;                               // leading byte offset (unused for swizzled K-major), bits [16, 30)
    desc |= (uint64_t)(1024 >> 4) << 32;                     // stride byte offset between 8-row groups, bits [32, 46)
    desc |= (uint64_t)1 << 46;                               // descriptor version (sm_100)
    desc |= (uint64_t)2 << 61;                               // layout type: SWIZZLE_128B
    return desc;
}
// instruction descriptor: D = f32, A = B = tf32, both K-major, N / 8 at [17, 23), M / 16 at [24, 29)
__host__ __device__ constexpr uint32_t umma_idesc(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct ProjectParams {
    float* Psrc;
    float* Pdst;
    int n, d, ld;        // rows of Z, features, leading dimension of Z / Psrc / Pdst (floats)
    int* error;          // set to 1 when a barrier wait timed out
};

// dynamic shared memory (1024-byte aligned): A [kb][128 rows][128 B] | B [kb][2d rows][128 B]
__global__ void __launch_bounds__(kThreads, 1)
k_asym_project(const __grid_constant__ CUtensorMap map_z, const __grid_constant__ CUtensorMap map_w, ProjectParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t full_bar[4];       // one per K block: its A and B pieces have landed
    __shared__ uint64_t mma_bar;           // the accumulator is complete
    __shared__ uint32_t tmem_base;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb = p.d / kBlockK;                       // K blocks (1..4)
    const int n2 = 2 * p.d;                              // columns of the accumulator
    const uint32_t tmem_cols = n2 <= 64 ? 64 : n2 <= 128 ? 128 : 256;
    uint8_t* sA = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);      // the swizzle atoms want 1024-byte alignment
    uint8_t* sB = sA + (size_t)nkb * kTileM * 128;
    const int row0 = blockIdx.x * kTileM;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(full_bar + i, 1);
        mbar_init(&mma_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {      // one warp allocates the tensor memory columns of the accumulator
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    bool ok = true;

    if (threadIdx.x == 0) {
        // ---- TMA producer: every K block of the Z tile and of the stacked weights, each on its own barrier ----
        for (int kb = 0; kb < nkb; ++kb) {
            mbar_expect_tx(full_bar + kb, (uint32_t)((kTileM + n2) * 128));
            tma_load_2d(sA + (size_t)kb * kTileM * 128, &map_z, kb * kBlockK, row0, full_bar + kb);
            tma_load_2d(sB + (size_t)kb * n2 * 128, &map_w, kb * kBlockK, 0, full_bar + kb);
        }
        // ---- MMA issuer: D[128, 2d] (+)= A[128, 8] x B[2d, 8]^T, four k-steps per K block ----
        const uint32_t idesc = umma_idesc(kTileM, n2);
        for (int kb = 0; kb < nkb && ok; ++kb) {
            ok = mbar_wait(full_bar + kb, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t a0 = smem_u32(sA + (size_t)kb * kTileM * 128), b0 = smem_u32(sB + (size_t)kb * n2 * 128);
            for (int k = 0; k < kBlockK / kUmmaK && ok; ++k) {
                const uint64_t da = umma_desc(a0 + k * kUmmaK * 4), db = umma_desc(b0 + k * kUmmaK * 4);
                const uint32_t accumulate = (kb | k) != 0;
                asm volatile(
                    "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                    ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
            }
        }
        // arrives on mma_bar once every MMA issued above has completed (implies fence::before_thread_sync)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&mma_bar)) : "memory");
    }
    __syncwarp();

    // ---- epilogue: warp w owns TMEM lanes 32w .. 32w + 31 = rows row0 + 32w + lane; 32 columns per tcgen05.ld ----
    // the give-up decision is the CTA's: every lane of a warp must take part in tcgen05.ld.sync.aligned, or none
    ok = __syncthreads_and(mbar_wait(&mma_bar, 0) && ok);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = row0 + warp * 32 + lane;
    if (ok) {
        for (int c0 = 0; c0 < n2; c0 += 32) {
            uint32_t v[32];
            const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                  "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                  "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr) : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (row < p.n) {
                float* dst = (c0 < p.d ? p.Psrc + (size_t)row * p.ld + c0 : p.Pdst + (size_t)row * p.ld + (c0 - p.d));
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(dst + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                                      __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
            }
        }
    } else if (threadIdx.x == 0) {
        *p.error = 1;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
}

// =============================================================================================
// fp32-faithful projection for any d (3xTF32): every operand x = hi + lo, hi = x rounded to TF32 (low 13 mantissa bits
// zero, so exact in TF32), lo = x - hi (exact in fp32, <= 12 significant bits, so reading it as TF32 drops at most
// 2^-23 |x| whether the tensor core truncates or rounds).  D = A_lo B_hi + A_hi B_lo + A_hi B_hi, dropping A_lo B_lo
// (<= 2^-22 |a b|): with the fp32 accumulation of 3d products every value is within (4 + 3d) 2^-23 sum_k |z_k w_k|.
// The tensor cores' fp32 accumulation is biased (a block of products is added to the accumulator without rounding to
// nearest), so the error grows with the number of MMAs that land on one accumulator: the two small cross terms go to a
// second accumulator and only A_hi B_hi to the main one (d / 8 instead of 3d / 8 biased steps on the large values;
// measured: P at arxiv shape 1.24e-5 from fp64 truth with one accumulator); the epilogue adds the two, rounded to nearest.
// =============================================================================================
constexpr int kMaxStages = 4;
constexpr int kMaxTileN = 256;                 // the MMA's largest N at M = 128
constexpr size_t kFp32SmemBudget = 200 * 1024; // dynamic shared memory of k_asym_project_fp32, alignment slack included

__device__ __forceinline__ float tf32_hi(float x) {       // round to nearest (ties away) at 10 mantissa bits
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

// 32 consecutive fp32 columns of the warp's 32 TMEM lanes (lane i: row i of the warp's quarter), waited for
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}

// W_hi / W_lo of the stacked weights [2d, ldw] (pad columns of W are zero, so are theirs)
__global__ void k_asym_split(const float* __restrict__ W, int64_t count, float* __restrict__ Whi, float* __restrict__ Wlo) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const float x = W[i], hi = tf32_hi(x);
    Whi[i] = hi;
    Wlo[i] = __fsub_rn(x, hi);
}

struct ProjectFp32Params {
    float* Psrc;
    float* Pdst;
    int n, d, ld;        // rows of Z, features, leading dimension of Z / Psrc / Pdst (floats)
    int tile_n;          // stacked output columns per CTA: a multiple of 16, <= 256
    int stages;          // depth of the K ring, 2..kMaxStages
    int* error;          // set to 1 when a barrier wait timed out
};

// CTA (x, y): rows [128 x, 128 x + 128) of Z, stacked columns [tile_n y, tile_n y + tile_n) of [P_src | P_dst].
// TMEM: two accumulators of tile_n columns (each rounded up to a power of two, <= 256): A_hi B_hi | A_lo B_hi + A_hi B_lo.
// Stage s of the K ring (dynamic shared memory, 1024-byte aligned):  A_hi [128][128 B] | A_lo | B_hi [tile_n][128 B] | B_lo.
// TMA fills A_hi (the raw Z block), B_hi and B_lo; the 128 threads split A_hi in place and write A_lo at the same swizzled
// offsets (the split is elementwise, the swizzle does not matter); thread 0 then issues 3 x 4 MMAs and, once they have
// drained the stage (tcgen05.commit -> empty barrier), refills it with the K block `stages` further on.
__global__ void __launch_bounds__(kThreads, 1)
k_asym_project_fp32(const __grid_constant__ CUtensorMap map_z, const __grid_constant__ CUtensorMap map_whi,
                    const __grid_constant__ CUtensorMap map_wlo, ProjectFp32Params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t full_bar[kMaxStages];     // the stage's copies have landed
    __shared__ uint64_t empty_bar[kMaxStages];    // the MMAs reading the stage have completed
    __shared__ uint64_t mma_bar;                  // the accumulator is complete
    __shared__ uint32_t tmem_base;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb = (p.d + kBlockK - 1) / kBlockK;       // the last block may be ragged: TMA fills it with zeros
    const int tn = p.tile_n, S = p.stages;
    const uint32_t acc_cols = tn <= 32 ? 32 : tn <= 64 ? 64 : tn <= 128 ? 128 : 256;
    const uint32_t tmem_cols = 2 * acc_cols;
    const size_t a_bytes = (size_t)kTileM * 128, b_bytes = (size_t)tn * 128, stage_bytes = 2 * (a_bytes + b_bytes);
    uint8_t* base = smem + ((1024u - (smem_u32(smem) & 1023u)) & 1023u);
    const int row0 = blockIdx.x * kTileM, n0 = blockIdx.y * tn;

    if (threadIdx.x == 0) {
        for (int i = 0; i < S; ++i) { mbar_init(full_bar + i, 1); mbar_init(empty_bar + i, 1); }
        mbar_init(&mma_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;

    auto load = [&](int kb) {           // thread 0: the Z block and both weight blocks of K block kb into its stage
        uint8_t* st = base + (size_t)(kb % S) * stage_bytes;
        uint64_t* bar = full_bar + kb % S;
        mbar_expect_tx(bar, (uint32_t)(a_bytes + 2 * b_bytes));
        tma_load_2d(st, &map_z, kb * kBlockK, row0, bar);
        tma_load_2d(st + 2 * a_bytes, &map_whi, kb * kBlockK, n0, bar);
        tma_load_2d(st + 2 * a_bytes + b_bytes, &map_wlo, kb * kBlockK, n0, bar);
    };
    if (threadIdx.x == 0)
        for (int kb = 0; kb < S && kb < nkb; ++kb) load(kb);

    bool ok = true;
    const uint32_t idesc = umma_idesc(kTileM, tn);
    for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % S;
        const uint32_t phase = (uint32_t)(kb / S) & 1u;
        uint8_t* st = base + (size_t)s * stage_bytes;
        const bool landed = mbar_wait(full_bar + s, phase);
        if (landed) {
            float4* hi = reinterpret_cast<float4*>(st);
            float4* lo = reinterpret_cast<float4*>(st + a_bytes);
#pragma unroll
            for (int i = threadIdx.x; i < (int)(a_bytes / 16); i += kThreads) {
                const float4 x = hi[i];
                const float4 h = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
                hi[i] = h;
                lo[i] = make_float4(__fsub_rn(x.x, h.x), __fsub_rn(x.y, h.y), __fsub_rn(x.z, h.z), __fsub_rn(x.w, h.w));
            }
        }
        // the split was written by the generic proxy; the tensor cores read through the async proxy
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        ok = __syncthreads_and(ok && landed);
        if (!ok) break;
        if (threadIdx.x == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t ahi = smem_u32(st), alo = ahi + (uint32_t)a_bytes;
            const uint32_t bhi = ahi + 2 * (uint32_t)a_bytes, blo = bhi + (uint32_t)b_bytes;
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                const uint32_t off = k * kUmmaK * 4;
                // the small products first (into the second accumulator), then A_hi B_hi
                const uint32_t pairs[3][2] = {{alo, bhi}, {ahi, blo}, {ahi, bhi}};
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const uint64_t da = umma_desc(pairs[t][0] + off), db = umma_desc(pairs[t][1] + off);
                    const uint32_t accumulate = (kb | k | (t == 1)) != 0;
                    const uint32_t acc = t < 2 ? tmem + acc_cols : tmem;
                    asm volatile(
                        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                        ::"r"(acc), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
                }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(empty_bar + s))
                         : "memory");
            if (kb + S < nkb) {
                ok = mbar_wait(empty_bar + s, phase);      // folded into the next iteration's CTA-wide decision
                if (ok) load(kb + S);
            }
        }
    }
    if (threadIdx.x == 0)      // also after a give-up: the MMAs already issued must finish before TMEM is released
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&mma_bar)) : "memory");
    ok = __syncthreads_and(mbar_wait(&mma_bar, 0) && ok);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue: warp w owns TMEM lanes 32w .. 32w + 31; stacked column c goes to P_src[:, c] or P_dst[:, c - d] ----
    const int row = row0 + warp * 32 + lane;
    if (ok) {
        const int n2 = 2 * p.d;
        const bool vec = (p.d & 3) == 0;               // then no group of 4 columns straddles P_src / P_dst
        for (int c0 = 0; c0 < tn; c0 += 32) {
            float v[32];
            const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0;
            tmem_ld32(taddr, v);
            {
                float w[32];
                tmem_ld32(taddr + acc_cols, w);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __fadd_rn(v[j], w[j]);
            }
            if (row < p.n) {
                float* psrc = p.Psrc + (size_t)row * p.ld;
                float* pdst = p.Pdst + (size_t)row * p.ld;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const int c = n0 + c0 + j;
                    if (c >= n2 || c0 + j >= tn) break;
                    if (vec) {
                        *reinterpret_cast<float4*>(c < p.d ? psrc + c : pdst + (c - p.d)) =
                            make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                    } else {
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int cu = c + u;
                            if (cu < n2) *(cu < p.d ? psrc + cu : pdst + (cu - p.d)) = v[j + u];
                        }
                    }
                }
            }
        }
    } else if (threadIdx.x == 0) {
        *p.error = 1;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// fp32 [rows, ld] row-major, boxes of 32 floats x box_rows rows, 128-byte swizzle, out-of-bounds rows read as zero
static int make_map(CUtensorMap* map, const float* base, int64_t rows, int d, int ld, int box_rows) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return CLANE_EUNSUPPORTED;
    const cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult rc = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return rc == CUDA_SUCCESS ? CLANE_OK : CLANE_EINVAL;
}

}  // namespace asym
}  // namespace clane

using namespace clane;

extern "C" {

int clane_asym_supported(int32_t d) { return d >= 32 && d <= 128 && d % 32 == 0; }

int clane_asym_project(const float* d_Z, int32_t n, int32_t d, int32_t ld, const float* d_W, float* d_Psrc, float* d_Pdst,
                       int32_t* d_error, clane_stream_t s) {
    if (!d_Z || !d_W || !d_Psrc || !d_Pdst || !d_error || n < 0 || ld < d || (ld & 3)) return CLANE_EINVAL;
    if (!clane_asym_supported(d)) return CLANE_EUNSUPPORTED;
    if (n == 0) return CLANE_OK;
    CUtensorMap map_z, map_w;
    int rc = asym::make_map(&map_z, d_Z, n, d, ld, asym::kTileM);
    if (rc != CLANE_OK) return rc;
    rc = asym::make_map(&map_w, d_W, 2 * d, d, d, 2 * d);       // the stacked weights [2d, d], contiguous
    if (rc != CLANE_OK) return rc;
    const size_t smem = (size_t)(d / asym::kBlockK) * (asym::kTileM + 2 * d) * 128 + 1024;
    static bool attr = false;
    if (!attr) {
        CLANE_CUDA(cudaFuncSetAttribute(asym::k_asym_project, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr = true;
    }
    asym::ProjectParams p{d_Psrc, d_Pdst, n, d, ld, d_error};
    asym::k_asym_project<<<(unsigned)((n + asym::kTileM - 1) / asym::kTileM), asym::kThreads, smem, (cudaStream_t)s>>>(map_z, map_w, p);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

int clane_asym_project_fp32(const float* d_Z, int32_t n, int32_t d, int32_t ld, const float* d_W, int32_t ldw, float* d_Psrc,
                            float* d_Pdst, float* d_work, int32_t* d_error, clane_stream_t s) {
    if (!d_Z || !d_W || !d_Psrc || !d_Pdst || !d_work || !d_error || n < 0 || d < 1 || ld < d || ldw < d) return CLANE_EINVAL;
    // TMA: 16-byte aligned bases and row strides
    if ((ld & 3) || (ldw & 3) || ((uintptr_t)d_Z & 15) || ((uintptr_t)d_work & 15)) return CLANE_EINVAL;
    if (n == 0) return CLANE_OK;
    cudaStream_t st = (cudaStream_t)s;
    const int64_t wcount = 2 * (int64_t)d * ldw;
    float* whi = d_work;
    float* wlo = d_work + wcount;
    asym::k_asym_split<<<(unsigned)((wcount + 255) / 256), 256, 0, st>>>(d_W, wcount, whi, wlo);
    CLANE_LAUNCH_CHECK();
    // the 2d stacked columns in the fewest tiles of <= 256, each padded to the MMA's N granularity of 16
    const int n_tiles = (2 * d + asym::kMaxTileN - 1) / asym::kMaxTileN;
    if (n_tiles > 65535) return CLANE_EUNSUPPORTED;
    const int tile_n = ((2 * d + n_tiles - 1) / n_tiles + 15) / 16 * 16;
    const size_t stage_bytes = 2 * (size_t)(asym::kTileM + tile_n) * 128;
    const int stages = (int)std::min<size_t>(asym::kMaxStages, (asym::kFp32SmemBudget - 1024) / stage_bytes);   // >= 2
    CUtensorMap map_z, map_whi, map_wlo;
    int rc = asym::make_map(&map_z, d_Z, n, d, ld, asym::kTileM);
    if (rc == CLANE_OK) rc = asym::make_map(&map_whi, whi, 2 * d, d, ldw, tile_n);
    if (rc == CLANE_OK) rc = asym::make_map(&map_wlo, wlo, 2 * d, d, ldw, tile_n);
    if (rc != CLANE_OK) return rc;
    static bool attr = false;
    if (!attr) {
        CLANE_CUDA(cudaFuncSetAttribute(asym::k_asym_project_fp32, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)asym::kFp32SmemBudget));
        attr = true;
    }
    asym::ProjectFp32Params p{d_Psrc, d_Pdst, n, d, ld, tile_n, stages, d_error};
    const dim3 grid((unsigned)((n + asym::kTileM - 1) / asym::kTileM), (unsigned)n_tiles);
    asym::k_asym_project_fp32<<<grid, asym::kThreads, stages * stage_bytes + 1024, st>>>(map_z, map_whi, map_wlo, p);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

}  // extern "C"
