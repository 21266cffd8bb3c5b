// libclane_b200.so -- device kernels and the kernel-level C-ABI (include/clane_b200.h).
// Hand-written CUDA for sm_100a.  HBM/L2-bound gather work: no tensor cores (SURVEY 8d).
//
// Reference call sites replaced (all under /root/reference/clane/):
//   graph.py:118-128  Graph.build_P          -> k_dots + cascade(ElemGatherSq2) + k_row_softmax
//   similarity.py:26-37 CosineSimilarity     -> k_dots + cascade(ElemGatherSq2)
//   embedder.py:84-94 Jacobi sweep + L1       -> k_sweep (sweep.cuh; fused L1 partials) + cascade levels 1-3
//   embedder.py:98-108 patience               -> patience_step (cascade.cuh)
#include <math_constants.h>

#include <cstring>
#include <vector>
#include <algorithm>

#include "cascade.cuh"
#include "common.cuh"
#include "plan.cuh"
#include "sweep.cuh"

namespace clane {

// ------------------------------------------------------------------------------------------
// edge -> source row (first row of A.indices(), graph.py:119)
// ------------------------------------------------------------------------------------------
__global__ void k_edge_rows(const int32_t* __restrict__ rowptr, int32_t n, int64_t e, int32_t* __restrict__ erow) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e) return;
    int lo = 0, hi = n;  // largest v with rowptr[v] <= i
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if ((int64_t)__ldg(rowptr + mid) <= i) lo = mid; else hi = mid;
    }
    erow[i] = lo;
}

// ------------------------------------------------------------------------------------------
// per-edge dot, sequential over the feature index (similarity.py:35-37)
//   d < 400 : ATen native bmm loop  acc = fl(acc + fl(a*b))
//   d >= 400: oneMKL                acc = fma(a, b, acc)
// The chain over the d features of one edge is inherently serial (one thread), the gathers want a whole warp per
// row.  So a warp takes 32 consecutive edges: phase A reads both rows of every edge with coalesced 128-bit loads
// (lane = float4 of columns, 128 columns at a time) and parks the products -- or, for the fma order, both operands --
// in a shared-memory tile; phase B gives every lane one edge, which it sums in feature order out of the tile (row
// pitch 132 floats: the 128-bit reads of a quarter warp cover all 32 banks).  The running sums stay in registers
// across the 128-column blocks, so any d works.
// ------------------------------------------------------------------------------------------
constexpr int kDotCols = 128, kDotPitch = kDotCols + 4;
template <bool kFma> __host__ __device__ constexpr int dot_warps() { return kFma ? 2 : 4; }
template <bool kFma> __host__ __device__ constexpr size_t dot_smem() { return (size_t)dot_warps<kFma>() * 32 * kDotPitch * sizeof(float) * (kFma ? 2 : 1); }

template <bool kFma>
__global__ void __launch_bounds__(32 * dot_warps<kFma>())
k_dots(const float* __restrict__ Za, const float* __restrict__ Zb, int ld, int d, const int32_t* __restrict__ erow,
       const int32_t* __restrict__ col, int64_t e_lo, int64_t e_hi, float* __restrict__ dots) {   // <Za[erow[e]], Zb[col[e]]>
    extern __shared__ __align__(16) float dot_tile[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* ta = dot_tile + (size_t)warp * 32 * kDotPitch * (kFma ? 2 : 1);
    float* tb = ta + 32 * kDotPitch;                     // kFma only
    const int64_t ntiles = (e_hi - e_lo + 31) / 32;
    for (int64_t tile = (int64_t)blockIdx.x * dot_warps<kFma>() + warp; tile < ntiles; tile += (int64_t)gridDim.x * dot_warps<kFma>()) {
        const int64_t e0 = e_lo + tile * 32;
        const int cnt = (int)min((int64_t)32, e_hi - e0);
        // lane i: the two rows of edge e0 + i as float4 indices, 32 bits unsigned (rows * ld <= 2^34, clane_plan_create)
        unsigned ra = 0, rb = 0;
        if (lane < cnt) {
            ra = (unsigned)__ldg(erow + e0 + lane) * (unsigned)(ld >> 2);
            rb = (unsigned)__ldg(col + e0 + lane) * (unsigned)(ld >> 2);
        }
        float acc = 0.0f;
        for (int c0 = 0; c0 < d; c0 += kDotCols) {
            const int c = c0 + 4 * lane;
            const bool in = c < ld;                      // rows are padded to a multiple of 4 floats: whole float4s are readable
            const float4* zc = reinterpret_cast<const float4*>(Za) + (in ? c >> 2 : 0);
            const float4* zd = reinterpret_cast<const float4*>(Zb) + (in ? c >> 2 : 0);
            // ---- phase A: 8 edges per round, 16 independent 128-bit loads in flight ----
            // (consecutive edges mostly share their source row -- CSR order: its piece is loaded once per run)
            unsigned prev = ~0u;                         // no row starts there: (rows - 1) * ld / 4 < 2^32 - 1
            float4 xprev = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int i = 0; i < cnt; i += 8) {
                float4 x[8], y[8];
                unsigned oa[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    oa[u] = __shfl_sync(kFull, ra, (i + u) & 31);
                    const unsigned ob = __shfl_sync(kFull, rb, (i + u) & 31);
                    y[u] = __ldg(zd + ob);
                    if (oa[u] != (u == 0 ? prev : oa[u - 1])) x[u] = __ldg(zc + oa[u]);     // uniform branch
                }
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (oa[u] == (u == 0 ? prev : oa[u - 1])) x[u] = u == 0 ? xprev : x[u - 1];
                prev = oa[7];
                xprev = x[7];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    if (kFma) {
                        *reinterpret_cast<float4*>(ta + (i + u) * kDotPitch + 4 * lane) = x[u];
                        *reinterpret_cast<float4*>(tb + (i + u) * kDotPitch + 4 * lane) = y[u];
                    } else {
                        *reinterpret_cast<float4*>(ta + (i + u) * kDotPitch + 4 * lane) =
                            make_float4(fmul(x[u].x, y[u].x), fmul(x[u].y, y[u].y), fmul(x[u].z, y[u].z), fmul(x[u].w, y[u].w));
                    }
                }
            }
            __syncwarp();
            // ---- phase B: lane i sums edge i over this block's columns, in order ----
            const int ncol = min(kDotCols, d - c0);
            const float* pa = ta + lane * kDotPitch;
            const float* pb = tb + lane * kDotPitch;
            int j = 0;
            for (; j + 4 <= ncol; j += 4) {
                const float4 p = *reinterpret_cast<const float4*>(pa + j);
                if (kFma) {
                    const float4 q = *reinterpret_cast<const float4*>(pb + j);
                    acc = ffma(p.x, q.x, acc); acc = ffma(p.y, q.y, acc); acc = ffma(p.z, q.z, acc); acc = ffma(p.w, q.w, acc);
                } else {
                    acc = fadd(acc, p.x); acc = fadd(acc, p.y); acc = fadd(acc, p.z); acc = fadd(acc, p.w);
                }
            }
            for (; j < ncol; ++j) acc = kFma ? ffma(pa[j], pb[j], acc) : fadd(acc, pa[j]);
            __syncwarp();
        }
        if (lane < cnt) dots[e0 + lane] = acc;
    }
}

// ------------------------------------------------------------------------------------------
// Sleef_expf_u10 (what ATen's vectorised softmax calls; SURVEY Appendix A.3)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float pow2if(int q) { return __int_as_float((q + 127) << 23); }

__device__ __forceinline__ float sleef_expf_u10(float d) {
    const float R_LN2f = 1.442695040888963407359924681001892137426645954152985934135449406931f;
    const float L2Uf = 0.693145751953125f, L2Lf = 1.428606765330187045e-06f;
    const float qf = rintf(fmul(d, R_LN2f));
    const int q = (int)qf;
    float s = ffma(qf, -L2Uf, d);
    s = ffma(qf, -L2Lf, s);
    float u = 0.000198527617612853646278381f;
    u = ffma(u, s, 0.00139304355252534151077271f);
    u = ffma(u, s, 0.00833336077630519866943359f);
    u = ffma(u, s, 0.0416664853692054748535156f);
    u = ffma(u, s, 0.166666671633720397949219f);
    u = ffma(u, s, 0.5f);
    u = fadd(1.0f, ffma(fmul(s, s), u, s));
    const int q1 = q >> 1;
    u = fmul(fmul(u, pow2if(q1)), pow2if(q - q1));
    if (d < -104.0f) u = 0.0f;
    if (d > 100.0f) u = CUDART_INF_F;
    return u;
}

// ------------------------------------------------------------------------------------------
// per-source softmax (graph.py:122-123): ATen last-dim softmax =
//   e_i = Sleef_expf_u10(s_i - max), sum by the 16-lane vec::reduce_all tree (sequential for
//   rows shorter than 16), p_i = e_i * (1 / sum).
// One warp per row.  Optional global divisor c = fl(sqrt(S1)) * fl(sqrt(S2)) (similarity.py:37).
// ------------------------------------------------------------------------------------------
constexpr int kSoftmaxShort = 64;   // rows shorter than this: one thread per row; the others: one warp per row

// Short rows (the bulk of a power-law graph: mean degree ~7): one THREAD per row.  The reference's order for k < 16 is a
// plain sequential sum -- exactly a one-thread loop; for 16 <= k < 64 the thread keeps the 16 lane accumulators of
// vec::reduce_all in registers and folds them with the xor-8/4/2/1 butterfly (only the nodes lane 0's result needs).
__global__ void __launch_bounds__(128)
k_row_softmax_short(const float* scores, const float* __restrict__ norms2, int32_t row_lo, int32_t row_hi,
                    const int32_t* __restrict__ rowptr, float* w) {   // scores and w may be the same array (in place)
    const int row = row_lo + (int)((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
    if (row >= row_hi) return;
    const int a = __ldg(rowptr + row), k = __ldg(rowptr + row + 1) - a;
    if (k == 0 || k >= kSoftmaxShort) return;
    const bool div = norms2 != nullptr;
    float c = 1.0f;
    if (div) c = fmul(__fsqrt_rn(__ldg(norms2)), __fsqrt_rn(__ldg(norms2 + 1)));
    float m = -CUDART_INF_F;
    for (int i = 0; i < k; ++i) {
        float s = scores[a + i];
        if (div) s = __fdiv_rn(s, c);
        m = fmaxf(m, s);
    }
    float sum;
    if (k < 16) {
        sum = 0.0f;
        for (int i = 0; i < k; ++i) {
            float s = scores[a + i];
            if (div) s = __fdiv_rn(s, c);
            const float e = sleef_expf_u10(fsub(s, m));
            w[a + i] = e;                       // position i is never read again as a score
            sum = i == 0 ? e : fadd(sum, e);
        }
    } else {
        float acc[16];
#pragma unroll
        for (int l = 0; l < 16; ++l) acc[l] = 0.0f;
        // lane l accumulates e_l, e_{l+16}, ... over the full 16-vectors, then the k mod 16 leftovers go to lanes 0..
        for (int base = 0; base < k; base += 16) {
#pragma unroll
            for (int l = 0; l < 16; ++l) {
                if (base + l < k) {
                    float s = scores[a + base + l];
                    if (div) s = __fdiv_rn(s, c);
                    const float e = sleef_expf_u10(fsub(s, m));
                    w[a + base + l] = e;
                    acc[l] = base == 0 ? e : fadd(acc[l], e);
                }
            }
        }
#pragma unroll
        for (int h = 8; h >= 1; h >>= 1)
#pragma unroll
            for (int l = 0; l < h; ++l) acc[l] = fadd(acc[l], acc[l + h]);
        sum = acc[0];
    }
    const float inv = __fdiv_rn(1.0f, sum);
    for (int i = 0; i < k; ++i) w[a + i] = fmul(w[a + i], inv);
}

// Long rows: one CTA per row.  Only the 16-lane accumulation is serial (k / 16 dependent adds per lane: microseconds
// even for a row of 10^5 neighbours); the maximum and the exponentials -- the expensive part -- are spread over the CTA.
// rows: a list of row ids (rows of >= kSoftmaxShort neighbours, from the plan), or null = row_lo + blockIdx.x.
constexpr int kSoftmaxLongThreads = 256;
__global__ void __launch_bounds__(kSoftmaxLongThreads)
k_row_softmax_long(const float* scores, const float* __restrict__ norms2, const int32_t* __restrict__ rows, int32_t row_lo,
                   const int32_t* __restrict__ rowptr, float* w) {   // scores and w may be the same array (in place)
    __shared__ float red[kSoftmaxLongThreads / 32];
    __shared__ float s_sum;
    const int row = rows != nullptr ? __ldg(rows + blockIdx.x) : row_lo + (int)blockIdx.x;
    const int a = __ldg(rowptr + row), k = __ldg(rowptr + row + 1) - a;
    if (k < kSoftmaxShort) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool div = norms2 != nullptr;
    float c = 1.0f;
    if (div) c = fmul(__fsqrt_rn(__ldg(norms2)), __fsqrt_rn(__ldg(norms2 + 1)));
    float m = -CUDART_INF_F;
    for (int i = tid; i < k; i += kSoftmaxLongThreads) {
        float s = scores[a + i];
        if (div) s = __fdiv_rn(s, c);
        m = fmaxf(m, s);
    }
#pragma unroll
    for (int h = 16; h >= 1; h >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, h));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
#pragma unroll
    for (int q = 1; q < kSoftmaxLongThreads / 32; ++q) m = fmaxf(m, red[q]);
    // every exponential, in parallel (element i is read as a score and written as e_i by the same thread)
    for (int i = tid; i < k; i += kSoftmaxLongThreads) {
        float s = scores[a + i];
        if (div) s = __fdiv_rn(s, c);
        w[a + i] = sleef_expf_u10(fsub(s, m));
    }
    __syncthreads();
    // lane l < 16 of warp 0: e_l, e_{l+16}, ... in order (the k mod 16 leftovers land in lanes 0..), then the butterfly
    if (warp == 0) {
        float acc = 0.0f;
        if (lane < 16) {
            int i = lane;
            for (; i + 7 * 16 < k; i += 8 * 16) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = w[a + i + 16 * u];
#pragma unroll
                for (int u = 0; u < 8; ++u) acc = (i == lane && u == 0) ? v[0] : fadd(acc, v[u]);
            }
            for (; i < k; i += 16) acc = i == lane ? w[a + i] : fadd(acc, w[a + i]);
        }
#pragma unroll
        for (int h = 8; h >= 1; h >>= 1) acc = fadd(acc, __shfl_xor_sync(kFull, acc, h));
        if (lane == 0) s_sum = acc;
    }
    __syncthreads();
    const float inv = __fdiv_rn(1.0f, s_sum);
    for (int i = tid; i < k; i += kSoftmaxLongThreads) w[a + i] = fmul(w[a + i], inv);
}

// col[e] * ld / 4: the float4 index the sweep gathers from (one multiply per edge, once per graph), as uint32 bits:
// n * ld <= 2^34 (clane_plan_create)
__global__ void k_col_offsets(const int32_t* __restrict__ col, int64_t e, int ld, int32_t* __restrict__ off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e) off[i] = (int32_t)((unsigned)col[i] * (unsigned)(ld >> 2));
}

__global__ void k_cosine_finalize(const float* __restrict__ dots, const float* __restrict__ norms2, int64_t e,
                                  float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e) return;
    const float c = fmul(__fsqrt_rn(__ldg(norms2)), __fsqrt_rn(__ldg(norms2 + 1)));
    out[i] = __fdiv_rn(dots[i], c);
}

__global__ void k_patience_reset(clane_patience* st, int tol, int max_sweeps) {
    st->minimum = CUDART_INF_F;
    st->patience = tol;
    st->tol = tol;
    st->sweeps = 0;
    st->max_sweeps = max_sweeps;
    st->stop = 0;
    st->last_amount = 0.0f;
    st->reserved = 0;
}

}  // namespace clane

namespace {

// kernel launch with an explicit priority: the attribute stays on the kernel node when the launch is captured into a
// graph (a captured node does not reliably inherit the priority of the stream it was captured from)
template <class... KArgs, class... Args>
cudaError_t launch_prio(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int prio, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributePriority;
    attr.val.priority = prio;
    cfg.attrs = &attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace

using namespace clane;

constexpr int kSweepBatch = 6;     // sweeps per replayed graph of clane_sweeps (a multiple of the three Z buffers)
constexpr int kWhileBatch = 6;     // sweeps per iteration of the conditional-WHILE body (until_stop); 12 / 24 measured
                                   // no better (arxiv shape, time to converge 0.105 / 0.107 / 0.115 s)
static_assert(kSweepBatch % 3 == 0 && kWhileBatch % 3 == 0, "a batch returns the three Z buffers to where it started");
// The L1 tail of sweep t runs while the span tasks of sweep t + 1 fill every SM (12 CTAs x 64 threads x 80 registers leave
// 4096 registers per SM): 64-thread CTAs of <= 64 registers are what still fits beside them.
constexpr int kTailThreads = 64;

// =============================================================================================
// C-ABI
// =============================================================================================
extern "C" {

int clane_version(void) { return 100; }

const char* clane_error_string(int code) {
    switch (code) {
        case CLANE_OK: return "ok";
        case CLANE_EINVAL: return "clane: invalid argument";
        case CLANE_ERANGE: return "clane: index out of range";
        case CLANE_EWORKSPACE: return "clane: workspace too small";
        case CLANE_ENODEVICE: return "clane: no sm_100 CUDA device";
        case CLANE_ENOENT: return "clane: cannot open file";
        case CLANE_EPARSE: return "clane: malformed edge line";
        case CLANE_EUNKNOWNID: return "clane: edge endpoint not in V";
        case CLANE_ENOMEM: return "clane: out of host memory";
        case CLANE_EUNSUPPORTED: return "clane: not supported by this driver";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "clane: unknown error";
    }
}

int clane_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    CLANE_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CLANE_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return CLANE_OK;
}

int32_t clane_padded_ld(int32_t d) { return (d + 3) & ~3; }

int clane_cascade_shape(int64_t n_elems, int64_t* n1_nodes, int64_t* elems_per_node) {
    if (n_elems < 0) return CLANE_EINVAL;
    CascadeShape sh = cascade_shape(n_elems);
    if (n1_nodes) *n1_nodes = sh.n1_nodes;
    if (elems_per_node) *elems_per_node = sh.node1_rows * 32;
    return CLANE_OK;
}

int clane_edge_rows(const int32_t* d_rowptr, int32_t n, int64_t e, int32_t* d_erow, clane_stream_t s) {
    if (!d_rowptr || !d_erow || n < 0 || e < 0) return CLANE_EINVAL;
    if (e == 0) return CLANE_OK;
    k_edge_rows<<<(unsigned)((e + 255) / 256), 256, 0, (cudaStream_t)s>>>(d_rowptr, n, e, d_erow);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

int clane_scores_cosine(clane_plan* plan, const float* d_Z, const int32_t* d_erow, const int32_t* d_col,
                        int64_t edge_lo, int64_t edge_hi, float* d_dots, float* d_norms2, clane_stream_t s) {
    if (!plan || !d_Z || !d_erow || !d_col || !d_dots) return CLANE_EINVAL;
    if (edge_lo < 0 || edge_hi > plan->e || edge_lo > edge_hi) return CLANE_EINVAL;
    cudaStream_t st = (cudaStream_t)s;
    // the dots and the norm cascade are independent and both latency-bound at partial occupancy: with a schedule plan (it
    // owns side streams) the dots run on a side stream beside the cascade on the caller's.  (One kernel gathering once for
    // both was measured slower at arxiv shape, 0.336 against 0.304 ms: profiles/r02_notes.md.)
    cudaStream_t caller = st;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    const bool beside = d_norms2 != nullptr && plan->side != nullptr && edge_hi > edge_lo;
    if (beside) {
        while (plan->evs.size() < 2) {
            cudaEvent_t ev = nullptr;
            CLANE_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            plan->evs.push_back(ev);
        }
        ev_fork = plan->evs[0]; ev_join = plan->evs[1];
        CLANE_CUDA(cudaEventRecord(ev_fork, caller));
        CLANE_CUDA(cudaStreamWaitEvent(plan->side, ev_fork, 0));
        st = plan->side;
    }
    if (edge_hi > edge_lo) {
        const int64_t ntiles = (edge_hi - edge_lo + 31) / 32;
        if (plan->d < 400) {
            const unsigned grid = (unsigned)std::min<int64_t>((ntiles + dot_warps<false>() - 1) / dot_warps<false>(), 148 * 24);
            k_dots<false><<<grid, 32 * dot_warps<false>(), dot_smem<false>(), st>>>(d_Z, d_Z, plan->ld, plan->d, d_erow, d_col, edge_lo, edge_hi, d_dots);
        } else {
            const unsigned grid = (unsigned)std::min<int64_t>((ntiles + dot_warps<true>() - 1) / dot_warps<true>(), 148 * 24);
            k_dots<true><<<grid, 32 * dot_warps<true>(), dot_smem<true>(), st>>>(d_Z, d_Z, plan->ld, plan->d, d_erow, d_col, edge_lo, edge_hi, d_dots);
        }
        CLANE_LAUNCH_CHECK();
    }
    if (!d_norms2) return CLANE_OK;       // dots only: a rank of a row-partitioned run reduces the norms by node range
    if (beside) CLANE_CUDA(cudaEventRecord(ev_join, plan->side));
    ElemGatherSq2 el{d_Z, d_erow, d_col, plan->d, plan->ld, plan->e};
    int rc = cascade_launch(el, plan->e * (int64_t)plan->d, plan->d_p1, plan->d_p2, d_norms2, nullptr, nullptr, 0, caller);
    if (beside) CLANE_CUDA(cudaStreamWaitEvent(caller, ev_join, 0));
    return rc;
}

int clane_norms_partial(clane_plan* plan, const float* d_Z, const int32_t* d_erow, const int32_t* d_col, int64_t node_lo,
                        int64_t node_hi, float* d_p1, clane_stream_t s) {
    if (!plan || !d_Z || !d_erow || !d_col || !d_p1) return CLANE_EINVAL;
    ElemGatherSq2 el{d_Z, d_erow, d_col, plan->d, plan->ld, plan->e};
    return cascade_launch_l01(el, plan->e * (int64_t)plan->d, node_lo, node_hi, d_p1, nullptr, (cudaStream_t)s);
}

int clane_norms_finish(clane_plan* plan, const float* d_Z, const int32_t* d_erow, const int32_t* d_col, const float* d_p1,
                       float* d_norms2, clane_stream_t s) {
    if (!plan || !d_Z || !d_erow || !d_col || !d_p1 || !d_norms2) return CLANE_EINVAL;
    ElemGatherSq2 el{d_Z, d_erow, d_col, plan->d, plan->ld, plan->e};
    return cascade_launch_finish(el, plan->e * (int64_t)plan->d, d_p1, plan->d_p2, d_norms2, nullptr, nullptr, 0, nullptr,
                                 (cudaStream_t)s);
}

int clane_row_softmax(const float* d_scores, const float* d_norms2, int32_t row_lo, int32_t row_hi,
                      const int32_t* d_rowptr, float* d_w, clane_stream_t s) {
    if (!d_scores || !d_rowptr || !d_w || row_lo < 0 || row_hi < row_lo) return CLANE_EINVAL;
    if (row_hi == row_lo) return CLANE_OK;
    // rows shorter than kSoftmaxShort: a thread each; the rest: a CTA each (without a plan's list of long rows the CTAs of
    // short rows exit at once)
    k_row_softmax_short<<<(unsigned)((row_hi - row_lo + 127) / 128), 128, 0, (cudaStream_t)s>>>(d_scores, d_norms2, row_lo, row_hi,
                                                                                             d_rowptr, d_w);
    CLANE_LAUNCH_CHECK();
    k_row_softmax_long<<<(unsigned)(row_hi - row_lo), kSoftmaxLongThreads, 0, (cudaStream_t)s>>>(d_scores, d_norms2, nullptr, row_lo,
                                                                                             d_rowptr, d_w);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

int clane_plan_softmax(clane_plan* plan, const float* d_scores, const float* d_norms2, const int32_t* d_rowptr, float* d_w,
                       clane_stream_t s) {
    if (!plan || !plan->has_schedule || !d_scores || !d_rowptr || !d_w) return CLANE_EINVAL;
    const int32_t rows = plan->row_hi - plan->row_lo;
    if (rows <= 0) return CLANE_OK;
    // the two kernels own disjoint rows: the long rows go beside the short ones on the plan's side stream
    cudaStream_t st = (cudaStream_t)s;
    const bool beside = plan->n_long_rows > 0 && plan->side != nullptr;
    if (beside) {
        while (plan->evs.size() < 2) {
            cudaEvent_t ev = nullptr;
            CLANE_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            plan->evs.push_back(ev);
        }
        CLANE_CUDA(cudaEventRecord(plan->evs[0], st));
        CLANE_CUDA(cudaStreamWaitEvent(plan->side, plan->evs[0], 0));
    }
    if (plan->n_long_rows > 0) {
        k_row_softmax_long<<<(unsigned)plan->n_long_rows, kSoftmaxLongThreads, 0, beside ? plan->side : st>>>(
            d_scores, d_norms2, plan->d_long_rows, plan->row_lo, d_rowptr, d_w);
        CLANE_LAUNCH_CHECK();
        if (beside) CLANE_CUDA(cudaEventRecord(plan->evs[1], plan->side));
    }
    k_row_softmax_short<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(d_scores, d_norms2, plan->row_lo, plan->row_hi, d_rowptr, d_w);
    CLANE_LAUNCH_CHECK();
    if (beside) CLANE_CUDA(cudaStreamWaitEvent(st, plan->evs[1], 0));
    return CLANE_OK;
}

int clane_build_p_asym(clane_plan* plan, const float* d_Z, const float* d_W, const int32_t* d_rowptr, const int32_t* d_erow,
                       const int32_t* d_col, float* d_w, float* d_work, int32_t* d_error, clane_stream_t s) {
    if (!plan || !plan->has_schedule || !d_Z || !d_W || !d_rowptr || !d_w || !d_work || !d_error) return CLANE_EINVAL;
    if (plan->e > 0 && (!d_erow || !d_col)) return CLANE_EINVAL;
    float* psrc = d_work;
    float* pdst = d_work + (size_t)plan->n * plan->ld;
    // every node projected once on the tensor cores: [P_src | P_dst] = Z [W_src ; W_dst]^T
    int rc = clane_asym_project(d_Z, plan->n, plan->d, plan->ld, d_W, psrc, pdst, d_error, s);
    if (rc != CLANE_OK) return rc;
    const int64_t e_lo = plan->edge_lo, e_hi = plan->edge_hi;
    if (e_hi > e_lo) {
        const int64_t ntiles = (e_hi - e_lo + 31) / 32;
        const unsigned grid = (unsigned)std::min<int64_t>((ntiles + dot_warps<false>() - 1) / dot_warps<false>(), 148 * 24);
        k_dots<false><<<grid, 32 * dot_warps<false>(), dot_smem<false>(), (cudaStream_t)s>>>(psrc, pdst, plan->ld, plan->d, d_erow, d_col,
                                                                                      e_lo, e_hi, d_w);
        CLANE_LAUNCH_CHECK();
    }
    return clane_plan_softmax(plan, d_w, nullptr, d_rowptr, d_w, s);     // graph.py:122-123: no norm divisor for this plugin
}

int clane_build_p_asym_fp32(clane_plan* plan, const float* d_Z, const float* d_W, int32_t ldw, const int32_t* d_rowptr,
                            const int32_t* d_erow, const int32_t* d_col, float* d_w, float* d_work, int32_t* d_error,
                            clane_stream_t s) {
    if (!plan || !plan->has_schedule || !d_Z || !d_W || !d_rowptr || !d_w || !d_work || !d_error) return CLANE_EINVAL;
    if (plan->e > 0 && (!d_erow || !d_col)) return CLANE_EINVAL;
    float* psrc = d_work;
    float* pdst = d_work + (size_t)plan->n * plan->ld;
    // every node projected once, 3xTF32 on the tensor cores; the weight split goes after the two projected matrices
    int rc = clane_asym_project_fp32(d_Z, plan->n, plan->d, plan->ld, d_W, ldw, psrc, pdst, pdst + (size_t)plan->n * plan->ld,
                                     d_error, s);
    if (rc != CLANE_OK) return rc;
    const int64_t e_lo = plan->edge_lo, e_hi = plan->edge_hi;
    if (e_hi > e_lo) {
        // the reference's bmm: mul + add below d = 400, fma from there on (as the cosine path)
        const int64_t ntiles = (e_hi - e_lo + 31) / 32;
        cudaStream_t st = (cudaStream_t)s;
        if (plan->d < 400) {
            const unsigned grid = (unsigned)std::min<int64_t>((ntiles + dot_warps<false>() - 1) / dot_warps<false>(), 148 * 24);
            k_dots<false><<<grid, 32 * dot_warps<false>(), dot_smem<false>(), st>>>(psrc, pdst, plan->ld, plan->d, d_erow, d_col, e_lo, e_hi, d_w);
        } else {
            const unsigned grid = (unsigned)std::min<int64_t>((ntiles + dot_warps<true>() - 1) / dot_warps<true>(), 148 * 24);
            k_dots<true><<<grid, 32 * dot_warps<true>(), dot_smem<true>(), st>>>(psrc, pdst, plan->ld, plan->d, d_erow, d_col, e_lo, e_hi, d_w);
        }
        CLANE_LAUNCH_CHECK();
    }
    return clane_plan_softmax(plan, d_w, nullptr, d_rowptr, d_w, s);
}

int clane_cosine_finalize(const float* d_dots, const float* d_norms2, int64_t e, float* d_out, clane_stream_t s) {
    if (!d_dots || !d_norms2 || !d_out || e < 0) return CLANE_EINVAL;
    if (e == 0) return CLANE_OK;
    k_cosine_finalize<<<(unsigned)((e + 255) / 256), 256, 0, (cudaStream_t)s>>>(d_dots, d_norms2, e, d_out);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

int clane_build_p_cosine(clane_plan* plan, const float* d_Z, const int32_t* d_rowptr, const int32_t* d_erow,
                         const int32_t* d_col, float* d_w, float* d_norms2, clane_stream_t s) {
    if (!plan || !d_rowptr || !plan->has_schedule) return CLANE_EINVAL;
    // rows [row_lo, row_hi) own the contiguous edge range [rowptr[row_lo], rowptr[row_hi])
    int rc = clane_scores_cosine(plan, d_Z, d_erow, d_col, plan->edge_lo, plan->edge_hi, d_w, d_norms2, s);
    if (rc != CLANE_OK) return rc;
    return clane_plan_softmax(plan, d_w, d_norms2, d_rowptr, d_w, s);
}

// timing bracket: an ordinary record, or -- while the sweep is being captured -- an external event-record node of
// the graph, so that the brackets measure the kernels as they run in the replayed graph
static cudaError_t prof_record(cudaEvent_t ev, cudaStream_t st) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    return cudaEventRecordWithFlags(ev, st, cap == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
}

namespace {

cudaError_t prof_mark(clane_plan* plan, int i, cudaStream_t st) {
    plan->prof_mask |= 1u << i;
    return prof_record(plan->ev_prof[i], st);
}

struct SweepArgs {
    const float* X;
    const int32_t* rowptr;
    const int32_t* col;
    const float* w;
    float gamma;
    float* amount;
    clane_patience* state;
    float* log;
    int32_t log_cap;
};

// tell a conditional-WHILE graph whether to run its body (a batch of sweeps) once more
__global__ void k_loop_condition(cudaGraphConditionalHandle handle, const clane_patience* st) {
    cudaGraphSetConditional(handle, st->stop ? 0u : 1u);
}

}  // namespace

// Enqueue `n_sweeps` consecutive sweeps.  Sweep t reads Z[(c0 + t) % nz] and writes Z[(c0 + t + 1) % nz].
//
// Streams of one sweep (all plan-owned except the caller's `st`; ordinary event dependencies, no flags):
//   st    : span tasks (k_sweep_rows over the span part of the task list)
//   side  : hub segment tasks (k_sweep_rows over the segment part), then the chains of the long hub rows
//   side2 : the chains of the short hub rows (after the segments)
//   tail  : the exact L1 change -- chunk fix-up, level 1, finish + patience
// Between sweeps (nz == 3, three rotating Z buffers): the spans / segments of sweep t + 1 only need the rows and
// chains of sweep t, so the whole L1 tail of sweep t runs beside sweep t + 1.  The patience flag a sweep sees is
// therefore one sweep old: at most one speculative sweep runs after the stop, into a buffer that is not the result
// (the result of the stopping sweep t is Z[(c0 + t + 1) % 3]; sweep t + 1 writes Z[(c0 + t + 2) % 3]; its tail is a
// no-op, so the state, the log and the sweep count are exactly the reference's).  With nz == 2 every sweep waits for
// the previous tail (its fix-up reads the buffer the next sweep overwrites).
static int enqueue_sweeps(clane_plan* plan, const SweepArgs& a, float* const* Z, int nz, int c0, int n_sweeps, cudaStream_t st) {
    const bool want_l1 = a.amount != nullptr || a.state != nullptr;
    size_t ne = 0;
    auto next_event = [&](cudaEvent_t* out) -> cudaError_t {
        if (ne == plan->evs.size()) {
            cudaEvent_t ev = nullptr;
            cudaError_t rc = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (rc != cudaSuccess) return rc;
            plan->evs.push_back(ev);
        }
        *out = plan->evs[ne++];
        return cudaSuccess;
    };
    auto mark = [&](cudaEvent_t* ev, cudaStream_t s) -> cudaError_t {       // *ev = a fresh event recorded on s
        cudaError_t rc = next_event(ev);
        return rc != cudaSuccess ? rc : cudaEventRecord(*ev, s);
    };
    const int per_row = plan->nslab32b + (plan->ntail4 > 0 ? 1 : 0);
    const int n_long = plan->n_long_hub_rows, n_short = plan->n_hub_rows - n_long;
    const bool hubs = plan->n_hub_rows > 0 && plan->n_seg_tasks > 0;
    const int64_t seg_ctas = ((int64_t)plan->n_seg_tasks * plan->nslab + kRowWarps - 1) / kRowWarps;
    const int64_t span_ctas = ((int64_t)(plan->n_tasks - plan->n_seg_tasks) * plan->nslab + kRowWarps - 1) / kRowWarps;
    const int64_t n_elems = (int64_t)plan->n * plan->d;
    const bool prof = plan->profile && n_sweeps == 1;
    if (prof) plan->prof_mask = 0;
    cudaEvent_t e_begin = nullptr;
    CLANE_CUDA(mark(&e_begin, st));
    if (prof) CLANE_CUDA(prof_mark(plan, 0, st));
    std::vector<cudaEvent_t> eR((size_t)n_sweeps, nullptr), eC(eR), eC2(eR), eF(eR), eL(eR);
    for (int t = 0; t < n_sweeps; ++t) {
        const float* Zc = Z[(c0 + t) % nz];
        float* Zn = Z[(c0 + t + 1) % nz];
        SweepParams p;
        p.X = a.X; p.Zc = Zc; p.Zn = Zn;
        p.ld = plan->ld; p.d = plan->d; p.n = plan->n;
        p.rowptr = a.rowptr; p.coloff = plan->d_coloff; p.w = a.w; p.gamma = a.gamma;
        p.tasks = static_cast<const SweepTask*>(plan->d_tasks); p.n_tasks = plan->n_tasks; p.task_lo = 0;
        p.row_lo = plan->row_lo;
        p.G = plan->G; p.nslab = plan->nslab;
        p.fuse = (plan->fuse && want_l1) ? 1 : 0;
        p.P0 = plan->d_P0 + (size_t)(t & 1) * plan->p0_stride;
        p.hub_info = static_cast<const int4*>(plan->d_hub_info); p.n_hub_rows = plan->n_hub_rows;
        p.limit = plan->limit; p.ntail4 = plan->ntail4; p.nslab32b = plan->nslab32b; p.sld = plan->nslab32b * 32;
        p.hubS = static_cast<float4*>(plan->d_hubS);
        p.hubT = static_cast<float4*>(plan->d_hubT);
        p.hub_first = 0;
        p.st = a.state;
        p.n_remote = 0;
        p.mc = nullptr;
        p.bulk = 0;
        p.trace = nullptr;
        unsigned long long* tr = (plan->d_trace != nullptr && t < kTraceSweeps) ? plan->d_trace + (size_t)t * kTraceSlots * 2 : nullptr;
        for (int q = 0; q < 3 && plan->n_peers > 1; ++q)
            if (plan->peers[q][plan->self_rank] == Zn) {
                if (plan->mc[q] != nullptr) { p.mc = plan->mc[q]; continue; }   // one multicast store instead of n - 1 unicast ones
                for (int r = 0; r < plan->n_peers; ++r)
                    if (r != plan->self_rank) p.peer[p.n_remote++] = plan->peers[q][r];
            }
        // whole rows per warp and unicast peers: the spans' rows leave as bulk stores (sweep.cuh, flush_rows)
        if (p.n_remote > 0 && plan->nslab == 1 && plan->G <= kStageRows) p.bulk = 1;
        // what the previous sweeps must have finished before this one may start
        cudaEvent_t prev_tail = nullptr;       // the tail whose inputs this sweep overwrites / whose flag it reads
        if (nz >= 3) { if (t >= 2) prev_tail = eL[t - 2]; }
        else if (t >= 1) prev_tail = eL[t - 1];
        // ---- side: hub segments, then the chains ----
        cudaEvent_t eS_cur = nullptr;
        if (hubs) {
            CLANE_CUDA(cudaStreamWaitEvent(plan->side, t == 0 ? e_begin : eR[t - 1], 0));
            if (t > 0 && eC2[t - 1]) CLANE_CUDA(cudaStreamWaitEvent(plan->side, eC2[t - 1], 0));
            if (prev_tail) CLANE_CUDA(cudaStreamWaitEvent(plan->side, prev_tail, 0));
            SweepParams ps = p;
            ps.n_tasks = plan->n_seg_tasks;
            ps.bulk = 0;
            ps.trace = tr;
            CLANE_CUDA(launch_prio(k_sweep_rows<false>, dim3((unsigned)seg_ctas), dim3(kRowThreads), 0, plan->side, plan->prio_hi, ps));
            cudaEvent_t eS = nullptr;
            CLANE_CUDA(mark(&eS, plan->side));
            eS_cur = eS;
            if (prof) CLANE_CUDA(prof_mark(plan, 4, plan->side));
            if (n_long > 0) {
                p.trace = tr ? tr + 2 : nullptr;
                CLANE_CUDA(launch_prio(k_hub_chain<false>, dim3((unsigned)(n_long * per_row)), dim3(kChainThreads), kHeavySmemBytes,
                                       plan->side, plan->prio_hi, p));
            }
            if (prof) CLANE_CUDA(prof_mark(plan, 5, plan->side));
            CLANE_CUDA(mark(&eC[t], plan->side));
            if (n_short > 0) {             // its own stream: not behind the long rows' chains
                CLANE_CUDA(cudaStreamWaitEvent(plan->side2, eS, 0));
                SweepParams pc = p;
                pc.hub_first = n_long;
                pc.trace = tr ? tr + 4 : nullptr;
                CLANE_CUDA(launch_prio(k_hub_chain<true>, dim3((unsigned)(n_short * per_row)), dim3(kChainThreads), kLightSmemBytes,
                                       plan->side2, plan->prio_hi, pc));
                CLANE_CUDA(mark(&eC2[t], plan->side2));
            }
        }
        // ---- caller's stream: the span tasks ----
        if (t > 0) {
            if (eC[t - 1]) CLANE_CUDA(cudaStreamWaitEvent(st, eC[t - 1], 0));
            if (eC2[t - 1]) CLANE_CUDA(cudaStreamWaitEvent(st, eC2[t - 1], 0));
        }
        if (prev_tail) CLANE_CUDA(cudaStreamWaitEvent(st, prev_tail, 0));
        // The segments and the light chains fit beside the span CTAs (sweep.cuh), so normally the spans do not wait for
        // them.  Heavy chains want an SM each: with long hub rows the spans start behind the segments, together with the
        // heavy chains, which the higher priority places first (the segments are microseconds of a millisecond sweep).
        if (eS_cur && n_long > 0) CLANE_CUDA(cudaStreamWaitEvent(st, eS_cur, 0));
        if (prof) CLANE_CUDA(prof_mark(plan, 1, st));
        if (span_ctas > 0) {
            SweepParams pr = p;
            pr.task_lo = plan->n_seg_tasks;
            pr.trace = tr ? tr + 6 : nullptr;
            if (pr.bulk)
                CLANE_CUDA(launch_prio(k_sweep_rows<true>, dim3((unsigned)span_ctas), dim3(kRowThreads), kRowWarps * kRowStageBytes, st,
                                       plan->prio_lo, pr));
            else
                CLANE_CUDA(launch_prio(k_sweep_rows<false>, dim3((unsigned)span_ctas), dim3(kRowThreads), 0, st, plan->prio_lo, pr));
        }
        if (prof) CLANE_CUDA(prof_mark(plan, 2, st));
        CLANE_CUDA(mark(&eR[t], st));
        // ---- tail: the exact L1 change of this sweep ----
        if (want_l1) {
            cudaStream_t tl = plan->tail;
            CLANE_CUDA(cudaStreamWaitEvent(tl, eR[t], 0));
            if (eC[t]) CLANE_CUDA(cudaStreamWaitEvent(tl, eC[t], 0));
            if (eC2[t]) CLANE_CUDA(cudaStreamWaitEvent(tl, eC2[t], 0));
            if (prof) CLANE_CUDA(prof_mark(plan, 6, tl));
            if (tr) k_trace_stamp<<<1, 1, 0, tl>>>(tr + 8, 0);
            ElemAbsDiff el{Zn, Zc, plan->d, plan->ld};
            int rc;
            if (p.fuse) {
                CascadeShape sh = cascade_shape(n_elems);
                if (plan->n_fix_groups > 0) {
                    CLANE_CUDA(launch_prio(k_fix_chunks, dim3((unsigned)(((int64_t)plan->n_fix_groups * 32 + kTailThreads - 1) / kTailThreads)),
                                           dim3(kTailThreads), 0, tl, plan->prio_hi, (const float*)Zn, Zc, plan->d, plan->n, plan->G,
                                           (const int32_t*)plan->d_fix_groups, plan->n_fix_groups, p.P0, (const clane_patience*)a.state));
                }
                CLANE_CUDA(mark(&eF[t], tl));
                if (sh.n1_nodes > 0) {
                    CLANE_CUDA(launch_prio(k_level1_from_p0, dim3((unsigned)((sh.n1_nodes * 32 + kTailThreads - 1) / kTailThreads)),
                                           dim3(kTailThreads), 0, tl, plan->prio_hi, sh, (const float*)p.P0, plan->d_p1,
                                           (const clane_patience*)a.state));
                }
                if (tr) k_trace_stamp<<<1, 1, 0, tl>>>(tr + 10, 0);
                rc = cascade_launch_finish(el, n_elems, plan->d_p1, plan->d_p2, a.amount, a.state, a.log, a.log_cap, nullptr, tl,
                                           n_sweeps > 1 ? kTailThreads : 1024);
                if (tr) k_trace_stamp<<<1, 1, 0, tl>>>(tr + 10, 1);
            } else {
                rc = cascade_launch_l01(el, n_elems, 0, cascade_shape(n_elems).n1_nodes, plan->d_p1, a.state, tl);
                CLANE_CUDA(mark(&eF[t], tl));      // Zn / Zc are not read after this point (the finish reads <= 31 tail elements:
                if (rc == CLANE_OK)               // they belong to the last rows, which the waits below still protect -- see eL)
                    rc = cascade_launch_finish(el, n_elems, plan->d_p1, plan->d_p2, a.amount, a.state, a.log, a.log_cap, nullptr, tl);
            }
            if (rc != CLANE_OK) return rc;
            if (tr) k_trace_stamp<<<1, 1, 0, tl>>>(tr + 8, 1);
            CLANE_CUDA(mark(&eL[t], tl));
        }
    }
    // join everything back into the caller's stream
    const int last = n_sweeps - 1;
    if (eC[last]) CLANE_CUDA(cudaStreamWaitEvent(st, eC[last], 0));
    if (eC2[last]) CLANE_CUDA(cudaStreamWaitEvent(st, eC2[last], 0));
    for (int t = std::max(0, n_sweeps - 2); t < n_sweeps; ++t)
        if (eL[t]) CLANE_CUDA(cudaStreamWaitEvent(st, eL[t], 0));
    if (prof) CLANE_CUDA(prof_mark(plan, 3, st));
    return CLANE_OK;
}

// enqueue through the CUDA-graph cache: capture once per argument set, replay afterwards.  loop != 0: the batch is the
// body of a conditional WHILE node that repeats it until the patience state machine stops (one launch = one propagate()).
static int launch_sweeps(clane_plan* plan, const SweepArgs& a, float* const* Z, int nz, int c0, int n_sweeps, int loop,
                         cudaStream_t st) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cap);
    if (!plan->use_graphs || cap != cudaStreamCaptureStatusNone || st == nullptr) {
        if (loop) return CLANE_EINVAL;   // the caller falls back to host-driven batches
        return enqueue_sweeps(plan, a, Z, nz, c0, n_sweeps, st);
    }
    const void* key[12] = {a.X, Z[0], Z[1], nz > 2 ? Z[2] : nullptr, a.rowptr, a.col, a.w, a.amount, a.state, a.log, st, nullptr};
    clane_plan::SweepGraph* slot = nullptr;
    for (auto& g : plan->graphs)
        if (g.exec && g.gamma == a.gamma && g.log_cap == a.log_cap && g.n_sweeps == n_sweeps && g.nz == nz && g.c0 == c0 &&
            g.loop == loop && memcmp(g.key, key, sizeof(key)) == 0)
            slot = &g;
    if (!slot) {
        slot = &plan->graphs[0];
        for (auto& g : plan->graphs)
            if (g.last_use < slot->last_use) slot = &g;
        if (slot->exec) { cudaGraphExecDestroy(slot->exec); slot->exec = nullptr; }
        cudaGraph_t graph = nullptr;
        int rc = CLANE_OK;
        cudaError_t ce = cudaSuccess;
        if (!loop) {
            CLANE_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            rc = enqueue_sweeps(plan, a, Z, nz, c0, n_sweeps, st);
            ce = cudaStreamEndCapture(st, &graph);
        } else {
            // graph = one conditional WHILE node; its body graph is filled by capturing the batch + the condition kernel
            cudaGraphConditionalHandle handle;
            cudaGraphNode_t node = nullptr;
            ce = cudaGraphCreate(&graph, 0);
            if (ce == cudaSuccess) ce = cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault);
            cudaGraphNodeParams np = {};
            np.type = cudaGraphNodeTypeConditional;
            np.conditional.handle = handle;
            np.conditional.type = cudaGraphCondTypeWhile;
            np.conditional.size = 1;
            if (ce == cudaSuccess) ce = cudaGraphAddNode(&node, graph, nullptr, 0, &np);
            if (ce == cudaSuccess) {
                cudaGraph_t body = np.conditional.phGraph_out[0];
                ce = cudaStreamBeginCaptureToGraph(st, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal);
                if (ce == cudaSuccess) {
                    rc = enqueue_sweeps(plan, a, Z, nz, c0, n_sweeps, st);
                    if (rc == CLANE_OK) {
                        k_loop_condition<<<1, 1, 0, st>>>(handle, a.state);
                        if (cudaGetLastError() != cudaSuccess) rc = CLANE_EINVAL;
                    }
                    cudaGraph_t same = nullptr;
                    ce = cudaStreamEndCapture(st, &same);
                }
            }
        }
        if (rc != CLANE_OK || ce != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            if (loop) { plan->while_ok = false; return CLANE_EINVAL; }
            if (rc != CLANE_OK) return rc;
            plan->use_graphs = false;   // capture unsupported here: direct launches from now on
            return enqueue_sweeps(plan, a, Z, nz, c0, n_sweeps, st);
        }
        // per-node priorities (launch_prio): without this flag every node runs at the priority of the launching stream and
        // the hub / tail kernels queue up behind the span tasks instead of running beside them
        ce = cudaGraphInstantiateWithFlags(&slot->exec, graph, cudaGraphInstantiateFlagUseNodePriority);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) {
            slot->exec = nullptr;
            cudaGetLastError();
            if (loop) { plan->while_ok = false; return CLANE_EINVAL; }
            return (int)ce;
        }
        memcpy(slot->key, key, sizeof(key));
        slot->gamma = a.gamma; slot->log_cap = a.log_cap; slot->n_sweeps = n_sweeps; slot->nz = nz; slot->c0 = c0;
        slot->loop = loop;
    }
    slot->last_use = ++plan->graph_clock;
    CLANE_CUDA(cudaGraphLaunch(slot->exec, st));
    return CLANE_OK;
}

static int ensure_coloff(clane_plan* plan, const int32_t* d_col, cudaStream_t st) {
    if (plan->e > 0 && plan->coloff_src != d_col) {   // first sweep with this column array
        k_col_offsets<<<(unsigned)((plan->e + 255) / 256), 256, 0, st>>>(d_col, plan->e, plan->ld, plan->d_coloff);
        CLANE_LAUNCH_CHECK();
        plan->coloff_src = d_col;
    }
    return CLANE_OK;
}

int clane_sweep(clane_plan* plan, const float* d_X, const float* d_Zcur, float* d_Znext, const int32_t* d_rowptr,
                const int32_t* d_col, const float* d_w, float gamma, float* d_amount, clane_patience* d_state,
                float* d_amounts_log, int32_t log_cap, clane_stream_t s) {
    if (!plan || !plan->has_schedule || !d_X || !d_Zcur || !d_Znext || !d_rowptr) return CLANE_EINVAL;
    if (plan->e > 0 && (!d_col || !d_w)) return CLANE_EINVAL;
    cudaStream_t st = (cudaStream_t)s;
    int rc = ensure_coloff(plan, d_col, st);
    if (rc != CLANE_OK) return rc;
    SweepArgs a{d_X, d_rowptr, d_col, d_w, gamma, d_amount, d_state, d_amounts_log, log_cap};
    float* Z[2] = {const_cast<float*>(d_Zcur), d_Znext};
    return launch_sweeps(plan, a, Z, 2, 0, 1, 0, st);
}

int clane_sweeps(clane_plan* plan, const float* d_X, float* const* d_Z3, int32_t cur, const int32_t* d_rowptr,
                 const int32_t* d_col, const float* d_w, float gamma, int32_t n_sweeps, int32_t until_stop,
                 clane_patience* d_state, float* d_amounts_log, int32_t log_cap, clane_stream_t s) {
    if (!plan || !plan->has_schedule || !d_X || !d_Z3 || !d_Z3[0] || !d_Z3[1] || !d_Z3[2] || !d_rowptr || !d_state ||
        cur < 0 || cur > 2 || n_sweeps < 0)
        return CLANE_EINVAL;
    if (plan->e > 0 && (!d_col || !d_w)) return CLANE_EINVAL;
    cudaStream_t st = (cudaStream_t)s;
    int rc = ensure_coloff(plan, d_col, st);
    if (rc != CLANE_OK) return rc;
    SweepArgs a{d_X, d_rowptr, d_col, d_w, gamma, nullptr, d_state, d_amounts_log, log_cap};
    if (until_stop) {
        if (!plan->while_ok) return CLANE_EUNSUPPORTED;
        // the WHILE body always starts at buffer `cur` (kWhileBatch is a multiple of 3)
        rc = launch_sweeps(plan, a, d_Z3, 3, cur, kWhileBatch, 1, st);
        return rc == CLANE_EINVAL ? CLANE_EUNSUPPORTED : rc;
    }
    // whole batches replay one cached graph per starting buffer (kSweepBatch is a multiple of 3: the rotation closes)
    int done = 0;
    while (n_sweeps - done >= kSweepBatch) {
        rc = launch_sweeps(plan, a, d_Z3, 3, (cur + done) % 3, kSweepBatch, 0, st);
        if (rc != CLANE_OK) return rc;
        done += kSweepBatch;
    }
    if (n_sweeps > done) rc = launch_sweeps(plan, a, d_Z3, 3, (cur + done) % 3, n_sweeps - done, 0, st);
    return rc;
}

// A bounded, short run of sweeps enqueued directly (no graph): what a propagate() of a few sweeps wants -- building and
// instantiating a graph costs ~1.2 ms at arxiv shape, the direct launches of 20 sweeps stay ahead of the device.  Same
// pipeline and the same device-side patience as clane_sweeps (sweeps after the stop are no-ops).  Library-internal
// (the session API); not part of include/clane_b200.h.
int clane_internal_sweeps_direct(clane_plan* plan, const float* d_X, float* const* d_Z3, int32_t cur, const int32_t* d_rowptr,
                                 const int32_t* d_col, const float* d_w, float gamma, int32_t n_sweeps, clane_patience* d_state,
                                 float* d_amounts_log, int32_t log_cap, clane_stream_t s) {
    if (!plan || !plan->has_schedule || !d_X || !d_Z3 || !d_rowptr || !d_state || cur < 0 || cur > 2 || n_sweeps < 0)
        return CLANE_EINVAL;
    cudaStream_t st = (cudaStream_t)s;
    int rc = ensure_coloff(plan, d_col, st);
    if (rc != CLANE_OK) return rc;
    SweepArgs a{d_X, d_rowptr, d_col, d_w, gamma, nullptr, d_state, d_amounts_log, log_cap};
    return enqueue_sweeps(plan, a, d_Z3, 3, cur, n_sweeps, st);
}

int clane_l1_diff(clane_plan* plan, const float* d_Za, const float* d_Zb, float* d_out, clane_stream_t s) {
    if (!plan || !d_Za || !d_Zb || !d_out) return CLANE_EINVAL;
    ElemAbsDiff el{d_Za, d_Zb, plan->d, plan->ld};
    return cascade_launch(el, (int64_t)plan->n * plan->d, plan->d_p1, plan->d_p2, d_out, nullptr, nullptr, 0,
                          (cudaStream_t)s);
}

int clane_l1_partial(clane_plan* plan, const float* d_Za, const float* d_Zb, int64_t node_lo, int64_t node_hi,
                     float* d_p1, clane_stream_t s) {
    if (!plan || !d_Za || !d_Zb || !d_p1) return CLANE_EINVAL;
    ElemAbsDiff el{d_Za, d_Zb, plan->d, plan->ld};
    return cascade_launch_l01(el, (int64_t)plan->n * plan->d, node_lo, node_hi, d_p1, nullptr, (cudaStream_t)s);
}

int clane_l1_finish(clane_plan* plan, const float* d_Za, const float* d_Zb, float* d_p1, float* d_out,
                    clane_patience* d_state, float* d_amounts_log, int32_t log_cap, clane_stream_t s) {
    if (!plan || !d_Za || !d_Zb || !d_p1) return CLANE_EINVAL;
    ElemAbsDiff el{d_Za, d_Zb, plan->d, plan->ld};
    return cascade_launch_finish(el, (int64_t)plan->n * plan->d, d_p1, plan->d_p2, d_out, d_state, d_amounts_log,
                                 log_cap, nullptr, (cudaStream_t)s);
}

int clane_plan_set_peers(clane_plan* plan, int32_t n_peers, int32_t self_rank, const uint64_t* h_ptrs_a,
                         const uint64_t* h_ptrs_b) {
    if (!plan || n_peers < 0 || n_peers > kMaxPeers + 1 || (n_peers > 0 && (self_rank < 0 || self_rank >= n_peers)))
        return CLANE_EINVAL;
    if (n_peers > 0 && (!h_ptrs_a || !h_ptrs_b)) return CLANE_EINVAL;
    plan->n_peers = n_peers;
    plan->self_rank = self_rank;
    for (int r = 0; r < 16; ++r) plan->peers[2][r] = nullptr;
    for (int r = 0; r < n_peers; ++r) {
        plan->peers[0][r] = reinterpret_cast<float*>(h_ptrs_a[r]);
        plan->peers[1][r] = reinterpret_cast<float*>(h_ptrs_b[r]);
    }
    for (auto& g : plan->graphs)   // cached sweeps were captured with the old peer set
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    return CLANE_OK;
}

int clane_plan_set_peers_third(clane_plan* plan, const uint64_t* h_ptrs_c) {
    if (!plan || !h_ptrs_c || plan->n_peers < 1) return CLANE_EINVAL;
    for (int r = 0; r < plan->n_peers; ++r) plan->peers[2][r] = reinterpret_cast<float*>(h_ptrs_c[r]);
    for (auto& g : plan->graphs)
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    return CLANE_OK;
}

int clane_plan_set_multicast(clane_plan* plan, uint64_t mc_a, uint64_t mc_b) {
    if (!plan) return CLANE_EINVAL;
    plan->mc[0] = reinterpret_cast<float*>(mc_a);
    plan->mc[1] = reinterpret_cast<float*>(mc_b);
    for (auto& g : plan->graphs)
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    return CLANE_OK;
}

int clane_l1_tail_values(clane_plan* plan, const float* d_Za, const float* d_Zb, float* d_vals, clane_stream_t s) {
    if (!plan || !d_Za || !d_Zb || !d_vals) return CLANE_EINVAL;
    ElemAbsDiff el{d_Za, d_Zb, plan->d, plan->ld};
    k_tail_values<<<1, 32, 0, (cudaStream_t)s>>>(el, cascade_shape((int64_t)plan->n * plan->d), d_vals);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

int clane_l1_finish_values(clane_plan* plan, float* d_p1, const float* d_vals, float* d_out, clane_patience* d_state,
                           float* d_amounts_log, int32_t log_cap, clane_stream_t s) {
    if (!plan || !d_p1 || !d_vals) return CLANE_EINVAL;
    ElemValues el{d_vals};
    return cascade_launch_finish(el, (int64_t)plan->n * plan->d, d_p1, plan->d_p2, d_out, d_state, d_amounts_log,
                                 log_cap, nullptr, (cudaStream_t)s);
}

int clane_plan_trace(clane_plan* plan, int enable, unsigned long long* h_out) {
    if (!plan) return CLANE_EINVAL;
    const size_t words = (size_t)kTraceSweeps * kTraceSlots * 2;
    if (h_out && plan->d_trace) {      // read back what the last enqueue left
        CLANE_CUDA(cudaDeviceSynchronize());
        CLANE_CUDA(cudaMemcpy(h_out, plan->d_trace, words * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
    if (enable) {
        if (!plan->d_trace) CLANE_CUDA(cudaMalloc(&plan->d_trace, words * sizeof(unsigned long long)));
        std::vector<unsigned long long> init(words);
        for (size_t i = 0; i < words; ++i) init[i] = (i & 1) ? 0ull : ~0ull;   // {min start, max end}
        CLANE_CUDA(cudaMemcpy(plan->d_trace, init.data(), words * sizeof(unsigned long long), cudaMemcpyHostToDevice));
    } else if (plan->d_trace) {
        cudaFree(plan->d_trace);
        plan->d_trace = nullptr;
    }
    for (auto& g : plan->graphs)       // the stamps are arguments of the captured kernels: re-capture
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    return CLANE_OK;
}

int clane_plan_profile(clane_plan* plan, int enable) {
    if (!plan) return CLANE_EINVAL;
    if (enable && !plan->ev_prof[0])
        for (int i = 0; i < 8; ++i) CLANE_CUDA(cudaEventCreate(&plan->ev_prof[i]));
    if (plan->profile != (enable != 0))   // the brackets are event-record nodes of the replayed sweep graphs: re-capture
        for (auto& g : plan->graphs)
            if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    plan->profile = enable != 0;
    return CLANE_OK;
}

int clane_plan_profile_read(clane_plan* plan, float* h_ms) {
    if (!plan || !h_ms || !plan->ev_prof[0]) return CLANE_EINVAL;
    CLANE_CUDA(cudaEventSynchronize(plan->ev_prof[3]));
    CLANE_CUDA(cudaEventElapsedTime(&h_ms[0], plan->ev_prof[1], plan->ev_prof[2]));   // row kernel
    CLANE_CUDA(cudaEventElapsedTime(&h_ms[1], plan->ev_prof[0], plan->ev_prof[3]));   // whole sweep
    h_ms[2] = h_ms[3] = 0.0f;
    if (plan->prof_mask & (1u << 6))
        CLANE_CUDA(cudaEventElapsedTime(&h_ms[2], plan->ev_prof[6], plan->ev_prof[3]));   // exact L1 tail
    if ((plan->prof_mask & (3u << 4)) == (3u << 4)) {
        CLANE_CUDA(cudaEventSynchronize(plan->ev_prof[5]));
        CLANE_CUDA(cudaEventElapsedTime(&h_ms[3], plan->ev_prof[4], plan->ev_prof[5]));   // chains of the long hub rows
    }
    return CLANE_OK;
}

int clane_patience_reset(clane_patience* d_state, int32_t tol, int32_t max_sweeps, clane_stream_t s) {
    if (!d_state) return CLANE_EINVAL;
    k_patience_reset<<<1, 1, 0, (cudaStream_t)s>>>(d_state, tol, max_sweeps);
    CLANE_LAUNCH_CHECK();
    return CLANE_OK;
}

// one-time: opt in to > 48 KB dynamic shared memory for the sweep kernel
int clane_internal_prepare_kernels(void) {
    static bool done = false;
    if (done) return CLANE_OK;
    CLANE_CUDA(cudaFuncSetAttribute(k_hub_chain<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kHeavySmemBytes));
    CLANE_CUDA(cudaFuncSetAttribute(k_dots<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dot_smem<false>()));
    CLANE_CUDA(cudaFuncSetAttribute(k_dots<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dot_smem<true>()));
    // the cascade level-0/1 kernel needs step*NQ*128 bytes (<= 32 KB for step = 128, NQ = 2)
    done = true;
    return CLANE_OK;
}

}  // extern "C"
