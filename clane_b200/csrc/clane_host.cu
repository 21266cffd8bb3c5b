// libclane_b200.so -- host side of the C-ABI: graph build, row schedule, host-buffer session.
//
// Reference call sites replaced (all under /root/reference/clane/):
//   graph.py:104-110  Graph.A (coalesce)              -> clane_csr_from_edges
//   graph.py:130-138  Graph.Z / set_Z                  -> clane_session_get_z / set_z
//   embedder.py:71-108 Embedder.propagate              -> clane_session_propagate
//   embedder.py:56-69  Embedder.iterate                -> clane_session_iterate
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <numeric>
#include <vector>

#include "common.cuh"
#include "plan.cuh"
#include "program.cuh"

namespace {

// host threads this process may run on (its affinity mask), capped by the amount of work
int host_threads(int64_t work_units) {
    int n = 1;
#ifdef __linux__
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
#else
    n = (int)std::thread::hardware_concurrency();
#endif
    return (int)std::max<int64_t>(1, std::min<int64_t>(std::min(n, 64), work_units));
}

// fn(lo, hi, t) over [0, total) cut into one contiguous chunk per thread t (the cut depends only on total and nthreads)
// Workers never let an exception escape their thread (that would be std::terminate across the C ABI): the first
// failure is flagged and re-raised as bad_alloc on the calling thread after the join; a thread that cannot be
// created leaves its share of the work to the caller.
template <class F>
void parallel_chunks(int64_t total, int nthreads, F&& fn) {
    if (nthreads <= 1 || total < 2) { fn((int64_t)0, total, 0); return; }
    std::vector<std::thread> th;
    std::atomic<int> failed{0};
    for (int t = 0; t < nthreads; ++t) {
        const int64_t lo = total * t / nthreads, hi = total * (t + 1) / nthreads;
        auto job = [&fn, &failed, lo, hi, t] {
            try { if (lo < hi) fn(lo, hi, t); } catch (...) { failed.store(1); }
        };
        try { th.emplace_back(job); } catch (...) { job(); }
    }
    for (auto& x : th) x.join();
    if (failed.load()) throw std::bad_alloc();
}

// fn(i) for every i in [0, total), items handed out dynamically (uneven items: buckets of a power-law graph)
template <class F>
void parallel_items(int64_t total, int nthreads, F&& fn) {
    if (nthreads <= 1 || total < 2) { for (int64_t i = 0; i < total; ++i) fn(i); return; }
    std::atomic<int64_t> next{0};
    std::atomic<int> failed{0};
    std::vector<std::thread> th;
    auto job = [&] {
        try { for (int64_t i; (i = next.fetch_add(1, std::memory_order_relaxed)) < total;) fn(i); }
        catch (...) { failed.store(1); }
    };
    for (int t = 0; t < nthreads; ++t) {
        try { th.emplace_back(job); } catch (...) { break; }
    }
    job();   // the caller works too (and does everything if no thread could be created)
    for (auto& x : th) x.join();
    if (failed.load()) throw std::bad_alloc();
}

}  // namespace

extern "C" {

int64_t clane_csr_from_edges(const int64_t* h_src, const int64_t* h_dst, int64_t e_raw, int64_t n, int32_t* h_rowptr,
                             int32_t* h_col) {
    if (e_raw < 0 || n < 0 || !h_rowptr || (e_raw > 0 && (!h_src || !h_dst || !h_col))) return CLANE_EINVAL;
    if (n > INT32_MAX || e_raw > INT32_MAX) return CLANE_ERANGE;
    try {
        // The order torch's coalesce() produces: row-major, ascending column, duplicates merged.  Two-level counting
        // sort on all host threads, no atomics and no random writes beyond a cache-sized window:
        //   1. rows are grouped into buckets of 2^shift rows; every thread histograms its chunk of the edge list;
        //   2. every thread scatters its chunk into per-(bucket, thread) regions (sequential writes per bucket);
        //   3. every bucket (a few 10^4 edges: cache resident) is counting-sorted by row, each row's destinations
        //      sorted and made unique; 4. a scan of the unique counts gives rowptr; 5. rows are compacted into col.
        int shift = 0;
        while ((n >> shift) > 4096) ++shift;
        const int64_t nbuckets = (n >> shift) + 1;
        const int nt = host_threads(std::max<int64_t>(e_raw, n) / 65536 + 1);
        std::vector<int64_t> hist((size_t)nt * nbuckets, 0);          // [thread][bucket] -> counts, then write cursors
        std::atomic<int> bad{0};
        parallel_chunks(e_raw, nt, [&](int64_t lo, int64_t hi, int t) {
            int64_t* h = hist.data() + (size_t)t * nbuckets;
            for (int64_t e = lo; e < hi; ++e) {
                const int64_t s = h_src[e], d = h_dst[e];
                if (s < 0 || s >= n || d < 0 || d >= n) { bad.store(1, std::memory_order_relaxed); return; }
                h[s >> shift]++;
            }
        });
        if (bad.load()) return CLANE_ERANGE;
        std::vector<int64_t> bstart((size_t)nbuckets + 1, 0);
        {
            int64_t run = 0;
            for (int64_t b = 0; b < nbuckets; ++b) {
                bstart[(size_t)b] = run;
                for (int t = 0; t < nt; ++t) {
                    const int64_t c = hist[(size_t)t * nbuckets + b];
                    hist[(size_t)t * nbuckets + b] = run;              // this thread's write cursor inside the bucket
                    run += c;
                }
            }
            bstart[(size_t)nbuckets] = run;
        }
        struct Pair { int32_t row, dst; };
        std::vector<Pair> staged((size_t)std::max<int64_t>(e_raw, 1));
        parallel_chunks(e_raw, nt, [&](int64_t lo, int64_t hi, int t) {
            int64_t* cur = hist.data() + (size_t)t * nbuckets;
            for (int64_t e = lo; e < hi; ++e) {
                const int64_t s = h_src[e];
                staged[(size_t)cur[s >> shift]++] = Pair{(int32_t)s, (int32_t)h_dst[e]};
            }
        });
        std::vector<int32_t> tmp((size_t)std::max<int64_t>(e_raw, 1));   // destinations, row-major, each row sorted + unique at its front
        std::vector<int32_t> start((size_t)n + 1, 0), uniq((size_t)n + 1, 0);
        parallel_items(nbuckets, nt, [&](int64_t bk) {
            const int64_t r0 = bk << shift, r1 = std::min<int64_t>(n, (bk + 1) << shift);
            if (r0 >= r1) return;
            const Pair* p = staged.data() + bstart[(size_t)bk];
            const int64_t cnt = bstart[(size_t)bk + 1] - bstart[(size_t)bk];
            std::vector<int32_t> c((size_t)(r1 - r0) + 1, 0);
            for (int64_t i = 0; i < cnt; ++i) c[(size_t)(p[i].row - r0) + 1]++;
            for (int64_t r = 0; r < r1 - r0; ++r) c[(size_t)r + 1] += c[(size_t)r];
            const int64_t base = bstart[(size_t)bk];
            for (int64_t r = 0; r < r1 - r0; ++r) start[(size_t)(r0 + r)] = (int32_t)(base + c[(size_t)r]);
            std::vector<int32_t> cur(c.begin(), c.end() - 1);
            for (int64_t i = 0; i < cnt; ++i) tmp[(size_t)(base + cur[(size_t)(p[i].row - r0)]++)] = p[i].dst;
            for (int64_t r = 0; r < r1 - r0; ++r) {
                int32_t* a = tmp.data() + base + c[(size_t)r];
                int32_t* b = tmp.data() + base + c[(size_t)r + 1];
                if (b - a > 1) std::sort(a, b);
                uniq[(size_t)(r0 + r)] = (int32_t)(std::unique(a, b) - a);
            }
        });
        int64_t out = 0;
        h_rowptr[0] = 0;
        for (int64_t v = 0; v < n; ++v) {
            out += uniq[(size_t)v];
            h_rowptr[v + 1] = (int32_t)out;
        }
        parallel_chunks(n, nt, [&](int64_t lo, int64_t hi, int) {
            for (int64_t v = lo; v < hi; ++v)
                if (uniq[(size_t)v])
                    memcpy(h_col + h_rowptr[v], tmp.data() + start[(size_t)v], (size_t)uniq[(size_t)v] * sizeof(int32_t));
        });
        return out;
    } catch (...) {
        return (int64_t)CLANE_ENOMEM;   // negative, like every error of this call (a positive value is an edge count)
    }
}

// ---------------------------------------------------------------------------------------------
// plan: degree-sorted row blocks + cascade scratch
// ---------------------------------------------------------------------------------------------
int clane_group_schedule(const int32_t* h_rowptr, int32_t n, int32_t d, int32_t row_lo, int32_t row_hi,
                         int32_t hub_threshold, int32_t span_edges, int32_t* h_span_row, int32_t* h_span_meta,
                         int32_t* n_spans, int32_t* h_fix_groups, int32_t* n_fix_groups, int32_t* h_hub_rows,
                         int32_t* n_hub_rows, int32_t* group_rows, int32_t* fused_l1) {
    if (!h_rowptr || n < 0 || d < 1 || row_lo < 0 || row_hi > n || row_lo > row_hi || hub_threshold < 8 ||
        span_edges < 8 || !h_span_row || !h_span_meta || !n_spans || !h_fix_groups || !n_fix_groups || !h_hub_rows ||
        !n_hub_rows || !group_rows || !fused_l1)
        return CLANE_EINVAL;
    // fused L1: a group of G rows is exactly one level-0 chunk of the cascade over n*d
    clane::CascadeShape sh = clane::cascade_shape((int64_t)n * d);
    const int64_t chunk = sh.step * 32;
    int32_t G = 8, fuse = 0;
    if ((d == 32 || d == 64 || d == 128) && row_lo == 0 && row_hi == n && chunk % d == 0 && chunk / d <= 32 &&
        chunk <= 1024) {   // a warp parks one chunk of |delta| in 4 KB of shared memory
        G = (int32_t)(chunk / d);
        fuse = 1;
    }
    const int32_t n_groups = (row_hi - row_lo + G - 1) / G;
    struct Span { int32_t row, nrows, direct; int64_t work; };
    std::vector<Span> spans;
    std::vector<int32_t> fix, hub_rows;
    spans.reserve((size_t)n_groups + 16);
    for (int32_t g = 0; g < n_groups; ++g) {
        const int32_t r0 = row_lo + g * G, r1 = std::min(r0 + G, row_hi);
        bool has_hub = false;
        const size_t first_span = spans.size();
        Span cur{r0, 0, 0, 0};
        for (int32_t v = r0; v < r1; ++v) {
            const int32_t k = h_rowptr[v + 1] - h_rowptr[v];
            if (k > hub_threshold) {      // hub rows are never inside a span: its edge stream stays contiguous
                has_hub = true;
                hub_rows.push_back(v);
                if (cur.work > 0) spans.push_back(cur);
                cur = Span{v + 1, 0, 0, 0};
                continue;
            }
            if (cur.work > 0 && cur.work + k > span_edges) {   // close the span before this row
                spans.push_back(cur);
                cur = Span{v, 0, 0, 0};
            }
            cur.nrows++;
            cur.work += k;
        }
        if (cur.work > 0) spans.push_back(cur);
        const size_t made = spans.size() - first_span;
        // one span covering the whole group and no hub row: the warp produces the chunk partial itself
        if (made == 1 && !has_hub && spans.back().row == r0 && spans.back().nrows == r1 - r0) spans.back().direct = 1;
        else if (fuse && (made > 0 || has_hub)) fix.push_back(g);
        // groups of sinks only are never updated (embedder.py:88-89): no span, partial stays +0
    }
    {   // spans by edge count, descending, ties in row order: a stable counting sort (the keys are <= a hub row's length)
        int64_t maxw = 0;
        for (const Span& sp : spans) maxw = std::max(maxw, sp.work);
        if (maxw <= (int64_t)1 << 22) {
            std::vector<uint32_t> first((size_t)maxw + 2, 0);
            for (const Span& sp : spans) first[(size_t)(maxw - sp.work) + 1]++;
            for (size_t i = 1; i < first.size(); ++i) first[i] += first[i - 1];
            std::vector<Span> sorted(spans.size());
            for (const Span& sp : spans) sorted[first[(size_t)(maxw - sp.work)]++] = sp;
            spans.swap(sorted);
        } else {
            std::stable_sort(spans.begin(), spans.end(), [](const Span& x, const Span& y) { return x.work > y.work; });
        }
    }
    auto by_degree_desc = [&](int32_t x, int32_t y) {
        const int32_t kx = h_rowptr[x + 1] - h_rowptr[x], ky = h_rowptr[y + 1] - h_rowptr[y];
        return kx != ky ? kx > ky : x < y;
    };
    std::sort(hub_rows.begin(), hub_rows.end(), by_degree_desc);
    for (size_t i = 0; i < spans.size(); ++i) {
        h_span_row[i] = spans[i].row;
        h_span_meta[i] = spans[i].nrows | (spans[i].direct << 8);
    }
    std::copy(fix.begin(), fix.end(), h_fix_groups);
    std::copy(hub_rows.begin(), hub_rows.end(), h_hub_rows);
    *n_spans = (int32_t)spans.size();
    *n_fix_groups = (int32_t)fix.size();
    *n_hub_rows = (int32_t)hub_rows.size();
    *group_rows = G;
    *fused_l1 = fuse;
    return CLANE_OK;
}

int clane_plan_destroy(clane_plan* plan) {
    if (!plan) return CLANE_OK;
    cudaFree(plan->d_tasks); cudaFree(plan->d_long_rows); cudaFree(plan->d_fix_groups); cudaFree(plan->d_hub_rows);
    cudaFree(plan->d_hub_info); cudaFree(plan->d_hubS); cudaFree(plan->d_hubT);
    for (cudaEvent_t ev : plan->evs) cudaEventDestroy(ev);
    if (plan->side) cudaStreamDestroy(plan->side);
    if (plan->side2) cudaStreamDestroy(plan->side2);
    if (plan->tail) cudaStreamDestroy(plan->tail);
    cudaFree(plan->d_P0); cudaFree(plan->d_coloff); cudaFree(plan->d_trace);
    for (auto& g : plan->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    for (int i = 0; i < 8; ++i) if (plan->ev_prof[i]) cudaEventDestroy(plan->ev_prof[i]);
    cudaFree(plan->d_p1); cudaFree(plan->d_p2);
    delete plan;
    return CLANE_OK;
}

#define PLAN_CUDA(x)                                               \
    do {                                                           \
        cudaError_t e__ = (x);                                     \
        if (e__ != cudaSuccess) { clane_plan_destroy(plan); return (int)e__; } \
    } while (0)

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// the sweep's program: every control decision of k_sweep_rows, made once per graph (sweep.cuh)
// ---------------------------------------------------------------------------------------------
namespace {

// hub segments (16 full blocks each, longest rows first), then the spans by edge count, descending
int build_program(const int32_t* h_rowptr, int fuse, const int32_t* srow, const int32_t* smeta, int32_t n_spans,
                  const int32_t* hrows, int32_t n_hrows, std::vector<clane::SweepTask>& tasks,
                  std::vector<int32_t>& blk0, int64_t* hub_blocks) {
    using namespace clane;
    try {
        blk0.assign((size_t)std::max(n_hrows, 1), 0);
        size_t n_seg = 0;
        for (int32_t h = 0; h < n_hrows; ++h)
            n_seg += (size_t)((h_rowptr[hrows[h] + 1] - h_rowptr[hrows[h]]) / 8 + kSegEdges / 8 - 1) / (kSegEdges / 8);
        tasks.reserve(tasks.size() + n_seg + (size_t)n_spans);
        int64_t blocks = 0;
        for (int32_t h = 0; h < n_hrows; ++h) {
            const int32_t v = hrows[h], a = h_rowptr[v], nblk = (h_rowptr[v + 1] - a) / 8;
            if (blocks + nblk > INT32_MAX || h >= (1 << 21)) return CLANE_ERANGE;
            blk0[h] = (int32_t)blocks;
            for (int32_t b0 = 0; b0 < nblk; b0 += kSegEdges / 8) {
                const int32_t nbk = std::min<int32_t>(kSegEdges / 8, nblk - b0);
                tasks.push_back(SweepTask{a + b0 * 8, nbk * 8, b0, kTaskSegment | (h << kTaskHubShift), nbk, (int32_t)blocks,
                                          nblk, 0});
            }
            blocks += (nblk + 1) & ~1;
        }
        *hub_blocks = blocks;
        for (int32_t i = 0; i < n_spans; ++i) {
            const int32_t r0 = srow[i], nrows = smeta[i] & 0xff, direct = (smeta[i] >> 8) && fuse;
            const int32_t e0 = h_rowptr[r0];
            tasks.push_back(SweepTask{e0, h_rowptr[r0 + nrows] - e0, r0, nrows | (direct ? kTaskDirect : 0), 0, 0, 0, 0});
        }
    } catch (const std::bad_alloc&) {
        return CLANE_ENOMEM;
    }
    return CLANE_OK;
}

}  // namespace

extern "C" {

int clane_sweep_program(const int32_t* h_rowptr, int32_t n, int32_t d, int32_t row_lo, int32_t row_hi,
                        int32_t hub_threshold, int32_t span_edges, int32_t* h_tasks, int64_t task_cap, int64_t* n_tasks) {
    if (!h_rowptr || !n_tasks || n < 0 || row_lo < 0 || row_hi > n || row_lo > row_hi) return CLANE_EINVAL;
    const size_t cap = (size_t)(row_hi - row_lo) + 1;
    try {
        std::vector<int32_t> srow(cap), smeta(cap), fix(cap), hrows(cap), blk0;
        std::vector<clane::SweepTask> tasks;
        int32_t n_spans = 0, n_fix = 0, n_hrows = 0, G = 0, fuse = 0;
        int rc = clane_group_schedule(h_rowptr, n, d, row_lo, row_hi, hub_threshold, span_edges, srow.data(), smeta.data(),
                                      &n_spans, fix.data(), &n_fix, hrows.data(), &n_hrows, &G, &fuse);
        if (rc != CLANE_OK) return rc;
        int64_t hub_blocks = 0;
        rc = build_program(h_rowptr, fuse, srow.data(), smeta.data(), n_spans, hrows.data(), n_hrows, tasks, blk0, &hub_blocks);
        if (rc != CLANE_OK) return rc;
        *n_tasks = (int64_t)tasks.size();
        if (h_tasks) {
            if (task_cap < (int64_t)tasks.size()) return CLANE_EWORKSPACE;
            memcpy(h_tasks, tasks.data(), tasks.size() * sizeof(clane::SweepTask));
        }
    } catch (const std::bad_alloc&) {
        return CLANE_ENOMEM;
    }
    return CLANE_OK;
}

int clane_plan_create(clane_plan** out, int32_t n, int64_t e, int32_t d, const int32_t* h_rowptr, int32_t row_lo,
                      int32_t row_hi, int32_t hub_threshold) {
    using namespace clane;
    if (!out || n < 0 || e < 0 || d < 1) return CLANE_EINVAL;
    if (h_rowptr && (row_lo < 0 || row_hi > n || row_lo > row_hi)) return CLANE_EINVAL;
    if (h_rowptr && h_rowptr[n] != e) return CLANE_EINVAL;
    int rc = clane_internal_prepare_kernels();
    if (rc != CLANE_OK) return rc;
    clane_plan* plan = new (std::nothrow) clane_plan();
    if (!plan) return (int)cudaErrorMemoryAllocation;
    plan->n = n; plan->e = e; plan->d = d; plan->ld = clane_padded_ld(d);
    // The kernels address rows of [n, ld] matrices by 32-bit unsigned float4 indices (the sweep's gathers and row
    // pieces, the per-edge dots): n * ld <= 2^34 floats, 64 GiB per matrix.  A sweep at that bound would need 256 GiB
    // for X and its three Z buffers, so the bound refuses no graph whose sweep fits a 180 GB device.
    if ((int64_t)n * plan->ld > CLANE_MAX_MATRIX_FLOATS) { delete plan; return CLANE_ERANGE; }
    // Hub rows bound the critical path of a sweep: a row of k neighbours is an in-order chain of k/8 batches on
    // one warp (~150 ns per neighbour), so rows longer than 1/4096 of the edges this plan sweeps (a few percent of
    // the row kernel's duration) go to the segment + chain path.
    const int64_t e_local = h_rowptr ? (int64_t)h_rowptr[row_hi] - h_rowptr[row_lo] : e;
    const int64_t auto_thr = std::min<int64_t>(16384, std::max<int64_t>(256, (e_local / 4096 + 7) / 8 * 8));
    plan->hub_threshold = hub_threshold > 0 ? std::min(std::max(hub_threshold, 8), 1 << 20) : (int32_t)auto_thr;
    plan->span_edges = 128;
    plan->nslab = (plan->ld + 127) / 128;
    plan->limit = (d / 16) * 16;
    plan->ntail4 = (plan->ld - plan->limit) / 4;
    plan->nslab32b = (plan->limit + 31) / 32;

    // cascade scratch: L1 over n*d (one quantity) and the norms over e*d (two quantities)
    const int64_t n_l1 = (int64_t)n * d, n_nrm = e * (int64_t)d;
    plan->p1_floats = std::max(clane::cascade_p1_floats(n_l1, 1), clane::cascade_p1_floats(n_nrm, 2)) + 64;
    plan->p2_floats = std::max(clane::cascade_p2_floats(n_l1, 1), clane::cascade_p2_floats(n_nrm, 2)) + 64;
    PLAN_CUDA(cudaMalloc(&plan->d_p1, plan->p1_floats * sizeof(float)));
    PLAN_CUDA(cudaMalloc(&plan->d_p2, plan->p2_floats * sizeof(float)));
    PLAN_CUDA(cudaMemset(plan->d_p1, 0, plan->p1_floats * sizeof(float)));
    PLAN_CUDA(cudaMemset(plan->d_p2, 0, plan->p2_floats * sizeof(float)));
    if (!h_rowptr) { *out = plan; return CLANE_OK; }

    plan->has_schedule = true;
    PLAN_CUDA(cudaMalloc(&plan->d_coloff, std::max<size_t>((size_t)e, 1) * sizeof(int32_t)));
    plan->row_lo = row_lo; plan->row_hi = row_hi;
    plan->edge_lo = h_rowptr[row_lo]; plan->edge_hi = h_rowptr[row_hi];
    const size_t cap = (size_t)(row_hi - row_lo) + 1;
    std::vector<int32_t> srow(cap), smeta(cap), fix(cap), hrows(cap);
    int32_t n_spans = 0, n_fix = 0, n_hrows = 0;
    rc = clane_group_schedule(h_rowptr, n, d, row_lo, row_hi, plan->hub_threshold, plan->span_edges, srow.data(),
                              smeta.data(), &n_spans, fix.data(), &n_fix, hrows.data(), &n_hrows, &plan->G, &plan->fuse);
    if (rc != CLANE_OK) { clane_plan_destroy(plan); return rc; }
    plan->n_groups = (row_hi - row_lo + plan->G - 1) / plan->G;
    plan->n_spans = n_spans;
    plan->n_fix_groups = n_fix;
    plan->n_hub_rows = n_hrows;
    plan->n_long_hub_rows = 0;
    for (int32_t h = 0; h < n_hrows; ++h)
        if ((h_rowptr[hrows[h] + 1] - h_rowptr[hrows[h]]) / 8 >= kLongBlocks) plan->n_long_hub_rows = h + 1;

    std::vector<SweepTask> tasks;
    std::vector<int32_t> blk0;
    rc = build_program(h_rowptr, plan->fuse, srow.data(), smeta.data(), n_spans, hrows.data(), n_hrows, tasks, blk0,
                       &plan->hub_blocks);
    if (rc != CLANE_OK) { clane_plan_destroy(plan); return rc; }
    plan->n_tasks = (int32_t)tasks.size();
    plan->n_seg_tasks = plan->n_tasks - n_spans;
    {   // rows the row softmax of build_P gives a whole CTA (>= 64 neighbours)
        std::vector<int32_t> longr;
        for (int32_t v = row_lo; v < row_hi; ++v)
            if (h_rowptr[v + 1] - h_rowptr[v] >= 64) longr.push_back(v);
        plan->n_long_rows = (int32_t)longr.size();
        if (!longr.empty()) {
            PLAN_CUDA(cudaMalloc(&plan->d_long_rows, longr.size() * sizeof(int32_t)));
            PLAN_CUDA(cudaMemcpy(plan->d_long_rows, longr.data(), longr.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        }
    }
    PLAN_CUDA(cudaMalloc(&plan->d_tasks, std::max<size_t>(tasks.size(), 1) * sizeof(SweepTask)));
    PLAN_CUDA(cudaMalloc(&plan->d_fix_groups, std::max<size_t>(n_fix, 1) * sizeof(int32_t)));
    PLAN_CUDA(cudaMalloc(&plan->d_hub_rows, std::max<size_t>(n_hrows, 1) * sizeof(int32_t)));
    PLAN_CUDA(cudaMalloc(&plan->d_hub_info, std::max<size_t>(n_hrows, 1) * sizeof(int4)));
    if (!tasks.empty()) PLAN_CUDA(cudaMemcpy(plan->d_tasks, tasks.data(), tasks.size() * sizeof(SweepTask), cudaMemcpyHostToDevice));
    if (n_fix) PLAN_CUDA(cudaMemcpy(plan->d_fix_groups, fix.data(), n_fix * sizeof(int32_t), cudaMemcpyHostToDevice));
    if (n_hrows) {
        PLAN_CUDA(cudaMemcpy(plan->d_hub_rows, hrows.data(), n_hrows * sizeof(int32_t), cudaMemcpyHostToDevice));
        std::vector<int4> info((size_t)n_hrows);
        for (int32_t h = 0; h < n_hrows; ++h) {
            const int32_t v = hrows[h];
            info[h] = make_int4(v, h_rowptr[v], h_rowptr[v + 1] - h_rowptr[v], blk0[h]);
        }
        PLAN_CUDA(cudaMemcpy(plan->d_hub_info, info.data(), n_hrows * sizeof(int4), cudaMemcpyHostToDevice));
        const size_t nb = (size_t)plan->hub_blocks;
        PLAN_CUDA(cudaMalloc(&plan->d_hubS, std::max<size_t>(nb * plan->nslab32b * 32, 1) * 16));
        if (plan->ntail4 > 0) PLAN_CUDA(cudaMalloc(&plan->d_hubT, nb * 8 * plan->ntail4 * 16));
    }
    {   // the segments + chains run beside the span tasks on their own streams, dispatched ahead of them
        int lo = 0, hi = 0;
        PLAN_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        plan->prio_hi = hi; plan->prio_lo = lo;
        PLAN_CUDA(cudaStreamCreateWithPriority(&plan->side, cudaStreamNonBlocking, hi));
        PLAN_CUDA(cudaStreamCreateWithPriority(&plan->side2, cudaStreamNonBlocking, hi));
        PLAN_CUDA(cudaStreamCreateWithPriority(&plan->tail, cudaStreamNonBlocking, hi));
    }
    if (plan->fuse) {
        plan->p0_stride = (size_t)(plan->n_groups + 1) * 32;
        const size_t p0 = 2 * plan->p0_stride * sizeof(float);
        PLAN_CUDA(cudaMalloc(&plan->d_P0, p0));
        PLAN_CUDA(cudaMemset(plan->d_P0, 0, p0));   // dropped (all-sink) groups contribute +0 forever
    }
    *out = plan;
    return CLANE_OK;
}

int clane_plan_info(const clane_plan* plan, int32_t* group_rows, int32_t* n_spans, int32_t* n_hub_rows,
                    int32_t* n_fix_groups, int32_t* fused_l1, int32_t* launches_per_sweep) {
    if (!plan) return CLANE_EINVAL;
    if (group_rows) *group_rows = plan->G;
    if (n_spans) *n_spans = plan->n_spans;
    if (n_hub_rows) *n_hub_rows = plan->n_hub_rows;
    if (n_fix_groups) *n_fix_groups = plan->n_fix_groups;
    if (fused_l1) *fused_l1 = plan->fuse;
    // spans, [hub segments, chains of long rows, chains of short rows], then the exact L1: fused = [chunk fix-up],
    // level 1, finish; otherwise level 0 + 1, finish
    if (launches_per_sweep) {
        const int n_long = plan->n_long_hub_rows, n_short = plan->n_hub_rows - n_long;
        const int hub = plan->n_hub_rows > 0 ? 1 + (n_long > 0 ? 1 : 0) + (n_short > 0 ? 1 : 0) : 0;
        const int l1 = plan->fuse ? 2 + (plan->n_fix_groups > 0 ? 1 : 0) : 2;
        *launches_per_sweep = 1 + hub + l1;
    }
    return CLANE_OK;
}

// ---------------------------------------------------------------------------------------------
// host-buffer session
// ---------------------------------------------------------------------------------------------
struct clane_session {
    int32_t n = 0, d = 0, ld = 0;
    int64_t e = 0;
    clane_plan* plan = nullptr;
    int32_t *rowptr = nullptr, *col = nullptr, *erow = nullptr;
    float *X = nullptr, *Z[3] = {nullptr, nullptr, nullptr}, *prev = nullptr, *w = nullptr, *norms2 = nullptr;
    float *amount = nullptr, *log = nullptr;
    clane_patience* state = nullptr;
    int cur = 0;  // Z[cur] holds the current embeddings (three rotating buffers: clane_sweeps)
    int32_t log_cap = 0;
    void* pool = nullptr;               // one device allocation behind all of the pointers above (prev excepted)
    cudaStream_t stream = nullptr;
    clane_patience* h_state = nullptr;  // pinned
    float* h_stage = nullptr;           // pinned staging for padded rows
    bool p_valid = false;
};

static int copy_rows_h2d(clane_session* s, float* d_dst, const float* h_src) {
    if (s->ld == s->d) {
        CLANE_CUDA(cudaMemcpyAsync(d_dst, h_src, (size_t)s->n * s->d * sizeof(float), cudaMemcpyHostToDevice, s->stream));
    } else {
        CLANE_CUDA(cudaMemsetAsync(d_dst, 0, (size_t)s->n * s->ld * sizeof(float), s->stream));
        CLANE_CUDA(cudaMemcpy2DAsync(d_dst, (size_t)s->ld * sizeof(float), h_src, (size_t)s->d * sizeof(float),
                                     (size_t)s->d * sizeof(float), (size_t)s->n, cudaMemcpyHostToDevice, s->stream));
    }
    return CLANE_OK;
}

static int copy_rows_d2h(clane_session* s, float* h_dst, const float* d_src) {
    if (s->ld == s->d) {
        CLANE_CUDA(cudaMemcpyAsync(h_dst, d_src, (size_t)s->n * s->d * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
        return CLANE_OK;
    }
    CLANE_CUDA(cudaMemcpy2DAsync(h_dst, (size_t)s->d * sizeof(float), d_src, (size_t)s->ld * sizeof(float),
                                 (size_t)s->d * sizeof(float), (size_t)s->n, cudaMemcpyDeviceToHost, s->stream));
    return CLANE_OK;
}

int clane_session_destroy(clane_session* s) {
    if (!s) return CLANE_OK;
    clane_plan_destroy(s->plan);
    cudaFree(s->pool); cudaFree(s->prev);
    if (s->h_state) cudaFreeHost(s->h_state);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
    return CLANE_OK;
}

#define SESSION_TRY(x)                                   \
    do {                                                 \
        int rc__ = (x);                                  \
        if (rc__ != CLANE_OK) { clane_session_destroy(s); return rc__; } \
    } while (0)
#define SESSION_CUDA(x) SESSION_TRY((int)(x))

int clane_session_create(clane_session** out, int32_t n, int64_t e, int32_t d, const int32_t* h_rowptr,
                         const int32_t* h_col, const float* h_X, int32_t hub_threshold) {
    if (!out || n < 0 || e < 0 || d < 1 || !h_rowptr || (e > 0 && !h_col) || (n > 0 && !h_X)) return CLANE_EINVAL;
    if (h_rowptr[n] != e) return CLANE_EINVAL;
    clane_session* s = new (std::nothrow) clane_session();
    if (!s) return (int)cudaErrorMemoryAllocation;
    s->n = n; s->e = e; s->d = d; s->ld = clane_padded_ld(d);
    s->log_cap = 1 << 16;
    const size_t zbytes = std::max<size_t>((size_t)n * s->ld * sizeof(float), 16);
    const size_t ebytes = std::max<size_t>((size_t)e * sizeof(int32_t), 16);
    SESSION_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    // ONE device allocation for everything the session owns (a dozen separate cudaMallocs cost milliseconds), carved
    // at 256-byte boundaries; `prev` (only iterate() needs it) is allocated on first use.
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t sizes[] = {up((size_t)(n + 1) * sizeof(int32_t)), up(ebytes), up(ebytes), up(zbytes), up(zbytes), up(zbytes),
                            up(zbytes), up(ebytes), 256, 256, up((size_t)s->log_cap * sizeof(float)), 256};
    size_t total = 0;
    for (size_t b : sizes) total += b;
    SESSION_CUDA(cudaMalloc(&s->pool, total));
    {
        char* p = static_cast<char*>(s->pool);
        auto take = [&](int i) { char* q = p; p += sizes[i]; return q; };
        s->rowptr = (int32_t*)take(0); s->col = (int32_t*)take(1); s->erow = (int32_t*)take(2);
        s->X = (float*)take(3); s->Z[0] = (float*)take(4); s->Z[1] = (float*)take(5); s->Z[2] = (float*)take(6);
        s->w = (float*)take(7); s->norms2 = (float*)take(8); s->amount = (float*)take(9); s->log = (float*)take(10);
        s->state = (clane_patience*)take(11);
    }
    SESSION_CUDA(cudaMallocHost(&s->h_state, sizeof(clane_patience)));
    // uploads first (asynchronous from pinned buffers), so that the host-side schedule build below overlaps them
    SESSION_CUDA(cudaMemcpyAsync(s->rowptr, h_rowptr, (size_t)(n + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream));
    if (e > 0) SESSION_CUDA(cudaMemcpyAsync(s->col, h_col, (size_t)e * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream));
    if (n > 0) {
        SESSION_TRY(copy_rows_h2d(s, s->X, h_X));
        SESSION_CUDA(cudaMemcpyAsync(s->Z[0], s->X, zbytes, cudaMemcpyDeviceToDevice, s->stream));
        SESSION_CUDA(cudaMemcpyAsync(s->Z[1], s->X, zbytes, cudaMemcpyDeviceToDevice, s->stream));
        SESSION_CUDA(cudaMemcpyAsync(s->Z[2], s->X, zbytes, cudaMemcpyDeviceToDevice, s->stream));
    }
    SESSION_TRY(clane_plan_create(&s->plan, n, e, d, h_rowptr, 0, n, hub_threshold));
    SESSION_TRY(clane_edge_rows(s->rowptr, n, e, s->erow, s->stream));
    SESSION_CUDA(cudaStreamSynchronize(s->stream));  // the host vectors above go out of scope
    *out = s;
    return CLANE_OK;
}

int clane_session_set_z(clane_session* s, const float* h_Z) {
    if (!s || !h_Z) return CLANE_EINVAL;
    int rc = copy_rows_h2d(s, s->Z[0], h_Z);
    if (rc != CLANE_OK) return rc;
    CLANE_CUDA(cudaMemcpyAsync(s->Z[1], s->Z[0], (size_t)s->n * s->ld * sizeof(float), cudaMemcpyDeviceToDevice, s->stream));
    CLANE_CUDA(cudaMemcpyAsync(s->Z[2], s->Z[0], (size_t)s->n * s->ld * sizeof(float), cudaMemcpyDeviceToDevice, s->stream));
    s->cur = 0;
    s->p_valid = false;
    CLANE_CUDA(cudaStreamSynchronize(s->stream));
    return CLANE_OK;
}

int clane_session_get_z(clane_session* s, float* h_Z) {
    if (!s || !h_Z) return CLANE_EINVAL;
    if (s->n == 0) return CLANE_OK;
    int rc = copy_rows_d2h(s, h_Z, s->Z[s->cur]);
    if (rc != CLANE_OK) return rc;
    CLANE_CUDA(cudaStreamSynchronize(s->stream));
    return CLANE_OK;
}

static int session_build_p(clane_session* s) {
    int rc = clane_build_p_cosine(s->plan, s->Z[s->cur], s->rowptr, s->erow, s->col, s->w, s->norms2, s->stream);
    if (rc == CLANE_OK) s->p_valid = true;
    return rc;
}

int clane_session_build_p(clane_session* s, float* h_w) {
    if (!s) return CLANE_EINVAL;
    int rc = session_build_p(s);
    if (rc != CLANE_OK) return rc;
    if (h_w && s->e > 0)
        CLANE_CUDA(cudaMemcpyAsync(h_w, s->w, (size_t)s->e * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    CLANE_CUDA(cudaStreamSynchronize(s->stream));
    return CLANE_OK;
}

static int session_sweep(clane_session* s, float gamma, bool with_state, float* d_amount) {
    const int nxt = (s->cur + 1) % 3;
    int rc = clane_sweep(s->plan, s->X, s->Z[s->cur], s->Z[nxt], s->rowptr, s->col, s->w, gamma, d_amount,
                         with_state ? s->state : nullptr, with_state ? s->log : nullptr, s->log_cap, s->stream);
    s->cur = nxt;
    return rc;
}

int clane_session_propagate(clane_session* s, float gamma, int32_t tol, int32_t max_sweeps, float* h_amounts,
                            int32_t cap, int32_t* sweeps) {
    if (!s || tol < 1 || max_sweeps < 0) return CLANE_EINVAL;
    int rc = session_build_p(s);
    if (rc != CLANE_OK) return rc;
    rc = clane_patience_reset(s->state, tol, max_sweeps, s->stream);
    if (rc != CLANE_OK) return rc;
    const int start = s->cur;
    // one graph launch for the whole call (conditional WHILE over batches of sweeps); without conditional nodes:
    // batches of 12 sweeps (whole buffer rotations), one host synchronisation per batch
    // ... except for a short bounded call (max_sweeps <= 24): its sweeps are enqueued directly, once -- no graph to build,
    // the device-side counter turns whatever follows the stop into no-ops
    if (max_sweeps > 0 && max_sweeps <= 24)
        rc = clane_internal_sweeps_direct(s->plan, s->X, s->Z, start, s->rowptr, s->col, s->w, gamma, max_sweeps, s->state, s->log,
                                          s->log_cap, s->stream);
    else
        rc = clane_sweeps(s->plan, s->X, s->Z, start, s->rowptr, s->col, s->w, gamma, 0, 1, s->state, s->log, s->log_cap, s->stream);
    if (rc != CLANE_OK && rc != CLANE_EUNSUPPORTED) return rc;
    const bool looped = rc == CLANE_OK;
    for (;;) {
        if (!looped) {
            rc = clane_sweeps(s->plan, s->X, s->Z, start, s->rowptr, s->col, s->w, gamma, 12, 0, s->state, s->log, s->log_cap,
                              s->stream);
            if (rc != CLANE_OK) return rc;
        }
        CLANE_CUDA(cudaMemcpyAsync(s->h_state, s->state, sizeof(clane_patience), cudaMemcpyDeviceToHost, s->stream));
        CLANE_CUDA(cudaStreamSynchronize(s->stream));
        if (s->h_state->stop) break;
        if (looped) return CLANE_EINVAL;   // the loop ended without the stop flag: cannot happen
    }
    const int done = s->h_state->sweeps;
    s->cur = (start + done) % 3;  // sweep i read Z[(start + i) % 3] and wrote the next buffer
    if (sweeps) *sweeps = done;
    if (h_amounts && cap > 0) {
        const int cnt = std::min(std::min(done, cap), s->log_cap);
        CLANE_CUDA(cudaMemcpyAsync(h_amounts, s->log, (size_t)cnt * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
        CLANE_CUDA(cudaStreamSynchronize(s->stream));
    }
    return CLANE_OK;
}

int clane_session_iterate(clane_session* s, float gamma, int32_t tol, int32_t max_outer, float* min_amount,
                          int32_t* h_sweeps_per_call, int32_t cap, int32_t* outer) {
    if (!s || tol < 1 || !min_amount) return CLANE_EINVAL;
    int patience = tol, calls = 0;
    const size_t zbytes = (size_t)s->n * s->ld * sizeof(float);
    if (!s->prev) CLANE_CUDA(cudaMalloc(&s->prev, std::max<size_t>(zbytes, 16)));
    for (;;) {
        CLANE_CUDA(cudaMemcpyAsync(s->prev, s->Z[s->cur], zbytes, cudaMemcpyDeviceToDevice, s->stream));
        int sweeps = 0;
        int rc = clane_session_propagate(s, gamma, tol, 0, nullptr, 0, &sweeps);
        if (rc != CLANE_OK) return rc;
        rc = clane_l1_diff(s->plan, s->Z[s->cur], s->prev, s->amount, s->stream);
        if (rc != CLANE_OK) return rc;
        float amt = 0.0f;
        CLANE_CUDA(cudaMemcpyAsync(&amt, s->amount, sizeof(float), cudaMemcpyDeviceToHost, s->stream));
        CLANE_CUDA(cudaStreamSynchronize(s->stream));
        if (h_sweeps_per_call && calls < cap) h_sweeps_per_call[calls] = sweeps;
        ++calls;
        if (*min_amount > amt) { patience = tol; *min_amount = amt; }
        else patience -= 1;
        if (patience == 0) break;
        if (max_outer > 0 && calls >= max_outer) break;
    }
    if (outer) *outer = calls;
    return CLANE_OK;
}

int clane_session_sweeps(clane_session* s, float gamma, int32_t sweeps, float* h_amount) {
    if (!s || sweeps < 0) return CLANE_EINVAL;
    if (!s->p_valid) {
        int rc = session_build_p(s);
        if (rc != CLANE_OK) return rc;
    }
    for (int i = 0; i < sweeps; ++i) {
        int rc = session_sweep(s, gamma, false, s->amount);
        if (rc != CLANE_OK) return rc;
    }
    if (h_amount) CLANE_CUDA(cudaMemcpyAsync(h_amount, s->amount, sizeof(float), cudaMemcpyDeviceToHost, s->stream));
    CLANE_CUDA(cudaStreamSynchronize(s->stream));
    return CLANE_OK;
}

}  // extern "C"
