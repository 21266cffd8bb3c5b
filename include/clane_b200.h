/*
 * clane_b200.h -- C-ABI of the B200-native CLANE hot path (libclane_b200.so).
 *
 * The reference (helloybz/CLANE) has no FFI boundary of its own: its hot path is Python
 * calling PyTorch-CPU (SURVEY.md section 8b).  Each entry point below therefore names the
 * reference *Python* interface it replaces; the Python host package (clane_b200/, mirroring
 * clane/graph.py, clane/similarity.py, clane/embedder.py) binds them with ctypes
 * (see INTEGRATION.md for the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - "d_" arguments are DEVICE pointers, "h_" arguments are HOST pointers;
 *   - every function returns 0 on success, a positive cudaError_t value, or a negative
 *     CLANE_E* code; nothing throws across the boundary (clane_error_string decodes both);
 *   - kernels are enqueued on the given stream (a cudaStream_t passed as void*) and do not
 *     synchronise unless the comment says so;
 *   - feature matrices are row-major fp32 [n, ld] with ld = clane_padded_ld(d) (rows 16-byte
 *     aligned); the pad columns must be zero and stay zero;
 *   - rowptr / col are int32 CSR of the coalesced (sorted-unique) adjacency, rows = sources.
 *
 * All floating-point work reproduces the reference's fp32 rounding sequence bit for bit
 * (SURVEY.md section 7.1): the kernels are compiled with -fmad=false and use explicit
 * __fmaf_rn / __fmul_rn / __fadd_rn where the reference's CPU kernels fuse or do not fuse.
 */
#ifndef CLANE_B200_H
#define CLANE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define CLANE_OK 0
#define CLANE_EINVAL (-1)      /* bad argument (null pointer, negative size, d < 1 ...) */
#define CLANE_ERANGE (-2)      /* edge endpoint outside [0, n) / n or e >= 2^31 / n * ld > CLANE_MAX_MATRIX_FLOATS */
#define CLANE_EWORKSPACE (-3)  /* caller-provided buffer too small */
#define CLANE_ENODEVICE (-4)   /* no CUDA device / not an sm_100 class device */
#define CLANE_ENOENT (-5)      /* file cannot be opened */
#define CLANE_EPARSE (-6)      /* edge line without exactly one TAB */
#define CLANE_EUNKNOWNID (-7)  /* edge endpoint that is not in V */
#define CLANE_ENOMEM (-8)      /* host allocation failed */
#define CLANE_EUNSUPPORTED (-9) /* not available with this driver (the caller has a fallback) */

typedef void* clane_stream_t;  /* cudaStream_t */

/* Device-resident patience ("tolerence") state machine of Embedder.propagate
 * (/root/reference/clane/embedder.py:78-79, :98-108).  32 bytes. */
typedef struct clane_patience {
    float   minimum;      /* running strict minimum of the per-sweep L1 amount (starts +inf) */
    int32_t patience;     /* current counter; reset to tol on a strict new minimum, else -1   */
    int32_t tol;          /* initial value ("tolerence")                                       */
    int32_t sweeps;       /* sweeps completed in this propagate() call                         */
    int32_t max_sweeps;   /* 0 = unbounded                                                     */
    int32_t stop;         /* 1 once patience hit 0 (or max_sweeps reached): later sweeps no-op */
    float   last_amount;  /* L1 amount of the last completed sweep                             */
    int32_t reserved;
} clane_patience;

/* ---- library / device ---------------------------------------------------------------- */
int         clane_version(void);
const char* clane_error_string(int code);
/* sm count and compute capability of the current device */
int         clane_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* leading dimension used for [n, d] fp32 matrices: d rounded up to a multiple of 4 */
int32_t     clane_padded_ld(int32_t d);

/* ---- graph build (host side) --------------------------------------------------------- */
/* Replaces Graph.A (/root/reference/clane/graph.py:104-110): coalesce the raw edge list --
 * sort by (src, dst), merge duplicates, keep self-loops.  h_rowptr has n+1 entries, h_col
 * capacity e_raw.  Returns the number of coalesced edges E >= 0, or CLANE_E* (< 0). */
int64_t clane_csr_from_edges(const int64_t* h_src, const int64_t* h_dst, int64_t e_raw, int64_t n,
                             int32_t* h_rowptr, int32_t* h_col);

/* Replaces the edge-file loop of Graph.__init__ (/root/reference/clane/graph.py:73-81):
 *   lines = io.read().strip().split("\n"); src_id, dst_id = line.split("\t"); vertex_ids.index(id)
 * -- text mode (universal newlines), the file's surrounding whitespace stripped, exactly one TAB
 * per line, ids resolved to their FIRST position in V -- with a hash map and one file piece per
 * thread instead of O(E*N) list.index calls.  v_ids = the n_vertices ids of V (parsed by the
 * caller with the reference's own expression) joined by "\n", v_bytes long.  threads <= 0:
 * all host threads.  On CLANE_EPARSE / CLANE_EUNKNOWNID *err_line is the 0-based line (the first
 * offending one in file order, as the reference's loop would hit it) and err_text the
 * reference's message / the unknown id; on CLANE_ENOENT err_text is the path.  The parsed
 * (src, dst) position pairs, in file order with duplicates and self-loops kept, are copied out
 * by clane_edges_read (capacity *e_raw each) and released by clane_edges_close. */
typedef struct clane_edge_file clane_edge_file;
int clane_edges_open(const char* v_ids, int64_t v_bytes, int64_t n_vertices, const char* e_path, int32_t threads,
                     clane_edge_file** out, int64_t* e_raw, int64_t* err_line, char* err_text, int32_t err_cap);
int clane_edges_read(const clane_edge_file* f, int64_t* h_src, int64_t* h_dst);
int clane_edges_close(clane_edge_file* f);

/* ---- plan: degree-sorted row blocks + scratch ----------------------------------------- */
/* A plan holds, on the device, the schedule of the sweep over rows [row_lo, row_hi) of an
 * n-row CSR (north_star: "degree-sorted row blocks") and the scratch of the exact reductions:
 *   - rows are cut into groups of `group_rows` consecutive rows (one level-0 chunk of the
 *     ATen cascade sum when d is 32, 64 or 128 and the plan covers all rows -- then the L1
 *     change is fused into the sweep; otherwise 8 rows and the L1 change is a second pass);
 *   - rows of degree > hub_threshold are "hub rows": cut into segments of 128 neighbours that any
 *     warp gathers and pre-reduces ({z6, z4, X, Y} per 8-neighbour block -- the part of the
 *     reference's summation order that does not involve the running sum); one warp per (hub
 *     row, 32 columns) then runs the short in-order chain over that contiguous stream;
 *   - the ordinary rows of a group are cut into spans of bounded edge count, sorted by edge
 *     count descending, one warp per (span, 128-column slab); groups of sinks only are dropped
 *     (embedder.py:88-89: such rows are never updated);
 * hub_threshold <= 0 selects the default: (edges of rows [row_lo, row_hi)) / 4096 rounded up to a
 * multiple of 8, clamped to [256, 16384] (a row is an in-order chain on one warp; this bounds it
 * to a few percent of a sweep).
 * h_rowptr may be NULL for a scores-only plan (clane_scores_cosine / clane_l1_*).
 * Every plan, scores-only included, needs n * clane_padded_ld(d) <= CLANE_MAX_MATRIX_FLOATS
 * (CLANE_ERANGE otherwise): the fp32 kernels address the rows of an [n, ld] matrix by 32-bit
 * unsigned float4 indices. */
typedef struct clane_plan clane_plan;
#define CLANE_MAX_MATRIX_FLOATS (1LL << 34)   /* 64 GiB of fp32 per [n, ld] matrix */
/* The schedule alone, on the host (what clane_plan_create uploads); every output has capacity
 * row_hi - row_lo + 1.
 *   spans       : runs of consecutive ordinary rows inside one group holding at most
 *                 span_edges edges (a single row may exceed it), sorted by edge count
 *                 descending; h_span_meta = rows | (1 << 8 when the span is the whole group and
 *                 the group has no hub row, i.e. its warp also produces the fused L1 partial)
 *   h_fix_groups: fused mode only -- groups (relative to row_lo) whose L1 partial is
 *                 recomputed from memory because they hold a hub row or several spans
 *   h_hub_rows  : rows of degree > hub_threshold, degree-descending */
int clane_group_schedule(const int32_t* h_rowptr, int32_t n, int32_t d, int32_t row_lo, int32_t row_hi,
                         int32_t hub_threshold, int32_t span_edges, int32_t* h_span_row, int32_t* h_span_meta,
                         int32_t* n_spans, int32_t* h_fix_groups, int32_t* n_fix_groups, int32_t* h_hub_rows,
                         int32_t* n_hub_rows, int32_t* group_rows, int32_t* fused_l1);
/* The sweep kernel's task list for that schedule, on the host (what clane_plan_create uploads).
 *   h_tasks : 8 int32 per task {first edge, edges, first row (span) or first 8-block within the hub row
 *             (segment), rows | direct << 8 | segment << 9 | hub row index << 10, 8-blocks of the segment,
 *             first scratch block of the hub row (segment), 8-blocks of the hub row (segment), 0};
 *             hub segments first (rows by degree, descending), then spans by edge count descending.
 *             A span's warp takes the row lengths from rowptr and walks the rows in order.
 * h_tasks may be NULL (size only); CLANE_EWORKSPACE if task_cap is too small. */
int clane_sweep_program(const int32_t* h_rowptr, int32_t n, int32_t d, int32_t row_lo, int32_t row_hi,
                        int32_t hub_threshold, int32_t span_edges, int32_t* h_tasks, int64_t task_cap,
                        int64_t* n_tasks);
int clane_plan_create(clane_plan** out, int32_t n, int64_t e, int32_t d, const int32_t* h_rowptr,
                      int32_t row_lo, int32_t row_hi, int32_t hub_threshold);
int clane_plan_destroy(clane_plan* plan);
/* any pointer may be NULL */
int clane_plan_info(const clane_plan* plan, int32_t* group_rows, int32_t* n_spans, int32_t* n_hub_rows,
                    int32_t* n_fix_groups, int32_t* fused_l1, int32_t* launches_per_sweep);
/* Shape of the exact L1 / norm reductions over a flattened array of n_elems fp32 values:
 * number of level-1 nodes of the ATen cascade and elements per node.  A caller that splits a
 * reduction over ranks exchanges [n1_nodes + 2] slots of 32 floats (see clane_l1_partial). */
int clane_cascade_shape(int64_t n_elems, int64_t* n1_nodes, int64_t* elems_per_node);

/* ---- device kernels ------------------------------------------------------------------ */
/* d_erow[e] = source row of coalesced edge e (the first row of A.indices(), graph.py:119) */
int clane_edge_rows(const int32_t* d_rowptr, int32_t n, int64_t e, int32_t* d_erow, clane_stream_t s);

/* CosineSimilarity.__call__ on (Z[src], Z[dst]) (/root/reference/clane/similarity.py:26-37),
 * split where the reference has its global reduction:
 *   d_dots[e]   = <z_src(e), z_dst(e)>   sequential over the feature index (mul+add for
 *                 d < 400, fma for d >= 400 -- the ATen / MKL switch), for edges
 *                 [edge_lo, edge_hi);
 *   d_norms2[0] = sum(Z[src]^2), d_norms2[1] = sum(Z[dst]^2) over the flattened [E*d]
 *                 gathered arrays in ATen cascade-sum order (all E edges); NULL: dots only. */
int clane_scores_cosine(clane_plan* plan, const float* d_Z, const int32_t* d_erow, const int32_t* d_col,
                        int64_t edge_lo, int64_t edge_hi, float* d_dots, float* d_norms2, clane_stream_t s);

/* The two global norms of similarity.py:37 split for a row-partitioned (multi-GPU) run, like clane_l1_partial: the
 * level-1 nodes of the cascade over the flattened [E*d] gathered arrays are independent, so each rank reduces nodes
 * [node_lo, node_hi) (of clane_cascade_shape(E*d)) into d_p1 -- layout [n1_nodes + 2][2][32] floats, zero elsewhere --
 * the ranks all-reduce(SUM) the slots (each is written by exactly one rank: exact), and clane_norms_finish combines
 * them in the one fixed order on every rank: d_norms2[0..1]. */
int clane_norms_partial(clane_plan* plan, const float* d_Z, const int32_t* d_erow, const int32_t* d_col, int64_t node_lo,
                        int64_t node_hi, float* d_p1, clane_stream_t s);
int clane_norms_finish(clane_plan* plan, const float* d_Z, const int32_t* d_erow, const int32_t* d_col, const float* d_p1,
                       float* d_norms2, clane_stream_t s);

/* The per-source softmax of Graph.build_P (/root/reference/clane/graph.py:122-123) for rows
 * [row_lo, row_hi).  If d_norms2 != NULL each score is first divided by
 * fl(fl(sqrt(norms2[0])) * fl(sqrt(norms2[1]))) (similarity.py:37); pass NULL for scores
 * produced by a user plugin.  d_w may alias d_scores. */
int clane_row_softmax(const float* d_scores, const float* d_norms2, int32_t row_lo, int32_t row_hi,
                      const int32_t* d_rowptr, float* d_w, clane_stream_t s);

/* The same softmax for the plan's rows, with the plan's list of long rows (one CTA per row of >= 64 neighbours, one
 * thread per shorter row). */
int clane_plan_softmax(clane_plan* plan, const float* d_scores, const float* d_norms2, const int32_t* d_rowptr, float* d_w,
                       clane_stream_t s);

/* AsymmertricSimilarity (/root/reference/clane/similarity.py:40-57): score(v -> u) = <Phi_src z_v, Phi_dst z_u>.
 * clane_asym_project: every node projected once, [P_src | P_dst] = Z [n, d] x [W_src ; W_dst]^T, d_W = the two nn.Linear
 * weights stacked ([2d, d] row-major, contiguous), on the tensor cores (tcgen05.mma kind::tf32, fp32 accumulation in TMEM,
 * TMA-staged operands); d in {32, 64, 96, 128} (clane_asym_supported), CLANE_EUNSUPPORTED otherwise -- the caller then
 * runs the plugin itself.  d_Psrc / d_Pdst: [n, ld]; *d_error is set to 1 if the kernel gave up waiting for its copies.
 * clane_build_p_asym: Graph.build_P with that scorer for the plan's rows -- projection, per-edge dots of the projected
 * rows, row softmax (no norm divisor); d_work: 2 * n * ld floats. */
int clane_asym_supported(int32_t d);
int clane_asym_project(const float* d_Z, int32_t n, int32_t d, int32_t ld, const float* d_W, float* d_Psrc, float* d_Pdst,
                       int32_t* d_error, clane_stream_t s);
int clane_build_p_asym(clane_plan* plan, const float* d_Z, const float* d_W, const int32_t* d_rowptr, const int32_t* d_erow,
                       const int32_t* d_col, float* d_w, float* d_work, int32_t* d_error, clane_stream_t s);

/* The same scorer at fp32 accuracy for any d >= 1 (3xTF32: each operand split into a TF32 high part and an fp32
 * remainder, three tcgen05 MMAs per K step into one fp32 accumulator; every projected value lies within
 * (4 + 3d) 2^-23 sum_k |z_k w_k| of the exact product).  d_W: the stacked weights [2d, ldw] row-major, ldw >= d a
 * multiple of 4 (clane_padded_ld(d)), pad columns zero.  ld, ldw multiples of 4; d_Z and d_work 16-byte aligned.
 * clane_asym_project_fp32: d_Psrc / d_Pdst [n, ld], only columns < d written; d_work: 4 * d * ldw floats (the split of W).
 * clane_build_p_asym_fp32: projection, per-edge dots (the reference bmm's order: mul + add below d = 400, fma from there
 * on), row softmax without the norm divisor; d_work: 2 * n * ld + 4 * d * ldw floats.
 * Both return CLANE_EINVAL for a null pointer, d < 1, ld < d or ldw < d; *d_error is set to 1 if the kernel gave up
 * waiting for its copies (it then writes no projected value). */
int clane_asym_project_fp32(const float* d_Z, int32_t n, int32_t d, int32_t ld, const float* d_W, int32_t ldw, float* d_Psrc,
                            float* d_Pdst, float* d_work, int32_t* d_error, clane_stream_t s);
int clane_build_p_asym_fp32(clane_plan* plan, const float* d_Z, const float* d_W, int32_t ldw, const int32_t* d_rowptr,
                            const int32_t* d_erow, const int32_t* d_col, float* d_w, float* d_work, int32_t* d_error,
                            clane_stream_t s);

/* The final division of CosineSimilarity.__call__ (similarity.py:37) for standalone plugin
 * calls: d_out[i] = d_dots[i] / fl(fl(sqrt(norms2[0])) * fl(sqrt(norms2[1]))).  May alias. */
int clane_cosine_finalize(const float* d_dots, const float* d_norms2, int64_t e, float* d_out, clane_stream_t s);

/* Graph.build_P with CosineSimilarity (graph.py:118-128) for the plan's rows:
 * clane_scores_cosine + clane_row_softmax. */
int clane_build_p_cosine(clane_plan* plan, const float* d_Z, const int32_t* d_rowptr, const int32_t* d_erow,
                         const int32_t* d_col, float* d_w, float* d_norms2, clane_stream_t s);

/* One Jacobi sweep of Embedder.propagate (/root/reference/clane/embedder.py:84-94) over the
 * plan's rows:  Znext[v] = X[v] + gamma * (w_v @ Zcur[nbrs(v)]) in oneMKL's summation order,
 * gamma*(.) and x+(.) rounded separately; rows without out-neighbours are not touched (Znext
 * must already hold their value).  If d_amount != NULL the L1 change sum|Znext - Zcur| over
 * the flattened [n*d] array (ATen cascade order, embedder.py:94) is written to d_amount[0];
 * if d_state != NULL the patience state machine (embedder.py:98-108) is advanced on the
 * device, d_amounts_log[sweep] (capacity log_cap) receives the amount, and the whole call is
 * a no-op once d_state->stop is set.  With both NULL only the row update runs (a rank of a
 * row-partitioned run: see clane_l1_partial). */
int clane_sweep(clane_plan* plan, const float* d_X, const float* d_Zcur, float* d_Znext,
                const int32_t* d_rowptr, const int32_t* d_col, const float* d_w, float gamma,
                float* d_amount, clane_patience* d_state, float* d_amounts_log, int32_t log_cap,
                clane_stream_t s);

/* Several sweeps of one Embedder.propagate call (/root/reference/clane/embedder.py:83-108) enqueued at once, with
 * the patience state machine on the device.  d_Z3 = three [n, ld] buffers (host array of three device pointers);
 * sweep t reads d_Z3[(cur + t) % 3] and writes d_Z3[(cur + t + 1) % 3] (rows without out-neighbours are never
 * written: all three buffers must hold their value).  With three buffers the exact L1 change + patience update of
 * sweep t runs beside the rows of sweep t + 1; a sweep therefore sees a patience flag that is one sweep old, and at
 * most ONE speculative sweep runs after the stop -- into a buffer that is not the result -- while its own L1 / patience
 * step is a no-op: d_state->sweeps, the amounts log and the result d_Z3[(cur + d_state->sweeps) % 3] are exactly the
 * reference's.
 *   until_stop == 0: exactly n_sweeps sweeps are enqueued (no-ops once d_state->stop is set).
 *   until_stop != 0: ONE graph launch whose conditional WHILE node repeats batches of sweeps until d_state->stop
 *                    (bound the number with clane_patience_reset's max_sweeps); CLANE_EUNSUPPORTED if conditional
 *                    graph nodes are not available -- call again with until_stop == 0 and poll d_state.
 * Returns as soon as the work is enqueued on stream s. */
int clane_sweeps(clane_plan* plan, const float* d_X, float* const* d_Z3, int32_t cur, const int32_t* d_rowptr,
                 const int32_t* d_col, const float* d_w, float gamma, int32_t n_sweeps, int32_t until_stop,
                 clane_patience* d_state, float* d_amounts_log, int32_t log_cap, clane_stream_t s);

/* Measurement aid: a timeline of the kernels of the next enqueued batch of sweeps.  enable != 0 arms it (and resets the
 * stamps); h_out (may be NULL) first receives the stamps of the previous batch: [64 sweeps][6 slots][2] unsigned 64-bit
 * globaltimer nanoseconds {first CTA start, last CTA end}; slots: hub segments, long-row chains, short-row chains, span
 * tasks, exact-L1 tail, unused.  Untouched slots read {2^64 - 1, 0}. */
int clane_plan_trace(clane_plan* plan, int enable, unsigned long long* h_out);

/* (Za - Zb).abs().sum() over the flattened [n*d] array in ATen cascade order
 * (/root/reference/clane/embedder.py:60).  Result in d_out[0]. */
int clane_l1_diff(clane_plan* plan, const float* d_Za, const float* d_Zb, float* d_out, clane_stream_t s);

/* The same reduction split for a row-partitioned (multi-GPU) run.  The cascade's level-1
 * nodes are independent: each rank reduces nodes [node_lo, node_hi) of the whole [n*d] array
 * into d_p1 (layout [n1_nodes + 2][32] floats, see clane_cascade_shape; slot n1_nodes - 1 may
 * be the trailing partial node, slot n1_nodes + 1 its leftover rows), the ranks all-gather
 * their slots, and clane_l1_finish combines them in the one fixed order on every rank. */
int clane_l1_partial(clane_plan* plan, const float* d_Za, const float* d_Zb, int64_t node_lo, int64_t node_hi,
                     float* d_p1, clane_stream_t s);
int clane_l1_finish(clane_plan* plan, const float* d_Za, const float* d_Zb, float* d_p1, float* d_out,
                    clane_patience* d_state, float* d_amounts_log, int32_t log_cap, clane_stream_t s);

/* The <= 31 elements of |Za - Zb| that clane_l1_finish reads itself (everything past the last
 * complete 32-element cascade row; the whole array when n*d < 8) -> d_vals[32] (rest +0), and a
 * finish that takes them from that buffer instead of from Za / Zb: a row-partitioned run
 * all-reduces the values with the level-1 slots, so that the finish never reads rows a faster
 * rank may already be overwriting with its next sweep. */
int clane_l1_tail_values(clane_plan* plan, const float* d_Za, const float* d_Zb, float* d_vals, clane_stream_t s);
int clane_l1_finish_values(clane_plan* plan, float* d_p1, const float* d_vals, float* d_out,
                           clane_patience* d_state, float* d_amounts_log, int32_t log_cap, clane_stream_t s);

/* Row-partitioned run on n_peers GPUs of one NVLink domain (SURVEY.md 8e): the device addresses
 * of every rank's two Z buffers (peer-mapped, e.g. CUDA VMM / torch symmetric memory;
 * entry self_rank = this rank's own buffers).  From then on clane_sweep stores every finished
 * row of Znext to all ranks' buffers from inside the sweep kernel (rows of one span as one bulk
 * store per rank when a row fits one warp pass) -- the exchange overlaps the sweep and needs no
 * collective; the caller only has to order the ranks between sweeps (an all-reduce of the L1
 * slots, or of a token, does).  n_peers = 0 turns it off. */
int clane_plan_set_peers(clane_plan* plan, int32_t n_peers, int32_t self_rank, const uint64_t* h_ptrs_a,
                         const uint64_t* h_ptrs_b);
/* Optional, after clane_plan_set_peers: every rank's address of a THIRD Z buffer.  With three rotating buffers the
 * caller can run the exact-L1 reduction of sweep t (own rows, all-reduce of the slots, finish) beside sweep t + 1:
 * the sweep that overwrites a buffer is two sweeps behind the one whose L1 pass reads it (clane_b200/dist.py). */
int clane_plan_set_peers_third(clane_plan* plan, const uint64_t* h_ptrs_c);

/* Optional, after clane_plan_set_peers: the multicast (NVLS) addresses of the two Z buffers (e.g.
 * torch symmetric memory's multicast_ptr; 0 = none).  The sweep then reaches all ranks with one
 * multimem.st per finished row piece (replicated inside the NVSwitch) instead of n_peers - 1
 * unicast stores; the local buffer is still written directly. */
int clane_plan_set_multicast(clane_plan* plan, uint64_t mc_a, uint64_t mc_b);

/* Measurement aid: when enabled, clane_sweep brackets its kernels with CUDA events on the
 * streams they are launched on; clane_plan_profile_read waits for the last sweep and returns
 * h_ms[0] = row kernel (k_sweep_rows), h_ms[1] = whole sweep, h_ms[2] = exact L1 tail (fix-up,
 * level-1, finish), h_ms[3] = hub chain kernel (k_hub_chain; ~0 if there are no hub rows). */
int clane_plan_profile(clane_plan* plan, int enable);
int clane_plan_profile_read(clane_plan* plan, float* h_ms);

/* Reset the device patience state for a new propagate() call (embedder.py:78-79). */
int clane_patience_reset(clane_patience* d_state, int32_t tol, int32_t max_sweeps, clane_stream_t s);

/* ---- float64 ------------------------------------------------------------------------- */
/* When the content embeddings are float64 the reference runs build_P, every sweep, the L1 change and
 * both patience loops in double (graph.py:51 keeps the dtype of C.npy).  These entry points reproduce
 * that run bit for bit (DESIGN.md, "fp64"): the row update is one sequential fma chain over the
 * neighbours for every column, torch.sum is the ATen cascade with 4 lanes x 4 ILP rows, softmax(0) is
 * Sleef expd u10 with an 8-lane reduce_all.  They take plain sizes instead of a clane_plan:
 *   - feature matrices are row-major fp64 [n, ld] with ld = clane_padded_ld_f64(d) (rows 16-byte
 *     aligned); the pad columns must be zero and stay zero;
 *   - d_work is caller-owned device scratch of clane_work_f64(m) doubles, m the largest reduction it
 *     serves: n * d for the sweeps and clane_l1_diff_f64, e * d for clane_build_p_cosine_f64. */
typedef struct clane_patience64 {
    double  minimum;      /* running strict minimum of the per-sweep L1 amount (starts +inf) */
    double  last_amount;  /* L1 amount of the last completed sweep                           */
    int32_t patience;     /* as in clane_patience                                             */
    int32_t tol;
    int32_t sweeps;
    int32_t max_sweeps;
    int32_t stop;
    int32_t reserved;
} clane_patience64;

/* d rounded up to a multiple of 2 */
int32_t clane_padded_ld_f64(int32_t d);
/* doubles of d_work that suffice for every reduction over at most n_elems elements (non-decreasing in
 * n_elems, so one buffer sized for the largest reduction serves the smaller ones) */
int64_t clane_work_f64(int64_t n_elems);
/* clane_patience_reset for the float64 state */
int clane_patience_reset_f64(clane_patience64* d_state, int32_t tol, int32_t max_sweeps, clane_stream_t s);
/* (Za - Zb).abs().sum() over the flattened [n*d] array (embedder.py:60) -> d_out[0] */
int clane_l1_diff_f64(int32_t n, int32_t d, const double* d_Za, const double* d_Zb, double* d_work, double* d_out,
                      clane_stream_t s);
/* clane_row_softmax in double; for scores a user plugin produced, pass d_norms2 = NULL.  d_w may alias d_scores. */
int clane_row_softmax_f64(const double* d_scores, const double* d_norms2, int32_t row_lo, int32_t row_hi,
                          const int32_t* d_rowptr, double* d_w, clane_stream_t s);
/* Graph.build_P with CosineSimilarity in double: per-edge dots, the two global norms (d_norms2[0..1]),
 * the division and the row softmax -> d_w[e]. */
int clane_build_p_cosine_f64(int32_t n, int64_t e, int32_t d, const double* d_Z, const int32_t* d_rowptr,
                             const int32_t* d_erow, const int32_t* d_col, double* d_w, double* d_norms2,
                             double* d_work, clane_stream_t s);
/* clane_sweep in double: Znext[v] = X[v] + gamma * (w_v @ Zcur[nbrs(v)]) for rows with out-neighbours;
 * the L1 change to d_amount (if not NULL) and the patience step (if d_state is not NULL; a no-op once
 * d_state->stop is set). */
int clane_sweep_f64(int32_t n, int32_t d, const int32_t* d_rowptr, const int32_t* d_col, const double* d_w,
                    const double* d_X, const double* d_Zcur, double* d_Znext, double gamma, double* d_amount,
                    clane_patience64* d_state, double* d_amounts_log, int32_t log_cap, double* d_work,
                    clane_stream_t s);
/* n_sweeps sweeps enqueued at once with the patience state on the device: sweep t reads d_Z3[(cur + t) % 3]
 * and writes d_Z3[(cur + t + 1) % 3].  Sweeps after the stop are device-side no-ops, so the caller polls
 * d_state once per batch; the result is d_Z3[(cur + d_state->sweeps) % 3]. */
int clane_sweeps_f64(int32_t n, int32_t d, const int32_t* d_rowptr, const int32_t* d_col, const double* d_w,
                     const double* d_X, double* const* d_Z3, int32_t cur, double gamma, int32_t n_sweeps,
                     clane_patience64* d_state, double* d_amounts_log, int32_t log_cap, double* d_work,
                     clane_stream_t s);

/* ---- host-buffer session API (pure C consumers; bench e2e) ---------------------------- */
typedef struct clane_session clane_session;

/* Upload a coalesced CSR graph and features from HOST memory.  h_X is [n, d] (unpadded).
 * Z starts as a copy of X (graph.py:18-19). */
int clane_session_create(clane_session** out, int32_t n, int64_t e, int32_t d, const int32_t* h_rowptr,
                         const int32_t* h_col, const float* h_X, int32_t hub_threshold);
int clane_session_destroy(clane_session* s);
/* replace Z (Graph.set_Z, graph.py:136-138) / read Z (Graph.Z, graph.py:130-134); [n, d] host */
int clane_session_set_z(clane_session* s, const float* h_Z);
int clane_session_get_z(clane_session* s, float* h_Z);
/* Graph.build_P values for the current Z -> h_w[e] (optional, may be NULL) */
int clane_session_build_p(clane_session* s, float* h_w);
/* One propagate() call (embedder.py:71-108): build_P once, sweep until the patience counter
 * reaches 0 (or max_sweeps > 0 sweeps).  h_amounts (capacity cap, may be NULL) receives the
 * per-sweep L1 amounts; *sweeps the count.  Synchronous. */
int clane_session_propagate(clane_session* s, float gamma, int32_t tol, int32_t max_sweeps,
                            float* h_amounts, int32_t cap, int32_t* sweeps);
/* Embedder.iterate() (embedder.py:56-69).  min_amount is the running minimum kept on the
 * Embedder object (embedder.py:43), in/out.  h_sweeps_per_call capacity cap. */
int clane_session_iterate(clane_session* s, float gamma, int32_t tol, int32_t max_outer, float* min_amount,
                          int32_t* h_sweeps_per_call, int32_t cap, int32_t* outer);
/* exactly `sweeps` sweeps with the current P (bench inner loop; no patience); returns the
 * last L1 amount in *h_amount (may be NULL).  Synchronous. */
int clane_session_sweeps(clane_session* s, float gamma, int32_t sweeps, float* h_amount);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* CLANE_B200_H */
