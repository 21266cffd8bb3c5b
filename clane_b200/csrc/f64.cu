// The float64 hot path: what the reference computes when the content embeddings are float64
// (graph.py:51 keeps the dtype of C.npy, so build_P, every sweep, the L1 change and both patience
// loops run in double on PyTorch-CPU).  The rounding orders (DESIGN.md, "fp64") are:
//   row update  w[1,k] @ Z[k,d]   one sequential fma chain over the neighbours, every column;
//               z = x + gamma * acc, gamma a double, two roundings;
//   torch.sum   the ATen cascade with 4 lanes x 4 ILP rows (16 accumulators);
//   bmm dots    mul then add for d < 400, fma for d >= 400;
//   softmax(0)  Sleef expd8_u10, an 8-lane reduce_all whose lanes are then added 0..7 in order,
//               one reciprocal, one multiply.
// Every operation is an explicit __fma_rn / __dmul_rn / __dadd_rn / __ddiv_rn / __dsqrt_rn
// (and the library is built with -fmad=false).
#include <algorithm>

#include "common.cuh"

namespace {

using clane::kFull;

constexpr int kLanes = 4;            // Vectorized<double>::size() of ATen's sum kernel
constexpr int kRow = 4 * kLanes;     // one cascade row: 4 ILP vectors
constexpr int kSoftLanes = 8;        // Vectorized<double>::size() of the softmax kernel
constexpr int kSlab = 64;            // columns per warp in the sweep: one double2 per lane

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dfma(double a, double b, double c) { return __fma_rn(a, b, c); }

// ---- ATen cascade sum (SURVEY Appendix A.2 with 4 lanes) -----------------------------------
// ni rows of 16 values; level-0 chunks of step = 2^p rows.  Every complete chunk, level-1 node
// and level-2 node is a sequential sum from zero of its children, so each level is one kernel;
// acc[3] is the sequential sum of the complete level-2 nodes, and the trailing partial node of
// each level is what acc[0..2] hold at the end.
struct Shape64 {
    int64_t n, nv, ni, step;
    int64_t m1, m2, m3;      // complete level-0 chunks / level-1 nodes / level-2 nodes
    int64_t n0, n1, n2;      // outputs of the three level kernels (complete + trailing partial)
};

Shape64 shape64(int64_t n) {
    Shape64 s{};
    s.n = n;
    s.nv = n / kLanes;
    s.ni = s.nv / 4;
    int p = clane::ceil_log2_i64(s.ni) / 4;
    if (p < 4) p = 4;
    s.step = (int64_t)1 << p;
    s.m1 = s.ni / s.step;
    s.n0 = (s.ni + s.step - 1) / s.step;
    s.m2 = s.m1 / s.step;
    s.n1 = (s.m1 + s.step - 1) / s.step;
    s.m3 = s.m2 / s.step;
    s.n2 = (s.m2 + s.step - 1) / s.step;
    return s;
}

int64_t work_exact(int64_t n) {
    const Shape64 s = shape64(n);
    return (s.n0 + s.n1 + s.n2 + 1) * kRow;
}

// Scratch for ANY reduction of at most n elements.  work_exact is not monotone: the chunk step doubles
// when ni passes 2^19, 2^23, 2^27, ... and the scratch needed just above such a boundary is about half
// of what it is just below.  Within one step it grows with ni, so the maximum over m <= n is reached
// at n or at the last ni of a smaller step.
int64_t work_doubles(int64_t n) {
    int64_t w = work_exact(n);
    const int64_t ni = n / kRow;
    for (int p = 5; 4 * p - 1 < 62; ++p) {
        const int64_t last = (int64_t)1 << (4 * p - 1);
        if (last >= ni) break;
        w = std::max(w, work_exact(last * kRow));
    }
    return w;
}

// element t of |Za - Zb| over the flattened [n, d] view of two [n, ld] matrices
struct AbsDiff {
    const double* a; const double* b; int32_t d, ld;
    __device__ double operator()(int64_t t) const {
        const int64_t r = t / d, c = t - r * d;
        return fabs(__dsub_rn(a[r * ld + c], b[r * ld + c]));
    }
};

// element t of Z[idx]^2 over the flattened [E, d] gathered array (similarity.py:37)
struct GatheredSq {
    const double* Z; const int32_t* idx; int32_t d, ld;
    __device__ double operator()(int64_t t) const {
        const int64_t e = t / d, c = t - e * d;
        const double v = Z[(int64_t)idx[e] * ld + c];
        return dmul(v, v);
    }
};

template <class F>
__global__ void k_cascade_level0_f64(F f, int64_t ni, int64_t step, int64_t n0, double* __restrict__ out,
                                     const clane_patience64* st) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (st && st->stop) return;
    if (t >= n0 * kRow) return;
    const int64_t c = t / kRow;
    const int l = (int)(t - c * kRow);
    const int64_t r0 = c * step, r1 = min(r0 + step, ni);
    double acc = 0.0;
    for (int64_t r = r0; r < r1; ++r) acc = dadd(acc, f(r * kRow + l));
    out[t] = acc;
}

__global__ void k_cascade_level_f64(const double* __restrict__ in, int64_t m, int64_t step, int64_t nout,
                                    double* __restrict__ out, const clane_patience64* st) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (st && st->stop) return;
    if (t >= nout * kRow) return;
    const int64_t c = t / kRow;
    const int l = (int)(t - c * kRow);
    const int64_t i0 = c * step, i1 = min(i0 + step, m);
    double acc = 0.0;
    for (int64_t i = i0; i < i1; ++i) acc = dadd(acc, in[i * kRow + l]);
    out[t] = acc;
}

__device__ void patience_step64(clane_patience64* st, double a, double* log, int32_t log_cap) {
    st->last_amount = a;
    if (log && st->sweeps < log_cap) log[st->sweeps] = a;
    st->sweeps += 1;
    if (st->minimum > a) { st->patience = st->tol; st->minimum = a; }   // embedder.py:98-102: strict '>'
    else st->patience -= 1;
    if (st->patience == 0 || (st->max_sweeps > 0 && st->sweeps >= st->max_sweeps)) st->stop = 1;
}

// One block of kRow threads: acc[3], the trailing partial nodes, the leftover vectors, the ILP
// rows, the scalar tail and the lanes, in ATen's order.  out may be null when st is given.
template <class F>
__global__ void k_cascade_finish_f64(F f, Shape64 s, const double* __restrict__ S0, const double* __restrict__ S1,
                                     const double* __restrict__ S2, double* out, clane_patience64* st, double* log,
                                     int32_t log_cap) {
    __shared__ double part[kRow];
    if (st && st->stop) return;
    const int l = threadIdx.x;
    if (s.n < kLanes) {
        if (l == 0) {
            double a = 0.0;
            for (int64_t i = 0; i < s.n; ++i) a = dadd(a, f(i));
            if (out) out[0] = a;
            if (st) patience_step64(st, a, log, log_cap);
        }
        return;
    }
    double acc3 = 0.0;
    for (int64_t k = 0; k < s.m3; ++k) acc3 = dadd(acc3, S2[k * kRow + l]);
    double a = (s.ni % s.step) ? S0[s.m1 * kRow + l] : 0.0;
    if (s.m1 % s.step) a = dadd(a, S1[s.m2 * kRow + l]);
    if (s.m2 % s.step) a = dadd(a, S2[s.m3 * kRow + l]);
    part[l] = s.ni > 0 ? dadd(a, acc3) : 0.0;
    __syncthreads();
    if (l != 0) return;
    for (int64_t v = s.ni * 4; v < s.nv; ++v)              // leftover vectors -> ILP row 0
        for (int j = 0; j < kLanes; ++j) part[j] = dadd(part[j], f(v * kLanes + j));
    for (int k = 1; k < 4; ++k)
        for (int j = 0; j < kLanes; ++j) part[j] = dadd(part[j], part[k * kLanes + j]);
    double r = 0.0;
    for (int64_t i = s.nv * kLanes; i < s.n; ++i) r = dadd(r, f(i));   // scalar tail first
    for (int j = 0; j < kLanes; ++j) r = dadd(r, part[j]);             // then the lanes, in order
    if (out) out[0] = r;
    if (st) patience_step64(st, r, log, log_cap);
}

template <class F>
int cascade_sum_f64(F f, int64_t n, double* work, double* out, clane_patience64* st, double* log, int32_t log_cap,
                    cudaStream_t s) {
    const Shape64 sh = shape64(n);
    double* S0 = work;
    double* S1 = S0 + sh.n0 * kRow;
    double* S2 = S1 + sh.n1 * kRow;
    const int T = 256;
    if (sh.n0 > 0) {
        const int64_t th = sh.n0 * kRow;
        k_cascade_level0_f64<F><<<(unsigned)((th + T - 1) / T), T, 0, s>>>(f, sh.ni, sh.step, sh.n0, S0, st);
        CLANE_LAUNCH_CHECK();
    }
    if (sh.n1 > 0) {
        const int64_t th = sh.n1 * kRow;
        k_cascade_level_f64<<<(unsigned)((th + T - 1) / T), T, 0, s>>>(S0, sh.m1, sh.step, sh.n1, S1, st);
        CLANE_LAUNCH_CHECK();
    }
    if (sh.n2 > 0) {
        const int64_t th = sh.n2 * kRow;
        k_cascade_level_f64<<<(unsigned)((th + T - 1) / T), T, 0, s>>>(S1, sh.m2, sh.step, sh.n2, S2, st);
        CLANE_LAUNCH_CHECK();
    }
    k_cascade_finish_f64<F><<<1, kRow, 0, s>>>(f, sh, S0, S1, S2, out, st, log, log_cap);
    CLANE_LAUNCH_CHECK();
    return 0;
}

// ---- the sweep ------------------------------------------------------------------------------
// One warp per (row, 64-column slab); lane i holds columns 64 * slab + 2i, 2i + 1 as one double2.
// The (col, w) of 32 neighbours are loaded at once, one per lane, and broadcast by shuffle; the
// gathers of a batch of 8 neighbours are issued before their fma chain runs, so the loads stay
// ahead of the (serial) chain.  Rows without out-neighbours are not touched (embedder.py:88-89).
constexpr int kAhead = 8;

__global__ void __launch_bounds__(256) k_sweep_rows_f64(int32_t n, int32_t ld, int32_t nslab,
                                                        const int32_t* __restrict__ rowptr,
                                                        const int32_t* __restrict__ col,
                                                        const double* __restrict__ w, const double* __restrict__ X,
                                                        const double* __restrict__ Zcur, double* __restrict__ Znext,
                                                        double gamma, const clane_patience64* st) {
    const int lane = threadIdx.x & 31;
    const int64_t task = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (task >= (int64_t)n * nslab) return;
    if (st && st->stop) return;
    const int32_t row = (int32_t)(task / nslab), slab = (int32_t)(task - (int64_t)row * nslab);
    const int32_t a = rowptr[row], b = rowptr[row + 1];
    if (b == a) return;
    const int32_t c = slab * kSlab + 2 * lane;
    const bool on = c < ld;                        // ld is even: both columns are in the row
    double2 acc = make_double2(0.0, 0.0);
    for (int32_t base = a; base < b; base += 32) {
        const int32_t cnt = min(32, b - base);
        int32_t my_col = 0;
        double my_w = 0.0;
        if (lane < cnt) { my_col = __ldg(col + base + lane); my_w = __ldg(w + base + lane); }
        for (int32_t t0 = 0; t0 < cnt; t0 += kAhead) {
            double2 v[kAhead];
            double wt[kAhead];
#pragma unroll
            for (int u = 0; u < kAhead; ++u) {
                const int32_t cu = __shfl_sync(kFull, my_col, (t0 + u) & 31);
                wt[u] = __shfl_sync(kFull, my_w, (t0 + u) & 31);
                v[u] = (on && t0 + u < cnt) ? __ldg(reinterpret_cast<const double2*>(Zcur + (int64_t)cu * ld + c))
                                            : make_double2(0.0, 0.0);
            }
#pragma unroll
            for (int u = 0; u < kAhead; ++u) {
                if (t0 + u < cnt) {
                    acc.x = dfma(wt[u], v[u].x, acc.x);
                    acc.y = dfma(wt[u], v[u].y, acc.y);
                }
            }
        }
    }
    if (!on) return;
    const double2 x = *reinterpret_cast<const double2*>(X + (int64_t)row * ld + c);
    double2 z;
    z.x = dadd(x.x, dmul(gamma, acc.x));
    z.y = dadd(x.y, dmul(gamma, acc.y));
    *reinterpret_cast<double2*>(Znext + (int64_t)row * ld + c) = z;
}

// ---- build_P --------------------------------------------------------------------------------
__global__ void k_dots_f64(const double* __restrict__ Z, int32_t d, int32_t ld, const int32_t* __restrict__ erow,
                           const int32_t* __restrict__ col, int64_t e, double* __restrict__ dots) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= e) return;
    const double* za = Z + (int64_t)erow[i] * ld;
    const double* zb = Z + (int64_t)col[i] * ld;
    double acc = 0.0;
    if (d < 400) { for (int32_t j = 0; j < d; ++j) acc = dadd(acc, dmul(za[j], zb[j])); }   // ATen bmm loop
    else         { for (int32_t j = 0; j < d; ++j) acc = dfma(za[j], zb[j], acc); }         // MKL
    dots[i] = acc;
}

__device__ __forceinline__ double pow2i(int q) { return __longlong_as_double((long long)(q + 1023) << 52); }

// Sleef_expd8_u10 (FMA variant): Cody-Waite reduction, Estrin polynomial of degree 10, three
// Horner steps, 2^q applied in two halves; 0 below -1000, inf above 709.78...
__device__ double sleef_expd_u10(double d) {
    const double R_LN2 = 1.442695040888963407359924681001892137426645954152985934135449406931;
    const double L2U = .69314718055966295651160180568695068359375;
    const double L2L = .28235290563031577122588448175013436025525412068e-12;
    const double qd = rint(dmul(d, R_LN2));
    const int q = (int)qd;
    double s = dfma(qd, -L2U, d);
    s = dfma(qd, -L2L, s);
    const double s2 = dmul(s, s), s4 = dmul(s2, s2), s8 = dmul(s4, s4);
    const double p98 = dfma(s, +0.2081276378237164457e-8, +0.2511210703042288022e-7);
    const double p76 = dfma(s, +0.2755762628169491192e-6, +0.2755723402025388239e-5);
    const double p54 = dfma(s, +0.2480158687479686264e-4, +0.1984126989855865850e-3);
    const double p32 = dfma(s, +0.1388888888914497797e-2, +0.8333333333314938210e-2);
    const double p10 = dfma(s, +0.4166666666666602598e-1, +0.1666666666666669072e+0);
    const double p8 = dfma(s4, dfma(s2, p76, p54), dfma(s2, p32, p10));
    double u = dfma(s8, p98, p8);
    u = dfma(u, s, 0.5);
    u = dfma(u, s, 1.0);
    u = dfma(u, s, 1.0);
    const int q1 = q >> 1;
    u = dmul(dmul(u, pow2i(q1)), pow2i(q - q1));
    if (d < -1000.0) u = 0.0;
    if (d > 709.78271114955742909217217426) u = __longlong_as_double(0x7ff0000000000000LL);
    return u;
}

// softmax(0) of each row (graph.py:123), one warp per row.  Scores are first divided by
// sqrt(norms2[0]) * sqrt(norms2[1]) when norms2 is given (similarity.py:37).  w may alias scores.
__global__ void k_row_softmax_f64(const double* scores, const double* __restrict__ norms2, int32_t row_lo,
                                  int32_t row_hi, const int32_t* __restrict__ rowptr, double* w) {
    const int lane = threadIdx.x & 31;
    const int64_t r = row_lo + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (r >= row_hi) return;
    const int32_t a = rowptr[r], k = rowptr[r + 1] - a;
    if (k == 0) return;
    double den = 1.0;
    if (norms2) den = dmul(__dsqrt_rn(norms2[0]), __dsqrt_rn(norms2[1]));
    double m = -__longlong_as_double(0x7ff0000000000000LL);
    for (int32_t i = lane; i < k; i += 32) {
        double v = scores[a + i];
        if (norms2) v = __ddiv_rn(v, den);
        m = fmax(m, v);
    }
    for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(kFull, m, o));
    for (int32_t i = lane; i < k; i += 32) {
        double v = scores[a + i];
        if (norms2) v = __ddiv_rn(v, den);
        w[a + i] = sleef_expd_u10(__dsub_rn(v, m));
    }
    __syncwarp();
    double sum = 0.0;
    if (k < kSoftLanes) {
        if (lane == 0) {
            sum = w[a];
            for (int32_t i = 1; i < k; ++i) sum = dadd(sum, w[a + i]);
        }
    } else {
        // lane j < 8 of reduce_all: w[j], w[j + 8], ... over the full vectors, then the leftovers
        double acc = 0.0;
        if (lane < kSoftLanes) {
            const int32_t full = k - k % kSoftLanes;
            acc = w[a + lane];
            for (int32_t p = kSoftLanes + lane; p < full; p += kSoftLanes) acc = dadd(acc, w[a + p]);
            if (full + lane < k) acc = dadd(acc, w[a + full + lane]);
        }
        sum = __shfl_sync(kFull, acc, 0);
        for (int j = 1; j < kSoftLanes; ++j) sum = dadd(sum, __shfl_sync(kFull, acc, j));
    }
    const double inv = __ddiv_rn(1.0, __shfl_sync(kFull, sum, 0));
    for (int32_t i = lane; i < k; i += 32) w[a + i] = dmul(w[a + i], inv);
}

__global__ void k_patience_reset64(clane_patience64* st, int32_t tol, int32_t max_sweeps) {
    st->minimum = __longlong_as_double(0x7ff0000000000000LL);
    st->last_amount = 0.0;
    st->patience = tol;
    st->tol = tol;
    st->sweeps = 0;
    st->max_sweeps = max_sweeps;
    st->stop = 0;
    st->reserved = 0;
}

int sweep_one(int32_t n, int32_t d, const int32_t* rowptr, const int32_t* col, const double* w, const double* X,
              const double* Zcur, double* Znext, double gamma, double* amount, clane_patience64* st, double* log,
              int32_t log_cap, double* work, cudaStream_t s) {
    const int32_t ld = clane_padded_ld_f64(d), nslab = (ld + kSlab - 1) / kSlab;
    const int64_t threads = (int64_t)n * nslab * 32;
    if (threads > 0) {
        k_sweep_rows_f64<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(n, ld, nslab, rowptr, col, w, X, Zcur, Znext,
                                                                           gamma, st);
        CLANE_LAUNCH_CHECK();
    }
    if (!amount && !st) return 0;
    return cascade_sum_f64(AbsDiff{Znext, Zcur, d, ld}, (int64_t)n * d, work, amount, st, log, log_cap, s);
}

}  // namespace

extern "C" {

int32_t clane_padded_ld_f64(int32_t d) { return d < 1 ? 2 : (d + 1) & ~1; }

int64_t clane_work_f64(int64_t n_elems) { return n_elems < 0 ? CLANE_EINVAL : work_doubles(n_elems); }

int clane_patience_reset_f64(clane_patience64* d_state, int32_t tol, int32_t max_sweeps, clane_stream_t s) {
    if (!d_state || tol < 1 || max_sweeps < 0) return CLANE_EINVAL;
    k_patience_reset64<<<1, 1, 0, (cudaStream_t)s>>>(d_state, tol, max_sweeps);
    CLANE_LAUNCH_CHECK();
    return 0;
}

int clane_l1_diff_f64(int32_t n, int32_t d, const double* d_Za, const double* d_Zb, double* d_work, double* d_out,
                      clane_stream_t s) {
    if (n < 0 || d < 1 || !d_Za || !d_Zb || !d_work || !d_out) return CLANE_EINVAL;
    const int32_t ld = clane_padded_ld_f64(d);
    return cascade_sum_f64(AbsDiff{d_Za, d_Zb, d, ld}, (int64_t)n * d, d_work, d_out, nullptr, nullptr, 0,
                           (cudaStream_t)s);
}

int clane_row_softmax_f64(const double* d_scores, const double* d_norms2, int32_t row_lo, int32_t row_hi,
                          const int32_t* d_rowptr, double* d_w, clane_stream_t s) {
    if (row_lo < 0 || row_hi < row_lo || !d_scores || !d_rowptr || !d_w) return CLANE_EINVAL;
    const int64_t threads = (int64_t)(row_hi - row_lo) * 32;
    if (threads == 0) return 0;
    k_row_softmax_f64<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)s>>>(d_scores, d_norms2, row_lo, row_hi,
                                                                                      d_rowptr, d_w);
    CLANE_LAUNCH_CHECK();
    return 0;
}

int clane_build_p_cosine_f64(int32_t n, int64_t e, int32_t d, const double* d_Z, const int32_t* d_rowptr,
                             const int32_t* d_erow, const int32_t* d_col, double* d_w, double* d_norms2,
                             double* d_work, clane_stream_t s) {
    if (n < 0 || e < 0 || d < 1 || !d_Z || !d_rowptr || !d_erow || !d_col || !d_w || !d_norms2 || !d_work)
        return CLANE_EINVAL;
    if (e == 0) return 0;
    const cudaStream_t st = (cudaStream_t)s;
    const int32_t ld = clane_padded_ld_f64(d);
    k_dots_f64<<<(unsigned)((e + 255) / 256), 256, 0, st>>>(d_Z, d, ld, d_erow, d_col, e, d_w);
    CLANE_LAUNCH_CHECK();
    int rc = cascade_sum_f64(GatheredSq{d_Z, d_erow, d, ld}, e * d, d_work, d_norms2, nullptr, nullptr, 0, st);
    if (rc) return rc;
    rc = cascade_sum_f64(GatheredSq{d_Z, d_col, d, ld}, e * d, d_work, d_norms2 + 1, nullptr, nullptr, 0, st);
    if (rc) return rc;
    return clane_row_softmax_f64(d_w, d_norms2, 0, n, d_rowptr, d_w, s);
}

int clane_sweep_f64(int32_t n, int32_t d, const int32_t* d_rowptr, const int32_t* d_col, const double* d_w,
                    const double* d_X, const double* d_Zcur, double* d_Znext, double gamma, double* d_amount,
                    clane_patience64* d_state, double* d_amounts_log, int32_t log_cap, double* d_work,
                    clane_stream_t s) {
    if (n < 0 || d < 1 || !d_rowptr || !d_col || !d_w || !d_X || !d_Zcur || !d_Znext || d_Zcur == d_Znext)
        return CLANE_EINVAL;
    if ((d_amount || d_state) && !d_work) return CLANE_EINVAL;
    return sweep_one(n, d, d_rowptr, d_col, d_w, d_X, d_Zcur, d_Znext, gamma, d_amount, d_state, d_amounts_log,
                     log_cap, d_work, (cudaStream_t)s);
}

int clane_sweeps_f64(int32_t n, int32_t d, const int32_t* d_rowptr, const int32_t* d_col, const double* d_w,
                     const double* d_X, double* const* d_Z3, int32_t cur, double gamma, int32_t n_sweeps,
                     clane_patience64* d_state, double* d_amounts_log, int32_t log_cap, double* d_work,
                     clane_stream_t s) {
    if (n < 0 || d < 1 || !d_rowptr || !d_col || !d_w || !d_X || !d_Z3 || !d_state || !d_work || n_sweeps < 0 ||
        cur < 0 || cur > 2)
        return CLANE_EINVAL;
    for (int32_t t = 0; t < n_sweeps; ++t) {
        const int rc = sweep_one(n, d, d_rowptr, d_col, d_w, d_X, d_Z3[(cur + t) % 3], d_Z3[(cur + t + 1) % 3], gamma,
                                 nullptr, d_state, d_amounts_log, log_cap, d_work, (cudaStream_t)s);
        if (rc) return rc;
    }
    return 0;
}

}  // extern "C"
