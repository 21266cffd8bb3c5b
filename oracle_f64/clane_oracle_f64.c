/*
 * oracle_f64/clane_oracle_f64.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The fp64 twin of oracle/clane_oracle.c: a CPU restatement (plain C, IEEE-754 binary64, no
 * fast-math, no contraction) of what the reference's hot path computes when the content embeddings
 * C.npy are float64 (graph.py:51 keeps the dtype, so build_P, every sweep, the L1 change and both
 * patience loops then run in double on PyTorch-CPU):
 *
 *   CosineSimilarity   similarity.py:26-37   per-edge dot: mul+add for d < 400, fma for d >= 400;
 *                                            global norms: ATen cascade sum, 4 lanes x 4 ILP
 *   Graph.build_P      graph.py:118-128      softmax(0): Sleef expd8_u10, 8-lane reduce_all whose
 *                                            lanes are combined sequentially, reciprocal multiply
 *   Embedder.propagate embedder.py:71-108    row update: one sequential fma chain over the
 *                                            neighbours for every column; z = x + gamma * acc with
 *                                            gamma a double; L1 change: the same cascade sum
 *   Embedder.iterate   embedder.py:56-69
 *
 * The orders are pinned by tests/golden/f64/ (tests/golden/make_golden_f64.py, torch on one thread)
 * in tests/test_oracle_f64.py.  Build: gcc -O2 -ffp-contract=off -mfma -fopenmp (oracle_f64.py).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define EXPORT __attribute__((visibility("default")))

static int g_threads = 1;

EXPORT void clane_oracle64_set_threads(int t) {
    g_threads = t < 1 ? 1 : t;
#ifdef _OPENMP
    omp_set_num_threads(g_threads);
#endif
}

/* ------------------------------------------------------------------------- */
/* ATen cascade sum in double: Vectorized<double> has 4 lanes, 4 ILP rows      */
/* (16 accumulators keyed by flat index mod 16), 4 levels, level_step = 2^p.   */
/* ------------------------------------------------------------------------- */
#define LANES 4
#define ROW (4 * LANES)
typedef void (*fetch_fn)(void* ctx, int64_t t0, int64_t cnt, double* out);

typedef struct {
    double acc[4][ROW];
    int64_t i;
    int p;
} cascade_t;

static int ceil_log2_i64(int64_t x) {
    if (x <= 1) return 0;
    int l = 0;
    int64_t v = x - 1;
    while (v > 0) { v >>= 1; ++l; }
    return l;
}

static int cascade_p(int64_t size_rows) {
    int p = ceil_log2_i64(size_rows) / 4;
    return p < 4 ? 4 : p;
}

static inline void cascade_push(cascade_t* c, const double* row) {
    for (int l = 0; l < ROW; ++l) c->acc[0][l] = c->acc[0][l] + row[l];
    c->i++;
    const int64_t step = (int64_t)1 << c->p, mask = step - 1;
    if ((c->i & mask) == 0) {
        for (int j = 1; j < 4; ++j) {
            for (int l = 0; l < ROW; ++l) {
                c->acc[j][l] = c->acc[j][l] + c->acc[j - 1][l];
                c->acc[j - 1][l] = 0.0;
            }
            if ((c->i & (mask << (j * c->p))) != 0) break;
        }
    }
}

#define FETCH_ROWS 256

static double aten_sum_stream(int64_t n, fetch_fn fetch, void* ctx) {
    if (n < LANES) {
        double x[LANES], out = 0.0;
        if (n > 0) fetch(ctx, 0, n, x);
        for (int64_t i = 0; i < n; ++i) out = out + x[i];
        return out;
    }
    const int64_t nv = n / LANES, ni = nv / 4;
    double part[ROW];
    memset(part, 0, sizeof(part));
    if (ni > 0) {
        const int p = cascade_p(ni);
        const int64_t seg = (int64_t)1 << (3 * p);           /* rows per level-2 node */
        const int64_t nseg = (ni + seg - 1) / seg;
        double* V = (double*)malloc((size_t)nseg * ROW * sizeof(double));
        cascade_t last;
        memset(&last, 0, sizeof(last));
#pragma omp parallel for schedule(dynamic, 1) num_threads(g_threads)
        for (int64_t k = 0; k < nseg; ++k) {
            cascade_t c;
            memset(&c, 0, sizeof(c));
            c.i = k * seg;
            c.p = p;
            int64_t r0 = k * seg, r1 = r0 + seg < ni ? r0 + seg : ni;
            double buf[FETCH_ROWS * ROW];
            for (int64_t r = r0; r < r1; r += FETCH_ROWS) {
                int64_t cnt = r1 - r < FETCH_ROWS ? r1 - r : FETCH_ROWS;
                fetch(ctx, r * ROW, cnt * ROW, buf);
                for (int64_t q = 0; q < cnt; ++q) cascade_push(&c, buf + q * ROW);
            }
            if (r1 - r0 == seg) memcpy(V + k * ROW, c.acc[3], ROW * sizeof(double));
            else last = c;
        }
        double acc3[ROW];
        memset(acc3, 0, sizeof(acc3));
        const int64_t nfull = ni / seg;
        for (int64_t k = 0; k < nfull; ++k)
            for (int l = 0; l < ROW; ++l) acc3[l] = acc3[l] + V[k * ROW + l];
        free(V);
        for (int l = 0; l < ROW; ++l) {
            double a = last.acc[0][l];
            a = a + last.acc[1][l];
            a = a + last.acc[2][l];
            a = a + acc3[l];
            part[l] = a;
        }
    }
    for (int64_t v = ni * 4; v < nv; ++v) {           /* leftover vectors -> ILP row 0 */
        double tmp[LANES];
        fetch(ctx, v * LANES, LANES, tmp);
        for (int l = 0; l < LANES; ++l) part[l] = part[l] + tmp[l];
    }
    for (int k = 1; k < 4; ++k)
        for (int l = 0; l < LANES; ++l) part[l] = part[l] + part[k * LANES + l];
    double out = 0.0;
    if (n > nv * LANES) {
        double tmp[LANES];
        fetch(ctx, nv * LANES, n - nv * LANES, tmp);
        for (int64_t k = 0; k < n - nv * LANES; ++k) out = out + tmp[k];
    }
    for (int l = 0; l < LANES; ++l) out = out + part[l];
    return out;
}

static void fetch_plain(void* ctx, int64_t t0, int64_t cnt, double* out) {
    memcpy(out, (const double*)ctx + t0, (size_t)cnt * sizeof(double));
}

EXPORT double clane_oracle64_aten_sum(const double* x, int64_t n) {
    return aten_sum_stream(n, fetch_plain, (void*)x);
}

typedef struct { const double* a; const double* b; } absdiff_ctx;
static void fetch_absdiff(void* vctx, int64_t t0, int64_t cnt, double* out) {
    const absdiff_ctx* c = (const absdiff_ctx*)vctx;
    for (int64_t k = 0; k < cnt; ++k) out[k] = fabs(c->a[t0 + k] - c->b[t0 + k]);
}

EXPORT double clane_oracle64_l1_diff(const double* za, const double* zb, int64_t n_elems) {
    absdiff_ctx c = { za, zb };
    return aten_sum_stream(n_elems, fetch_absdiff, &c);
}

typedef struct { const double* Z; int64_t d; const int32_t* idx; } gsq_ctx;
static void fetch_gathered_sq(void* vctx, int64_t t0, int64_t cnt, double* out) {
    const gsq_ctx* c = (const gsq_ctx*)vctx;
    int64_t e = t0 / c->d, j = t0 % c->d;
    const double* row = c->Z + (int64_t)c->idx[e] * c->d;
    for (int64_t k = 0; k < cnt; ++k) {
        double a = row[j];
        out[k] = a * a;
        if (++j == c->d) { j = 0; ++e; if (k + 1 < cnt) row = c->Z + (int64_t)c->idx[e] * c->d; }
    }
}

/* similarity.py:35-37: per-edge dot, sequential over the feature index */
static inline double dot_seq(const double* a, const double* b, int64_t d) {
    double acc = 0.0;
    if (d < 400) { for (int64_t j = 0; j < d; ++j) { double p = a[j] * b[j]; acc = acc + p; } }
    else         { for (int64_t j = 0; j < d; ++j) acc = fma(a[j], b[j], acc); }
    return acc;
}

static int32_t* edge_rows(int64_t n, const int64_t* rowptr) {
    int64_t E = rowptr[n];
    int32_t* er = (int32_t*)malloc((size_t)(E > 0 ? E : 1) * sizeof(int32_t));
    for (int64_t v = 0; v < n; ++v)
        for (int64_t k = rowptr[v]; k < rowptr[v + 1]; ++k) er[k] = (int32_t)v;
    return er;
}

EXPORT void clane_oracle64_scores_raw(const double* Z, int64_t n, int64_t d, const int64_t* rowptr,
                                      const int32_t* col, double* dots, double* s1, double* s2) {
    const int64_t E = rowptr[n];
    int32_t* er = edge_rows(n, rowptr);
#pragma omp parallel for schedule(static) num_threads(g_threads)
    for (int64_t e = 0; e < E; ++e)
        dots[e] = dot_seq(Z + (int64_t)er[e] * d, Z + (int64_t)col[e] * d, d);
    gsq_ctx c1 = { Z, d, er }, c2 = { Z, d, col };
    *s1 = aten_sum_stream(E * d, fetch_gathered_sq, &c1);
    *s2 = aten_sum_stream(E * d, fetch_gathered_sq, &c2);
    free(er);
}

/* ------------------------------------------------------------------------- */
/* graph.py:123 in double: Sleef_expd8_u10 (FMA variant, Estrin polynomial),   */
/* then Vectorized<double> reduce_all (8 lanes, combined lane 0..7 in order).  */
/* ------------------------------------------------------------------------- */
static inline double pow2i(int q) {
    union { uint64_t u; double f; } v;
    v.u = (uint64_t)(q + 1023) << 52;
    return v.f;
}

static inline double sleef_expd_u10(double d) {
    const double R_LN2 = 1.442695040888963407359924681001892137426645954152985934135449406931;
    const double L2U = .69314718055966295651160180568695068359375;
    const double L2L = .28235290563031577122588448175013436025525412068e-12;
    double qd = rint(d * R_LN2);
    int q = (int)qd;
    double s = fma(qd, -L2U, d);
    s = fma(qd, -L2L, s);
    double s2 = s * s, s4 = s2 * s2, s8 = s4 * s4;
    double p98 = fma(s, +0.2081276378237164457e-8, +0.2511210703042288022e-7);
    double p76 = fma(s, +0.2755762628169491192e-6, +0.2755723402025388239e-5);
    double p54 = fma(s, +0.2480158687479686264e-4, +0.1984126989855865850e-3);
    double p32 = fma(s, +0.1388888888914497797e-2, +0.8333333333314938210e-2);
    double p10 = fma(s, +0.4166666666666602598e-1, +0.1666666666666669072e+0);
    double p7654 = fma(s2, p76, p54), p3210 = fma(s2, p32, p10);
    double p8 = fma(s4, p7654, p3210);
    double u = fma(s8, p98, p8);
    u = fma(u, s, 0.5);
    u = fma(u, s, 1.0);
    u = fma(u, s, 1.0);
    int q1 = q >> 1;
    u = (u * pow2i(q1)) * pow2i(q - q1);
    if (d < -1000.0) u = 0.0;
    if (d > 709.78271114955742909217217426) u = INFINITY;
    return u;
}

EXPORT void clane_oracle64_exp(const double* in, double* out, int64_t n) {
    for (int64_t i = 0; i < n; ++i) out[i] = sleef_expd_u10(in[i]);
}

#define RLANES 8
static double reduce_all_sum8(const double* e, int64_t k) {
    double acc[RLANES];
    int64_t p;
    if (k < RLANES) {
        double a = e[0];
        for (int64_t i = 1; i < k; ++i) a = a + e[i];
        return a;
    }
    for (int l = 0; l < RLANES; ++l) acc[l] = e[l];
    const int64_t full = k - (k % RLANES);
    for (p = RLANES; p < full; p += RLANES)
        for (int l = 0; l < RLANES; ++l) acc[l] = acc[l] + e[p + l];
    for (int64_t l = 0; p + l < k; ++l) acc[l] = acc[l] + e[p + l];
    double out = acc[0];
    for (int l = 1; l < RLANES; ++l) out = out + acc[l];
    return out;
}

static void softmax_row(const double* s, double* w, int64_t k) {
    double m = s[0];
    for (int64_t i = 1; i < k; ++i) if (s[i] > m) m = s[i];
    for (int64_t i = 0; i < k; ++i) w[i] = sleef_expd_u10(s[i] - m);
    double inv = 1.0 / reduce_all_sum8(w, k);
    for (int64_t i = 0; i < k; ++i) w[i] = w[i] * inv;
}

EXPORT void clane_oracle64_softmax_rows(const double* scores, int64_t n, const int64_t* rowptr, double* w) {
#pragma omp parallel for schedule(dynamic, 256) num_threads(g_threads)
    for (int64_t v = 0; v < n; ++v) {
        int64_t a = rowptr[v], b = rowptr[v + 1];
        if (b > a) softmax_row(scores + a, w + a, b - a);
    }
}

EXPORT void clane_oracle64_build_p(const double* Z, int64_t n, int64_t d, const int64_t* rowptr,
                                   const int32_t* col, double* w) {
    const int64_t E = rowptr[n];
    double s1, s2;
    clane_oracle64_scores_raw(Z, n, d, rowptr, col, w, &s1, &s2);
    double c = sqrt(s1) * sqrt(s2);
#pragma omp parallel for schedule(static) num_threads(g_threads)
    for (int64_t e = 0; e < E; ++e) w[e] = w[e] / c;
    clane_oracle64_softmax_rows(w, n, rowptr, w);
}

/* embedder.py:92 in double: w[1,k] @ Z[k,d] is one sequential fma chain per column */
static void row_update(const double* x, const double* Zcur, double* znew, int64_t d, const int32_t* cols,
                       const double* w, int64_t k, double gamma) {
    for (int64_t j = 0; j < d; ++j) {
        double acc = 0.0;
        for (int64_t t = 0; t < k; ++t) acc = fma(w[t], Zcur[(int64_t)cols[t] * d + j], acc);
        double g = gamma * acc;
        znew[j] = x[j] + g;
    }
}

EXPORT void clane_oracle64_sweep(const double* X, const double* Zcur, double* Znext, int64_t n, int64_t d,
                                 const int64_t* rowptr, const int32_t* col, const double* w, double gamma) {
#pragma omp parallel for schedule(dynamic, 64) num_threads(g_threads)
    for (int64_t v = 0; v < n; ++v) {
        int64_t a = rowptr[v], b = rowptr[v + 1];
        if (b > a) row_update(X + v * d, Zcur, Znext + v * d, d, col + a, w + a, b - a, gamma);
        else memcpy(Znext + v * d, Zcur + v * d, (size_t)d * sizeof(double));
    }
}

EXPORT int64_t clane_oracle64_propagate(const double* X, double* Z, int64_t n, int64_t d, const int64_t* rowptr,
                                        const int32_t* col, double gamma, int64_t tol, int64_t max_sweeps,
                                        double* amounts, int64_t cap, double* w_out) {
    const int64_t E = rowptr[n];
    double* w = (double*)malloc((size_t)(E > 0 ? E : 1) * sizeof(double));
    double* Zn = (double*)malloc((size_t)(n * d > 0 ? n * d : 1) * sizeof(double));
    clane_oracle64_build_p(Z, n, d, rowptr, col, w);
    if (w_out) memcpy(w_out, w, (size_t)E * sizeof(double));
    double minimum = INFINITY;
    int64_t patience = tol, sweeps = 0;
    for (;;) {
        clane_oracle64_sweep(X, Z, Zn, n, d, rowptr, col, w, gamma);
        double amt = clane_oracle64_l1_diff(Zn, Z, n * d);
        memcpy(Z, Zn, (size_t)n * d * sizeof(double));
        if (amounts && sweeps < cap) amounts[sweeps] = amt;
        ++sweeps;
        if (minimum > amt) { patience = tol; minimum = amt; }
        else patience -= 1;
        if (patience == 0) break;
        if (max_sweeps > 0 && sweeps >= max_sweeps) break;
    }
    free(w); free(Zn);
    return sweeps;
}

EXPORT int64_t clane_oracle64_iterate(const double* X, double* Z, int64_t n, int64_t d, const int64_t* rowptr,
                                      const int32_t* col, double gamma, int64_t tol, int64_t max_outer,
                                      int64_t* sweeps_per_call, double* outer_amounts, int64_t cap) {
    double* prev = (double*)malloc((size_t)(n * d > 0 ? n * d : 1) * sizeof(double));
    double g_min = INFINITY;
    int64_t g_tol = tol, outer = 0;
    for (;;) {
        memcpy(prev, Z, (size_t)n * d * sizeof(double));
        int64_t s = clane_oracle64_propagate(X, Z, n, d, rowptr, col, gamma, tol, 0, NULL, 0, NULL);
        double amt = clane_oracle64_l1_diff(Z, prev, n * d);
        if (outer < cap) {
            if (sweeps_per_call) sweeps_per_call[outer] = s;
            if (outer_amounts) outer_amounts[outer] = amt;
        }
        ++outer;
        if (g_min > amt) { g_tol = tol; g_min = amt; }
        else g_tol -= 1;
        if (g_tol == 0) break;
        if (max_outer > 0 && outer >= max_outer) break;
    }
    free(prev);
    return outer;
}
