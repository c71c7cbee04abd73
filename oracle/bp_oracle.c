/*
 * bp_oracle.c -- CPU restatement of LDPCDecoders.jl's belief-propagation hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path (ldpcdecoders.jl_b200/,
 * libldpcb200.so) may include, link or call this file.  It is used by tests/,
 * __graft_entry__.smoke() and the cpu_baseline / --impl reference legs of bench.py.
 *
 * PARITY UNPINNED: the reference (pure Julia) cannot be executed in this image
 * (no julia binary, no network) and its test-suite holds no golden vectors for this
 * path (all inputs come from an unseeded RNG, /root/reference/test/test_bp_decoder.jl:7-9).
 * This restatement is therefore pinned only by (i) line-by-line correspondence with the
 * cited reference lines, (ii) brute-force marginal KATs on cycle-free graphs,
 * (iii) an independent dense transliteration (oracle/bp_dense.py) and (iv) the
 * reference's statistical acceptance thresholds.  oracle/dump_golden.jl loads the text
 * twins of the golden fixtures (tests/golden/julia_twins/) into the REAL package, runs
 * batchdecode! for the BP and BP+OSD-0 decoders, compares bit for bit and exits non-zero
 * on any difference: the one command that pins this file for anyone who has Julia.
 *
 * What is restated (all citations relative to /root/reference/):
 *   src/decoders/belief_propagation.jl:83-91    reset!   (scratch zeroed, priors refilled)
 *   src/decoders/belief_propagation.jl:127-131  message initialisation  b2c = p/(1-p)
 *   src/decoders/belief_propagation.jl:135-150  check update (ratio domain, prefix/suffix)
 *   src/decoders/belief_propagation.jl:152-178  variable update, hard decision, NaN clamp
 *   src/decoders/belief_propagation.jl:180-184  syndrome re-check and early break
 *   src/decoders/belief_propagation.jl:220-231  batchdecode! column loop
 *
 * Arithmetic: IEEE-754 binary64, round-to-nearest, every operation rounded
 * separately (compile with -O2 -ffp-contract=off -fno-fast-math on x86-64/SSE2).
 *
 * Two storage modes with bit-identical results:
 *   dense = 0 : messages stored per edge (E doubles each direction)
 *   dense = 1 : "faithful cost" -- two dense s*n column-major matrices that are
 *               zero-filled on every decode and a per-iteration H*err mat-vec with
 *               fresh allocations, mimicking what the Julia package does per call.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct {
    int64_t s, n, E;
    const int64_t *colptr;   /* n+1, 0-based: column j of H = edges [colptr[j], colptr[j+1]) */
    const int64_t *rowval;   /* E, 0-based check index, ascending inside a column (SparseMatrixCSC invariant) */
    int64_t *rowptr;         /* s+1: row i of H (= column i of sparse_HT) */
    int64_t *rowvar;         /* E: variable index, ascending inside a row */
    int64_t *rowedge;        /* E: CSC position of that (i,j) entry */
} graph_t;

static int build_graph(graph_t *g, int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval)
{
    g->s = s; g->n = n; g->E = colptr[n];
    g->colptr = colptr; g->rowval = rowval;
    g->rowptr = (int64_t *)calloc((size_t)s + 1, sizeof(int64_t));
    g->rowvar = (int64_t *)malloc(sizeof(int64_t) * (size_t)(g->E ? g->E : 1));
    g->rowedge = (int64_t *)malloc(sizeof(int64_t) * (size_t)(g->E ? g->E : 1));
    if (!g->rowptr || !g->rowvar || !g->rowedge) return -1;
    for (int64_t e = 0; e < g->E; ++e) {
        if (rowval[e] < 0 || rowval[e] >= s) return -2;
        g->rowptr[rowval[e] + 1]++;
    }
    for (int64_t i = 0; i < s; ++i) g->rowptr[i + 1] += g->rowptr[i];
    int64_t *fill = (int64_t *)malloc(sizeof(int64_t) * (size_t)(s ? s : 1));
    if (!fill) return -1;
    memcpy(fill, g->rowptr, sizeof(int64_t) * (size_t)s);
    /* columns visited in ascending j => variables ascending inside every row,
       which is the order nzrange(sparse_HT, i) walks (belief_propagation.jl:137). */
    for (int64_t j = 0; j < n; ++j)
        for (int64_t e = colptr[j]; e < colptr[j + 1]; ++e) {
            int64_t i = rowval[e];
            g->rowvar[fill[i]] = j;
            g->rowedge[fill[i]] = e;
            fill[i]++;
        }
    free(fill);
    return 0;
}

static void free_graph(graph_t *g) { free(g->rowptr); free(g->rowvar); free(g->rowedge); }

/* One decode!, edge-indexed storage.  b2c/c2b are indexed by CSC edge position.
 * syn: s bytes (0/1).  err: n bytes out.  ratio: n doubles out or NULL (posterior
 * ratio R_j; the reference stores log(1/R_j), belief_propagation.jl:163).
 * Returns converged flag; *iters_out = iterations executed. */
static int decode_edge(const graph_t *g, double per, int max_iters, const uint8_t *syn,
                       double *b2c, double *c2b, uint8_t *err, double *ratio, int32_t *iters_out)
{
    const int64_t s = g->s, n = g->n;
    /* reset! : belief_propagation.jl:83-91 (err .= 0; messages are fully rewritten below) */
    memset(err, 0, (size_t)n);
    if (ratio) for (int64_t j = 0; j < n; ++j) ratio[j] = 1.0; /* log_probabs .= 0  <=> ratio 1 */
    /* init : belief_propagation.jl:127-131 */
    for (int64_t j = 0; j < n; ++j)
        for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e)
            b2c[e] = per / (1 - per);

    int converged = 0;
    int32_t it = 0;
    for (int iter = 1; iter <= max_iters; ++iter) {            /* :134 */
        it = iter;
        for (int64_t i = 0; i < s; ++i) {                      /* :135 */
            double temp = syn[i] ? -1.0 : 1.0;                 /* (-1)^syndrome[i], :136 */
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) {      /* :137-141 */
                int64_t e = g->rowedge[k];
                c2b[e] = temp;
                temp *= 2 / (1 + b2c[e]) - 1;
            }
            temp = 1.0;                                        /* :143 */
            for (int64_t k = g->rowptr[i + 1] - 1; k >= g->rowptr[i]; --k) { /* :144-149 */
                int64_t e = g->rowedge[k];
                c2b[e] *= temp;
                c2b[e] = (1 - c2b[e]) / (1 + c2b[e]);
                temp *= 2 / (1 + b2c[e]) - 1;
            }
        }
        for (int64_t j = 0; j < n; ++j) {                      /* :152 */
            double temp = per / (1 - per);                     /* :153 */
            for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e) {      /* :155-161 */
                b2c[e] = temp;
                temp *= c2b[e];
                if (temp != temp) temp = 1.0;
            }
            if (ratio) ratio[j] = temp;                        /* :163 stores log(1/temp) */
            err[j] = (temp >= 1) ? 1 : 0;                      /* :164-168 */
            temp = 1.0;                                        /* :170 */
            for (int64_t e = g->colptr[j + 1] - 1; e >= g->colptr[j]; --e) { /* :171-177 */
                b2c[e] *= temp;
                temp *= c2b[e];
                if (temp != temp) temp = 1.0;
            }
        }
        /* :180-184  (sparse_H * err) .% 2 == syndrome */
        int ok = 1;
        for (int64_t i = 0; i < s && ok; ++i) {
            unsigned par = 0;
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) par ^= err[g->rowvar[k]];
            if (par != (unsigned)syn[i]) ok = 0;
        }
        if (ok) { converged = 1; break; }
    }
    if (iters_out) *iters_out = (max_iters > 0) ? it : 0;
    return converged;
}

/* Min-sum variant (LDPCB200_VARIANT_MINSUM).  NOT a restatement of the reference -- the package's
 * BeliefPropagationDecoder is sum-product only -- but the definition the CUDA min-sum kernels are
 * checked against: flooding schedule, early stop, tie rule and outputs as in decode_edge(),
 * messages are log-likelihood ratios L = log(P0/P1), prior L0 = log((1-per)/per).
 *   check i : out_k = (-1)^{s_i} * prod_{j!=k} sgn(L_j) * (alpha * min_{j!=k} |L_j|)   (first minimum wins ties;
 *             alpha = normalisation factor, default 0.875, bp_oracle_set_minsum_scale)
 *   var j   : T_0 = L0, T_{k+1} = T_k + M_k; U_last = 0, U_{k-1} = U_k + M_k; out_k = T_k + U_k
 *   decision: 1 iff posterior T_D <= 0.   ratio[] receives the posterior LLR. */
static double g_minsum_scale = 0.875;
void bp_oracle_set_minsum_scale(double a) { g_minsum_scale = a; }

static int decode_edge_minsum(const graph_t *g, double per, int max_iters, const uint8_t *syn,
                              double *b2c, double *c2b, uint8_t *err, double *ratio, int32_t *iters_out)
{
    const int64_t s = g->s, n = g->n;
    volatile double one_minus = 1.0 - per;
    volatile double r = one_minus / per;
    const double L0 = log(r);
    memset(err, 0, (size_t)n);
    if (ratio) for (int64_t j = 0; j < n; ++j) ratio[j] = 0.0;
    for (int64_t e = 0; e < g->E; ++e) b2c[e] = L0;
    int converged = 0;
    int32_t it = 0;
    for (int iter = 1; iter <= max_iters; ++iter) {
        it = iter;
        for (int64_t i = 0; i < s; ++i) {
            int par = syn[i] ? 1 : 0;
            double m1 = INFINITY, m2 = INFINITY;
            int64_t idx = -1;
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) {
                const double L = b2c[g->rowedge[k]];
                par ^= signbit(L) ? 1 : 0;
                const double a = fabs(L);
                if (a < m1) { m2 = m1; m1 = a; idx = k; }
                else if (a < m2) m2 = a;
            }
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) {
                const int64_t e = g->rowedge[k];
                const double mag = ((k == idx) ? m2 : m1) * g_minsum_scale;
                const int sk = par ^ (signbit(b2c[e]) ? 1 : 0);
                c2b[e] = sk ? -mag : mag;
            }
        }
        for (int64_t j = 0; j < n; ++j) {
            double run = L0;
            for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e) {
                b2c[e] = run;
                run = run + c2b[e];
            }
            if (ratio) ratio[j] = run;
            err[j] = (run <= 0) ? 1 : 0;
            double U = 0.0;
            for (int64_t e = g->colptr[j + 1] - 1; e >= g->colptr[j]; --e) {
                b2c[e] = b2c[e] + U;
                U = U + c2b[e];
            }
        }
        int ok = 1;
        for (int64_t i = 0; i < s && ok; ++i) {
            unsigned par = 0;
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) par ^= err[g->rowvar[k]];
            if (par != (unsigned)syn[i]) ok = 0;
        }
        if (ok) { converged = 1; break; }
    }
    if (iters_out) *iters_out = (max_iters > 0) ? it : 0;
    return converged;
}

/* Fast FP32 variant (LDPCB200_VARIANT_FAST32).  NOT a restatement of the BP decoder -- the reference's BP decoder works in the
 * ratio domain in Float64 -- but the definition the CUDA fast kernels are compared with: the clamped tanh/atanh check update
 * of the only LLR-domain BP in the package (src/decoders/bpots_decoder.jl:182-211: tanh(nu/2) clamped to +-0.99999, product
 * clamped to +-0.99999, 2 atanh) on the BP decoder's flooding schedule, priors log((1-per)/per), early stop and tie rule, all
 * in float.  tanh(L/2) = (1-u)/(1+u), u = 2^(-|L| log2 e); 2 atanh(x) = ln 2 * log2((1+x)/(1-x)).  The kernels evaluate
 * 2^x, 1/x and log2 x with the GPU's special-function unit, so agreement is statistical (the tests bound it), not bitwise. */
static float fast_tanh_half(float L)
{
    float u = exp2f(-fabsf(L) * 1.4426950408889634f);
    float t = (1.0f - u) / (1.0f + u);
    if (t > 0.99999f) t = 0.99999f;
    return copysignf(t, L);
}
static float fast_two_atanh(float x)
{
    if (x > 0.99999f) x = 0.99999f;
    if (x < -0.99999f) x = -0.99999f;
    return log2f((1.0f + x) / (1.0f - x)) * 0.6931471805599453f;
}

static int decode_edge_fast32(const graph_t *g, double per, int max_iters, const uint8_t *syn,
                              double *b2c_d, double *c2b_d, uint8_t *err, double *ratio, int32_t *iters_out)
{
    const int64_t s = g->s, n = g->n;
    float *b2c = (float *)b2c_d, *c2b = (float *)c2b_d;         /* the double buffers are large enough */
    volatile double one_minus = 1.0 - per;
    volatile double r = one_minus / per;
    const float L0 = (float)log(r);
    float t[128], S[128];
    memset(err, 0, (size_t)n);
    if (ratio) for (int64_t j = 0; j < n; ++j) ratio[j] = 0.0;
    for (int64_t e = 0; e < g->E; ++e) b2c[e] = L0;
    int converged = 0;
    int32_t it = 0;
    for (int iter = 1; iter <= max_iters; ++iter) {
        it = iter;
        for (int64_t i = 0; i < s; ++i) {
            const int64_t r0 = g->rowptr[i], d = g->rowptr[i + 1] - r0;
            if (d == 0) continue;
            for (int64_t k = 0; k < d; ++k) t[k] = fast_tanh_half(b2c[g->rowedge[r0 + k]]);
            S[d - 1] = 1.0f;
            for (int64_t k = d - 2; k >= 0; --k) S[k] = S[k + 1] * t[k + 1];
            float P = syn[i] ? -1.0f : 1.0f;
            for (int64_t k = 0; k < d; ++k) {
                c2b[g->rowedge[r0 + k]] = fast_two_atanh(P * S[k]);
                P *= t[k];
            }
        }
        for (int64_t j = 0; j < n; ++j) {
            float run = L0;
            for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e) {
                b2c[e] = run;
                run = run + c2b[e];
            }
            if (ratio) ratio[j] = (double)run;
            err[j] = (run <= 0) ? 1 : 0;
            float U = 0.0f;
            for (int64_t e = g->colptr[j + 1] - 1; e >= g->colptr[j]; --e) {
                b2c[e] = b2c[e] + U;
                U = U + c2b[e];
            }
        }
        int ok = 1;
        for (int64_t i = 0; i < s && ok; ++i) {
            unsigned par = 0;
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) par ^= err[g->rowvar[k]];
            if (par != (unsigned)syn[i]) ok = 0;
        }
        if (ok) { converged = 1; break; }
    }
    if (iters_out) *iters_out = (max_iters > 0) ? it : 0;
    return converged;
}

/* One decode!, dense "faithful cost" storage: two s*n column-major matrices exactly like
 * BeliefPropagationScratchSpace (belief_propagation.jl:3-22), full reset per call (:83-91),
 * and the allocating mat-vec of :180-181. */
static int decode_dense(const graph_t *g, double per, int max_iters, const uint8_t *syn,
                        double *B2C, double *C2B, double *errd, double *chan, double *logp,
                        uint8_t *err, double *ratio, int32_t *iters_out)
{
    const int64_t s = g->s, n = g->n;
    for (int64_t j = 0; j < n; ++j) logp[j] = 0.0;
    for (int64_t j = 0; j < n; ++j) chan[j] = per;
    memset(B2C, 0, sizeof(double) * (size_t)s * (size_t)n);
    memset(C2B, 0, sizeof(double) * (size_t)s * (size_t)n);
    for (int64_t j = 0; j < n; ++j) errd[j] = 0.0;
    if (ratio) for (int64_t j = 0; j < n; ++j) ratio[j] = 1.0;
#define AT(M, i, j) (M)[(size_t)(i) + (size_t)(j) * (size_t)s]
    for (int64_t j = 0; j < n; ++j)
        for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e)
            AT(B2C, g->rowval[e], j) = chan[j] / (1 - chan[j]);
    int converged = 0;
    int32_t it = 0;
    for (int iter = 1; iter <= max_iters; ++iter) {
        it = iter;
        for (int64_t i = 0; i < s; ++i) {
            double temp = syn[i] ? -1.0 : 1.0;
            for (int64_t k = g->rowptr[i]; k < g->rowptr[i + 1]; ++k) {
                int64_t j = g->rowvar[k];
                AT(C2B, i, j) = temp;
                temp *= 2 / (1 + AT(B2C, i, j)) - 1;
            }
            temp = 1.0;
            for (int64_t k = g->rowptr[i + 1] - 1; k >= g->rowptr[i]; --k) {
                int64_t j = g->rowvar[k];
                AT(C2B, i, j) *= temp;
                AT(C2B, i, j) = (1 - AT(C2B, i, j)) / (1 + AT(C2B, i, j));
                temp *= 2 / (1 + AT(B2C, i, j)) - 1;
            }
        }
        for (int64_t j = 0; j < n; ++j) {
            double temp = chan[j] / (1 - chan[j]);
            for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e) {
                int64_t i = g->rowval[e];
                AT(B2C, i, j) = temp;
                temp *= AT(C2B, i, j);
                if (temp != temp) temp = 1.0;
            }
            logp[j] = log(1 / temp);
            if (ratio) ratio[j] = temp;
            errd[j] = (temp >= 1) ? 1.0 : 0.0;
            temp = 1.0;
            for (int64_t e = g->colptr[j + 1] - 1; e >= g->colptr[j]; --e) {
                int64_t i = g->rowval[e];
                AT(B2C, i, j) *= temp;
                temp *= AT(C2B, i, j);
                if (temp != temp) temp = 1.0;
            }
        }
#undef AT
        /* syndrome_decoded = (sparse_H * err) .% 2 ; all(syndrome_decoded .== syndrome) */
        double *prod = (double *)calloc((size_t)(s ? s : 1), sizeof(double));
        double *mod2 = (double *)malloc(sizeof(double) * (size_t)(s ? s : 1));
        uint8_t *eq = (uint8_t *)malloc((size_t)(s ? s : 1));
        for (int64_t j = 0; j < n; ++j)
            for (int64_t e = g->colptr[j]; e < g->colptr[j + 1]; ++e)
                prod[g->rowval[e]] += errd[j];
        int ok = 1;
        for (int64_t i = 0; i < s; ++i) mod2[i] = fmod(prod[i], 2.0);
        for (int64_t i = 0; i < s; ++i) eq[i] = (mod2[i] == (double)syn[i]);
        for (int64_t i = 0; i < s; ++i) ok &= eq[i];
        free(prod); free(mod2); free(eq);
        if (ok) { converged = 1; break; }
    }
    for (int64_t j = 0; j < n; ++j) err[j] = (uint8_t)(errd[j] != 0.0);
    if (iters_out) *iters_out = (max_iters > 0) ? it : 0;
    return converged;
}

/* batchdecode! : belief_propagation.jl:220-231.
 * syn  : s x B bytes, column-major (column b = syndrome b), values 0/1
 * err  : n x B bytes out, column-major
 * conv : B bytes out
 * iters: B int32 out or NULL ; ratio: n x B doubles out or NULL
 * nthreads: 1 = what the reference does (serial); >1 = one private scratch per thread.
 * Returns 0 on success. */
int bp_oracle_batch(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval,
                    double per, int32_t max_iters, int64_t B,
                    const uint8_t *syn, uint8_t *err, uint8_t *conv,
                    int32_t *iters, double *ratio, int32_t nthreads, int32_t dense)
{
    /* dense: 0 = edge-indexed, 1 = dense faithful cost, 2 = min-sum variant (edge-indexed), 3 = fast FP32 variant */
    graph_t g;
    int rc = build_graph(&g, s, n, colptr, rowval);
    if (rc) return rc;
    if (nthreads < 1) nthreads = 1;
    int fail = 0;
#ifdef _OPENMP
#pragma omp parallel num_threads(nthreads)
#endif
    {
        double *a = NULL, *b = NULL, *errd = NULL, *chan = NULL, *logp = NULL;
        size_t msz = (dense == 1) ? (size_t)s * (size_t)n : (size_t)g.E;
        if (msz == 0) msz = 1;
        a = (double *)malloc(sizeof(double) * msz);
        b = (double *)malloc(sizeof(double) * msz);
        errd = (double *)malloc(sizeof(double) * (size_t)(n ? n : 1));
        chan = (double *)malloc(sizeof(double) * (size_t)(n ? n : 1));
        logp = (double *)malloc(sizeof(double) * (size_t)(n ? n : 1));
        if (!a || !b || !errd || !chan || !logp) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
            fail = 1;
        } else {
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 16)
#endif
            for (int64_t c = 0; c < B; ++c) {
                const uint8_t *sc = syn + (size_t)c * (size_t)s;
                uint8_t *ec = err + (size_t)c * (size_t)n;
                double *rc_ = ratio ? ratio + (size_t)c * (size_t)n : NULL;
                int32_t itc = 0;
                int cv = (dense == 1) ? decode_dense(&g, per, max_iters, sc, a, b, errd, chan, logp, ec, rc_, &itc)
                       : (dense == 2) ? decode_edge_minsum(&g, per, max_iters, sc, a, b, ec, rc_, &itc)
                       : (dense == 3) ? decode_edge_fast32(&g, per, max_iters, sc, a, b, ec, rc_, &itc)
                                      : decode_edge(&g, per, max_iters, sc, a, b, ec, rc_, &itc);
                conv[c] = (uint8_t)cv;
                if (iters) iters[c] = itc;
            }
        }
        free(a); free(b); free(errd); free(chan); free(logp);
    }
    free_graph(&g);
    return fail ? -1 : 0;
}

/* ------------------------------------------------------------------------------------
 * Synthetic inputs: i.i.d. Bernoulli(per) bit-flips from Philox4x32-10, keyed by the global
 * syndrome index so that any sharding of the batch sees the same inputs
 * (SURVEY.md section 8d).  counter = (b_lo, b_hi, g, 0), key = (seed_lo, seed_hi);
 * the four 32-bit outputs decide bits 4g..4g+3:  e = (out < floor(per * 2^32)).
 * The CUDA sampler in the library (ldpcb200_sample) implements the same stream and is
 * checked against this one.
 * ---------------------------------------------------------------------------------- */
static inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                 uint32_t k0, uint32_t k1, uint32_t out[4])
{
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

uint32_t bp_oracle_threshold(double per)
{
    double t = floor(per * 4294967296.0);
    if (!(t > 0)) return 0;
    if (t >= 4294967295.0) return 0xFFFFFFFFu;
    return (uint32_t)t;
}

/* Fills true errors (n x B bytes, column-major) and syndromes (s x B bytes) for global
 * syndrome indices first .. first+B-1. */
int bp_oracle_sample(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval,
                     double per, uint64_t seed, int64_t first, int64_t B,
                     uint8_t *errs, uint8_t *syn)
{
    uint32_t thr = bp_oracle_threshold(per);
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int64_t c = 0; c < B; ++c) {
        uint64_t gb = (uint64_t)(first + c);
        uint8_t *ec = errs + (size_t)c * (size_t)n;
        uint8_t *sc = syn + (size_t)c * (size_t)s;
        memset(sc, 0, (size_t)s);
        for (int64_t g = 0; 4 * g < n; ++g) {
            uint32_t o[4];
            philox4x32_10((uint32_t)gb, (uint32_t)(gb >> 32), (uint32_t)g, 0u, k0, k1, o);
            for (int i = 0; i < 4 && 4 * g + i < n; ++i) ec[4 * g + i] = (uint8_t)(o[i] < thr);
        }
        for (int64_t j = 0; j < n; ++j)
            if (ec[j])
                for (int64_t e = colptr[j]; e < colptr[j + 1]; ++e) sc[rowval[e]] ^= 1;
    }
    return 0;
}

int bp_oracle_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* ------------------------------------------------------------------------------------
 * OSD-0 post-processing, the consumer of the BP stage in BASELINE config 4:
 * decode!(::BeliefPropagationOSDDecoder, syndrome)  belief_propagation_osd.jl:49-61 and
 * osd(H, syndrome, bp_err, Val(0))                  belief_propagation_osd.jl:63-125.
 * Control flow follows the reference statement by statement (physical row swaps, the early
 * break on an all-zero remaining target, the reverse back-substitution); rows of H_work are
 * bit-packed (uint64 words over the SORTED column positions), which changes no result.
 *
 * One stated deviation: the reference sorts on max(r, 1-r) with r = exp(log_probabs) and
 * log_probabs = log(1/R) (belief_propagation.jl:163, belief_propagation_osd.jl:52-55), using
 * Julia's own exp/log.  Those cannot be reproduced bit for bit here, so r = RN(1/R) is used
 * (the value exp(log(.)) approximates to a few ulp).  The order can differ from Julia's only
 * between two posteriors that agree to ~2^-45 relative without being equal; exact ties (the
 * common case, by symmetry) are broken by index exactly as Julia's stable sortperm does.
 * PARITY UNPINNED like the rest of this file.
 * ------------------------------------------------------------------------------------ */
typedef struct { double key; int64_t idx; } keyidx_t;

/* Sort key of the reliability order: 0 (default, what the CUDA kernel computes) r = RN(1/R); 1 r = exp(log(1/R)) with this
 * libm's exp/log -- the reference's own expression exp.(log_probabs), log_probabs = log(1/R) (belief_propagation.jl:163,
 * belief_propagation_osd.jl:53), evaluated with glibc instead of Julia's exp/log.  Mode 1 exists to MEASURE how often the
 * composition changes the order (tools/osd_key_study.py): it is not bit-identical to Julia either. */
static int g_osd_key_mode = 0;
void bp_oracle_set_osd_key_mode(int m) { g_osd_key_mode = m; }

static int cmp_keyidx_desc(const void *a, const void *b)
{
    const keyidx_t *x = (const keyidx_t *)a, *y = (const keyidx_t *)b;
    if (x->key > y->key) return -1;           /* rev=true: larger key first              */
    if (x->key < y->key) return 1;
    return (x->idx > y->idx) - (x->idx < y->idx);   /* stable: equal keys keep index order */
}

#define OSD_BIT(row, j) (((row)[(j) >> 6] >> ((j) & 63)) & 1ull)

static int osd0_one(const graph_t *g, const int64_t *colptr, const int64_t *rowval,
                    const uint8_t *syn, const uint8_t *bp_err, const double *ratio,
                    uint8_t *out, keyidx_t *ki, uint64_t *Hw, uint8_t *tgt,
                    uint8_t *err_sorted, uint8_t *corr, int64_t *piv_r, int64_t *piv_c)
{
    const int64_t m = g->s, n = g->n, nw = (n + 63) / 64;
    /* :53-55  reliability order */
    for (int64_t j = 0; j < n; ++j) {
        double r = 1.0 / ratio[j];
        if (g_osd_key_mode == 1) r = exp(log(r));
        double q = 1.0 - r;
        ki[j].key = (r > q) ? r : q;
        ki[j].idx = j;
    }
    qsort(ki, (size_t)n, sizeof(keyidx_t), cmp_keyidx_desc);
    /* :56-57  H_sorted (bit-packed rows), bp_err_sorted */
    memset(Hw, 0, sizeof(uint64_t) * (size_t)(m * nw));
    for (int64_t j = 0; j < n; ++j) {
        int64_t c = ki[j].idx;
        err_sorted[j] = bp_err[c];
        for (int64_t e = colptr[c]; e < colptr[c + 1]; ++e)
            Hw[rowval[e] * nw + (j >> 6)] |= 1ull << (j & 63);
    }
    /* :66-71  s_target = syndrome xor H*bp_err */
    for (int64_t i = 0; i < m; ++i) tgt[i] = syn[i] & 1;
    for (int64_t j = 0; j < n; ++j)
        if (err_sorted[j] == 1)
            for (int64_t i = 0; i < m; ++i) tgt[i] ^= (uint8_t)OSD_BIT(Hw + i * nw, j);
    int any = 0;
    for (int64_t i = 0; i < m; ++i) any |= tgt[i];
    memcpy(corr, err_sorted, (size_t)n);
    int64_t np = 0;
    if (any) {                                   /* :72-74 returns bp_err otherwise */
        int64_t i = 0;
        for (int64_t j = 0; j < n; ++j) {        /* :81-107 */
            if (i >= m) break;
            int rest = 0;
            for (int64_t ii = i; ii < m; ++ii) rest |= tgt[ii];
            if (!rest) break;
            int64_t k = -1;
            for (int64_t ii = i; ii < m; ++ii) if (OSD_BIT(Hw + ii * nw, j)) { k = ii; break; }
            if (k < 0) continue;
            if (err_sorted[j] == 1)
                for (int64_t ii = 0; ii < m; ++ii) tgt[ii] ^= (uint8_t)OSD_BIT(Hw + ii * nw, j);
            if (k != i) {
                for (int64_t w = 0; w < nw; ++w) {
                    uint64_t t = Hw[i * nw + w]; Hw[i * nw + w] = Hw[k * nw + w]; Hw[k * nw + w] = t;
                }
                uint8_t t = tgt[i]; tgt[i] = tgt[k]; tgt[k] = t;
            }
            for (int64_t ii = i + 1; ii < m; ++ii)
                if (OSD_BIT(Hw + ii * nw, j)) {
                    for (int64_t w = 0; w < nw; ++w) Hw[ii * nw + w] ^= Hw[i * nw + w];
                    tgt[ii] ^= tgt[i];
                }
            piv_r[np] = i; piv_c[np] = j; ++np;
            ++i;
        }
        for (int64_t q = np - 1; q >= 0; --q) {  /* :110-121 */
            int64_t r = piv_r[q], c = piv_c[q];
            corr[c] = tgt[r];
            if (corr[c])
                for (int64_t ii = 0; ii < r; ++ii)
                    if (OSD_BIT(Hw + ii * nw, c)) tgt[ii] ^= 1;
        }
    }
    for (int64_t j = 0; j < n; ++j) out[ki[j].idx] = corr[j];   /* :60 err[invperm(...)] */
    return (int)np;
}

/* osd(H, syndrome, bp_err, Val{O}) for O > 0: belief_propagation_osd.jl:127-209, statement by statement (physical row
 * swaps, full Gauss-Jordan without early exit, the exhaustive 2^O search over the first O non-pivot columns with the
 * strict `<` on the weight, so the first minimum wins).  Rows are bit-packed over the SORTED column positions.  Applied to
 * EVERY syndrome -- decode! has no shortcut for converged ones when osd_order > 0 (:49-61).  out: n bytes in the
 * original column order (:60).  Returns the rank r. */
static int osdk_one(const graph_t *g, const int64_t *colptr, const int64_t *rowval, const uint8_t *syn, const uint8_t *bp_err,
                    const double *ratio, int order, uint8_t *out, keyidx_t *ki, uint64_t *Hw, uint8_t *sv, uint8_t *err,
                    uint8_t *best, int64_t *piv_r, int64_t *piv_c, int64_t *mrc)
{
    const int64_t m = g->s, n = g->n, nw = (n + 63) / 64;
    for (int64_t j = 0; j < n; ++j) {                      /* :53-55 reliability order (same key as osd0_one) */
        double r = 1.0 / ratio[j];
        if (g_osd_key_mode == 1) r = exp(log(r));
        double q = 1.0 - r;
        ki[j].key = (r > q) ? r : q;
        ki[j].idx = j;
    }
    qsort(ki, (size_t)n, sizeof(keyidx_t), cmp_keyidx_desc);
    memset(Hw, 0, sizeof(uint64_t) * (size_t)(m * nw));
    for (int64_t j = 0; j < n; ++j) {                      /* :56-57 */
        int64_t c = ki[j].idx;
        err[j] = bp_err[c];
        for (int64_t e = colptr[c]; e < colptr[c + 1]; ++e) Hw[rowval[e] * nw + (j >> 6)] |= 1ull << (j & 63);
    }
    for (int64_t i = 0; i < m; ++i) sv[i] = syn[i] & 1;    /* :137 s = copy(syndrome) */
    int64_t np = 0, i = 0, j = 0;
    while (i < m && j < n) {                               /* :139-160 */
        int64_t k = -1;
        for (int64_t ii = i; ii < m; ++ii) if (OSD_BIT(Hw + ii * nw, j)) { k = ii; break; }
        if (k < 0) { ++j; continue; }
        if (k != i) {
            for (int64_t w = 0; w < nw; ++w) { uint64_t t = Hw[i * nw + w]; Hw[i * nw + w] = Hw[k * nw + w]; Hw[k * nw + w] = t; }
            uint8_t t = sv[i]; sv[i] = sv[k]; sv[k] = t;
        }
        for (int64_t ii = i + 1; ii < m; ++ii)
            if (OSD_BIT(Hw + ii * nw, j)) {
                for (int64_t w = 0; w < nw; ++w) Hw[ii * nw + w] ^= Hw[i * nw + w];
                sv[ii] ^= sv[i];
            }
        piv_r[np] = i; piv_c[np] = j; ++np;
        ++i; ++j;
    }
    for (int64_t q = np - 1; q >= 0; --q) {                /* :163-170 diagonalise */
        const int64_t pi = piv_r[q], pj = piv_c[q];
        for (int64_t ii = 0; ii < pi; ++ii)
            if (OSD_BIT(Hw + ii * nw, pj)) {
                for (int64_t w = 0; w < nw; ++w) Hw[ii * nw + w] ^= Hw[pi * nw + w];
                sv[ii] ^= sv[pi];
            }
    }
    if (order > n - np) order = (int)(n - np);            /* :172-175 */
    int64_t nm = 0;                                        /* most_reliable_cols = setdiff(1:n, pivot columns), ascending */
    {
        int64_t q = 0;
        for (int64_t c = 0; c < n; ++c) {
            if (q < np && piv_c[q] == c) { ++q; continue; }
            mrc[nm++] = c;
        }
    }
    memcpy(best, err, (size_t)n);                          /* best_err = copy(bp_err) */
    int64_t min_weight = n + 1;
    for (uint64_t x = 0; x < (1ull << order); ++x) {       /* :182-206 */
        if (x != 0)
            for (int b = 0; b < order; ++b) err[mrc[b]] = (uint8_t)((x >> b) & 1);
        for (int64_t q = 0; q < np; ++q) {
            const int64_t pi = piv_r[q], pj = piv_c[q];
            uint8_t v = sv[pi];
            for (int64_t t = 0; t < nm; ++t) v ^= (uint8_t)(OSD_BIT(Hw + pi * nw, mrc[t]) & err[mrc[t]]);
            err[pj] = v;
        }
        int64_t weight = 0;
        for (int64_t c = 0; c < n; ++c) weight += err[c];
        if (weight < min_weight) { min_weight = weight; memcpy(best, err, (size_t)n); }
    }
    for (int64_t c = 0; c < n; ++c) out[ki[c].idx] = best[c];   /* :60 err[invperm(...)] */
    return (int)np;
}

/* BP followed by OSD of order `order` > 0 on every column (decode!(::BeliefPropagationOSDDecoder, ...) with osd_order = order). */
int bp_oracle_bposd_order_batch(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval, double per, int32_t max_iters,
                                int32_t order, int64_t B, const uint8_t *syn, uint8_t *err, uint8_t *conv, int32_t nthreads)
{
    graph_t g;
    int rc = build_graph(&g, s, n, colptr, rowval);
    if (rc) return rc;
    if (nthreads < 1) nthreads = 1;
    int fail = 0;
    const size_t nn = (size_t)(n ? n : 1), ss = (size_t)(s ? s : 1), nw = (size_t)((n + 63) / 64 + 1);
#ifdef _OPENMP
#pragma omp parallel num_threads(nthreads)
#endif
    {
        size_t msz = g.E ? (size_t)g.E : 1;
        double *a = (double *)malloc(sizeof(double) * msz), *b = (double *)malloc(sizeof(double) * msz);
        double *ratio = (double *)malloc(sizeof(double) * nn);
        uint8_t *bp = (uint8_t *)malloc(nn), *sv = (uint8_t *)malloc(ss), *e1 = (uint8_t *)malloc(nn), *best = (uint8_t *)malloc(nn);
        keyidx_t *ki = (keyidx_t *)malloc(sizeof(keyidx_t) * nn);
        uint64_t *Hw = (uint64_t *)malloc(sizeof(uint64_t) * ss * nw);
        int64_t *pr = (int64_t *)malloc(sizeof(int64_t) * ss), *pc = (int64_t *)malloc(sizeof(int64_t) * ss);
        int64_t *mrc = (int64_t *)malloc(sizeof(int64_t) * nn);
        if (!a || !b || !ratio || !bp || !sv || !e1 || !best || !ki || !Hw || !pr || !pc || !mrc) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
            fail = 1;
        } else {
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 4)
#endif
            for (int64_t c = 0; c < B; ++c) {
                const uint8_t *sc = syn + (size_t)c * (size_t)s;
                int32_t itc = 0;
                conv[c] = (uint8_t)decode_edge(&g, per, max_iters, sc, a, b, bp, ratio, &itc);
                osdk_one(&g, colptr, rowval, sc, bp, ratio, order, err + (size_t)c * (size_t)n, ki, Hw, sv, e1, best, pr, pc, mrc);
            }
        }
        free(a); free(b); free(ratio); free(bp); free(sv); free(e1); free(best); free(ki); free(Hw); free(pr); free(pc); free(mrc);
    }
    free_graph(&g);
    return fail ? -1 : 0;
}

/* BP followed by OSD-0 on every column of the batch (decode! of the BP+OSD decoder applied per
 * column).  err: n x B bytes out (the OSD result), conv: BP's converged flag (:60), bp_err:
 * optional n x B bytes (BP's own decisions), pivots: optional B int32 (pivots used). */
int bp_oracle_bposd_batch(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval,
                          double per, int32_t max_iters, int64_t B, const uint8_t *syn,
                          uint8_t *err, uint8_t *conv, uint8_t *bp_err_out, int32_t *pivots,
                          int32_t nthreads)
{
    graph_t g;
    int rc = build_graph(&g, s, n, colptr, rowval);
    if (rc) return rc;
    if (nthreads < 1) nthreads = 1;
    int fail = 0;
    const size_t nn = (size_t)(n ? n : 1), ss = (size_t)(s ? s : 1), nw = (size_t)((n + 63) / 64 + 1);
#ifdef _OPENMP
#pragma omp parallel num_threads(nthreads)
#endif
    {
        size_t msz = g.E ? (size_t)g.E : 1;
        double *a = (double *)malloc(sizeof(double) * msz), *b = (double *)malloc(sizeof(double) * msz);
        double *ratio = (double *)malloc(sizeof(double) * nn);
        uint8_t *bp = (uint8_t *)malloc(nn), *tgt = (uint8_t *)malloc(ss);
        uint8_t *es = (uint8_t *)malloc(nn), *corr = (uint8_t *)malloc(nn);
        keyidx_t *ki = (keyidx_t *)malloc(sizeof(keyidx_t) * nn);
        uint64_t *Hw = (uint64_t *)malloc(sizeof(uint64_t) * ss * nw);
        int64_t *pr = (int64_t *)malloc(sizeof(int64_t) * ss), *pc = (int64_t *)malloc(sizeof(int64_t) * ss);
        if (!a || !b || !ratio || !bp || !tgt || !es || !corr || !ki || !Hw || !pr || !pc) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
            fail = 1;
        } else {
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 4)
#endif
            for (int64_t c = 0; c < B; ++c) {
                const uint8_t *sc = syn + (size_t)c * (size_t)s;
                int32_t itc = 0;
                int cv = decode_edge(&g, per, max_iters, sc, a, b, bp, ratio, &itc);
                conv[c] = (uint8_t)cv;
                if (bp_err_out) memcpy(bp_err_out + (size_t)c * (size_t)n, bp, (size_t)n);
                int np = 0;
                /* max_iters = 0 leaves log_probabs = 0, i.e. ratio 1 everywhere (decode_edge does that) */
                np = osd0_one(&g, colptr, rowval, sc, bp, ratio, err + (size_t)c * (size_t)n,
                              ki, Hw, tgt, es, corr, pr, pc);
                if (pivots) pivots[c] = np;
            }
        }
        free(a); free(b); free(ratio); free(bp); free(tgt); free(es); free(corr); free(ki); free(Hw); free(pr); free(pc);
    }
    free_graph(&g);
    return fail ? -1 : 0;
}

/* OSD-0 (osd0_one) on caller-supplied BP decisions and posterior ratios, every column: osd(..., Val(0)) as a function of
 * (syndrome, bp_err, ratio) alone, whatever produced them.  syn: s x B, bp_err: n x B bytes, ratio: n x B doubles, all
 * column-major; err_out: n x B bytes, pivots_out: optional B int32 (pivots used; 0 where bp_err already satisfies the
 * syndrome). */
int bp_oracle_osd0_given(int64_t s, int64_t n, const int64_t *colptr, const int64_t *rowval, int64_t B, const uint8_t *syn,
                         const uint8_t *bp_err, const double *ratio, uint8_t *err_out, int32_t *pivots_out, int32_t nthreads)
{
    graph_t g;
    int rc = build_graph(&g, s, n, colptr, rowval);
    if (rc) return rc;
    if (nthreads < 1) nthreads = 1;
    int fail = 0;
    const size_t nn = (size_t)(n ? n : 1), ss = (size_t)(s ? s : 1), nw = (size_t)((n + 63) / 64 + 1);
#ifdef _OPENMP
#pragma omp parallel num_threads(nthreads)
#endif
    {
        uint8_t *tgt = (uint8_t *)malloc(ss), *es = (uint8_t *)malloc(nn), *corr = (uint8_t *)malloc(nn);
        keyidx_t *ki = (keyidx_t *)malloc(sizeof(keyidx_t) * nn);
        uint64_t *Hw = (uint64_t *)malloc(sizeof(uint64_t) * ss * nw);
        int64_t *pr = (int64_t *)malloc(sizeof(int64_t) * ss), *pc = (int64_t *)malloc(sizeof(int64_t) * ss);
        if (!tgt || !es || !corr || !ki || !Hw || !pr || !pc) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
            fail = 1;
        } else {
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 4)
#endif
            for (int64_t c = 0; c < B; ++c) {
                const int np = osd0_one(&g, colptr, rowval, syn + (size_t)c * (size_t)s, bp_err + (size_t)c * (size_t)n,
                                        ratio + (size_t)c * (size_t)n, err_out + (size_t)c * (size_t)n, ki, Hw, tgt, es, corr, pr, pc);
                if (pivots_out) pivots_out[c] = np;
            }
        }
        free(tgt); free(es); free(corr); free(ki); free(Hw); free(pr); free(pc);
    }
    free_graph(&g);
    return fail ? -1 : 0;
}
