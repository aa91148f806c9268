/*
 * Per-query drivers: JSON in -> device seam -> JSON out.
 *
 * Each driver mirrors the reference's _parse / _query / _nd_accum_update trio
 * (arbplfll.c:110-323, arbplfderiv.c:210-531, arbplfmarginal.c:111-446,
 * arbplfdwell.c:116-610, arbplftrans.c:115-660) except that the loop nest
 * over sites x categories x nodes and the precision loop are replaced by one
 * call into the CUDA engine (include/plf.h).  What stays on the host is the
 * reference's outer, precision-agnostic layer: schema validation, selection /
 * aggregation weights and the output table.
 */
#include <fenv.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <time.h>

#include "arbplf.h"
#include "plf.h"
#include "json.h"
#include "model.h"
#include "reduce.h"
#include "dd.h"

/* One engine per process, shared by every arbplf_* call.  The reference's functions are re-entrant (all state on
 * the caller's stack, runjson.c:10-66); here calls from several host threads are serialised on this lock, held from
 * the moment a call takes the engine (ctx_load) until it has built its result (ctx_clear). */
static plf_engine *g_engine = NULL;
static int g_device = -1;
static pthread_mutex_t g_engine_lock = PTHREAD_MUTEX_INITIALIZER;

/* what the shared engine holds from the previous call (guarded by g_engine_lock, like the engine) */
static struct {
    plf_engine *e;
    int N, n, K;
    int *indptr, *indices, *preorder;
    double *defs;
    jv_codes *data;
} g_resident;

static void resident_forget_data(void)
{
    if (g_resident.data) json_codes_release(g_resident.data);
    free(g_resident.defs);
    g_resident.data = NULL; g_resident.defs = NULL; g_resident.K = 0;
}

static void resident_forget(void)
{
    resident_forget_data();
    free(g_resident.indptr); free(g_resident.indices); free(g_resident.preorder);
    memset(&g_resident, 0, sizeof g_resident);
}

static int *copy_ints(const int *src, size_t n)
{
    int *p = malloc(sizeof(int) * (n ? n : 1));
    if (p) memcpy(p, src, sizeof(int) * n);
    return p;
}

void arbplf_set_device(int device)
{
    pthread_mutex_lock(&g_engine_lock);
    if (g_engine && device != g_device) { plf_destroy(g_engine); g_engine = NULL; resident_forget(); }
    g_device = device;
    pthread_mutex_unlock(&g_engine_lock);
}

static plf_engine *get_engine(void)
{
    if (g_engine) return g_engine;
    if (g_device < 0) {
        const char *s = getenv("ARBPLF_DEVICE");
        g_device = s ? atoi(s) : 0;
    }
    if (plf_create(&g_engine, g_device)) {
        fprintf(stderr, "error: cannot create the CUDA engine on device %d (this build has no CPU path)\n", g_device);
        g_engine = NULL;
    }
    return g_engine;
}

/* wall-clock phases of the most recent call: parse (JSON + schema), model + upload, compute, emit */
static double g_phase[4];
static double now_s(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
void arbplf_last_timing(double out[4]) { memcpy(out, g_phase, sizeof g_phase); }

typedef struct {
    jv *root;
    plf_model m;
    plf_derived d;
    plf_engine *e;
    int loaded;
    int locked;         /* this call holds g_engine_lock */
    double t_mark;      /* start of the phase in progress */
} ctx;

static void ctx_clear(ctx *c)
{
    json_free(c->root);
    plf_model_clear(&c->m);
    plf_derived_clear(&c->d);
    if (c->locked) pthread_mutex_unlock(&g_engine_lock);
    memset(c, 0, sizeof(*c));
}

/* parse the document and the model; keys: NULL-terminated list for the strict top-level unpack */
static int ctx_parse(ctx *c, const char *json_in, const char *const *keys, const jv **out)
{
    char err[256];
    memset(c, 0, sizeof(*c));
    c->t_mark = now_s();
    memset(g_phase, 0, sizeof g_phase);
    plf_model_init(&c->m);
    c->root = json_parse(json_in, err, sizeof err);
    if (!c->root) { fprintf(stderr, "%s\n", err); return -1; }
    if (jv_unpack_strict(c->root, keys, out)) return -1;
    if (plf_model_parse(&c->m, out[0])) return -1;
    g_phase[0] = now_s() - c->t_mark; c->t_mark = now_s();
    return 0;
}

/* push tree, model and data to the device */
static int ctx_load(ctx *c)
{
    if (plf_derive(&c->d, &c->m)) return -1;
    if (!c->locked) { pthread_mutex_lock(&g_engine_lock); c->locked = 1; }
    c->e = get_engine();
    if (!c->e) return -1;
    const plf_model *m = &c->m;
    const plf_derived *d = &c->d;
#define EK(call) do { if (call) { fprintf(stderr, "error: %s\n", plf_last_error(c->e)); return -1; } } while (0)
    /* What the engine already holds from the previous call stays there: the tree if it is the same, and the alignment
     * if the reader recognised its text (json.h: the codes are then the very buffer that was uploaded last time) and the
     * definitions are the same -- an optimiser that varies the edge rates re-sends both with every call. */
    const int same_tree = g_resident.e == c->e && g_resident.N == m->N && g_resident.indptr &&
                          !memcmp(g_resident.indptr, m->indptr, sizeof(int) * (size_t)(m->N + 1)) &&
                          !memcmp(g_resident.indices, m->indices, sizeof(int) * (size_t)m->E) &&
                          !memcmp(g_resident.preorder, m->preorder, sizeof(int) * (size_t)m->N);
    if (!same_tree) {
        resident_forget();
        EK(plf_set_tree(c->e, m->N, m->indptr, m->indices, m->preorder));
        g_resident.e = c->e; g_resident.N = m->N;
        g_resident.indptr = copy_ints(m->indptr, (size_t)m->N + 1);
        g_resident.indices = copy_ints(m->indices, (size_t)m->E);
        g_resident.preorder = copy_ints(m->preorder, (size_t)m->N);
        if (!g_resident.indptr || !g_resident.indices || !g_resident.preorder) resident_forget();
    }
    if (g_resident.n != m->n) resident_forget_data();       /* plf_set_model drops the data when the state count changes */
    EK(plf_set_model(c->e, m->n, d->C, d->q_hi, d->q_lo, d->edge_rates_csr, d->cat_rates, d->cat_prior,
                     m->root_mode, d->root_vec));
    g_resident.n = m->n;
    const int same_data = same_tree && m->S > 0 && m->codes_shared && m->codes_shared == g_resident.data &&
                          g_resident.K == m->K && g_resident.defs &&
                          !memcmp(g_resident.defs, m->defs, sizeof(double) * (size_t)m->K * (size_t)m->n);
    if (same_data) {
        if (getenv("ARBPLF_JSON_TRACE")) fprintf(stderr, "drivers: alignment already on the device, no upload\n");
    } else {
        resident_forget_data();
        /* the codes travel in chunks behind which the first query starts (they stay valid until ctx_clear) */
        if (m->S > 0) EK(plf_set_data_async(c->e, m->S, m->K, m->defs, m->codes, m->code_bytes, NULL));
        if (m->S > 0 && m->codes_shared && g_resident.e == c->e) {
            g_resident.defs = malloc(sizeof(double) * ((size_t)m->K * (size_t)m->n + 1));
            if (g_resident.defs) {
                memcpy(g_resident.defs, m->defs, sizeof(double) * (size_t)m->K * (size_t)m->n);
                g_resident.K = m->K;
                json_codes_retain(m->codes_shared);
                g_resident.data = m->codes_shared;
            }
        }
    }
    c->loaded = 1;
    g_phase[1] = now_s() - c->t_mark; c->t_mark = now_s();
    return 0;
}

static void phase_compute_done(ctx *c)
{
    g_phase[2] = now_s() - c->t_mark; c->t_mark = now_s();
}

static unsigned char *edge_mask_csr(const plf_model *m, const axis *edge_axis)
{
    unsigned char *mask = calloc(m->E > 0 ? m->E : 1, 1);
    for (int e = 0; e < m->E; e++) mask[m->order[e]] = edge_axis->requested[e];
    return mask;
}

static char *finish(ctx *c, char *out, int rc, int *retcode)
{
    /* callers mark the end of the compute phase with phase_compute_done(); whatever follows is output formatting */
    if (c->t_mark > 0) g_phase[3] = now_s() - c->t_mark;
    if (rc && c->locked) resident_forget();     /* after a failed call nothing is assumed about what the engine holds */
    ctx_clear(c);
    *retcode = rc;
    if (rc) { free(out); return NULL; }
    return out;
}

/* ------------------------------------------------------------------ */
/* arbplf-ll                                                           */
/* ------------------------------------------------------------------ */

char *arbplf_ll(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", NULL};
    const jv *v[2];
    ctx c;
    reduction r_site; reduction_init(&r_site);
    axis ax[1]; memset(ax, 0, sizeof ax);
    double *val = NULL, *site_ll = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site)) goto done;
    val = calloc(ax[0].aggregated ? 1 : (S > 0 ? S : 1), sizeof(double));
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        if (ax[0].aggregated) {
            if (plf_set_site_weights(c.e, ax[0].w) || plf_ll(c.e, NULL, &val[0])) {
                fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done;
            }
        } else {
            site_ll = malloc(sizeof(double) * S);
            if (plf_set_site_weights(c.e, NULL) || plf_ll(c.e, site_ll, NULL)) {
                fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done;
            }
            for (int64_t s = 0; s < S; s++) {
                if (!ax[0].requested[s]) continue;
                if (!isfinite(site_ll[s])) { fprintf(stderr, "error: site %lld has zero likelihood\n", (long long)s); goto done; }
                val[s] = site_ll[s];
            }
        }
    }
    phase_compute_done(&c);
    out = table_to_json(ax, 1, val);
    rc = 0;
done:
    free(val); free(site_ll);
    axis_clear(&ax[0]); reduction_clear(&r_site);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* shared by deriv / dwell / trans: values over (site, edge[, third])  */
/* ------------------------------------------------------------------ */

/*
 * One engine call producing edge values for all sites (kind < 0: derivative).
 * Fills val over (site, user edge) at third-axis coordinate `third` (stride 1,
 * extent third_n), applying the site / edge aggregation weights.
 */
static int edge_pass(ctx *c, int kind, const double *l_hi, const double *l_lo,
                     const axis *ax_site, const axis *ax_edge, const unsigned char *mask,
                     double *val, int third, int third_n)
{
    const plf_model *m = &c->m;
    const int E = m->E;
    const int64_t S = m->S;
    int rc = -1;
    double *sum = NULL, *per_site = NULL, *site_ll = NULL;
    const size_t edge_ext = ax_edge->aggregated ? 1 : (size_t)E;
    if (ax_site->aggregated) {
        sum = calloc(E > 0 ? E : 1, sizeof(double));
        double dummy = 0;
        int r;
        if (plf_set_site_weights(c->e, ax_site->w)) goto engine_error;
        if (kind < 0) r = plf_deriv(c->e, mask, NULL, &dummy, NULL, sum);
        else r = plf_edge_expect(c->e, kind, l_hi, l_lo, mask, NULL, sum);
        if (r) goto engine_error;
        for (int e = 0; e < E; e++) {
            if (!ax_edge->requested[e]) continue;
            double x = sum[m->order[e]];
            if (!isfinite(x)) { fprintf(stderr, "error: a requested site has zero likelihood\n"); goto done; }
            if (ax_edge->aggregated) val[third] += x * ax_edge->w[e];
            else val[(size_t)e * third_n + third] = x;
        }
    } else {
        per_site = malloc(sizeof(double) * (size_t)S * (E > 0 ? E : 1));
        int r;
        if (plf_set_site_weights(c->e, NULL)) goto engine_error;
        if (kind < 0) r = plf_deriv(c->e, mask, NULL, NULL, per_site, NULL);
        else r = plf_edge_expect(c->e, kind, l_hi, l_lo, mask, per_site, NULL);
        if (r) goto engine_error;
        for (int64_t s = 0; s < S; s++) {
            if (!ax_site->requested[s]) continue;
            for (int e = 0; e < E; e++) {
                if (!ax_edge->requested[e]) continue;
                double x = per_site[(size_t)s * E + m->order[e]];
                if (!isfinite(x)) { fprintf(stderr, "error: site %lld has zero likelihood\n", (long long)s); goto done; }
                if (ax_edge->aggregated) val[(size_t)s * third_n + third] += x * ax_edge->w[e];
                else val[((size_t)s * edge_ext + e) * third_n + third] = x;
            }
        }
    }
    rc = 0;
    goto done;
engine_error:
    fprintf(stderr, "error: %s\n", plf_last_error(c->e));
done:
    free(sum); free(per_site); free(site_ll);
    return rc;
}

char *arbplf_deriv(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?edge_reduction", NULL};
    const jv *v[3];
    ctx c;
    reduction r_site, r_edge; reduction_init(&r_site); reduction_init(&r_edge);
    axis ax[2]; memset(ax, 0, sizeof ax);
    double *val = NULL;
    unsigned char *mask = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    if (reduction_parse(&r_site, (int)c.m.S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, c.m.E, "edge", v[2])) goto done;
    if (axis_init(&ax[0], "site", (int)c.m.S, &r_site) || axis_init(&ax[1], "edge", c.m.E, &r_edge)) goto done;
    {
        size_t cells = (ax[0].aggregated ? 1 : (size_t)c.m.S) * (ax[1].aggregated ? 1 : (size_t)c.m.E);
        val = calloc(cells ? cells : 1, sizeof(double));
    }
    if (c.m.S > 0) {
        if (ctx_load(&c)) goto done;
        mask = edge_mask_csr(&c.m, &ax[1]);
        if (edge_pass(&c, -1, NULL, NULL, &ax[0], &ax[1], mask, val, 0, 1)) goto done;
    }
    phase_compute_done(&c);
    out = table_to_json(ax, 2, val);
    rc = 0;
done:
    free(val); free(mask);
    axis_clear(&ax[0]); axis_clear(&ax[1]);
    reduction_clear(&r_site); reduction_clear(&r_edge);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* arbplf-marginal                                                     */
/* ------------------------------------------------------------------ */

char *arbplf_marginal(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?node_reduction", "?state_reduction", NULL};
    const jv *v[4];
    ctx c;
    reduction r_site, r_node, r_state;
    reduction_init(&r_site); reduction_init(&r_node); reduction_init(&r_state);
    axis ax[3]; memset(ax, 0, sizeof ax);
    double *val = NULL, *buf = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int N = c.m.N, n = c.m.n;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_node, N, "node", v[2])) goto done;
    if (reduction_parse(&r_state, n, "state", v[3])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "node", N, &r_node) ||
        axis_init(&ax[2], "state", n, &r_state)) goto done;
    const size_t e1 = ax[1].aggregated ? 1 : (size_t)N, e2 = ax[2].aggregated ? 1 : (size_t)n;
    val = calloc((ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * e1 * e2, sizeof(double));
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        const int64_t rows = ax[0].aggregated ? 1 : S;
        buf = malloc(sizeof(double) * (size_t)rows * N * n);
        int r;
        if (ax[0].aggregated) r = plf_set_site_weights(c.e, ax[0].w) || plf_marginal(c.e, NULL, buf);
        else r = plf_set_site_weights(c.e, NULL) || plf_marginal(c.e, buf, NULL);
        if (r) { fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done; }
        for (int64_t s = 0; s < rows; s++) {
            if (!ax[0].aggregated && !ax[0].requested[s]) continue;
            for (int a = 0; a < N; a++) {
                if (!ax[1].requested[a]) continue;
                for (int j = 0; j < n; j++) {
                    if (!ax[2].requested[j]) continue;
                    double x = buf[((size_t)s * N + a) * n + j];
                    if (!isfinite(x)) { fprintf(stderr, "error: a requested site has zero likelihood\n"); goto done; }
                    if (ax[1].aggregated) x *= ax[1].w[a];
                    if (ax[2].aggregated) x *= ax[2].w[j];
                    size_t off = ((size_t)s * e1 + (ax[1].aggregated ? 0 : a)) * e2 + (ax[2].aggregated ? 0 : j);
                    val[off] += x;
                }
            }
        }
    }
    phase_compute_done(&c);
    out = table_to_json(ax, 3, val);
    rc = 0;
done:
    free(val); free(buf);
    for (int i = 0; i < 3; i++) axis_clear(&ax[i]);
    reduction_clear(&r_site); reduction_clear(&r_node); reduction_clear(&r_state);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* arbplf-dwell / arbplf-trans                                         */
/* ------------------------------------------------------------------ */

char *arbplf_dwell(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?edge_reduction", "?state_reduction", NULL};
    const jv *v[4];
    ctx c;
    reduction r_site, r_edge, r_state;
    reduction_init(&r_site); reduction_init(&r_edge); reduction_init(&r_state);
    axis ax[3]; memset(ax, 0, sizeof ax);
    double *val = NULL, *L = NULL;
    unsigned char *mask = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int n = c.m.n, E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, E, "edge", v[2])) goto done;
    if (reduction_parse(&r_state, n, "state", v[3])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "edge", E, &r_edge) ||
        axis_init(&ax[2], "state", n, &r_state)) goto done;
    /* state aggregation is folded into the Frechet direction: ndim = 2 (arbplfdwell.c:462-468) */
    const int state_agg = ax[2].aggregated;
    const int third_n = state_agg ? 1 : n;
    {
        size_t cells = (ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * (ax[1].aggregated ? 1 : (size_t)E) * third_n;
        val = calloc(cells ? cells : 1, sizeof(double));
    }
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        mask = edge_mask_csr(&c.m, &ax[1]);
        L = calloc((size_t)n * n, sizeof(double));
        if (state_agg) {
            for (int s = 0; s < n; s++) L[s * n + s] = ax[2].w[s];     /* arbplfdwell.c:173-178 */
            if (edge_pass(&c, PLF_KIND_DWELL, L, NULL, &ax[0], &ax[1], mask, val, 0, 1)) goto done;
        } else {
            for (int s = 0; s < n; s++) {
                if (!ax[2].requested[s]) continue;
                memset(L, 0, sizeof(double) * n * n);
                L[s * n + s] = 1.0;                                     /* arbplfdwell.c:133 */
                if (edge_pass(&c, PLF_KIND_DWELL, L, NULL, &ax[0], &ax[1], mask, val, s, n)) goto done;
            }
        }
    }
    phase_compute_done(&c);
    out = table_to_json(ax, state_agg ? 2 : 3, val);
    rc = 0;
done:
    free(val); free(L); free(mask);
    for (int i = 0; i < 3; i++) axis_clear(&ax[i]);
    reduction_clear(&r_site); reduction_clear(&r_edge); reduction_clear(&r_state);
    return finish(&c, out, rc, retcode);
}

char *arbplf_trans(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?edge_reduction", "?trans_reduction", NULL};
    const jv *v[4];
    ctx c;
    reduction r_site, r_edge, r_trans;
    reduction_init(&r_site); reduction_init(&r_edge); reduction_init(&r_trans);
    axis ax[3]; memset(ax, 0, sizeof ax);
    double *val = NULL, *Lh = NULL, *Ll = NULL;
    unsigned char *mask = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int n = c.m.n, E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, E, "edge", v[2])) goto done;
    if (reduction_parse_pairs(&r_trans, n, "trans", v[3])) goto done;
    const int T = r_trans.selection_len;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "edge", E, &r_edge) ||
        axis_init(&ax[2], "trans", T, &r_trans)) goto done;
    ax[2].ncomp = 2;
    ax[2].comp_name[0] = "first_state"; ax[2].comp_name[1] = "second_state";
    ax[2].comp_idx[0] = r_trans.first_idx; ax[2].comp_idx[1] = r_trans.second_idx;
    const int trans_agg = ax[2].aggregated;
    const int third_n = trans_agg ? 1 : (T > 0 ? T : 1);
    {
        size_t cells = (ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * (ax[1].aggregated ? 1 : (size_t)E) * third_n;
        val = calloc(cells ? cells : 1, sizeof(double));
    }
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        mask = edge_mask_csr(&c.m, &ax[1]);
        Lh = calloc((size_t)n * n, sizeof(double));
        Ll = calloc((size_t)n * n, sizeof(double));
        if (trans_agg) {
            /* L = (sum_k w_k E_{a_k b_k}) .* Q / divisor  (arbplftrans.c:179-193) */
            double *W = calloc((size_t)n * n, sizeof(double));
            for (int k = 0; k < T; k++) W[r_trans.first_idx[k] * n + r_trans.second_idx[k]] += ax[2].w[k];
            for (int i = 0; i < n * n; i++) {
                dd_t q = dd_mul_d(dd_make(c.d.q_hi[i], c.d.q_lo[i]), W[i]);
                Lh[i] = q.hi; Ll[i] = q.lo;
            }
            free(W);
            if (edge_pass(&c, PLF_KIND_TRANS, Lh, Ll, &ax[0], &ax[1], mask, val, 0, 1)) goto done;
        } else {
            for (int k = 0; k < T; k++) {
                if (!ax[2].requested[k]) continue;
                memset(Lh, 0, sizeof(double) * n * n); memset(Ll, 0, sizeof(double) * n * n);
                int idx = r_trans.first_idx[k] * n + r_trans.second_idx[k];
                Lh[idx] = c.d.q_hi[idx]; Ll[idx] = c.d.q_lo[idx];      /* arbplftrans.c:133-134 */
                if (edge_pass(&c, PLF_KIND_TRANS, Lh, Ll, &ax[0], &ax[1], mask, val, k, third_n)) goto done;
            }
        }
    }
    phase_compute_done(&c);
    out = table_to_json(ax, trans_agg ? 2 : 3, val);
    rc = 0;
done:
    free(val); free(Lh); free(Ll); free(mask);
    for (int i = 0; i < 3; i++) axis_clear(&ax[i]);
    reduction_clear(&r_site); reduction_clear(&r_edge); reduction_clear(&r_trans);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* arbplf-em-update                                                    */
/* ------------------------------------------------------------------ */

/*
 * One EM update of the edge rate coefficients (arbplfem.c).  The reference accumulates, per edge,
 *   trans = sum_s w_s/L_s sum_c prior_c rate_c fe^T Frechet(offdiag Q) L_b     (arbplfem.c:122-128,351-353)
 *   dwell = sum_s w_s/L_s sum_c prior_c rate_c fe^T Frechet(diag -Q_ii) L_b     (arbplfem.c:117-120)
 * and returns t_e * trans / dwell (0 when trans is exactly 0, :434-458).  Both sums are what the device
 * seam's PLF_KIND_TRANS query returns for those two directions up to a common factor t_e, which cancels in
 * the ratio.  Site aggregation is required (:566-571); all edges are reported in the user's order.
 */
char *arbplf_em_update(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", NULL};
    const jv *v[2];
    ctx c;
    reduction r_site, r_edge;
    reduction_init(&r_site); reduction_init(&r_edge);
    axis ax_site, ax_edge;
    memset(&ax_site, 0, sizeof ax_site); memset(&ax_edge, 0, sizeof ax_edge);
    double *val = NULL, *Lh = NULL, *Ll = NULL, *sum_d = NULL, *sum_t = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int n = c.m.n, E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, E, "edge", NULL)) goto done;
    if (axis_init(&ax_site, "site", (int)S, &r_site) || axis_init(&ax_edge, "edge", E, &r_edge)) goto done;
    if (!ax_site.aggregated) { fprintf(stderr, "error: aggregation over sites is required\n"); goto done; }
    val = calloc(E > 0 ? E : 1, sizeof(double));
    if (S > 0 && E > 0) {
        if (ctx_load(&c)) goto done;
        Lh = calloc((size_t)n * n, sizeof(double));
        Ll = calloc((size_t)n * n, sizeof(double));
        sum_d = calloc(E, sizeof(double));
        sum_t = calloc(E, sizeof(double));
        if (plf_set_site_weights(c.e, ax_site.w)) { fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done; }
        /* exit rates on the diagonal */
        for (int i = 0; i < n; i++) { Lh[i * n + i] = -c.d.q_hi[i * n + i]; Ll[i * n + i] = -c.d.q_lo[i * n + i]; }
        if (plf_edge_expect(c.e, PLF_KIND_TRANS, Lh, Ll, NULL, NULL, sum_d)) { fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done; }
        /* rates off the diagonal */
        for (int i = 0; i < n; i++)
            for (int j = 0; j < n; j++) {
                Lh[i * n + j] = (i == j) ? 0.0 : c.d.q_hi[i * n + j];
                Ll[i * n + j] = (i == j) ? 0.0 : c.d.q_lo[i * n + j];
            }
        if (plf_edge_expect(c.e, PLF_KIND_TRANS, Lh, Ll, NULL, NULL, sum_t)) { fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done; }
        for (int e = 0; e < E; e++) {
            const int idx = c.m.order[e];
            double x = 0.0;
            if (sum_t[idx] != 0.0) x = sum_t[idx] / sum_d[idx] * c.d.edge_rates_csr[idx];
            if (!isfinite(x)) { fprintf(stderr, "error: the EM update of edge %d is not finite\n", e); goto done; }
            val[e] = x;
        }
    }
    phase_compute_done(&c);
    out = table_to_json(&ax_edge, 1, val);
    rc = 0;
done:
    free(val); free(Lh); free(Ll); free(sum_d); free(sum_t);
    axis_clear(&ax_site); axis_clear(&ax_edge);
    reduction_clear(&r_site); reduction_clear(&r_edge);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* model summary, stdio shell                                          */
/* ------------------------------------------------------------------ */

static void put_darray(jbuf *b, const char *key, const double *x, size_t n)
{
    jbuf_puts(b, "\""); jbuf_puts(b, key); jbuf_puts(b, "\": ");
    if (!x) { jbuf_puts(b, "null"); return; }
    jbuf_puts(b, "[");
    for (size_t i = 0; i < n; i++) { if (i) jbuf_puts(b, ", "); jbuf_real(b, x[i]); }
    jbuf_puts(b, "]");
}

static void put_iarray(jbuf *b, const char *key, const int *x, size_t n)
{
    jbuf_puts(b, "\""); jbuf_puts(b, key); jbuf_puts(b, "\": [");
    for (size_t i = 0; i < n; i++) { if (i) jbuf_puts(b, ", "); jbuf_int(b, x[i]); }
    jbuf_puts(b, "]");
}

char *arbplf_model_summary(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", NULL};
    const jv *v[1];
    ctx c;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    if (plf_derive(&c.d, &c.m)) goto done;
    {
        jbuf b; jbuf_init(&b);
        const int n = c.m.n;
        jbuf_puts(&b, "{\"state_count\": "); jbuf_int(&b, n);
        jbuf_puts(&b, ", \"category_count\": "); jbuf_int(&b, c.d.C);
        jbuf_puts(&b, ", \"site_count\": "); jbuf_int(&b, c.m.S);
        jbuf_puts(&b, ", \"root_mode\": "); jbuf_int(&b, c.m.root_mode);
        jbuf_puts(&b, ", \"rate_mix_expect\": "); jbuf_real(&b, c.d.expect);
        jbuf_puts(&b, ", "); put_darray(&b, "cat_rates", c.d.cat_rates, c.d.C);
        jbuf_puts(&b, ", "); put_darray(&b, "cat_prior", c.d.cat_prior, c.d.C);
        jbuf_puts(&b, ", "); put_darray(&b, "equilibrium", c.d.equilibrium, n);
        jbuf_puts(&b, ", "); put_darray(&b, "root_vec", c.d.root_vec, n);
        jbuf_puts(&b, ", "); put_darray(&b, "q_hi", c.d.q_hi, (size_t)n * n);
        jbuf_puts(&b, ", "); put_darray(&b, "q_lo", c.d.q_lo, (size_t)n * n);
        jbuf_puts(&b, ", "); put_darray(&b, "edge_rates_csr", c.d.edge_rates_csr, c.m.E);
        jbuf_puts(&b, ", "); put_iarray(&b, "indptr", c.m.indptr, c.m.N + 1);
        jbuf_puts(&b, ", "); put_iarray(&b, "indices", c.m.indices, c.m.E);
        jbuf_puts(&b, ", "); put_iarray(&b, "preorder", c.m.preorder, c.m.N);
        jbuf_puts(&b, ", "); put_iarray(&b, "order", c.m.order, c.m.E);
        {
            /* what the site data was read as: definition rows, and two sums over the codes in row-major order
             * (plain, and weighted by position + 1; both modulo 2^64, printed as strings) */
            unsigned long long plain = 0, weighted = 0;
            const size_t total = (size_t)c.m.S * c.m.N;
            for (size_t i = 0; i < total; i++) {
                unsigned long long code = c.m.code_bytes == 1 ? ((const unsigned char *)c.m.codes)[i] : (unsigned long long)((const int *)c.m.codes)[i];
                plain += code; weighted += (unsigned long long)(i + 1) * code;
            }
            char t[96];
            jbuf_puts(&b, ", \"definition_count\": "); jbuf_int(&b, c.m.K);
            snprintf(t, sizeof t, ", \"codes_sum\": \"%llu\", \"codes_weighted_sum\": \"%llu\"", plain, weighted);
            jbuf_puts(&b, t);
        }
        jbuf_puts(&b, "}");
        out = jbuf_take(&b);
    }
    rc = 0;
done:
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* arbplf-ll, certified mode                                           */
/* ------------------------------------------------------------------ */

/*
 * The same request as arbplf-ll, answered with an enclosure: {"lower": <table>, "upper": <table>}, both tables in the
 * format of arbplf-ll, lower <= log-likelihood <= upper entry by entry (directed rounding on the device,
 * csrc/certified.cuh).  The reference certifies every output through Arb balls (arbplfll.c:206-224); this is the fp64
 * counterpart for the log-likelihood.  Weighted aggregation with negative weights swaps the bounds of those sites.
 */
char *arbplf_ll_certified(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", NULL};
    const jv *v[2];
    ctx c;
    reduction r_site; reduction_init(&r_site);
    axis ax[1]; memset(ax, 0, sizeof ax);
    double *lo = NULL, *hi = NULL, *slo = NULL, *shi = NULL;
    char *out = NULL, *t_lo = NULL, *t_hi = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site)) goto done;
    lo = calloc(ax[0].aggregated ? 1 : (S > 0 ? S : 1), sizeof(double));
    hi = calloc(ax[0].aggregated ? 1 : (S > 0 ? S : 1), sizeof(double));
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        const double d_rate = 4e-15, d_q = 8.673617379884035e-19;       /* 2^-60 */
        if (ax[0].aggregated) {
            if (plf_set_site_weights(c.e, ax[0].w) || plf_ll_certified(c.e, d_rate, d_q, NULL, NULL, &lo[0], &hi[0])) {
                fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done;
            }
        } else {
            slo = malloc(sizeof(double) * S); shi = malloc(sizeof(double) * S);
            if (plf_set_site_weights(c.e, NULL) || plf_ll_certified(c.e, d_rate, d_q, slo, shi, NULL, NULL)) {
                fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done;
            }
            for (int64_t s = 0; s < S; s++) {
                if (!ax[0].requested[s]) continue;
                if (!isfinite(slo[s]) || !isfinite(shi[s])) { fprintf(stderr, "error: site %lld has zero likelihood\n", (long long)s); goto done; }
                lo[s] = slo[s]; hi[s] = shi[s];
            }
        }
    }
    phase_compute_done(&c);
    t_lo = table_to_json(ax, 1, lo);
    t_hi = table_to_json(ax, 1, hi);
    {
        jbuf b; jbuf_init(&b);
        jbuf_puts(&b, "{\"lower\": "); jbuf_puts(&b, t_lo); jbuf_puts(&b, ", \"upper\": "); jbuf_puts(&b, t_hi); jbuf_puts(&b, "}");
        out = jbuf_take(&b);
    }
    rc = 0;
done:
    free(lo); free(hi); free(slo); free(shi); free(t_lo); free(t_hi);
    axis_clear(&ax[0]); reduction_clear(&r_site);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* arbplf-deriv, certified mode                                        */
/* ------------------------------------------------------------------ */

/* [*lo, *hi] += w [xlo, xhi], rounded outwards on the host (a negative weight swaps the bounds it multiplies) */
static void acc_bounds(double *lo, double *hi, double w, double xlo, double xhi)
{
    const int old = fegetround();
    volatile double t;
    fesetround(FE_DOWNWARD);
    t = w * (w >= 0.0 ? xlo : xhi);
    t = *lo + t;
    *lo = t;
    fesetround(FE_UPWARD);
    t = w * (w >= 0.0 ? xhi : xlo);
    t = *hi + t;
    *hi = t;
    fesetround(old);
}

/* {"lower": <table>, "upper": <table>} */
static char *bounds_to_json(const axis *ax, int ndim, const double *lo, const double *hi)
{
    char *t_lo = table_to_json(ax, ndim, lo), *t_hi = table_to_json(ax, ndim, hi);
    jbuf b; jbuf_init(&b);
    jbuf_puts(&b, "{\"lower\": "); jbuf_puts(&b, t_lo); jbuf_puts(&b, ", \"upper\": "); jbuf_puts(&b, t_hi); jbuf_puts(&b, "}");
    free(t_lo); free(t_hi);
    return jbuf_take(&b);
}

/* the relative input uncertainties of every certified program (plf.h): rate_c t_e, and Q and the priors (2^-60) */
#define CERT_D_RATE 4e-15
#define CERT_D_Q 8.673617379884035e-19

/*
 * The certified counterpart of edge_pass: one engine call (kind < 0: plf_deriv_certified, else plf_edge_expect_certified
 * with direction L) fills [lo, hi] over (site, user edge) at third-axis coordinate `third` (extent third_n); site
 * aggregation is the engine's weighted sum, edge aggregation acc_bounds.
 */
static int edge_pass_certified(ctx *c, int kind, const double *l_hi, const double *l_lo, const axis *ax_site,
                               const axis *ax_edge, const unsigned char *mask, double *lo, double *hi, int third, int third_n)
{
    const plf_model *m = &c->m;
    const int E = m->E;
    const int64_t rows = ax_site->aggregated ? 1 : m->S;
    const size_t edge_ext = ax_edge->aggregated ? 1 : (size_t)E;
    double *blo = malloc(sizeof(double) * (size_t)rows * (E > 0 ? E : 1)), *bhi = malloc(sizeof(double) * (size_t)rows * (E > 0 ? E : 1));
    int rc = -1, r;
    double *slo = ax_site->aggregated ? NULL : blo, *shi = ax_site->aggregated ? NULL : bhi;
    double *tlo = ax_site->aggregated ? blo : NULL, *thi = ax_site->aggregated ? bhi : NULL;
    if (plf_set_site_weights(c->e, ax_site->aggregated ? ax_site->w : NULL)) r = -1;
    else if (kind < 0) r = plf_deriv_certified(c->e, CERT_D_RATE, CERT_D_Q, mask, slo, shi, tlo, thi);
    else r = plf_edge_expect_certified(c->e, CERT_D_RATE, CERT_D_Q, kind, l_hi, l_lo, mask, slo, shi, tlo, thi);
    if (r) { fprintf(stderr, "error: %s\n", plf_last_error(c->e)); goto done; }
    for (int64_t s = 0; s < rows; s++) {
        if (!ax_site->aggregated && !ax_site->requested[s]) continue;
        for (int e = 0; e < E; e++) {
            if (!ax_edge->requested[e]) continue;
            const double xl = blo[(size_t)s * E + m->order[e]], xh = bhi[(size_t)s * E + m->order[e]];
            if (!isfinite(xl) || !isfinite(xh)) {
                if (ax_site->aggregated) fprintf(stderr, "error: a requested site has zero likelihood\n");
                else fprintf(stderr, "error: site %lld has zero likelihood\n", (long long)s);
                goto done;
            }
            if (ax_edge->aggregated) acc_bounds(&lo[(size_t)s * third_n + third], &hi[(size_t)s * third_n + third], ax_edge->w[e], xl, xh);
            else { lo[((size_t)s * edge_ext + e) * third_n + third] = xl; hi[((size_t)s * edge_ext + e) * third_n + third] = xh; }
        }
    }
    rc = 0;
done:
    free(blo); free(bhi);
    return rc;
}

/*
 * The same request as arbplf-deriv, answered with an enclosure: {"lower": <table>, "upper": <table>}, both tables in
 * the format of arbplf-deriv (plf_deriv_certified).  Site aggregation is the engine's weighted sum; edge aggregation
 * combines the per-edge bounds here with directed rounding.  As in arbplf-ll-certified the weights are the doubles of
 * the reduction step (an "avg" weight 1 / count included).
 */
char *arbplf_deriv_certified(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?edge_reduction", NULL};
    const jv *v[3];
    ctx c;
    reduction r_site, r_edge; reduction_init(&r_site); reduction_init(&r_edge);
    axis ax[2]; memset(ax, 0, sizeof ax);
    double *lo = NULL, *hi = NULL;
    unsigned char *mask = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, E, "edge", v[2])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "edge", E, &r_edge)) goto done;
    {
        size_t cells = (ax[0].aggregated ? 1 : (size_t)S) * (ax[1].aggregated ? 1 : (size_t)E);
        lo = calloc(cells ? cells : 1, sizeof(double));
        hi = calloc(cells ? cells : 1, sizeof(double));
    }
    if (S > 0 && E > 0) {
        if (ctx_load(&c)) goto done;
        mask = edge_mask_csr(&c.m, &ax[1]);
        if (edge_pass_certified(&c, -1, NULL, NULL, &ax[0], &ax[1], mask, lo, hi, 0, 1)) goto done;
    }
    phase_compute_done(&c);
    out = bounds_to_json(ax, 2, lo, hi);
    rc = 0;
done:
    free(lo); free(hi); free(mask);
    axis_clear(&ax[0]); axis_clear(&ax[1]);
    reduction_clear(&r_site); reduction_clear(&r_edge);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* arbplf-marginal / arbplf-dwell / arbplf-trans, certified mode       */
/* ------------------------------------------------------------------ */

/*
 * The same request as arbplf-marginal, answered with {"lower", "upper"} tables in its format (plf_marginal_certified).
 * Site aggregation is the engine's weighted sum; node and state aggregation multiply the bounds by each weight in turn
 * and add them up with directed rounding.
 */
char *arbplf_marginal_certified(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?node_reduction", "?state_reduction", NULL};
    const jv *v[4];
    ctx c;
    reduction r_site, r_node, r_state;
    reduction_init(&r_site); reduction_init(&r_node); reduction_init(&r_state);
    axis ax[3]; memset(ax, 0, sizeof ax);
    double *lo = NULL, *hi = NULL, *blo = NULL, *bhi = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int N = c.m.N, n = c.m.n;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_node, N, "node", v[2])) goto done;
    if (reduction_parse(&r_state, n, "state", v[3])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "node", N, &r_node) ||
        axis_init(&ax[2], "state", n, &r_state)) goto done;
    const size_t e1 = ax[1].aggregated ? 1 : (size_t)N, e2 = ax[2].aggregated ? 1 : (size_t)n;
    lo = calloc((ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * e1 * e2, sizeof(double));
    hi = calloc((ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * e1 * e2, sizeof(double));
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        const int64_t rows = ax[0].aggregated ? 1 : S;
        blo = malloc(sizeof(double) * (size_t)rows * N * n);
        bhi = malloc(sizeof(double) * (size_t)rows * N * n);
        int r;
        if (ax[0].aggregated) r = plf_set_site_weights(c.e, ax[0].w) || plf_marginal_certified(c.e, CERT_D_RATE, CERT_D_Q, NULL, NULL, blo, bhi);
        else r = plf_set_site_weights(c.e, NULL) || plf_marginal_certified(c.e, CERT_D_RATE, CERT_D_Q, blo, bhi, NULL, NULL);
        if (r) { fprintf(stderr, "error: %s\n", plf_last_error(c.e)); goto done; }
        for (int64_t s = 0; s < rows; s++) {
            if (!ax[0].aggregated && !ax[0].requested[s]) continue;
            for (int a = 0; a < N; a++) {
                if (!ax[1].requested[a]) continue;
                for (int j = 0; j < n; j++) {
                    if (!ax[2].requested[j]) continue;
                    double xl = blo[((size_t)s * N + a) * n + j], xh = bhi[((size_t)s * N + a) * n + j];
                    if (!isfinite(xl) || !isfinite(xh)) { fprintf(stderr, "error: a requested site has zero likelihood\n"); goto done; }
                    if (ax[1].aggregated) { double tl = 0.0, th = 0.0; acc_bounds(&tl, &th, ax[1].w[a], xl, xh); xl = tl; xh = th; }
                    const size_t off = ((size_t)s * e1 + (ax[1].aggregated ? 0 : a)) * e2 + (ax[2].aggregated ? 0 : j);
                    acc_bounds(&lo[off], &hi[off], ax[2].aggregated ? ax[2].w[j] : 1.0, xl, xh);
                }
            }
        }
    }
    phase_compute_done(&c);
    out = bounds_to_json(ax, 3, lo, hi);
    rc = 0;
done:
    free(lo); free(hi); free(blo); free(bhi);
    for (int i = 0; i < 3; i++) axis_clear(&ax[i]);
    reduction_clear(&r_site); reduction_clear(&r_node); reduction_clear(&r_state);
    return finish(&c, out, rc, retcode);
}

/* The same request as arbplf-dwell, answered with {"lower", "upper"} tables in its format (plf_edge_expect_certified);
 * state aggregation is folded into the direction as arbplf-dwell folds it, signed weights included. */
char *arbplf_dwell_certified(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?edge_reduction", "?state_reduction", NULL};
    const jv *v[4];
    ctx c;
    reduction r_site, r_edge, r_state;
    reduction_init(&r_site); reduction_init(&r_edge); reduction_init(&r_state);
    axis ax[3]; memset(ax, 0, sizeof ax);
    double *lo = NULL, *hi = NULL, *L = NULL;
    unsigned char *mask = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int n = c.m.n, E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, E, "edge", v[2])) goto done;
    if (reduction_parse(&r_state, n, "state", v[3])) goto done;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "edge", E, &r_edge) ||
        axis_init(&ax[2], "state", n, &r_state)) goto done;
    const int state_agg = ax[2].aggregated;
    const int third_n = state_agg ? 1 : n;
    {
        size_t cells = (ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * (ax[1].aggregated ? 1 : (size_t)E) * third_n;
        lo = calloc(cells ? cells : 1, sizeof(double));
        hi = calloc(cells ? cells : 1, sizeof(double));
    }
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        mask = edge_mask_csr(&c.m, &ax[1]);
        L = calloc((size_t)n * n, sizeof(double));
        if (state_agg) {
            for (int s = 0; s < n; s++) L[s * n + s] = ax[2].w[s];     /* arbplfdwell.c:173-178 */
            if (edge_pass_certified(&c, PLF_KIND_DWELL, L, NULL, &ax[0], &ax[1], mask, lo, hi, 0, 1)) goto done;
        } else {
            for (int s = 0; s < n; s++) {
                if (!ax[2].requested[s]) continue;
                memset(L, 0, sizeof(double) * n * n);
                L[s * n + s] = 1.0;                                     /* arbplfdwell.c:133 */
                if (edge_pass_certified(&c, PLF_KIND_DWELL, L, NULL, &ax[0], &ax[1], mask, lo, hi, s, n)) goto done;
            }
        }
    }
    phase_compute_done(&c);
    out = bounds_to_json(ax, state_agg ? 2 : 3, lo, hi);
    rc = 0;
done:
    free(lo); free(hi); free(L); free(mask);
    for (int i = 0; i < 3; i++) axis_clear(&ax[i]);
    reduction_clear(&r_site); reduction_clear(&r_edge); reduction_clear(&r_state);
    return finish(&c, out, rc, retcode);
}

/* The same request as arbplf-trans, answered with {"lower", "upper"} tables in its format (plf_edge_expect_certified);
 * transition aggregation is folded into the direction (sum_k w_k E_{a_k b_k}) .* Q as arbplf-trans folds it, signed
 * weights included.  The weights of a repeated pair are added in double-double, so that the direction stays within the
 * engine's relative delta_q of the exact one. */
char *arbplf_trans_certified(const char *json_in, int *retcode)
{
    static const char *const keys[] = {"model_and_data", "?site_reduction", "?edge_reduction", "?trans_reduction", NULL};
    const jv *v[4];
    ctx c;
    reduction r_site, r_edge, r_trans;
    reduction_init(&r_site); reduction_init(&r_edge); reduction_init(&r_trans);
    axis ax[3]; memset(ax, 0, sizeof ax);
    double *lo = NULL, *hi = NULL, *Lh = NULL, *Ll = NULL;
    dd_t *W = NULL;
    unsigned char *mask = NULL;
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int n = c.m.n, E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (reduction_parse(&r_edge, E, "edge", v[2])) goto done;
    if (reduction_parse_pairs(&r_trans, n, "trans", v[3])) goto done;
    const int T = r_trans.selection_len;
    if (axis_init(&ax[0], "site", (int)S, &r_site) || axis_init(&ax[1], "edge", E, &r_edge) ||
        axis_init(&ax[2], "trans", T, &r_trans)) goto done;
    ax[2].ncomp = 2;
    ax[2].comp_name[0] = "first_state"; ax[2].comp_name[1] = "second_state";
    ax[2].comp_idx[0] = r_trans.first_idx; ax[2].comp_idx[1] = r_trans.second_idx;
    const int trans_agg = ax[2].aggregated;
    const int third_n = trans_agg ? 1 : (T > 0 ? T : 1);
    {
        size_t cells = (ax[0].aggregated ? 1 : (size_t)(S > 0 ? S : 1)) * (ax[1].aggregated ? 1 : (size_t)E) * third_n;
        lo = calloc(cells ? cells : 1, sizeof(double));
        hi = calloc(cells ? cells : 1, sizeof(double));
    }
    if (S > 0) {
        if (ctx_load(&c)) goto done;
        mask = edge_mask_csr(&c.m, &ax[1]);
        Lh = calloc((size_t)n * n, sizeof(double));
        Ll = calloc((size_t)n * n, sizeof(double));
        if (trans_agg) {
            /* L = (sum_k w_k E_{a_k b_k}) .* Q / divisor  (arbplftrans.c:179-193) */
            W = calloc((size_t)n * n, sizeof(dd_t));
            for (int k = 0; k < T; k++) {
                dd_t *x = &W[r_trans.first_idx[k] * n + r_trans.second_idx[k]];
                *x = dd_add(*x, dd_make(ax[2].w[k], 0.0));
            }
            for (int i = 0; i < n * n; i++) {
                dd_t q = dd_mul(dd_make(c.d.q_hi[i], c.d.q_lo[i]), W[i]);
                Lh[i] = q.hi; Ll[i] = q.lo;
            }
            if (edge_pass_certified(&c, PLF_KIND_TRANS, Lh, Ll, &ax[0], &ax[1], mask, lo, hi, 0, 1)) goto done;
        } else {
            for (int k = 0; k < T; k++) {
                if (!ax[2].requested[k]) continue;
                memset(Lh, 0, sizeof(double) * n * n); memset(Ll, 0, sizeof(double) * n * n);
                int idx = r_trans.first_idx[k] * n + r_trans.second_idx[k];
                Lh[idx] = c.d.q_hi[idx]; Ll[idx] = c.d.q_lo[idx];      /* arbplftrans.c:133-134 */
                if (edge_pass_certified(&c, PLF_KIND_TRANS, Lh, Ll, &ax[0], &ax[1], mask, lo, hi, k, third_n)) goto done;
            }
        }
    }
    phase_compute_done(&c);
    out = bounds_to_json(ax, trans_agg ? 2 : 3, lo, hi);
    rc = 0;
done:
    free(lo); free(hi); free(Lh); free(Ll); free(W); free(mask);
    for (int i = 0; i < 3; i++) axis_clear(&ax[i]);
    reduction_clear(&r_site); reduction_clear(&r_edge); reduction_clear(&r_trans);
    return finish(&c, out, rc, retcode);
}

/* ------------------------------------------------------------------ */
/* second order programs (arbplfhess.c)                                */
/* ------------------------------------------------------------------ */

/* A x = b by Gaussian elimination with partial pivoting in long double, nrhs right-hand sides (columns of B, row major
 * [n][nrhs]); returns -1 when A is singular to working precision. */
static int solve_ld(int n, const double *A, const double *B, int nrhs, double *X)
{
    long double *M = malloc(sizeof(long double) * (size_t)n * (n + nrhs) + 16);
    const int W = n + nrhs;
    int rc = 0;
    for (int i = 0; i < n; i++) {
        for (int j = 0; j < n; j++) M[(size_t)i * W + j] = A[(size_t)i * n + j];
        for (int j = 0; j < nrhs; j++) M[(size_t)i * W + n + j] = B[(size_t)i * nrhs + j];
    }
    for (int k = 0; k < n && !rc; k++) {
        int piv = k;
        long double best = fabsl(M[(size_t)k * W + k]);
        for (int i = k + 1; i < n; i++) if (fabsl(M[(size_t)i * W + k]) > best) { best = fabsl(M[(size_t)i * W + k]); piv = i; }
        if (!(best > 0.0L)) { rc = -1; break; }
        if (piv != k) for (int j = 0; j < W; j++) { long double t = M[(size_t)k * W + j]; M[(size_t)k * W + j] = M[(size_t)piv * W + j]; M[(size_t)piv * W + j] = t; }
        for (int i = k + 1; i < n; i++) {
            const long double f = M[(size_t)i * W + k] / M[(size_t)k * W + k];
            if (f == 0.0L) continue;
            for (int j = k; j < W; j++) M[(size_t)i * W + j] -= f * M[(size_t)k * W + j];
        }
    }
    if (!rc) {
        for (int r = 0; r < nrhs; r++)
            for (int i = n - 1; i >= 0; i--) {
                long double t = M[(size_t)i * W + n + r];
                for (int j = i + 1; j < n; j++) t -= M[(size_t)i * W + j] * M[(size_t)j * W + n + r];
                M[(size_t)i * W + n + r] = t / M[(size_t)i * W + i];
            }
        for (int i = 0; i < n; i++) for (int r = 0; r < nrhs; r++) X[(size_t)i * nrhs + r] = (double)M[(size_t)i * W + n + r];
    }
    free(M);
    return rc;
}

enum { SO_HESS, SO_INV_HESS, SO_DELTA, SO_UPDATE, SO_REFINE };

/*
 * hess_query / inv_hess_query / newton_delta_query / newton_point_query (arbplfhess.c:1208-1452): the site reduction is
 * required and must aggregate (arbplfhess.c:1162-1207); outputs in the user's edge order.  newton-refine here is a
 * plain (uncertified) Newton iteration from the given rates to a stationary point; the reference's trust-region search
 * followed by interval-Newton certification (arbplfhess.c:1454-1733) is not reproduced.
 */
static char *second_order(const char *json_in, int *retcode, int which)
{
    static const char *const keys[] = {"model_and_data", "site_reduction", NULL};
    const jv *v[2];
    ctx c;
    reduction r_site; reduction_init(&r_site);
    axis ax_site; memset(&ax_site, 0, sizeof ax_site);
    double *H = NULL, *g = NULL, *X = NULL, *B = NULL, *rates = NULL;
    jbuf jb; jbuf_init(&jb);
    char *out = NULL;
    int rc = -1;
    if (ctx_parse(&c, json_in, keys, v)) goto done;
    const int E = c.m.E;
    const int64_t S = c.m.S;
    if (reduction_parse(&r_site, (int)S, "site", v[1])) goto done;
    if (axis_init(&ax_site, "site", (int)S, &r_site)) goto done;
    if (!ax_site.aggregated) { fprintf(stderr, "error: aggregation over sites is required\n"); goto done; }
    H = calloc((size_t)E * E + 1, sizeof(double));
    g = calloc(E + 1, sizeof(double));
    X = calloc((size_t)E * E + 1, sizeof(double));
    B = calloc((size_t)E * E + 1, sizeof(double));
    rates = calloc(E + 1, sizeof(double));
    if (S > 0 && E > 0) {
        if (ctx_load(&c)) goto done;
        if (plf_set_site_weights(c.e, ax_site.w)) goto engine_error;
        for (int i = 0; i < E; i++) rates[i] = c.d.edge_rates_csr[i];
        const int iters = which == SO_REFINE ? 100 : 1;
        for (int it = 0; it < iters; it++) {
            if (it > 0 && plf_set_edge_rates(c.e, rates)) goto engine_error;
            if (plf_hess(c.e, NULL, g, H)) goto engine_error;
            if (which == SO_HESS) break;
            if (which == SO_INV_HESS) {
                for (int i = 0; i < E; i++) B[(size_t)i * E + i] = 1.0;
                if (solve_ld(E, H, B, E, X)) { fprintf(stderr, "error: the hessian is singular\n"); goto done; }
                break;
            }
            if (solve_ld(E, H, g, 1, X)) { fprintf(stderr, "error: the hessian is singular\n"); goto done; }
            if (which != SO_REFINE) break;
            /* x <- x - inv(H) g, kept positive; stop when the step no longer changes the rates */
            double big = 0.0;
            for (int i = 0; i < E; i++) {
                double step = -X[i], lim = 0.5 * rates[i];
                if (step < -lim) step = -lim;
                rates[i] += step;
                if (fabs(step) > big * fabs(rates[i])) big = fabs(step) / (fabs(rates[i]) > 0 ? fabs(rates[i]) : 1.0);
            }
            if (big < 1e-15) break;
        }
    }
    phase_compute_done(&c);
    if (which == SO_HESS || which == SO_INV_HESS) {
        const double *M = which == SO_HESS ? H : X;
        jbuf_puts(&jb, "{\"columns\": [\"first_edge\", \"second_edge\", \"value\"], \"data\": [");
        for (int a = 0; a < E; a++)
            for (int b = 0; b < E; b++) {
                const int i = c.m.order[a], j = c.m.order[b];
                const double x = (j < i) ? M[(size_t)i * E + j] : M[(size_t)j * E + i];
                if (!isfinite(x)) { fprintf(stderr, "error: a requested site has zero likelihood\n"); goto done; }
                if (a || b) jbuf_puts(&jb, ", ");
                jbuf_puts(&jb, "["); jbuf_int(&jb, a); jbuf_puts(&jb, ", "); jbuf_int(&jb, b); jbuf_puts(&jb, ", ");
                jbuf_real(&jb, x); jbuf_puts(&jb, "]");
            }
        jbuf_puts(&jb, "]}");
    } else {
        jbuf_puts(&jb, "{\"columns\": [\"edge\", \"value\"], \"data\": [");
        for (int a = 0; a < E; a++) {
            const int i = c.m.order[a];
            double x = -X[i];                                      /* newton delta = -inv(hess) grad (arbplfhess.c:203-234) */
            if (which == SO_UPDATE) x += c.d.edge_rates_csr[i];    /* arbplfhess.c:236-245 */
            if (which == SO_REFINE) x = rates[i];
            if (!isfinite(x)) { fprintf(stderr, "error: a requested site has zero likelihood\n"); goto done; }
            if (a) jbuf_puts(&jb, ", ");
            jbuf_puts(&jb, "["); jbuf_int(&jb, a); jbuf_puts(&jb, ", "); jbuf_real(&jb, x); jbuf_puts(&jb, "]");
        }
        jbuf_puts(&jb, "]}");
    }
    out = jbuf_take(&jb);
    rc = 0;
    goto done;
engine_error:
    fprintf(stderr, "error: %s\n", plf_last_error(c.e));
done:
    if (rc) free(jbuf_take(&jb));
    free(H); free(g); free(X); free(B); free(rates);
    axis_clear(&ax_site);
    reduction_clear(&r_site);
    return finish(&c, out, rc, retcode);
}

char *arbplf_hess(const char *j, int *rc) { return second_order(j, rc, SO_HESS); }
char *arbplf_inv_hess(const char *j, int *rc) { return second_order(j, rc, SO_INV_HESS); }
char *arbplf_newton_delta(const char *j, int *rc) { return second_order(j, rc, SO_DELTA); }
char *arbplf_newton_update(const char *j, int *rc) { return second_order(j, rc, SO_UPDATE); }
char *arbplf_newton_refine(const char *j, int *rc) { return second_order(j, rc, SO_REFINE); }

/* runjson.c:88-147 */
/* An arbplf-* process answers one document: creating the CUDA context (a few tenths of a second) overlaps reading and
 * parsing the document instead of following it.  Failure here is silent -- the call itself tries again and reports. */
static void *warm_engine(void *unused)
{
    (void)unused;
    const char *s = getenv("ARBPLF_DEVICE");
    plf_warmup(g_device >= 0 ? g_device : (s ? atoi(s) : 0));
    return NULL;
}

int arbplf_run_stdio(char *(*f)(const char *, int *))
{
    pthread_t warm;
    const int warming = !getenv("ARBPLF_NO_WARMUP") && pthread_create(&warm, NULL, warm_engine, NULL) == 0;
    size_t cap = 1 << 16, len = 0;
    char *s = malloc(cap);
    if (!s) { if (warming) pthread_join(warm, NULL); return -1; }
    for (;;) {
        size_t got = fread(s + len, 1, cap - len - 1, stdin);
        len += got;
        if (got == 0) break;
        if (len + 1 >= cap) {
            cap *= 2;
            char *t = realloc(s, cap);
            if (!t) { fprintf(stderr, "failed to read string from stdin\n"); free(s); if (warming) pthread_join(warm, NULL); return -1; }
            s = t;
        }
    }
    s[len] = 0;
    int rc = 0;
    char *out = f(s, &rc);
    free(s);
    if (out) { puts(out); free(out); }
    if (warming) pthread_join(warm, NULL);
    return rc;
}
