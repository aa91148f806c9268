/*
 * Generic (any state count, any data) per-site kernels.
 *
 * These restate evaluate_site_lhood (evaluate_site_lhood.c:6-63),
 * evaluate_site_forward (evaluate_site_forward.c:31-105),
 * evaluate_site_marginal_unnormalized (evaluate_site_marginal.c:6-21) and
 * evaluate_site_frechet (evaluate_site_frechet.c:4-42) with one GPU thread per
 * site (x rate category for the inside pass).  All per-node vectors live in HBM
 * with the site index fastest, so every load and store of a warp is one
 * contiguous 256-byte run.  Per-site power-of-two rescaling (exponents counted
 * in units of 2^256) replaces the reference's growing precision.
 *
 * Layouts (Sc = sites in the current chunk, s = site within the chunk):
 *   Lg [C][N][n][Sc]  inside ("lhood node") vectors, mantissas
 *   Kg [C][N][Sc]     their exponents (int32, <= 0), true = mant * 2^(256 K)
 *   Cg [C][N][Sc]     1 if the vector is an exact constant column
 *                     (arb_mat_extras.c:35-51), tracked symbolically
 *   Eg [C][E][n][Sc]  edge vectors P_e L_b (mantissas; exponent = K of the child)
 *   Fg [C][N][n][Sc]  outside ("forward node") vectors, FK [C][N][Sc] exponents
 */
#pragma once
#include <stdint.h>

#include "plf_consts.h"
#define PLF_TS 128   /* threads (sites) per CTA in the generic kernels */

struct TreeDev {
    int N, E, root;
    const int *indptr;     /* [N+1] */
    const int *indices;    /* [E]   */
    const int *preorder;   /* [N]   */
    const unsigned char *node_has_data;  /* [N] */
};

struct GenericArgs {
    TreeDev t;
    int n, C, K;
    int64_t S;            /* total sites */
    int64_t s0;           /* first site of the chunk */
    int Sc;               /* sites in the chunk */
    const void *codes;    /* [N][S] node-major, uint8 or int32 */
    int code_bytes;
    const double *defs;   /* [K][n] */
    const unsigned char *def_const;   /* [K] row is constant */
    const double *P;      /* [C][E][n][n] */
    const double *Fm;     /* [C][E][n][n] matrices of the edge bilinear form (or NULL) */
    int f_zero_rowsum;    /* Fm has zero row sums: constant columns map to exact 0 (util.c:338-344) */
    const double *edge_coef; /* [C][E] extra factor per (category, edge) on the edge form, or NULL */
    const unsigned char *edge_mask;  /* [E] or NULL */
    const double *cat_prior; /* [C] */
    int root_mode;
    const double *root_vec;  /* [n] */
    double *Lg; int *Kg; unsigned char *Cg; double *Eg; double *Fg; int *FK;
    double *cat_lh;       /* [C][Sc] mantissa of root-prior expectation */
    int *cat_k;           /* [C][Sc] */
    double *site_m;       /* [Sc] mantissa of site likelihood */
    int *site_k;          /* [Sc] */
    double *site_ll;      /* [S]  (global site index) */
    double *edge_out;     /* [E][Sc] per-site edge forms (already divided by site lhood) or NULL */
    double *marg_out;     /* [N][n][Sc] or NULL */
    int want_edge, want_marg;
    /* tip tables for the tile kernel: TP[c][tip edge][k][i] = (P_e def_k)_i, tip_of_edge[csr idx] = tip edge or -1 */
    const double *TP;
    const double *TF;             /* the same with the edge-form matrices (F_e def_k), or NULL */
    const int *tip_of_edge;
    int Et;
    /* csr indices of the edges whose child goes through the GEMM, in the order tile_inside_kernel meets them */
    const int *int_seq;
    int n_int_seq;
    /* tile_inside_kernel stages the tile's tip codes in shared memory (1-byte codes, Et * 64 bytes) */
    int tip_stage;
    const int *tip_edge_csr;      /* [Et] csr index of each tip edge */
    /* plf_edge_expect_all: the outside pass writes the scaled outside edge vectors w_s prior_c fe / L_s (exponents
     * applied, the child's included) to fe_out [C][E][n][Sc]; generic_gmat_kernel multiplies them into the L_b */
    double *fe_out;
    const double *site_w;         /* [S] or NULL, read with fe_out */
};

__device__ __forceinline__ int plf_code_at(const void *codes, int code_bytes, int64_t S, int node, int64_t site)
{
    if (code_bytes == 1) return ((const unsigned char *)codes)[(size_t)node * S + site];
    return ((const int *)codes)[(size_t)node * S + site];
}


/* inside pass: thread = (site, category) ; blockIdx.y = category */
__global__ void __launch_bounds__(PLF_TS) generic_inside_kernel(GenericArgs a)
{
    extern __shared__ double gsm[];
    const int tid = threadIdx.x;
    const int s = blockIdx.x * PLF_TS + tid;
    const int c = blockIdx.y;
    if (s >= a.Sc) return;
    const int n = a.n, Sc = a.Sc;
    const int64_t gs = a.s0 + s;
    double *acc = gsm + tid;                  /* acc[i*PLF_TS] */
    double *v = gsm + (size_t)n * PLF_TS + tid;
    const size_t cN = (size_t)c * a.t.N;
    const size_t cE = (size_t)c * a.t.E;

    for (int u = a.t.N - 1; u >= 0; u--) {
        const int nd = a.t.preorder[u];
        const int start = a.t.indptr[nd], stop = a.t.indptr[nd + 1];
        int accK = 0;
        int cst = 1;
        if (a.t.node_has_data[nd]) {
            int code = plf_code_at(a.codes, a.code_bytes, a.S, nd, gs);
            for (int i = 0; i < n; i++) acc[i * PLF_TS] = a.defs[(size_t)code * n + i];
            cst = a.def_const[code];
        } else {
            for (int i = 0; i < n; i++) acc[i * PLF_TS] = 1.0;
        }
        for (int idx = start; idx < stop; idx++) {
            const int b = a.t.indices[idx];
            const double *Lb = a.Lg + ((cN + b) * n) * Sc + s;
            for (int k = 0; k < n; k++) v[k * PLF_TS] = Lb[(size_t)k * Sc];
            const int kb = a.Kg[(cN + b) * Sc + s];
            const int bc = a.Cg[(cN + b) * Sc + s];
            const double *Pm = a.P + (cE + idx) * n * n;
            double *Eo = a.Eg + ((cE + idx) * n) * Sc + s;
            double mx = 0.0;
            for (int i = 0; i < n; i++) {
                double em;
                if (bc) {
                    em = v[0];
                } else {
                    em = 0.0;
                    for (int k = 0; k < n; k++) em = fma(Pm[i * n + k], v[k * PLF_TS], em);
                }
                Eo[(size_t)i * Sc] = em;
                double x = acc[i * PLF_TS] * em;
                acc[i * PLF_TS] = x;
                mx = fmax(mx, x);
            }
            accK += kb;
            cst &= bc;
            while (mx > 0.0 && mx < PLF_TWO_M256) {
                for (int i = 0; i < n; i++) acc[i * PLF_TS] *= PLF_TWO_P256;
                mx *= PLF_TWO_P256;
                accK -= 1;
            }
        }
        double *La = a.Lg + ((cN + nd) * n) * Sc + s;
        for (int i = 0; i < n; i++) La[(size_t)i * Sc] = acc[i * PLF_TS];
        a.Kg[(cN + nd) * Sc + s] = accK;
        a.Cg[(cN + nd) * Sc + s] = (unsigned char)cst;
        if (nd == a.t.root) {
            /* root_prior_expectation, model.c:282-350 */
            double lh = 0.0;
            if (a.root_mode == PLF_ROOT_NONE) {
                for (int i = 0; i < n; i++) lh += acc[i * PLF_TS];
            } else if (a.root_mode == PLF_ROOT_UNIFORM) {
                if (cst) lh = acc[0];
                else { for (int i = 0; i < n; i++) lh += acc[i * PLF_TS]; lh /= (double)n; }
            } else if (a.root_mode == PLF_ROOT_EQUILIBRIUM && cst) {
                lh = acc[0];
            } else {
                for (int i = 0; i < n; i++) lh = fma(a.root_vec[i], acc[i * PLF_TS], lh);
            }
            a.cat_lh[(size_t)c * Sc + s] = lh;
            a.cat_k[(size_t)c * Sc + s] = accK;
        }
    }
}

/* combine categories: site likelihood and log-likelihood (arbplfll.c:149-169) */
__global__ void generic_site_kernel(GenericArgs a)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.Sc) return;
    const int Sc = a.Sc;
    int k0 = INT_MIN;
    for (int c = 0; c < a.C; c++) {
        double v = a.cat_prior[c] * a.cat_lh[(size_t)c * Sc + s];
        if (v > 0.0) k0 = max(k0, a.cat_k[(size_t)c * Sc + s]);
    }
    double m = 0.0;
    if (k0 != INT_MIN) {
        for (int c = 0; c < a.C; c++) {
            double v = a.cat_prior[c] * a.cat_lh[(size_t)c * Sc + s];
            if (v > 0.0) m += scalbn(v, PLF_SCALE_BITS * (a.cat_k[(size_t)c * Sc + s] - k0));
        }
    } else {
        k0 = 0;
    }
    a.site_m[s] = m;
    a.site_k[s] = k0;
    /* log(m * 2^(256 k0)) ; 256*ln2 split in two parts */
    const double c_hi = 177.445678223346, c_lo = 5.936759843446527e-15;  /* 256*ln(2) = hi + lo */
    double ll = log(m);
    ll = fma((double)k0, c_hi, ll);
    ll = fma((double)k0, c_lo, ll);
    a.site_ll[a.s0 + s] = ll;
}

/*
 * outside pass: thread = site, categories looped inside (their contributions to
 * the same output cell are summed without atomics).
 */
__global__ void __launch_bounds__(PLF_TS) generic_outside_kernel(GenericArgs a)
{
    extern __shared__ double gsm[];
    const int tid = threadIdx.x;
    const int s = blockIdx.x * PLF_TS + tid;
    if (s >= a.Sc) return;
    const int n = a.n, Sc = a.Sc;
    const int64_t gs = a.s0 + s;
    double *tmp = gsm + tid;
    double *fe = gsm + (size_t)n * PLF_TS + tid;
    double *y = gsm + (size_t)2 * n * PLF_TS + tid;
    const double site_m = a.site_m[s];
    const int site_k = a.site_k[s];

    for (int c = 0; c < a.C; c++) {
        const size_t cN = (size_t)c * a.t.N;
        const size_t cE = (size_t)c * a.t.E;
        const double prior = a.cat_prior[c];
        /* arbplfmarginal.c:184-191: skip categories whose posterior is exactly zero */
        if (!(prior * a.cat_lh[(size_t)c * Sc + s] > 0.0)) continue;
        const double coef = prior / site_m;
        /* forward vector at the root: root_prior_mul_col_vec, model.c:225-280 */
        {
            double *Fr = a.Fg + ((cN + a.t.root) * n) * Sc + s;
            for (int i = 0; i < n; i++) {
                double r = 1.0;
                if (a.root_mode == PLF_ROOT_UNIFORM) r = 1.0 / (double)n;
                else if (a.root_mode == PLF_ROOT_EQUILIBRIUM || a.root_mode == PLF_ROOT_CUSTOM) r = a.root_vec[i];
                Fr[(size_t)i * Sc] = r;
            }
            a.FK[(cN + a.t.root) * Sc + s] = 0;
        }
        for (int u = 0; u < a.t.N; u++) {
            const int nd = a.t.preorder[u];
            const int start = a.t.indptr[nd], stop = a.t.indptr[nd + 1];
            const double *Fa = a.Fg + ((cN + nd) * n) * Sc + s;
            const int ka = a.FK[(cN + nd) * Sc + s];
            if (a.want_marg) {
                /* marg_a += prior * fn_a .* L_a / site_L */
                const double *La = a.Lg + ((cN + nd) * n) * Sc + s;
                const int kl = a.Kg[(cN + nd) * Sc + s];
                const int sh = PLF_SCALE_BITS * (ka + kl - site_k);
                double *Mo = a.marg_out + ((size_t)nd * n) * Sc + s;
                for (int i = 0; i < n; i++)
                    Mo[(size_t)i * Sc] += scalbn(coef * Fa[(size_t)i * Sc] * La[(size_t)i * Sc], sh);
            }
            if (start == stop) continue;
            if (a.t.node_has_data[nd]) {
                int code = plf_code_at(a.codes, a.code_bytes, a.S, nd, gs);
                for (int i = 0; i < n; i++) tmp[i * PLF_TS] = Fa[(size_t)i * Sc] * a.defs[(size_t)code * n + i];
            } else {
                for (int i = 0; i < n; i++) tmp[i * PLF_TS] = Fa[(size_t)i * Sc];
            }
            for (int idx = start; idx < stop; idx++) {
                const int b = a.t.indices[idx];
                int kfe = ka;
                for (int i = 0; i < n; i++) fe[i * PLF_TS] = tmp[i * PLF_TS];
                for (int idx2 = start; idx2 < stop; idx2++) {
                    if (idx2 == idx) continue;
                    const double *Es = a.Eg + ((cE + idx2) * n) * Sc + s;
                    double mx = 0.0;
                    for (int i = 0; i < n; i++) {
                        double x = fe[i * PLF_TS] * Es[(size_t)i * Sc];
                        fe[i * PLF_TS] = x;
                        mx = fmax(mx, x);
                    }
                    kfe += a.Kg[(cN + a.t.indices[idx2]) * Sc + s];
                    while (mx > 0.0 && mx < PLF_TWO_M256) {
                        for (int i = 0; i < n; i++) fe[i * PLF_TS] *= PLF_TWO_P256;
                        mx *= PLF_TWO_P256; kfe -= 1;
                    }
                    while (mx > PLF_TWO_P256) {
                        for (int i = 0; i < n; i++) fe[i * PLF_TS] *= PLF_TWO_M256;
                        mx *= PLF_TWO_M256; kfe += 1;
                    }
                }
                const double *Lb = a.Lg + ((cN + b) * n) * Sc + s;
                const int kb = a.Kg[(cN + b) * Sc + s];
                const int bc = a.Cg[(cN + b) * Sc + s];
                if (a.fe_out) {
                    const double wv = a.site_w ? a.site_w[gs] : 1.0;
                    double *Fo = a.fe_out + ((cE + idx) * n) * Sc + s;
                    const int sh = PLF_SCALE_BITS * (kfe + kb - site_k);
                    for (int i = 0; i < n; i++) Fo[(size_t)i * Sc] = (wv == 0.0) ? 0.0 : scalbn(fe[i * PLF_TS] * coef * wv, sh);
                }
                if (a.want_edge && (!a.edge_mask || a.edge_mask[idx])) {
                    /* evaluate_site_frechet.c:18-39: fe^T F L_b */
                    double x = 0.0;
                    if (!(a.f_zero_rowsum && bc)) {
                        const double *Fm = a.Fm + (cE + idx) * n * n;
                        for (int k = 0; k < n; k++) y[k * PLF_TS] = Lb[(size_t)k * Sc];
                        for (int i = 0; i < n; i++) {
                            double acc = 0.0;
                            for (int k = 0; k < n; k++) acc = fma(Fm[i * n + k], y[k * PLF_TS], acc);
                            x = fma(fe[i * PLF_TS], acc, x);
                        }
                    }
                    double ec = a.edge_coef ? a.edge_coef[cE + idx] : 1.0;
                    a.edge_out[(size_t)idx * Sc + s] += scalbn(x * coef * ec, PLF_SCALE_BITS * (kfe + kb - site_k));
                }
                /* forward node vector of b: P^T fe  (util.c:464-498) */
                {
                    const double *Pm = a.P + (cE + idx) * n * n;
                    double *Fb = a.Fg + ((cN + b) * n) * Sc + s;
                    double mx = 0.0;
                    for (int j = 0; j < n; j++) {
                        double acc = 0.0;
                        for (int i = 0; i < n; i++) acc = fma(Pm[i * n + j], fe[i * PLF_TS], acc);
                        y[j * PLF_TS] = acc;
                        mx = fmax(mx, acc);
                    }
                    int kfb = kfe;
                    double sc = 1.0;
                    while (mx * sc > PLF_TWO_P256) { sc *= PLF_TWO_M256; kfb += 1; }
                    while (mx > 0.0 && mx * sc < PLF_TWO_M256) { sc *= PLF_TWO_P256; kfb -= 1; }
                    for (int j = 0; j < n; j++) Fb[(size_t)j * Sc] = y[j * PLF_TS] * sc;
                    a.FK[(cN + b) * Sc + s] = kfb;
                }
            }
        }
    }
}

/*
 * plf_edge_expect_all: G[c][e][i][j] += sum_s fe_out[c][e][i][s] L_b[c][b][j][s] over the sites of a chunk (b = child of
 * edge e).  One CTA per (edge, category); the entries in blocks of 4 x 4, every thread a fixed slice of the sites, the
 * slices added in a fixed tree order, the chunks in order: the same bits on every run.
 */
__global__ void __launch_bounds__(256) generic_gmat_kernel(GenericArgs a, double *G)
{
    __shared__ double red[16][256];
    const int e = blockIdx.x, c = blockIdx.y, tid = threadIdx.x, n = a.n, Sc = a.Sc;
    const int b = a.t.indices[e];
    const double *FE = a.fe_out + (((size_t)c * a.t.E + e) * n) * Sc;
    const double *Lb = a.Lg + (((size_t)c * a.t.N + b) * n) * Sc;
    double *Ge = G + ((size_t)c * a.t.E + e) * n * n;
    for (int i0 = 0; i0 < n; i0 += 4) {
        for (int j0 = 0; j0 < n; j0 += 4) {
            double acc[16];
#pragma unroll
            for (int k = 0; k < 16; k++) acc[k] = 0.0;
            for (int s = tid; s < Sc; s += 256) {
                double f[4], l[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    f[k] = (i0 + k < n) ? FE[(size_t)(i0 + k) * Sc + s] : 0.0;
                    l[k] = (j0 + k < n) ? Lb[(size_t)(j0 + k) * Sc + s] : 0.0;
                }
#pragma unroll
                for (int ii = 0; ii < 4; ii++)
#pragma unroll
                    for (int jj = 0; jj < 4; jj++) acc[4 * ii + jj] = fma(f[ii], l[jj], acc[4 * ii + jj]);
            }
#pragma unroll
            for (int k = 0; k < 16; k++) red[k][tid] = acc[k];
            __syncthreads();
            for (int o = 128; o > 0; o >>= 1) {
                if (tid < o)
#pragma unroll
                    for (int k = 0; k < 16; k++) red[k][tid] += red[k][tid + o];
                __syncthreads();
            }
            if (tid < 16) {
                const int i = i0 + (tid >> 2), j = j0 + (tid & 3);
                if (i < n && j < n) Ge[(size_t)i * n + j] += red[tid][0];
            }
            __syncthreads();
        }
    }
}

/* leaves: write their base vectors as "inside" vectors once per chunk (so that
 * parents read every child the same way). blockIdx.y = category.  write_vectors = 0 writes the
 * exponents and constant flags only (the tile kernels take the vectors of tips from tip tables). */
__global__ void generic_leaf_kernel(GenericArgs a, int write_vectors)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (s >= a.Sc) return;
    const int n = a.n, Sc = a.Sc;
    const size_t cN = (size_t)c * a.t.N;
    for (int nd = 0; nd < a.t.N; nd++) {
        if (a.t.indptr[nd] != a.t.indptr[nd + 1]) continue;
        double *La = a.Lg + ((cN + nd) * n) * Sc + s;
        int cst = 1;
        if (a.t.node_has_data[nd]) {
            int code = plf_code_at(a.codes, a.code_bytes, a.S, nd, a.s0 + s);
            if (write_vectors) for (int i = 0; i < n; i++) La[(size_t)i * Sc] = a.defs[(size_t)code * n + i];
            cst = a.def_const[code];
        } else if (write_vectors) {
            for (int i = 0; i < n; i++) La[(size_t)i * Sc] = 1.0;
        }
        a.Kg[(cN + nd) * Sc + s] = 0;
        a.Cg[(cN + nd) * Sc + s] = (unsigned char)cst;
    }
}

/* ------------------------------------------------------------------ */
/* second order: Hessian of the log likelihood w.r.t. the edge rates   */
/* ------------------------------------------------------------------ */

/*
 * The reference (arbplfhess.c:502-829) obtains d^2 L / dt_i dt_j by substituting Q P for P on both edges and
 * re-walking the two root paths for every pair of edges, O(E^2 depth) prune updates per (site, category).  The
 * site likelihood is multilinear in the per-edge matrices, so the same numbers come out of ONE tangent sweep per
 * edge j on top of the stored inside / outside vectors (O(E^2) updates per (site, category) in total):
 *
 *   - v = rate Q em_j is the tangent of edge j's vector; carried up j's root path, v <- P_p (base_a . v . prod
 *     sibling vectors), it gives the pairs (ancestor edge p, j) as fe_p . (rate Q v);
 *   - at every node a of that path the tangent also enters the OTHER children's subtrees through their outside
 *     vectors, dfe_e' = fn_a . base_a . v . prod(other sibling vectors), and travels down like the outside pass
 *     (dfn_b = P^T dfe); every edge i met on the way gives the pair (i, j) as dfe_i . (rate Q em_i);
 *   - the diagonal is fe_j . (rate^2 Q Q em_j).
 * Each unordered pair is accumulated once, into H[max(i,j)][min(i,j)] (csr indices): a disjoint pair is met from
 * both sides, only the side where i ranks above j (BFS position of the child node) counts, and subtrees that hold no
 * rank above j's are not entered.
 *
 * The kernel adds sum_s w_s [ sum_c prior_c rate_c^2 H_c ] / L_s into Hpart[cta][E][E]; the g g^T / L^2 part of
 * _lhood_hess_to_ll_hess (arbplfhess.c:455-495) is a weighted Gram matrix of the per-site derivatives
 * (gram_rows_kernel).  thread = site, categories looped inside; all control flow is uniform over the CTA.
 */
struct HessTree {
    const int *parent_node;   /* [E]  node above csr edge idx (idx_to_a, util.c:369-389) */
    const int *parent_edge;   /* [N]  csr edge above a node, -1 at the root (b_to_idx) */
    const int *dfs_nodes;     /* [N]  nodes in depth-first pre-order */
    const int *dfs_pos;       /* [N]  position of a node in dfs_nodes */
    const int *sub_end;       /* [N]  end (exclusive) of the node's subtree in dfs_nodes */
    const int *erank;         /* [E]  rank of an edge = position of its child node in the BFS order: ancestors rank lower */
    const int *sub_max;       /* [E]  largest rank in the subtree hanging from edge idx (idx itself included) */
};

__device__ __forceinline__ double hess_warp_sum(double x)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

/* |max| rescale of a signed per-thread vector v[i * PLF_TS] into [2^-256, 2^256] */
__device__ __forceinline__ void hess_rescale(double *v, int n, int &k)
{
    double mx = 0.0;
    for (int i = 0; i < n; i++) mx = fmax(mx, fabs(v[i * PLF_TS]));
    if (!(mx > 0.0) || !isfinite(mx)) return;
    double sc = 1.0;
    while (mx * sc > PLF_TWO_P256) { sc *= PLF_TWO_M256; k += 1; }
    while (mx * sc < PLF_TWO_M256) { sc *= PLF_TWO_P256; k -= 1; }
    if (sc != 1.0) for (int i = 0; i < n; i++) v[i * PLF_TS] *= sc;
}

__global__ void __launch_bounds__(PLF_TS) generic_hess_kernel(GenericArgs a, HessTree ht, const double *Q /*[n][n] scaled*/,
                                                              const double *cat_rates, const double *site_w /*[S] or NULL*/,
                                                              double *Yg /*[C][E][n][Sc] scratch*/, double *dFg /*[N][n][Sc] scratch*/,
                                                              int *dFk /*[N][Sc]*/, double *Hpart /*[grid][E][E]*/, int *err)
{
    extern __shared__ double gsm[];
    const int tid = threadIdx.x, lane = tid & 31;
    const int n = a.n, Sc = a.Sc, E = a.t.E;
    double *v = gsm + tid;                              /* tangent of the edge vector on j's root path */
    double *t1 = gsm + (size_t)n * PLF_TS + tid;        /* work: dfe / dL */
    double *t2 = gsm + (size_t)2 * n * PLF_TS + tid;    /* work: matrix-vector results */
    double *buf = gsm + (size_t)3 * n * PLF_TS;         /* [E] this CTA's sums for the current j */
    double *myH = Hpart + (size_t)blockIdx.x * E * E;

    for (int tile = blockIdx.x; tile * PLF_TS < Sc; tile += gridDim.x) {
        const int s_raw = tile * PLF_TS + tid;
        const bool valid = s_raw < Sc;
        const int s = valid ? s_raw : Sc - 1;
        const int64_t gs = a.s0 + s;
        const double site_m = a.site_m[s];
        const int site_k = a.site_k[s];
        const double w = valid ? (site_w ? site_w[gs] : 1.0) : 0.0;

        /* y_idx = rate Q em_idx for every edge and category (exponent: that of the child) */
        for (int c = 0; c < a.C; c++) {
            const double rate = cat_rates[c];
            const size_t cE = (size_t)c * E;
            for (int idx = 0; idx < E; idx++) {
                const double *Em = a.Eg + ((cE + idx) * n) * Sc + s;
                double *Y = Yg + ((cE + idx) * n) * Sc + s;
                const int bc = a.Cg[((size_t)c * a.t.N + a.t.indices[idx]) * Sc + s];
                for (int k = 0; k < n; k++) t1[k * PLF_TS] = Em[(size_t)k * Sc];
                for (int i = 0; i < n; i++) {
                    double acc = 0.0;
                    if (!bc) for (int k = 0; k < n; k++) acc = fma(Q[i * n + k], t1[k * PLF_TS], acc);   /* util.c:338-344 */
                    Y[(size_t)i * Sc] = acc * rate;
                }
            }
        }

        for (int j = 0; j < E; j++) {
            const int rank_j = ht.erank[j];
            for (int i = tid; i < E; i += PLF_TS) buf[i] = 0.0;
            __syncthreads();
            for (int c = 0; c < a.C; c++) {
                const size_t cN = (size_t)c * a.t.N, cE = (size_t)c * E;
                const double rate = cat_rates[c];
                const double lhc = a.cat_prior[c] * a.cat_lh[(size_t)c * Sc + s];
                if (valid && w != 0.0 && !(lhc > 0.0) && rate != 0.0) atomicOr(err, 2);      /* arbplfhess.c:640-660: infeasible */
                const double coef = (lhc > 0.0 && site_m > 0.0) ? w * a.cat_prior[c] / site_m : 0.0;
                if (rate == 0.0) continue;          /* uniform over the CTA: a zero-rate category has no derivatives */

                /* fe of an edge, rebuilt from fn of its parent and the siblings' vectors: into t1, exponent returned */
                auto build_fe = [&](int idx, double *dst) -> int {
                    const int p = ht.parent_node[idx];
                    const double *Fa = a.Fg + ((cN + p) * n) * Sc + s;
                    int k = a.FK[(cN + p) * Sc + s];
                    if (a.t.node_has_data[p]) {
                        const int code = plf_code_at(a.codes, a.code_bytes, a.S, p, gs);
                        for (int i = 0; i < n; i++) dst[i * PLF_TS] = Fa[(size_t)i * Sc] * a.defs[(size_t)code * n + i];
                    } else {
                        for (int i = 0; i < n; i++) dst[i * PLF_TS] = Fa[(size_t)i * Sc];
                    }
                    for (int idx2 = a.t.indptr[p]; idx2 < a.t.indptr[p + 1]; idx2++) {
                        if (idx2 == idx) continue;
                        const double *Es = a.Eg + ((cE + idx2) * n) * Sc + s;
                        for (int i = 0; i < n; i++) dst[i * PLF_TS] *= Es[(size_t)i * Sc];
                        k += a.Kg[(cN + a.t.indices[idx2]) * Sc + s];
                        hess_rescale(dst, n, k);
                    }
                    return k;
                };

                /* ---- the edge itself: v = y_j, diagonal term ---- */
                const int bj = a.t.indices[j];
                const int kbj = a.Kg[(cN + bj) * Sc + s];
                {
                    const double *Y = Yg + ((cE + j) * n) * Sc + s;
                    for (int i = 0; i < n; i++) v[i * PLF_TS] = Y[(size_t)i * Sc];
                }
                int kv = kbj;
                {
                    const int kfe = build_fe(j, t1);
                    double x = 0.0;
                    for (int i = 0; i < n; i++) {
                        double acc = 0.0;
                        for (int k = 0; k < n; k++) acc = fma(Q[i * n + k], v[k * PLF_TS], acc);
                        x = fma(t1[i * PLF_TS], acc * rate, x);
                    }
                    x = hess_warp_sum(scalbn(x * coef, PLF_SCALE_BITS * max(-16, min(16, kfe + kv - site_k))));
                    if (lane == 0 && x != 0.0) atomicAdd(&buf[j], x);
                }

                /* ---- up the root path of j ---- */
                int cur = j;
                while (true) {
                    const int an = ht.parent_node[cur];
                    const int start = a.t.indptr[an], stop = a.t.indptr[an + 1];
                    const double *Fa = a.Fg + ((cN + an) * n) * Sc + s;
                    const int kFa = a.FK[(cN + an) * Sc + s];
                    int code_a = -1;
                    if (a.t.node_has_data[an]) code_a = plf_code_at(a.codes, a.code_bytes, a.S, an, gs);
                    /* the tangent enters the other children's subtrees */
                    for (int e1 = start; e1 < stop; e1++) {
                        if (e1 == cur || ht.sub_max[e1] <= rank_j) continue;
                        /* dfe_e1 = fn_a . base_a . v . prod(siblings other than e1 and cur) */
                        int kd = kFa + kv;
                        for (int i = 0; i < n; i++) {
                            double x = Fa[(size_t)i * Sc] * v[i * PLF_TS];
                            if (code_a >= 0) x *= a.defs[(size_t)code_a * n + i];
                            t1[i * PLF_TS] = x;
                        }
                        for (int e2 = start; e2 < stop; e2++) {
                            if (e2 == e1 || e2 == cur) continue;
                            const double *Es = a.Eg + ((cE + e2) * n) * Sc + s;
                            for (int i = 0; i < n; i++) t1[i * PLF_TS] *= Es[(size_t)i * Sc];
                            kd += a.Kg[(cN + a.t.indices[e2]) * Sc + s];
                        }
                        hess_rescale(t1, n, kd);
                        /* edge e1 itself, then its subtree in depth-first order; dfe of the edge being handled is in t1 */
                        const int b1 = a.t.indices[e1];
                        const int lo = ht.dfs_pos[b1], hi = ht.sub_end[b1];
                        int edge = e1, child = b1, kde = kd;
                        int pos = lo, cidx = 0, cstop = 0;      /* iteration state over (node at pos, its child edges) */
                        while (true) {
                            /* pair (edge, j) */
                            if (ht.erank[edge] > rank_j) {
                                const double *Y = Yg + ((cE + edge) * n) * Sc + s;
                                double x = 0.0;
                                for (int i = 0; i < n; i++) x = fma(t1[i * PLF_TS], Y[(size_t)i * Sc], x);
                                const int kc = a.Kg[(cN + child) * Sc + s];
                                x = hess_warp_sum(scalbn(x * coef, PLF_SCALE_BITS * max(-16, min(16, kde + kc - site_k))));
                                if (lane == 0 && x != 0.0) atomicAdd(&buf[edge], x);
                            }
                            /* dfn_child = P^T dfe (kept only for internal children) */
                            if (a.t.indptr[child] != a.t.indptr[child + 1]) {
                                const double *Pm = a.P + (cE + edge) * n * n;
                                double *dF = dFg + ((size_t)child * n) * Sc + s;
                                for (int jj = 0; jj < n; jj++) {
                                    double acc = 0.0;
                                    for (int i = 0; i < n; i++) acc = fma(Pm[i * n + jj], t1[i * PLF_TS], acc);
                                    t2[jj * PLF_TS] = acc;
                                }
                                int kk = kde;
                                hess_rescale(t2, n, kk);
                                for (int jj = 0; jj < n; jj++) dF[(size_t)jj * Sc] = t2[jj * PLF_TS];
                                dFk[(size_t)child * Sc + s] = kk;
                            }
                            /* next (node, child edge) of the subtree */
                            bool found = false;
                            while (!found) {
                                if (cidx < cstop) { found = true; break; }
                                if (pos >= hi) break;
                                const int x = ht.dfs_nodes[pos++];
                                cidx = a.t.indptr[x]; cstop = a.t.indptr[x + 1];
                            }
                            if (!found) break;
                            edge = cidx++;
                            child = a.t.indices[edge];
                            {
                                /* dfe_edge = dfn_x . base_x . prod(sibling vectors) */
                                const int x = ht.parent_node[edge];
                                const double *dF = dFg + ((size_t)x * n) * Sc + s;
                                kde = dFk[(size_t)x * Sc + s];
                                int code_x = -1;
                                if (a.t.node_has_data[x]) code_x = plf_code_at(a.codes, a.code_bytes, a.S, x, gs);
                                for (int i = 0; i < n; i++) {
                                    double y = dF[(size_t)i * Sc];
                                    if (code_x >= 0) y *= a.defs[(size_t)code_x * n + i];
                                    t1[i * PLF_TS] = y;
                                }
                                for (int e2 = a.t.indptr[x]; e2 < a.t.indptr[x + 1]; e2++) {
                                    if (e2 == edge) continue;
                                    const double *Es = a.Eg + ((cE + e2) * n) * Sc + s;
                                    for (int i = 0; i < n; i++) t1[i * PLF_TS] *= Es[(size_t)i * Sc];
                                    kde += a.Kg[(cN + a.t.indices[e2]) * Sc + s];
                                }
                                hess_rescale(t1, n, kde);
                            }
                        }
                    }
                    /* tangent of the node vector of an, then of the edge above it */
                    const int p = ht.parent_edge[an];
                    if (p < 0) break;
                    for (int i = 0; i < n; i++) {
                        double x = v[i * PLF_TS];
                        if (code_a >= 0) x *= a.defs[(size_t)code_a * n + i];
                        t1[i * PLF_TS] = x;
                    }
                    for (int e2 = start; e2 < stop; e2++) {
                        if (e2 == cur) continue;
                        const double *Es = a.Eg + ((cE + e2) * n) * Sc + s;
                        for (int i = 0; i < n; i++) t1[i * PLF_TS] *= Es[(size_t)i * Sc];
                        kv += a.Kg[(cN + a.t.indices[e2]) * Sc + s];
                    }
                    hess_rescale(t1, n, kv);
                    {
                        const double *Pm = a.P + (cE + p) * n * n;
                        for (int i = 0; i < n; i++) {
                            double acc = 0.0;
                            for (int k = 0; k < n; k++) acc = fma(Pm[i * n + k], t1[k * PLF_TS], acc);
                            v[i * PLF_TS] = acc;
                        }
                    }
                    /* pair (ancestor edge p, j): fe_p . (rate Q v) */
                    {
                        const int kfe = build_fe(p, t1);
                        double x = 0.0;
                        for (int i = 0; i < n; i++) {
                            double acc = 0.0;
                            for (int k = 0; k < n; k++) acc = fma(Q[i * n + k], v[k * PLF_TS], acc);
                            x = fma(t1[i * PLF_TS], acc * rate, x);
                        }
                        x = hess_warp_sum(scalbn(x * coef, PLF_SCALE_BITS * max(-16, min(16, kfe + kv - site_k))));
                        if (lane == 0 && x != 0.0) atomicAdd(&buf[p], x);
                    }
                    cur = p;
                }
            }
            __syncthreads();
            for (int i = tid; i < E; i += PLF_TS) {
                const double x = buf[i];
                if (x != 0.0) {
                    const int r = i > j ? i : j, cl = i > j ? j : i;
                    myH[(size_t)r * E + cl] += x;
                }
            }
            __syncthreads();
        }
    }
}

/* out[i][j] += sum_s w_s rows[i][s] rows[j][s] for j <= i: the g g^T / L^2 part of the Hessian of log L.
 * grid (ceil(E/16), ceil(E/16), splits over sites), 16 x 16 threads. */
__global__ void gram_rows_kernel(const double *rows, const double *w, int64_t w_off, int E, int cols, double *out)
{
    __shared__ double A[16][17], B[16][17];
    const int bi = blockIdx.x, bj = blockIdx.y;
    if (bj > bi) return;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int per = ((cols + gridDim.z - 1) / gridDim.z + 15) / 16 * 16;
    const int c0 = blockIdx.z * per, c1 = min(cols, c0 + per);
    double acc = 0.0;
    for (int c = c0; c < c1; c += 16) {
        const int col = c + tx;
        const double wv = (col < c1) ? (w ? w[w_off + col] : 1.0) : 0.0;
        const int ri = bi * 16 + ty, rj = bj * 16 + ty;
        A[ty][tx] = (ri < E && col < c1 && wv != 0.0) ? rows[(size_t)ri * cols + col] * wv : 0.0;
        B[ty][tx] = (rj < E && col < c1 && wv != 0.0) ? rows[(size_t)rj * cols + col] : 0.0;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; k++) acc = fma(A[ty][k], B[tx][k], acc);
        __syncthreads();
    }
    const int i = bi * 16 + ty, j = bj * 16 + tx;
    if (i < E && j < E && j <= i && acc != 0.0) atomicAdd(&out[(size_t)i * E + j], acc);
}
