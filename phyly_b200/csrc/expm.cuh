/*
 * K1/K2: batched matrix exponentials in double-double, one CTA per
 * (rate category, edge).
 *
 * Replaces arb_mat_exp in _update_transition_matrices (cross_site_ws.c:150-168)
 * and the 2n x 2n block exponential of _arb_mat_exp_frechet (util.c:500-548).
 *
 * Algorithm (not Arb's): A = r_c t_e Q is a rate matrix (off-diagonal >= 0, rows
 * sum to 0).  With mu = max_i |A_ii| and s = ceil(log2 mu)^+,
 *     exp(A) = ( e^{-mu/2^s} exp(B) )^(2^s),      B = (A + mu I)/2^s >= 0 .
 * exp(B) is a Taylor series of non-negative terms (no cancellation, so every
 * entry keeps full relative accuracy) and the squarings multiply non-negative
 * matrices.  The Frechet block exp([[A,L],[0,A]]) keeps its block-triangular
 * structure through both stages:
 *     X_k = B X_{k-1}/k,  Y_k = (B Y_{k-1} + L_s X_{k-1})/k ;  (X,Y)^2 = (X X, X Y + Y X).
 * Everything runs in double-double and is rounded to fp64 on output, together
 * with D = scale * Q * P (the derivative matrices), which needs the extra
 * digits when P is close to its stationary limit.
 */
#pragma once
#include "dd.h"

struct ExpmArgs {
    int n, E, C;
    const double *q_hi, *q_lo;       /* scaled rate matrix, n*n */
    const double *l_hi, *l_lo;       /* Frechet direction or NULL */
    const double *edge_rate;         /* [E] */
    const double *cat_rate;          /* [C] */
    const unsigned char *edge_mask;  /* [E] or NULL */
    double *P;                       /* [C][E][n][n] or NULL */
    double *D;                       /* [C][E][n][n] = cat_rate * Q * P, or NULL */
    double *F;                       /* [C][E][n][n] Frechet block, or NULL */
    int f_scale_mode;                /* 0: F ; 1: F * cat_rate * edge_rate */
    dd_t *ws;                        /* global workspace (8*n*n dd per CTA) or NULL => shared */
    /* adjoint form (plf_edge_expect_all): a direction per matrix, l_per[C][E][n][n] (fp64, replaces l_hi / l_lo),
     * and the Frechet derivative taken at A^T = r_c t_e Q^T -- the adjoint of L -> Frechet(A, L) */
    const double *l_per = nullptr;
    int q_transpose = 0;
};

__device__ __forceinline__ void dd_matmul(dd_t *Cm, const dd_t *A, const dd_t *B, int n, dd_t scale, bool use_scale)
{
    for (int idx = threadIdx.x; idx < n * n; idx += blockDim.x) {
        int i = idx / n, j = idx - i * n;
        dd_t acc = dd_make(0.0, 0.0);
        for (int k = 0; k < n; k++) {
            dd_t a = A[i * n + k];
            if (a.hi == 0.0) continue;
            acc = dd_add(acc, dd_mul(a, B[k * n + j]));
        }
        if (use_scale) acc = dd_mul(acc, scale);
        Cm[idx] = acc;
    }
}

/* Cm = (A*B + A2*B2) * scale */
__device__ __forceinline__ void dd_matmul2(dd_t *Cm, const dd_t *A, const dd_t *B, const dd_t *A2, const dd_t *B2,
                                           int n, dd_t scale, bool use_scale)
{
    for (int idx = threadIdx.x; idx < n * n; idx += blockDim.x) {
        int i = idx / n, j = idx - i * n;
        dd_t acc = dd_make(0.0, 0.0);
        for (int k = 0; k < n; k++) {
            dd_t a = A[i * n + k];
            if (a.hi != 0.0) acc = dd_add(acc, dd_mul(a, B[k * n + j]));
            dd_t a2 = A2[i * n + k];
            if (a2.hi != 0.0) acc = dd_add(acc, dd_mul(a2, B2[k * n + j]));
        }
        if (use_scale) acc = dd_mul(acc, scale);
        Cm[idx] = acc;
    }
}

/* e^{-x} for 0 <= x <= 1 in double-double (Taylor of e^{x}, then reciprocal) */
__device__ __forceinline__ dd_t dd_exp_neg_small(dd_t x)
{
    dd_t term = dd_make(1.0, 0.0), sum = dd_make(1.0, 0.0);
    for (int k = 1; k <= 34; k++) {
        term = dd_div_d(dd_mul(term, x), (double)k);
        sum = dd_add(sum, term);
        if (term.hi < 1e-36) break;
    }
    return dd_div(dd_make(1.0, 0.0), sum);
}

__global__ void __launch_bounds__(256) expm_dd_kernel(ExpmArgs a)
{
    extern __shared__ __align__(16) unsigned char expm_smem[];
    const int n = a.n, nn = n * n;
    const int e = blockIdx.x, c = blockIdx.y;
    if (a.edge_mask && !a.edge_mask[e]) {
        /* unrequested edge: leave zeros in F (evaluate_site_frechet.c:24-38 never uses them) */
        if (a.F) for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) a.F[((size_t)c * a.E + e) * nn + idx] = 0.0;
        if (!a.P && !a.D) return;
    }
    const bool want_f = (a.F != nullptr) && !(a.edge_mask && !a.edge_mask[e]);
    dd_t *base = a.ws ? a.ws + ((size_t)(c * a.E + e)) * 8 * nn : reinterpret_cast<dd_t *>(expm_smem);
    dd_t *B = base, *X = base + nn, *SX = base + 2 * nn, *T = base + 3 * nn;
    dd_t *Ls = base + 4 * nn, *Y = base + 5 * nn, *SY = base + 6 * nn, *T2 = base + 7 * nn;

    const double r = a.cat_rate[c], t = a.edge_rate[e];
    const dd_t rt = dd_two_prod(r, t);

    __shared__ double sh_mu;
    __shared__ int sh_s;
    /* A = rt * Q ; find mu */
    if (threadIdx.x == 0) {
        double mu = 0.0;
        for (int i = 0; i < n; i++) {
            dd_t q = dd_make(a.q_hi[i * n + i], a.q_lo ? a.q_lo[i * n + i] : 0.0);
            double v = fabs(dd_to_d(dd_mul(q, rt)));
            if (v > mu) mu = v;
        }
        int s = 0;
        if (mu > 1.0) { int ex; frexp(mu, &ex); s = ex; /* mu < 2^ex */ }
        /* Every extra halving of B costs one squaring and saves Taylor terms; both are one matrix product on the
         * critical path (the kernel is latency bound: a handful of warps per SM), a squaring being the cheaper one.
         * Take the number of halvings (<= 8) that minimises terms + squarings: 31 + 0 becomes about 14 + 6 at mu = 1.
         * Squaring non-negative matrices keeps the relative accuracy; 8 squarings cost 2^8 dd roundings, 1e-29. */
        if (mu > 0.0) {
            int best = 1 << 30, best_j = 0;
            for (int j = 0; j <= 8; j++) {
                const double m = scalbn(mu, -(s + j));
                double bound = 1.0;
                int k = 1;
                while (k < 40) { bound *= m / k; if (bound < 1.9e-34 && k >= 2) break; k++; }
                if (k + j < best) { best = k + j; best_j = j; }
            }
            s += best_j;
        }
        sh_mu = mu; sh_s = s;
    }
    __syncthreads();
    const double mu = sh_mu;
    const int s = sh_s;
    const double inv2s = scalbn(1.0, -s);
    const dd_t mus = dd_make(mu * inv2s, 0.0);   /* exact: power of two scaling */

    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        int i = idx / n, j = idx - i * n;
        const int qidx = a.q_transpose ? j * n + i : idx;
        dd_t q = dd_make(a.q_hi[qidx], a.q_lo ? a.q_lo[qidx] : 0.0);
        dd_t v = dd_mul_pwr2(dd_mul(q, rt), inv2s);
        if (i == j) v = dd_add(v, mus);
        if (v.hi < 0.0) v = dd_make(0.0, 0.0);   /* the diagonal entry that defines mu */
        B[idx] = v;
        dd_t id = dd_make(i == j ? 1.0 : 0.0, 0.0);
        X[idx] = id; SX[idx] = id;
        if (want_f) {
            dd_t l = a.l_per ? dd_make(a.l_per[((size_t)c * a.E + e) * nn + idx], 0.0)
                             : dd_make(a.l_hi[idx], a.l_lo ? a.l_lo[idx] : 0.0);
            Ls[idx] = dd_mul_pwr2(l, inv2s);
            Y[idx] = dd_make(0.0, 0.0); SY[idx] = dd_make(0.0, 0.0);
        }
    }
    __syncthreads();

    /* number of Taylor terms: mus^k/k! < 2^-112 (mus <= 1 -> at most 32) */
    int nterms = 1;
    {
        double bound = 1.0, m = mus.hi;
        /* for the Frechet block the norm of the shifted block matrix is mus + |L_s|; be generous */
        while (nterms < 40) { bound *= (m > 0.0 ? m : 0.0) / nterms; if (bound < 1.9e-34 && nterms >= 2) break; nterms++; }
        if (m == 0.0) nterms = 2;
        if (want_f) nterms += 4;
    }
    for (int k = 1; k <= nterms; k++) {
        dd_t invk = dd_div(dd_make(1.0, 0.0), dd_make((double)k, 0.0));
        /* T = B X / k ; T2 = (B Y + Ls X)/k */
        dd_matmul(T, B, X, n, invk, true);
        if (want_f) dd_matmul2(T2, B, Y, Ls, X, n, invk, true);
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            X[idx] = T[idx]; SX[idx] = dd_add(SX[idx], T[idx]);
            if (want_f) { Y[idx] = T2[idx]; SY[idx] = dd_add(SY[idx], T2[idx]); }
        }
        __syncthreads();
    }
    /* multiply by e^{-mus} */
    {
        dd_t em = dd_exp_neg_small(mus);
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            SX[idx] = dd_mul(SX[idx], em);
            if (want_f) SY[idx] = dd_mul(SY[idx], em);
        }
        __syncthreads();
    }
    /* squarings: (X,Y) <- (X X, X Y + Y X) */
    for (int it = 0; it < s; it++) {
        dd_matmul(T, SX, SX, n, dd_make(1.0, 0.0), false);
        if (want_f) dd_matmul2(T2, SX, SY, SY, SX, n, dd_make(1.0, 0.0), false);
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            SX[idx] = T[idx];
            if (want_f) SY[idx] = T2[idx];
        }
        __syncthreads();
    }
    const size_t off = ((size_t)c * a.E + e) * nn;
    if (a.P) for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) a.P[off + idx] = dd_to_d(SX[idx]);
    if (want_f) {
        dd_t fsd = (a.f_scale_mode == 1) ? rt : dd_make(1.0, 0.0);
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) a.F[off + idx] = dd_to_d(dd_mul(SY[idx], fsd));
    }
    if (a.D) {
        /* D = r * Q * P in dd, T as scratch holding Q */
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) T[idx] = dd_make(a.q_hi[idx], a.q_lo ? a.q_lo[idx] : 0.0);
        __syncthreads();
        dd_matmul(T2, T, SX, n, dd_make(r, 0.0), true);
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) a.D[off + idx] = dd_to_d(T2[idx]);
    }
}

/*
 * The 4-state case without a Frechet block (P and D of every ll / deriv / marginal step): the same arithmetic in the same
 * order as expm_dd_kernel -- the two give identical bits -- but 16 lanes per matrix (lane = 4 i + j holds entry (i, j)),
 * operands exchanged by shuffles inside the half-warp, no shared-memory round trips and no block barrier in the loops.  The
 * generic kernel spends 40 us on the 504 matrices of cfg2 (a chain of ~20 dependent dd products, each between two
 * barriers; the search for the number of halvings on one thread; 1/k by a dd division per term); this one 10 us, which is
 * 4 % of a step at 8 GPUs.
 */
__device__ __forceinline__ dd_t dd_shfl16(unsigned mask, dd_t v, int src)
{
    return dd_make(__shfl_sync(mask, v.hi, src, 16), __shfl_sync(mask, v.lo, src, 16));
}

__global__ void __launch_bounds__(128) expm4_dd_kernel(ExpmArgs a)
{
    __shared__ dd_t s_invk[48];
    for (int k = threadIdx.x; k < 48; k += blockDim.x) s_invk[k] = dd_div(dd_make(1.0, 0.0), dd_make((double)(k + 1), 0.0));
    __syncthreads();
    const int l16 = threadIdx.x & 15, i = l16 >> 2, j = l16 & 3;
    const unsigned mask = 0xffffu << (threadIdx.x & 16);
    const int total = a.C * a.E;
    const int m_raw = blockIdx.x * (blockDim.x >> 4) + (threadIdx.x >> 4);
    const bool live = m_raw < total;
    const int m_idx = live ? m_raw : total - 1;          /* spare half-warps redo the last matrix and write nothing */
    const int c = m_idx / a.E, e = m_idx - c * a.E;
    const double r = a.cat_rate[c], t = a.edge_rate[e];
    const dd_t rt = dd_two_prod(r, t);

    double mu = 0.0;
#pragma unroll
    for (int d = 0; d < 4; d++) {
        dd_t q = dd_make(a.q_hi[d * 5], a.q_lo ? a.q_lo[d * 5] : 0.0);
        double v = fabs(dd_to_d(dd_mul(q, rt)));
        if (v > mu) mu = v;
    }
    int s = 0;
    if (mu > 1.0) { int ex; frexp(mu, &ex); s = ex; }
    if (mu > 0.0) {
        /* halvings 0..8 tried by nine lanes at once (expm_dd_kernel tries them one after the other) */
        const int jj = min(l16, 8);
        const double mm = scalbn(mu, -(s + jj));
        double bound = 1.0;
        int k = 1;
        while (k < 40) { bound *= mm / k; if (bound < 1.9e-34 && k >= 2) break; k++; }
        int key = (k + jj) * 16 + jj;
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) key = min(key, __shfl_xor_sync(mask, key, o, 16));
        s += key & 15;
    }
    const double inv2s = scalbn(1.0, -s);
    const dd_t mus = dd_make(mu * inv2s, 0.0);

    dd_t Bij;
    {
        dd_t q = dd_make(a.q_hi[l16], a.q_lo ? a.q_lo[l16] : 0.0);
        dd_t v = dd_mul_pwr2(dd_mul(q, rt), inv2s);
        if (i == j) v = dd_add(v, mus);
        if (v.hi < 0.0) v = dd_make(0.0, 0.0);
        Bij = v;
    }
    dd_t Brow[4];
#pragma unroll
    for (int k = 0; k < 4; k++) Brow[k] = dd_shfl16(mask, Bij, i * 4 + k);
    dd_t X = dd_make(i == j ? 1.0 : 0.0, 0.0), SX = X;

    int nterms = 1;
    {
        double bound = 1.0, mm = mus.hi;
        while (nterms < 40) { bound *= (mm > 0.0 ? mm : 0.0) / nterms; if (bound < 1.9e-34 && nterms >= 2) break; nterms++; }
        if (mm == 0.0) nterms = 2;
    }
    for (int k = 1; k <= nterms; k++) {
        dd_t acc = dd_make(0.0, 0.0);
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            const dd_t x = dd_shfl16(mask, X, kk * 4 + j);
            if (Brow[kk].hi != 0.0) acc = dd_add(acc, dd_mul(Brow[kk], x));
        }
        acc = dd_mul(acc, s_invk[k - 1]);
        X = acc;
        SX = dd_add(SX, acc);
    }
    SX = dd_mul(SX, dd_exp_neg_small(mus));
    for (int it = 0; it < s; it++) {
        dd_t acc = dd_make(0.0, 0.0);
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            const dd_t av = dd_shfl16(mask, SX, i * 4 + kk), bv = dd_shfl16(mask, SX, kk * 4 + j);
            if (av.hi != 0.0) acc = dd_add(acc, dd_mul(av, bv));
        }
        SX = acc;
    }
    const size_t off = (size_t)m_idx * 16;
    if (a.P && live) a.P[off + l16] = dd_to_d(SX);
    if (a.D) {
        dd_t acc = dd_make(0.0, 0.0);
#pragma unroll
        for (int kk = 0; kk < 4; kk++) {
            const dd_t qv = dd_make(a.q_hi[i * 4 + kk], a.q_lo ? a.q_lo[i * 4 + kk] : 0.0);
            const dd_t pv = dd_shfl16(mask, SX, kk * 4 + j);
            if (qv.hi != 0.0) acc = dd_add(acc, dd_mul(qv, pv));
        }
        acc = dd_mul(acc, dd_make(r, 0.0));
        if (live) a.D[off + l16] = dd_to_d(acc);
    }
}
