/*
 * Certified mode: enclosures [lower, upper] of the site log-likelihoods with directed rounding.
 *
 * The reference computes in Arb's midpoint-radius arithmetic and raises the precision until every output is a ball
 * that rounds to a unique double (util.c:12-50, arbplfll.c:206-224).  Here the same pruning recursion
 * (evaluate_site_lhood.c:21-57, arbplfll.c:139-170) is run in fp64 INTERVAL arithmetic: every quantity on the path is
 * non-negative, so a lower bound is obtained by rounding every operation down (__dmul_rd, __fma_rd, __dadd_rd) and an
 * upper bound by rounding every operation up; scaling by powers of two is exact.  The enclosure is rigorous with
 * respect to the inputs the device receives, given as intervals themselves:
 *   - rate_c * t_e  within a relative delta_rate (the host's gamma quantiles are accurate to 1e-14, not certified);
 *   - the scaled rate matrix Q and the derived priors within a relative delta_q (long-double host arithmetic);
 *   - exp / log of the CUDA math library within their documented 1 ulp (3 ulps are taken).
 *
 * cert_expm_kernel encloses exp(x Q), x in [x_lo, x_hi]:  with mu >= max_i |x Q_ii| and B = (x Q + mu I) / 2^s >= 0,
 * exp(x Q) = (e^{-beta} exp(B))^(2^s), beta = mu / 2^s <= 1.  The Taylor polynomial of degree K of exp(B) with all
 * operations rounded down is a lower bound; rounded up and increased by the bound beta^(K+1)/(K+1)!/(1 - beta/(K+2)) of
 * the remainder (B has row sums beta) it is an upper bound; squaring keeps both (non-negative matrices).
 *
 * Derivatives (plf_deriv_certified) are signed: d L_c / d t_e = r_c fe^T Q P_e L_b.  Q P is not formed from [Plo, Phi],
 * whose width on a long branch is as large as Q P itself.  With R(y) = P(y) - 1 P_0(y) (row 0 subtracted from every
 * row; R 1 = 0), R(y)^2 = R(2y) and Q P = Q R, so R is enclosed at the scaled level y = x / 2^s, where its entries are
 * O(beta) and not O(e^{-lambda x}), squared s times in signed interval arithmetic (cert_imul), and D = r_c Q R(x).
 * cert_outside_kernel restates generic_outside_kernel on non-negative intervals (one exponent for both bounds, as in
 * cert_inside_kernel); only the edge form fe^T D L_b is signed.  cert_deriv_site_kernel sums the categories and
 * divides by the site likelihood enclosure of cert_site_kernel.
 *
 * Edge expectations (plf_edge_expect_certified) take the Frechet matrices of cert_frechet_kernel in place of D, without
 * D's literal-zero shortcuts; marginals (plf_marginal_certified) replace every node's outside vector by fa_v .* L_v in
 * the outside pass.  Both are non-negative apart from a signed direction L = L+ - L-.
 */
#pragma once
#include <stdint.h>
#include "plf_consts.h"

#define CERT_TS 64          /* sites per CTA in cert_inside_kernel and cert_outside_kernel */
#define CERT_TAYLOR 26
#define CERT_GROUP 1024     /* sites per partial sum of the certified outside queries: chunks are multiples of it */

__device__ __forceinline__ double cert_down(double x, int ulps)
{
    for (int i = 0; i < ulps; i++) x = nextafter(x, -__longlong_as_double(0x7ff0000000000000LL));
    return x;
}
__device__ __forceinline__ double cert_up(double x, int ulps)
{
    for (int i = 0; i < ulps; i++) x = nextafter(x, __longlong_as_double(0x7ff0000000000000LL));
    return x;
}

/* [lo, hi] = [alo, ahi] * [blo, bhi], signs arbitrary */
__device__ __forceinline__ void cert_imul(double alo, double ahi, double blo, double bhi, double &lo, double &hi)
{
    lo = fmin(fmin(__dmul_rd(alo, blo), __dmul_rd(alo, bhi)), fmin(__dmul_rd(ahi, blo), __dmul_rd(ahi, bhi)));
    hi = fmax(fmax(__dmul_ru(alo, blo), __dmul_ru(alo, bhi)), fmax(__dmul_ru(ahi, blo), __dmul_ru(ahi, bhi)));
}

/* [lo, hi] = [alo, ahi] * [blo, bhi] with blo >= 0 */
__device__ __forceinline__ void cert_mul_pos(double alo, double ahi, double blo, double bhi, double &lo, double &hi)
{
    lo = __dmul_rd(alo, alo >= 0.0 ? blo : bhi);
    hi = __dmul_ru(ahi, ahi >= 0.0 ? bhi : blo);
}

/*
 * D = r Q R(x) from R at the scaled level (in Rlo / Rhi, s squarings to go); W: 2 n^2 doubles of workspace.  Q is the
 * interval matrix of cert_expm_kernel without the factor x: off the diagonal the enclosure of q_ij, on it minus the sum
 * of that row's enclosures.  r = 0 gives D = 0 exactly.
 */
__device__ void cert_deriv_matrix(int n, int s, double r, double delta_rate, double delta_q, const double *q_hi, const double *q_lo,
                                  double *Rlo, double *Rhi, double *Wlo, double *Whi, double *Dlo, double *Dhi)
{
    const int nn = n * n;
    if (r == 0.0) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { Dlo[idx] = 0.0; Dhi[idx] = 0.0; }
        return;
    }
    for (int q = 0; q < s; q++) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            double lo = 0.0, hi = 0.0;
            for (int m = 0; m < n; m++) {
                double pl, ph;
                cert_imul(Rlo[i * n + m], Rhi[i * n + m], Rlo[m * n + j], Rhi[m * n + j], pl, ph);
                lo = __dadd_rd(lo, pl); hi = __dadd_ru(hi, ph);
            }
            Wlo[idx] = lo; Whi[idx] = hi;
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { Rlo[idx] = Wlo[idx]; Rhi[idx] = Whi[idx]; }
    }
    __syncthreads();
    /* the enclosure of Q into W */
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        const int i = idx / n, j = idx - i * n;
        if (i != j) {
            const double qd = __dadd_rd(q_hi[idx], q_lo ? q_lo[idx] : 0.0), qu = __dadd_ru(q_hi[idx], q_lo ? q_lo[idx] : 0.0);
            Wlo[idx] = fmax(0.0, __dmul_rd(qd, __dsub_rd(1.0, delta_q)));
            Whi[idx] = __dmul_ru(fmax(0.0, qu), __dadd_ru(1.0, delta_q));
        } else {
            double rlo = 0.0, rhi = 0.0;
            for (int k = 0; k < n; k++) {
                if (k == i) continue;
                const double qd = __dadd_rd(q_hi[i * n + k], q_lo ? q_lo[i * n + k] : 0.0), qu = __dadd_ru(q_hi[i * n + k], q_lo ? q_lo[i * n + k] : 0.0);
                rlo = __dadd_rd(rlo, fmax(0.0, __dmul_rd(qd, __dsub_rd(1.0, delta_q))));
                rhi = __dadd_ru(rhi, __dmul_ru(fmax(0.0, qu), __dadd_ru(1.0, delta_q)));
            }
            Wlo[idx] = -rhi; Whi[idx] = -rlo;
        }
    }
    __syncthreads();
    const double rl = __dmul_rd(r, __dsub_rd(1.0, delta_rate)), rh = __dmul_ru(r, __dadd_ru(1.0, delta_rate));
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        const int i = idx / n, j = idx - i * n;
        double lo = 0.0, hi = 0.0;
        for (int m = 0; m < n; m++) {
            double pl, ph;
            cert_imul(Wlo[i * n + m], Whi[i * n + m], Rlo[m * n + j], Rhi[m * n + j], pl, ph);
            lo = __dadd_rd(lo, pl); hi = __dadd_ru(hi, ph);
        }
        double dl, dh;
        cert_mul_pos(lo, hi, rl, rh, dl, dh);
        Dlo[idx] = dl; Dhi[idx] = dh;
    }
}

/* thread 0 of the CTA: x = r t in [xlo, xhi] and mu >= max_i x sum_{j != i} q_ij, both rounded up */
__device__ __forceinline__ void cert_shift(int n, const double *q_hi, const double *q_lo, double r, double t, double delta_rate,
                                           double delta_q, double &xlo, double &xhi, double &mu)
{
    xlo = __dmul_rd(__dmul_rd(r, __dsub_rd(1.0, delta_rate)), t);
    xhi = __dmul_ru(__dmul_ru(r, __dadd_ru(1.0, delta_rate)), t);
    mu = 0.0;
    for (int i = 0; i < n; i++) {
        double rs = 0.0;
        for (int j = 0; j < n; j++) {
            if (j == i) continue;
            const double q = __dmul_ru(__dadd_ru(q_hi[i * n + j], q_lo ? q_lo[i * n + j] : 0.0), __dadd_ru(1.0, delta_q));
            rs = __dadd_ru(rs, q);
        }
        mu = fmax(mu, __dmul_ru(xhi, rs));
    }
}

/* [Blo, Bhi] = (x Q + mu I) sc, sc a power of two */
__device__ __forceinline__ void cert_shifted_matrix(int n, const double *q_hi, const double *q_lo, double delta_q, double xlo,
                                                    double xhi, double mu, double sc, double *Blo, double *Bhi)
{
    for (int idx = threadIdx.x; idx < n * n; idx += blockDim.x) {
        const int i = idx / n, j = idx - i * n;
        double lo, hi;
        if (i != j) {
            const double qd = __dadd_rd(q_hi[idx], q_lo ? q_lo[idx] : 0.0), qu = __dadd_ru(q_hi[idx], q_lo ? q_lo[idx] : 0.0);
            lo = __dmul_rd(xlo, fmax(0.0, __dmul_rd(qd, __dsub_rd(1.0, delta_q))));
            hi = __dmul_ru(xhi, __dmul_ru(fmax(0.0, qu), __dadd_ru(1.0, delta_q)));
        } else {
            double rlo = 0.0, rhi = 0.0;
            for (int k = 0; k < n; k++) {
                if (k == i) continue;
                const double qd = __dadd_rd(q_hi[i * n + k], q_lo ? q_lo[i * n + k] : 0.0), qu = __dadd_ru(q_hi[i * n + k], q_lo ? q_lo[i * n + k] : 0.0);
                rlo = __dadd_rd(rlo, fmax(0.0, __dmul_rd(qd, __dsub_rd(1.0, delta_q))));
                rhi = __dadd_ru(rhi, __dmul_ru(fmax(0.0, qu), __dadd_ru(1.0, delta_q)));
            }
            lo = fmax(0.0, __dsub_rd(mu, __dmul_ru(xhi, rhi)));
            hi = __dsub_ru(mu, __dmul_rd(xlo, rlo));
        }
        Blo[idx] = lo * sc; Bhi[idx] = hi * sc;               /* exact: a power of two */
    }
}

/* b^(K+1) / (K+1)! / (1 - b / (K+2)), rounded up: the remainder of the Taylor series of exp(M), M >= 0 of row sums <= b <= 1 */
__device__ __forceinline__ double cert_taylor_rem(double b)
{
    double rem = 1.0;
    for (int k = 1; k <= CERT_TAYLOR + 1; k++) rem = __ddiv_ru(__dmul_ru(rem, b), (double)k);
    return __ddiv_ru(rem, __dsub_rd(1.0, __ddiv_ru(b, (double)(CERT_TAYLOR + 2))));
}

/* one CTA per (edge, category); ws: 8 n^2 doubles per CTA.  Dlo / Dhi (or NULL): enclosure of r_c Q P_e as well. */
__global__ void __launch_bounds__(128) cert_expm_kernel(int n, int E, int C, const double *q_hi, const double *q_lo,
                                                        const double *edge_rate, const double *cat_rate, double delta_rate,
                                                        double delta_q, double *ws, double *Plo, double *Phi,
                                                        double *Dlo, double *Dhi)
{
    const int e = blockIdx.x, c = blockIdx.y, nn = n * n;
    double *base = ws + ((size_t)c * E + e) * 8 * nn;
    double *Blo = base, *Bhi = base + nn, *Tlo = base + 2 * nn, *Thi = base + 3 * nn;
    double *Slo = base + 4 * nn, *Shi = base + 5 * nn, *Ulo = base + 6 * nn, *Uhi = base + 7 * nn;
    double *outlo = Plo + ((size_t)c * E + e) * nn, *outhi = Phi + ((size_t)c * E + e) * nn;
    __shared__ double sh_mu, sh_xlo, sh_xhi;
    __shared__ int sh_s;
    const double r = cat_rate[c], t = edge_rate[e];
    if (threadIdx.x == 0) {
        double xlo, xhi, mu;
        cert_shift(n, q_hi, q_lo, r, t, delta_rate, delta_q, xlo, xhi, mu);
        int s = 0;
        if (mu > 1.0) { int ex; frexp(mu, &ex); s = ex; }
        sh_mu = mu; sh_s = s; sh_xlo = xlo; sh_xhi = xhi;
    }
    __syncthreads();
    const double mu = sh_mu, xlo = sh_xlo, xhi = sh_xhi;
    const int s = sh_s;
    if (!(mu > 0.0)) {          /* zero rate or zero length: the identity, exactly */
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { const double v = (idx / n == idx % n) ? 1.0 : 0.0; outlo[idx] = v; outhi[idx] = v; }
        if (!Dlo) return;
        /* R = I - 1 e_0^T, exactly */
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            const double v = (i == j ? 1.0 : 0.0) - (j == 0 ? 1.0 : 0.0);
            Blo[idx] = v; Bhi[idx] = v;
        }
        cert_deriv_matrix(n, 0, r, delta_rate, delta_q, q_hi, q_lo, Blo, Bhi, Tlo, Thi,
                          Dlo + ((size_t)c * E + e) * nn, Dhi + ((size_t)c * E + e) * nn);
        return;
    }
    const double sc = scalbn(1.0, -s);
    /* B, term_0 = sum_0 = I */
    cert_shifted_matrix(n, q_hi, q_lo, delta_q, xlo, xhi, mu, sc, Blo, Bhi);
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        const double id = (idx / n == idx % n) ? 1.0 : 0.0;
        Tlo[idx] = id; Thi[idx] = id; Slo[idx] = id; Shi[idx] = id;
    }
    __syncthreads();
    for (int k = 1; k <= CERT_TAYLOR; k++) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            double lo = 0.0, hi = 0.0;
            for (int m = 0; m < n; m++) {
                lo = __fma_rd(Tlo[i * n + m], Blo[m * n + j], lo);
                hi = __fma_ru(Thi[i * n + m], Bhi[m * n + j], hi);
            }
            Ulo[idx] = __ddiv_rd(lo, (double)k); Uhi[idx] = __ddiv_ru(hi, (double)k);
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            Tlo[idx] = Ulo[idx]; Thi[idx] = Uhi[idx];
            Slo[idx] = __dadd_rd(Slo[idx], Ulo[idx]); Shi[idx] = __dadd_ru(Shi[idx], Uhi[idx]);
        }
        __syncthreads();
    }
    /* remainder of the series and the scalar e^{-beta} */
    const double beta = mu * sc;                               /* exact, <= 1 */
    const double rem = cert_taylor_rem(beta);
    const double ev = exp(-beta);
    const double elo = cert_down(ev, 3), ehi = cert_up(ev, 3);
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        Slo[idx] = __dmul_rd(Slo[idx], elo);
        Shi[idx] = __dmul_ru(__dadd_ru(Shi[idx], rem), ehi);
    }
    __syncthreads();
    if (Dlo) {
        /* R(y) = P(y) - 1 P_0(y) at the scaled level into B (free after the Taylor stage); row 0 is exactly 0 */
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            Blo[idx] = i == 0 ? 0.0 : __dsub_rd(Slo[idx], Shi[j]);
            Bhi[idx] = i == 0 ? 0.0 : __dsub_ru(Shi[idx], Slo[j]);
        }
    }
    for (int q = 0; q < s; q++) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            double lo = 0.0, hi = 0.0;
            for (int m = 0; m < n; m++) {
                lo = __fma_rd(Slo[i * n + m], Slo[m * n + j], lo);
                hi = __fma_ru(Shi[i * n + m], Shi[m * n + j], hi);
            }
            Ulo[idx] = lo; Uhi[idx] = hi;
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { Slo[idx] = Ulo[idx]; Shi[idx] = Uhi[idx]; }
        __syncthreads();
    }
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { outlo[idx] = fmax(0.0, Slo[idx]); outhi[idx] = fmin(1.0, Shi[idx]); }
    if (Dlo) cert_deriv_matrix(n, s, r, delta_rate, delta_q, q_hi, q_lo, Blo, Bhi, Tlo, Thi,
                               Dlo + ((size_t)c * E + e) * nn, Dhi + ((size_t)c * E + e) * nn);
}

/*
 * [Ylo, Yhi] encloses the Frechet block F(L) = the top-right block of exp([[A, L], [0, A]]), A = x Q, for a direction
 * [Llo, Lhi] >= 0 of row sums <= lnorm.  With B = (A + mu I) / 2^s >= 0 and L_s = L / 2^s, the shifted block matrix
 * [[B, L_s], [0, B]] is non-negative with row sums <= b = (mu + lnorm) / 2^s <= 1; its Taylor terms are X_k = B X_{k-1} / k
 * and Y_k = (B Y_{k-1} + L_s X_{k-1}) / k, the remainder of every entry is cert_taylor_rem(b), and e^{-beta} (X, Y) is
 * squared s times as (X, Y) <- (X X, X Y + Y X).  Everything is non-negative: round down for Ylo, up for Yhi.
 * W: 14 n^2 doubles of workspace.  mu = 0 (x = 0, or Q = 0) gives F = L exactly.
 */
__device__ void cert_frechet_pos(int n, const double *q_hi, const double *q_lo, double delta_q, double xlo, double xhi,
                                 double mu, double lnorm, const double *Llo, const double *Lhi, double *W, double *Ylo, double *Yhi)
{
    const int nn = n * n;
    if (!(mu > 0.0)) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { Ylo[idx] = Llo[idx]; Yhi[idx] = Lhi[idx]; }
        __syncthreads();
        return;
    }
    double *Blo = W, *Bhi = W + nn, *Xlo = W + 2 * nn, *Xhi = W + 3 * nn, *Tlo = W + 4 * nn, *Thi = W + 5 * nn;
    double *SXlo = W + 6 * nn, *SXhi = W + 7 * nn, *Ulo = W + 8 * nn, *Uhi = W + 9 * nn, *Vlo = W + 10 * nn, *Vhi = W + 11 * nn;
    double *Lslo = W + 12 * nn, *Lshi = W + 13 * nn;
    const double bsum = __dadd_ru(mu, lnorm);
    int s = 0;
    if (bsum > 1.0) { int ex; frexp(bsum, &ex); s = ex; }
    const double sc = scalbn(1.0, -s);
    cert_shifted_matrix(n, q_hi, q_lo, delta_q, xlo, xhi, mu, sc, Blo, Bhi);
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        const double id = (idx / n == idx % n) ? 1.0 : 0.0;
        Xlo[idx] = id; Xhi[idx] = id; SXlo[idx] = id; SXhi[idx] = id;
        Tlo[idx] = 0.0; Thi[idx] = 0.0; Ylo[idx] = 0.0; Yhi[idx] = 0.0;
        Lslo[idx] = __dmul_rd(Llo[idx], sc); Lshi[idx] = __dmul_ru(Lhi[idx], sc);
    }
    __syncthreads();
    /* Taylor terms: X in (X, SX), Y_k in T, their sum in Y */
    for (int k = 1; k <= CERT_TAYLOR; k++) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            double xl = 0.0, xh = 0.0, yl = 0.0, yh = 0.0;
            for (int m = 0; m < n; m++) {
                xl = __fma_rd(Blo[i * n + m], Xlo[m * n + j], xl);
                xh = __fma_ru(Bhi[i * n + m], Xhi[m * n + j], xh);
                yl = __fma_rd(Blo[i * n + m], Tlo[m * n + j], yl);
                yh = __fma_ru(Bhi[i * n + m], Thi[m * n + j], yh);
                yl = __fma_rd(Lslo[i * n + m], Xlo[m * n + j], yl);
                yh = __fma_ru(Lshi[i * n + m], Xhi[m * n + j], yh);
            }
            Ulo[idx] = __ddiv_rd(xl, (double)k); Uhi[idx] = __ddiv_ru(xh, (double)k);
            Vlo[idx] = __ddiv_rd(yl, (double)k); Vhi[idx] = __ddiv_ru(yh, (double)k);
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            Xlo[idx] = Ulo[idx]; Xhi[idx] = Uhi[idx]; Tlo[idx] = Vlo[idx]; Thi[idx] = Vhi[idx];
            SXlo[idx] = __dadd_rd(SXlo[idx], Ulo[idx]); SXhi[idx] = __dadd_ru(SXhi[idx], Uhi[idx]);
            Ylo[idx] = __dadd_rd(Ylo[idx], Vlo[idx]); Yhi[idx] = __dadd_ru(Yhi[idx], Vhi[idx]);
        }
        __syncthreads();
    }
    /* remainder of both blocks and the scalar e^{-beta} */
    const double rem = cert_taylor_rem(bsum * sc);             /* bsum * sc: exact, <= 1 */
    const double ev = exp(-(mu * sc));
    const double elo = cert_down(ev, 3), ehi = cert_up(ev, 3);
    for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
        SXlo[idx] = __dmul_rd(SXlo[idx], elo); SXhi[idx] = __dmul_ru(__dadd_ru(SXhi[idx], rem), ehi);
        Ylo[idx] = __dmul_rd(Ylo[idx], elo); Yhi[idx] = __dmul_ru(__dadd_ru(Yhi[idx], rem), ehi);
    }
    __syncthreads();
    for (int q = 0; q < s; q++) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            double xl = 0.0, xh = 0.0, yl = 0.0, yh = 0.0;
            for (int m = 0; m < n; m++) {
                xl = __fma_rd(SXlo[i * n + m], SXlo[m * n + j], xl);
                xh = __fma_ru(SXhi[i * n + m], SXhi[m * n + j], xh);
                yl = __fma_rd(SXlo[i * n + m], Ylo[m * n + j], yl);
                yh = __fma_ru(SXhi[i * n + m], Yhi[m * n + j], yh);
                yl = __fma_rd(Ylo[i * n + m], SXlo[m * n + j], yl);
                yh = __fma_ru(Yhi[i * n + m], SXhi[m * n + j], yh);
            }
            Ulo[idx] = xl; Uhi[idx] = fmin(1.0, xh); Vlo[idx] = yl; Vhi[idx] = yh;
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            SXlo[idx] = Ulo[idx]; SXhi[idx] = Uhi[idx]; Ylo[idx] = Vlo[idx]; Yhi[idx] = Vhi[idx];
        }
        __syncthreads();
    }
}

/*
 * Enclosures of the Frechet matrices of plf_edge_expect: one CTA per (edge, category), ws: 18 n^2 doubles per CTA.
 * F is linear in L = L+ - L-; each entry l_hi + l_lo is widened by the relative delta_q (a TRANS direction holds entries
 * of the scaled Q), and F(L-) is formed only when L has a negative entry.  trans: F x, x in [xlo, xhi] (f_scale_mode 1
 * of expm_dd_kernel); x = 0 gives F = L (DWELL) or F = 0 (TRANS) exactly.  Unrequested edges are 0.
 */
__global__ void __launch_bounds__(128) cert_frechet_kernel(int n, int E, int C, const double *q_hi, const double *q_lo,
                                                           const double *edge_rate, const double *cat_rate, double delta_rate,
                                                           double delta_q, const double *l_hi, const double *l_lo, int trans,
                                                           const unsigned char *edge_mask, double *ws, double *Flo, double *Fhi)
{
    const int e = blockIdx.x, c = blockIdx.y, nn = n * n;
    double *outlo = Flo + ((size_t)c * E + e) * nn, *outhi = Fhi + ((size_t)c * E + e) * nn;
    if (edge_mask && !edge_mask[e]) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { outlo[idx] = 0.0; outhi[idx] = 0.0; }
        return;
    }
    double *base = ws + ((size_t)c * E + e) * 18 * nn;
    double *Ylo = base + 14 * nn, *Yhi = base + 15 * nn, *Llo = base + 16 * nn, *Lhi = base + 17 * nn;
    __shared__ double sh_mu, sh_xlo, sh_xhi, sh_lnorm;
    if (threadIdx.x == 0) {
        double xlo, xhi, mu;
        cert_shift(n, q_hi, q_lo, cat_rate[c], edge_rate[e], delta_rate, delta_q, xlo, xhi, mu);
        sh_mu = mu; sh_xlo = xlo; sh_xhi = xhi;
    }
    __syncthreads();
    const double mu = sh_mu, xlo = sh_xlo, xhi = sh_xhi;
    if (trans && !(xhi > 0.0)) {
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) { outlo[idx] = 0.0; outhi[idx] = 0.0; }
        return;
    }
    for (int neg = 0; neg < 2; neg++) {
        /* [Llo, Lhi]: the enclosure of L+ (neg = 0) or of L- (neg = 1) */
        int any = 0;
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            const double vd = __dadd_rd(l_hi[idx], l_lo ? l_lo[idx] : 0.0), vu = __dadd_ru(l_hi[idx], l_lo ? l_lo[idx] : 0.0);
            const double pd = neg ? -vu : vd, pu = neg ? -vd : vu;
            Llo[idx] = fmax(0.0, __dmul_rd(pd, __dsub_rd(1.0, delta_q)));
            Lhi[idx] = __dmul_ru(fmax(0.0, pu), __dadd_ru(1.0, delta_q));
            any |= Lhi[idx] > 0.0;
        }
        if (!__syncthreads_or(any) && neg) break;
        if (threadIdx.x == 0) {
            double ln = 0.0;
            for (int i = 0; i < n; i++) {
                double rs = 0.0;
                for (int j = 0; j < n; j++) rs = __dadd_ru(rs, Lhi[i * n + j]);
                ln = fmax(ln, rs);
            }
            sh_lnorm = ln;
        }
        __syncthreads();
        cert_frechet_pos(n, q_hi, q_lo, delta_q, xlo, xhi, mu, sh_lnorm, Llo, Lhi, base, Ylo, Yhi);
        for (int idx = threadIdx.x; idx < nn; idx += blockDim.x) {
            double lo = Ylo[idx], hi = Yhi[idx];
            if (trans) cert_mul_pos(lo, hi, xlo, xhi, lo, hi);
            if (!neg) { outlo[idx] = lo; outhi[idx] = hi; }
            else { outlo[idx] = __dsub_rd(outlo[idx], hi); outhi[idx] = __dsub_ru(outhi[idx], lo); }
        }
        __syncthreads();
    }
}

struct CertArgs {
    TreeDev t;
    int n, C, K;
    int64_t S, s0;
    int Sc;
    const void *codes; int code_bytes;
    const double *defs; const unsigned char *def_const;
    const double *Plo, *Phi;           /* [C][E][n][n] */
    int root_mode;
    const double *root_lo, *root_hi;   /* [n] enclosure of the root prior weights */
    const double *prior_lo, *prior_hi; /* [C] enclosure of the category priors */
    double *Llo, *Lhi;                 /* [C][N][n][Sc] node vectors (mantissas), one exponent for both bounds */
    int *Kg; unsigned char *Cg;        /* [C][N][Sc] */
    double *cat_lo, *cat_hi; int *cat_k;   /* [C][Sc] */
    double *site_lo, *site_hi;         /* [S] enclosures of the site log-likelihoods */
    /* the outside queries only: plf_deriv_certified, plf_edge_expect_certified, plf_marginal_certified (NULL otherwise) */
    double *site_mlo, *site_mhi; int *site_k;   /* [Sc] the site likelihood enclosure [mlo, mhi] 2^(256 k) */
    const double *Dlo, *Dhi;           /* [C][E][n][n] enclosures of the edge matrices: r_c Q P_e, or Frechet matrices */
    int deriv;                         /* the edge matrices are r_c Q P_e: D 1 = 0 and D = 0 at rate 0 (literal zeros) */
    int marg;                          /* replace every node's outside vector (leaves included) by fa_v .* L_v */
    const double *cat_rate;            /* [C] */
    const unsigned char *edge_mask;    /* [E] or NULL */
    double *Flo, *Fhi; int *FK;        /* [C][N][n][Sc] outside vectors (mantissas), [C][N][Sc] their exponents */
    double *xlo, *xhi; int *xk;        /* [C][E][Sc] edge forms fe^T D L_b (mantissas), [C][E][Sc] exponents; NULL: none */
    const double *site_w;              /* [S] or NULL */
    double *out_lo, *out_hi;           /* [cols][Sc] per-site enclosures (columns: edges, or node x state) */
    int *err;                          /* bit 0: a site of non-zero weight whose likelihood enclosure reaches 0 */
};

/* interval restatement of generic_inside_kernel: thread = (site, category), blockIdx.y = category */
__global__ void __launch_bounds__(CERT_TS) cert_inside_kernel(CertArgs a)
{
    extern __shared__ double csm[];
    const int tid = threadIdx.x;
    const int s = blockIdx.x * CERT_TS + tid;
    const int c = blockIdx.y;
    if (s >= a.Sc) return;
    const int n = a.n, Sc = a.Sc;
    const int64_t gs = a.s0 + s;
    double *alo = csm + tid, *ahi = csm + (size_t)n * CERT_TS + tid;
    double *vlo = csm + (size_t)2 * n * CERT_TS + tid, *vhi = csm + (size_t)3 * n * CERT_TS + tid;
    const size_t cN = (size_t)c * a.t.N, cE = (size_t)c * a.t.E;

    for (int u = a.t.N - 1; u >= 0; u--) {
        const int nd = a.t.preorder[u];
        const int start = a.t.indptr[nd], stop = a.t.indptr[nd + 1];
        int accK = 0, cst = 1;
        if (a.t.node_has_data[nd]) {
            const int code = plf_code_at(a.codes, a.code_bytes, a.S, nd, gs);
            for (int i = 0; i < n; i++) { const double d = a.defs[(size_t)code * n + i]; alo[i * CERT_TS] = d; ahi[i * CERT_TS] = d; }
            cst = a.def_const[code];
        } else {
            for (int i = 0; i < n; i++) { alo[i * CERT_TS] = 1.0; ahi[i * CERT_TS] = 1.0; }
        }
        for (int idx = start; idx < stop; idx++) {
            const int b = a.t.indices[idx];
            const double *Lbl = a.Llo + ((cN + b) * n) * Sc + s, *Lbh = a.Lhi + ((cN + b) * n) * Sc + s;
            for (int k = 0; k < n; k++) { vlo[k * CERT_TS] = Lbl[(size_t)k * Sc]; vhi[k * CERT_TS] = Lbh[(size_t)k * Sc]; }
            const int kb = a.Kg[(cN + b) * Sc + s];
            const int bc = a.Cg[(cN + b) * Sc + s];
            const double *Pl = a.Plo + (cE + idx) * n * n, *Ph = a.Phi + (cE + idx) * n * n;
            double mx = 0.0;
            for (int i = 0; i < n; i++) {
                double elo, ehi;
                if (bc) {                    /* exact constant column under a stochastic matrix (arb_mat_extras.c:84-91) */
                    elo = vlo[0]; ehi = vhi[0];
                } else {
                    elo = 0.0; ehi = 0.0;
                    for (int k = 0; k < n; k++) {
                        elo = __fma_rd(Pl[i * n + k], vlo[k * CERT_TS], elo);
                        ehi = __fma_ru(Ph[i * n + k], vhi[k * CERT_TS], ehi);
                    }
                }
                const double xl = __dmul_rd(alo[i * CERT_TS], elo), xh = __dmul_ru(ahi[i * CERT_TS], ehi);
                alo[i * CERT_TS] = xl; ahi[i * CERT_TS] = xh;
                mx = fmax(mx, xh);
            }
            accK += kb;
            cst &= bc;
            while (mx > 0.0 && mx < PLF_TWO_M256) {      /* exact rescaling of both bounds */
                for (int i = 0; i < n; i++) { alo[i * CERT_TS] *= PLF_TWO_P256; ahi[i * CERT_TS] *= PLF_TWO_P256; }
                mx *= PLF_TWO_P256;
                accK -= 1;
            }
        }
        double *Ll = a.Llo + ((cN + nd) * n) * Sc + s, *Lh = a.Lhi + ((cN + nd) * n) * Sc + s;
        for (int i = 0; i < n; i++) { Ll[(size_t)i * Sc] = alo[i * CERT_TS]; Lh[(size_t)i * Sc] = ahi[i * CERT_TS]; }
        a.Kg[(cN + nd) * Sc + s] = accK;
        a.Cg[(cN + nd) * Sc + s] = (unsigned char)cst;
        if (nd == a.t.root) {
            /* root_prior_expectation, model.c:282-350 */
            double lo = 0.0, hi = 0.0;
            if (cst && (a.root_mode == PLF_ROOT_UNIFORM || a.root_mode == PLF_ROOT_EQUILIBRIUM)) {
                lo = alo[0]; hi = ahi[0];
            } else {
                for (int i = 0; i < n; i++) {
                    lo = __fma_rd(a.root_lo[i], alo[i * CERT_TS], lo);
                    hi = __fma_ru(a.root_hi[i], ahi[i * CERT_TS], hi);
                }
            }
            a.cat_lo[(size_t)c * Sc + s] = lo;
            a.cat_hi[(size_t)c * Sc + s] = hi;
            a.cat_k[(size_t)c * Sc + s] = accK;
        }
    }
}

/* x 2^(256 k), k <= 0, rounded towards zero (down = 1) or away from it, for x >= 0 */
__device__ __forceinline__ double cert_scale(double x, int k, int down)
{
    if (x == 0.0 || k == 0) return x;
    const double y = scalbn(x, PLF_SCALE_BITS * max(k, -16));
    if (scalbn(y, -PLF_SCALE_BITS * max(k, -16)) == x && k >= -16) return y;       /* exact */
    return down ? (y > 0.0 ? cert_down(y, 1) : 0.0) : cert_up(y, 1);
}

/* combine the categories (arbplfll.c:149-169): enclosure of log(sum_c prior_c L_c) */
__global__ void cert_site_kernel(CertArgs a)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.Sc) return;
    const int Sc = a.Sc;
    int k0 = INT_MIN;
    for (int c = 0; c < a.C; c++)
        if (a.prior_hi[c] * a.cat_hi[(size_t)c * Sc + s] > 0.0) k0 = max(k0, a.cat_k[(size_t)c * Sc + s]);
    double lo = 0.0, hi = 0.0;
    if (k0 != INT_MIN) {
        for (int c = 0; c < a.C; c++) {
            const int dk = a.cat_k[(size_t)c * Sc + s] - k0;
            if (a.prior_hi[c] * a.cat_hi[(size_t)c * Sc + s] > 0.0) {
                lo = __dadd_rd(lo, cert_scale(__dmul_rd(a.prior_lo[c], a.cat_lo[(size_t)c * Sc + s]), dk, 1));
                hi = __dadd_ru(hi, cert_scale(__dmul_ru(a.prior_hi[c], a.cat_hi[(size_t)c * Sc + s]), dk, 0));
            }
        }
    } else {
        k0 = 0;
    }
    /* log(m 2^(256 k0)): 256 ln 2 lies in [c_lo, c_hi]; k0 <= 0 */
    const double c_lo = 177.445678223346, c_hi = 177.44567822334602;
    const double kd = (double)k0;
    double llo = (lo > 0.0) ? cert_down(log(lo), 3) : -INFINITY;
    double lhi = (hi > 0.0) ? cert_up(log(hi), 3) : -INFINITY;
    llo = __dadd_rd(llo, __dmul_rd(kd, k0 <= 0 ? c_hi : c_lo));
    lhi = __dadd_ru(lhi, __dmul_ru(kd, k0 <= 0 ? c_lo : c_hi));
    a.site_lo[a.s0 + s] = llo;
    a.site_hi[a.s0 + s] = lhi;
    if (a.site_mlo) { a.site_mlo[s] = lo; a.site_mhi[s] = hi; a.site_k[s] = k0; }
}

/* x 2^(256 k), any sign and any k, rounded down (down = 1) or up; exact whenever the result is representable */
__device__ __forceinline__ double cert_scale_signed(double x, int k, int down)
{
    if (x == 0.0 || k == 0) return x;
    const int kk = max(-16, min(16, k));
    const double y = scalbn(x, PLF_SCALE_BITS * kk);
    if (kk == k && isfinite(y) && scalbn(y, -PLF_SCALE_BITS * kk) == x) return y;
    if (y == 0.0) return (down == (x < 0.0)) ? (down ? -__longlong_as_double(1LL) : __longlong_as_double(1LL)) : 0.0;
    return down ? cert_down(y, 1) : cert_up(y, 1);
}

/* rescale a non-negative interval vector (stride CERT_TS) by powers of 2^256 until max(hi) lies in [2^-256, 2^256] */
__device__ __forceinline__ void cert_rescale(double *lo, double *hi, int n, double mx, int &k)
{
    while (mx > 0.0 && mx < PLF_TWO_M256) {            /* exact */
        for (int i = 0; i < n; i++) { lo[i * CERT_TS] *= PLF_TWO_P256; hi[i * CERT_TS] *= PLF_TWO_P256; }
        mx *= PLF_TWO_P256; k -= 1;
    }
    while (mx > PLF_TWO_P256 && mx < INFINITY) {        /* the low bounds may lose bits: round them down */
        for (int i = 0; i < n; i++) { lo[i * CERT_TS] = __dmul_rd(lo[i * CERT_TS], PLF_TWO_M256); hi[i * CERT_TS] = __dmul_ru(hi[i * CERT_TS], PLF_TWO_M256); }
        mx *= PLF_TWO_M256; k += 1;
    }
}

/*
 * Interval restatement of generic_outside_kernel: thread = (site, category), blockIdx.y = category.  Writes the edge
 * form fe^T D L_b of every requested edge to xlo / xhi / xk (unless xlo is NULL).  A category with zero likelihood at
 * the site writes nothing (cert_deriv_site_kernel skips it); for the derivative (deriv) a category of rate 0 and a child
 * whose vector is an exact constant column (D 1 = 0) give 0 exactly -- properties of D that a Frechet matrix does not
 * have.  With marg, every node's outside vector fa_v is replaced by the marginal product fa_v .* L_v (exponent
 * k_a + k_v) once its children have used it; the leaves get outside vectors too.  The sibling edge vectors P L are
 * recomputed from the inside vectors.
 */
__global__ void __launch_bounds__(CERT_TS) cert_outside_kernel(CertArgs a)
{
    extern __shared__ double csm[];
    const int tid = threadIdx.x;
    const int s = blockIdx.x * CERT_TS + tid;
    const int c = blockIdx.y;
    if (s >= a.Sc) return;
    const int n = a.n, Sc = a.Sc;
    const int64_t gs = a.s0 + s;
    if (!(a.prior_hi[c] * a.cat_hi[(size_t)c * Sc + s] > 0.0)) return;
    double *tlo = csm + tid, *thi = csm + (size_t)n * CERT_TS + tid;
    double *flo = csm + (size_t)2 * n * CERT_TS + tid, *fhi = csm + (size_t)3 * n * CERT_TS + tid;
    double *ylo = csm + (size_t)4 * n * CERT_TS + tid, *yhi = csm + (size_t)5 * n * CERT_TS + tid;
    const size_t cN = (size_t)c * a.t.N, cE = (size_t)c * a.t.E, nn = (size_t)n * n;
    const bool zero_rate = a.deriv && a.cat_rate[c] == 0.0;
    {
        double *Fl = a.Flo + ((cN + a.t.root) * n) * Sc + s, *Fh = a.Fhi + ((cN + a.t.root) * n) * Sc + s;
        for (int i = 0; i < n; i++) { Fl[(size_t)i * Sc] = a.root_lo[i]; Fh[(size_t)i * Sc] = a.root_hi[i]; }
        a.FK[(cN + a.t.root) * Sc + s] = 0;
    }
    for (int u = 0; u < a.t.N; u++) {
        const int nd = a.t.preorder[u];
        const int start = a.t.indptr[nd], stop = a.t.indptr[nd + 1];
        if (start == stop && !a.marg) continue;
        double *Fl = a.Flo + ((cN + nd) * n) * Sc + s, *Fh = a.Fhi + ((cN + nd) * n) * Sc + s;
        const int ka = a.FK[(cN + nd) * Sc + s];
        if (start != stop) {
            if (a.t.node_has_data[nd]) {
                const int code = plf_code_at(a.codes, a.code_bytes, a.S, nd, gs);
                for (int i = 0; i < n; i++) {
                    const double d = a.defs[(size_t)code * n + i];
                    tlo[i * CERT_TS] = __dmul_rd(Fl[(size_t)i * Sc], d); thi[i * CERT_TS] = __dmul_ru(Fh[(size_t)i * Sc], d);
                }
            } else {
                for (int i = 0; i < n; i++) { tlo[i * CERT_TS] = Fl[(size_t)i * Sc]; thi[i * CERT_TS] = Fh[(size_t)i * Sc]; }
            }
        }
        if (a.marg) {
            /* fa_v .* L_v in place of fa_v, which the children below take from t */
            const double *Ll = a.Llo + ((cN + nd) * n) * Sc + s, *Lh = a.Lhi + ((cN + nd) * n) * Sc + s;
            for (int i = 0; i < n; i++) {
                Fl[(size_t)i * Sc] = __dmul_rd(Fl[(size_t)i * Sc], Ll[(size_t)i * Sc]);
                Fh[(size_t)i * Sc] = __dmul_ru(Fh[(size_t)i * Sc], Lh[(size_t)i * Sc]);
            }
            a.FK[(cN + nd) * Sc + s] = ka + a.Kg[(cN + nd) * Sc + s];
            if (start == stop) continue;
        }
        for (int idx = start; idx < stop; idx++) {
            const int b = a.t.indices[idx];
            int kfe = ka;
            for (int i = 0; i < n; i++) { flo[i * CERT_TS] = tlo[i * CERT_TS]; fhi[i * CERT_TS] = thi[i * CERT_TS]; }
            for (int idx2 = start; idx2 < stop; idx2++) {
                if (idx2 == idx) continue;
                const int b2 = a.t.indices[idx2];
                const double *Lbl = a.Llo + ((cN + b2) * n) * Sc + s, *Lbh = a.Lhi + ((cN + b2) * n) * Sc + s;
                for (int k = 0; k < n; k++) { ylo[k * CERT_TS] = Lbl[(size_t)k * Sc]; yhi[k * CERT_TS] = Lbh[(size_t)k * Sc]; }
                const int bc = a.Cg[(cN + b2) * Sc + s];
                const double *Pl = a.Plo + (cE + idx2) * nn, *Ph = a.Phi + (cE + idx2) * nn;
                double mx = 0.0;
                for (int i = 0; i < n; i++) {
                    double elo, ehi;
                    if (bc) {
                        elo = ylo[0]; ehi = yhi[0];
                    } else {
                        elo = 0.0; ehi = 0.0;
                        for (int k = 0; k < n; k++) {
                            elo = __fma_rd(Pl[i * n + k], ylo[k * CERT_TS], elo);
                            ehi = __fma_ru(Ph[i * n + k], yhi[k * CERT_TS], ehi);
                        }
                    }
                    const double xl = __dmul_rd(flo[i * CERT_TS], elo), xh = __dmul_ru(fhi[i * CERT_TS], ehi);
                    flo[i * CERT_TS] = xl; fhi[i * CERT_TS] = xh;
                    mx = fmax(mx, xh);
                }
                kfe += a.Kg[(cN + b2) * Sc + s];
                cert_rescale(flo, fhi, n, mx, kfe);
            }
            const int kb = a.Kg[(cN + b) * Sc + s];
            if (a.xlo && (!a.edge_mask || a.edge_mask[idx])) {
                /* fe^T (D L_b): first the signed interval vector D L_b, then its product with the non-negative fe */
                double xl = 0.0, xh = 0.0;
                if (!zero_rate && !(a.deriv && a.Cg[(cN + b) * Sc + s])) {
                    const double *Lbl = a.Llo + ((cN + b) * n) * Sc + s, *Lbh = a.Lhi + ((cN + b) * n) * Sc + s;
                    for (int k = 0; k < n; k++) { ylo[k * CERT_TS] = Lbl[(size_t)k * Sc]; yhi[k * CERT_TS] = Lbh[(size_t)k * Sc]; }
                    const double *Dl = a.Dlo + (cE + idx) * nn, *Dh = a.Dhi + (cE + idx) * nn;
                    for (int i = 0; i < n; i++) {
                        double vl = 0.0, vh = 0.0;
                        for (int k = 0; k < n; k++) {
                            double pl, ph;
                            cert_mul_pos(Dl[i * n + k], Dh[i * n + k], ylo[k * CERT_TS], yhi[k * CERT_TS], pl, ph);
                            vl = __dadd_rd(vl, pl); vh = __dadd_ru(vh, ph);
                        }
                        double pl, ph;
                        cert_mul_pos(vl, vh, flo[i * CERT_TS], fhi[i * CERT_TS], pl, ph);
                        xl = __dadd_rd(xl, pl); xh = __dadd_ru(xh, ph);
                    }
                }
                a.xlo[(cE + idx) * Sc + s] = xl;
                a.xhi[(cE + idx) * Sc + s] = xh;
                a.xk[(cE + idx) * Sc + s] = kfe + kb;
            }
            /* outside vector of b: P^T fe (internal children only, unless marg) */
            if (a.marg || a.t.indptr[b] != a.t.indptr[b + 1]) {
                const double *Pl = a.Plo + (cE + idx) * nn, *Ph = a.Phi + (cE + idx) * nn;
                double mx = 0.0;
                for (int j = 0; j < n; j++) {
                    double lo = 0.0, hi = 0.0;
                    for (int i = 0; i < n; i++) {
                        lo = __fma_rd(Pl[i * n + j], flo[i * CERT_TS], lo);
                        hi = __fma_ru(Ph[i * n + j], fhi[i * CERT_TS], hi);
                    }
                    ylo[j * CERT_TS] = lo; yhi[j * CERT_TS] = hi;
                    mx = fmax(mx, hi);
                }
                int kfb = kfe;
                cert_rescale(ylo, yhi, n, mx, kfb);
                double *Fbl = a.Flo + ((cN + b) * n) * Sc + s, *Fbh = a.Fhi + ((cN + b) * n) * Sc + s;
                for (int j = 0; j < n; j++) { Fbl[(size_t)j * Sc] = ylo[j * CERT_TS]; Fbh[(size_t)j * Sc] = yhi[j * CERT_TS]; }
                a.FK[(cN + b) * Sc + s] = kfb;
            }
        }
    }
}

/*
 * Per (site, column): sum_c prior_c x_c 2^(256 (xk_c - k0)) over the categories of non-zero likelihood, divided by the
 * site likelihood enclosure [mlo, mhi] 2^(256 k0).  Column e of category c has its mantissas at x[(c cols + e) Sc + s]
 * and its exponent at xk[(c cols / cpk + e / cpk) Sc + s]: the edge forms (cols = E, cpk = 1) or the marginal products
 * (cols = N n, cpk = n).  grid (sites / 128, columns e0..).  Unrequested edges are 0 exactly; a site whose likelihood
 * enclosure reaches 0 gets [-inf, +inf] (and bit 0 of err if its weight is not 0).
 */
__global__ void cert_deriv_site_kernel(CertArgs a, const double *x_lo, const double *x_hi, const int *x_k, int cols, int cpk, int e0)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int e = e0 + blockIdx.y;
    if (s >= a.Sc) return;
    const int Sc = a.Sc;
    const double mlo = a.site_mlo[s], mhi = a.site_mhi[s];
    const int k0 = a.site_k[s];
    if (e == 0 && !(mlo > 0.0) && (a.site_w ? a.site_w[a.s0 + s] : 1.0) != 0.0) atomicOr(a.err, 1);
    double lo = 0.0, hi = 0.0;
    if (!a.edge_mask || a.edge_mask[e]) {
        if (!(mlo > 0.0)) {
            lo = -INFINITY; hi = INFINITY;
        } else {
            double nlo = 0.0, nhi = 0.0;
            for (int c = 0; c < a.C; c++) {
                if (!(a.prior_hi[c] * a.cat_hi[(size_t)c * Sc + s] > 0.0)) continue;
                const size_t at = ((size_t)c * cols + e) * Sc + s;
                double tl, th;
                cert_mul_pos(x_lo[at], x_hi[at], a.prior_lo[c], a.prior_hi[c], tl, th);
                const int dk = x_k[((size_t)c * (cols / cpk) + e / cpk) * Sc + s] - k0;
                nlo = __dadd_rd(nlo, cert_scale_signed(tl, dk, 1));
                nhi = __dadd_ru(nhi, cert_scale_signed(th, dk, 0));
            }
            lo = __ddiv_rd(nlo, nlo >= 0.0 ? mhi : mlo);
            hi = __ddiv_ru(nhi, nhi >= 0.0 ? mlo : mhi);
            if (lo == 0.0) lo = 0.0;            /* no -0.0 */
            if (hi == 0.0) hi = 0.0;
        }
    }
    a.out_lo[(size_t)e * Sc + s] = lo;
    a.out_hi[(size_t)e * Sc + s] = hi;
}

/*
 * Weighted sums of the enclosures, per group of CERT_GROUP sites and column, in a fixed order (the same bits on every
 * call, whatever the chunking): grid (groups of the chunk, columns e0..), one warp.  A negative weight swaps the bounds.
 */
__global__ void __launch_bounds__(32) cert_deriv_group_sum_kernel(CertArgs a, int cols, int e0, double *part_lo, double *part_hi)
{
    const int g = blockIdx.x, e = e0 + blockIdx.y, lane = threadIdx.x, Sc = a.Sc;
    const int s1 = min(Sc, (g + 1) * CERT_GROUP);
    double lo = 0.0, hi = 0.0;
    for (int s = g * CERT_GROUP + lane; s < s1; s += 32) {
        const double w = a.site_w ? a.site_w[a.s0 + s] : 1.0;
        if (w == 0.0) continue;
        const double l = a.out_lo[(size_t)e * Sc + s], h = a.out_hi[(size_t)e * Sc + s];
        lo = __dadd_rd(lo, __dmul_rd(w, w > 0.0 ? l : h));
        hi = __dadd_ru(hi, __dmul_ru(w, w > 0.0 ? h : l));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = __dadd_rd(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = __dadd_ru(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) {
        const size_t at = (size_t)(a.s0 / CERT_GROUP + g) * cols + e;
        part_lo[at] = lo; part_hi[at] = hi;
    }
}

/* sum_lo[e] / sum_hi[e]: the groups' partial sums in order */
__global__ void cert_deriv_total_kernel(const double *part_lo, const double *part_hi, int groups, int E, double *sum_lo, double *sum_hi)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double lo = 0.0, hi = 0.0;
    for (int g = 0; g < groups; g++) {
        lo = __dadd_rd(lo, part_lo[(size_t)g * E + e]);
        hi = __dadd_ru(hi, part_hi[(size_t)g * E + e]);
    }
    sum_lo[e] = lo == 0.0 ? 0.0 : lo;           /* no -0.0 (a rounded-down sum of zeros) */
    sum_hi[e] = hi == 0.0 ? 0.0 : hi;
}
