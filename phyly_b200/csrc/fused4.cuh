/*
 * Fused 4-state (DNA) pruning kernel: the hot path of arbplf-ll / arbplf-deriv
 * (and of dwell / trans, which only change the per-edge matrices).
 *
 * Reference loop nest being replaced (arbplfll.c:139-170, arbplfderiv.c:274-357):
 *   for site: for category: evaluate_site_lhood (evaluate_site_lhood.c:21-57,
 *   _prune_update_prob util.c:241-301), then per requested edge a root-path
 *   recomputation (arbplfderiv.c:144-205).
 *
 * B200 design
 *   - one thread owns one site pattern and walks the whole tree; all rate
 *     categories are advanced together (compile-time C, unrolled), so tree
 *     decoding, tip codes and addresses are shared by the categories and each
 *     thread carries 4*C independent fp64 chains.
 *   - the tree is compiled on the host into a post-order program with
 *     Sethi-Ullman child ordering; the program, the transition / derivative
 *     matrices of the internal edges and the tip tables (P_e.def_k, F_e.def_k
 *     per character k) are staged in shared memory once per CTA; the tile's tip
 *     codes are staged in shared memory once per tile (coalesced 1-byte loads).
 *   - the newest partial of each category lives in shared memory ("cur");
 *     inside partials of internal nodes are written once to a per-thread slab
 *     in HBM ([slot][category][thread] double4: every warp access is one
 *     contiguous 1 KB run) and read once by the outside pass.
 *   - derivative / dwell / trans outputs come from an outside (pre-order) pass
 *     that runs the same program backwards with the identity
 *         d L_c / d t_e = rate_c * fe_e^T (Q P_e) L_b ,
 *     replacing the reference's O(depth) walk per edge.  Per-edge values are
 *     summed over categories in registers, over the 32 sites of a warp with
 *     shuffles, over the warps of the CTA in shared memory, and over CTAs by a
 *     deterministic second-stage kernel.
 * Algorithmic HBM traffic: 1 byte per (site, tip) of codes plus, when the
 * outside pass runs, 2 x 33 bytes per (internal node, category, site).
 */
#pragma once
#include <stdint.h>

#include "f4prog.h"

#include "../../include/plf.h"
#include "plf_consts.h"
#include "fused4_args.h"

__constant__ double f4_cP[F4_CM_MAXD];
__constant__ double f4_cF[F4_CM_MAXD];


__device__ __forceinline__ void f4_matvec(const double *__restrict__ M, const double v[4], double out[4])
{
    const double2 *M2 = reinterpret_cast<const double2 *>(M);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        double2 a = M2[2 * i], b = M2[2 * i + 1];
        double r = a.x * v[0];
        r = fma(a.y, v[1], r);
        r = fma(b.x, v[2], r);
        r = fma(b.y, v[3], r);
        out[i] = r;
    }
}

/* out = M^T v */
__device__ __forceinline__ void f4_matvec_t(const double *__restrict__ M, const double v[4], double out[4])
{
    const double2 *M2 = reinterpret_cast<const double2 *>(M);
    double2 a0 = M2[0], b0 = M2[1];
    out[0] = a0.x * v[0]; out[1] = a0.y * v[0]; out[2] = b0.x * v[0]; out[3] = b0.y * v[0];
#pragma unroll
    for (int i = 1; i < 4; i++) {
        double2 a = M2[2 * i], b = M2[2 * i + 1];
        out[0] = fma(a.x, v[i], out[0]);
        out[1] = fma(a.y, v[i], out[1]);
        out[2] = fma(b.x, v[i], out[2]);
        out[3] = fma(b.y, v[i], out[3]);
    }
}

/* out = M v with M = base[off..] (shared / global memory) or, for CM, the constant set WHICH (0 = P, 1 = F) */
template <bool CM, int WHICH>
__device__ __forceinline__ void f4_mv(const double *__restrict__ base, int off, const double v[4], double out[4])
{
    if (CM) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            double r;
            if (WHICH) {
                r = f4_cF[off + 4 * i] * v[0];
                r = fma(f4_cF[off + 4 * i + 1], v[1], r);
                r = fma(f4_cF[off + 4 * i + 2], v[2], r);
                r = fma(f4_cF[off + 4 * i + 3], v[3], r);
            } else {
                r = f4_cP[off + 4 * i] * v[0];
                r = fma(f4_cP[off + 4 * i + 1], v[1], r);
                r = fma(f4_cP[off + 4 * i + 2], v[2], r);
                r = fma(f4_cP[off + 4 * i + 3], v[3], r);
            }
            out[i] = r;
        }
    } else {
        f4_matvec(base + off, v, out);
    }
}

/* out = P^T v */
template <bool CM>
__device__ __forceinline__ void f4_mvt(const double *__restrict__ base, int off, const double v[4], double out[4])
{
    if (CM) {
#pragma unroll
        for (int j = 0; j < 4; j++) out[j] = f4_cP[off + j] * v[0];
#pragma unroll
        for (int i = 1; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) out[j] = fma(f4_cP[off + 4 * i + j], v[i], out[j]);
    } else {
        f4_matvec_t(base + off, v, out);
    }
}

__device__ __forceinline__ void f4_ld4(const double *__restrict__ p, double out[4])
{
    const double2 *p2 = reinterpret_cast<const double2 *>(p);
    double2 a = p2[0], b = p2[1];
    out[0] = a.x; out[1] = a.y; out[2] = b.x; out[3] = b.y;
}

/* number of 2^256 up-scalings applied so that max(v) >= 2^-256 (v >= 0) */
__device__ __forceinline__ int f4_rescale_up(double v[4])
{
    /* non-negative doubles order like their high words */
    int h = max(max(__double2hiint(v[0]), __double2hiint(v[1])), max(__double2hiint(v[2]), __double2hiint(v[3])));
    int s = 0;
    if (h < 0x2FF00000) {          /* high word of 2^-256 */
        double m = fmax(fmax(v[0], v[1]), fmax(v[2], v[3]));
        while (m > 0.0 && m < PLF_TWO_M256 && s < 3) {
#pragma unroll
            for (int i = 0; i < 4; i++) v[i] *= PLF_TWO_P256;
            m *= PLF_TWO_P256;
            s++;
        }
    }
    return s;
}

__device__ __forceinline__ double f4_warp_sum(double x)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

/* character code of this thread's site for tile row r */
template <int BD, bool PACK>
__device__ __forceinline__ int f4_code(const unsigned char *tile, int r, int tid)
{
    if (PACK) return (tile[(r >> 1) * BD + tid] >> ((r & 1) * 4)) & 15;
    return tile[r * BD + tid];
}

__device__ __forceinline__ void f4_prefetch(const void *p)
{
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}


/*
 * Unstaged kernels (trees whose tables exceed shared memory): fetch what the coming node will read into L1 --
 * the 4x4 matrices of its internal-child edges (one 128-byte line per category, lanes 0..C-1 of each warp)
 * and, per thread, the tip-table rows its own character codes select.
 */
template <int C, int BD, bool PACK, bool WITH_F>
__device__ __forceinline__ void f4_prefetch_tables(const F4Args &a, const F4Child &nc, const unsigned char *tile,
                                                   const double *Pint, const double *Fint, const double *TP, const double *TF,
                                                   int pstride, int tpstride, int tid, int lane)
{
    if (nc.kind == F4_KIND_TIP) {
        const int code = f4_code<BD, PACK>(tile, nc.code_row, tid);
        const double *tp = TP + (nc.mat * a.K + code) * 4;
#pragma unroll
        for (int c = 0; c < C; c++) f4_prefetch(tp + c * tpstride);
        if (WITH_F) {
            const double *tf = TF + (nc.mat * a.K + code) * 4;
#pragma unroll
            for (int c = 0; c < C; c++) f4_prefetch(tf + c * tpstride);
        }
    } else if (lane < C) {
        f4_prefetch(Pint + lane * pstride + nc.mat * 16);
        if (WITH_F) f4_prefetch(Fint + lane * pstride + nc.mat * 16);
    }
}

/* slab accesses: every line is written once and read once, so they are marked streaming (evict-first) and do
 * not displace the tables and prefetched lines in L1 / L2 */
__device__ __forceinline__ double4 f4_slab_ld(const double4 *p)
{
    const double2 *q = reinterpret_cast<const double2 *>(p);
    const double2 a = __ldcs(q), b = __ldcs(q + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void f4_slab_st(double4 *p, double x, double y, double z, double w)
{
    double2 *q = reinterpret_cast<double2 *>(p);
    __stcs(q, make_double2(x, y));
    __stcs(q + 1, make_double2(z, w));
}

/* sums of two values over the warp in one butterfly: sum(a) lands in lanes < 16, sum(b) in lanes >= 16 */
__device__ __forceinline__ double f4_warp_sum2(double a, double b, int lane)
{
    const bool hi = lane >= 16;
    double keep = hi ? b : a, send = hi ? a : b;
    keep += __shfl_xor_sync(0xffffffffu, send, 16);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    return keep;
}

/*
 * Mode 3 (plf_edge_expect_all): adds the warp's sum of the outer product fe (x) lb -- entry 4 i + j = fe_i lb_j -- to the
 * 16 accumulators at row.  A reduce-scatter butterfly halves the live products at every step (16 shuffles instead of
 * 16 x 5) and leaves the sum of entry m = lane >> 1 in lanes lane and lane ^ 1; the even lanes add it.  Every lane
 * stores entry k ^ m at position k (fe and lb permuted by the bits of m), so that at every step the half it keeps is
 * its lower half and the half it sends its upper one: no selects.  Fixed order: the bits do not depend on timing.
 */
__device__ __forceinline__ void f4_gm_add(double *row, const double fe[4], const double lb[4], int lane)
{
    const int m = (lane >> 1) & 15;
    double f[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const double f1 = (m & 4) ? fe[i ^ 1] : fe[i], l1 = (m & 1) ? lb[i ^ 1] : lb[i];
        f[i] = f1; l[i] = l1;
    }
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const double fa = f[i], fb = f[i + 2], la = l[i], lbv = l[i + 2];
        if (m & 8) { f[i] = fb; f[i + 2] = fa; }
        if (m & 2) { l[i] = lbv; l[i + 2] = la; }
    }
    double v[16];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) v[4 * i + j] = f[i] * l[j];
#pragma unroll
    for (int h = 8; h >= 1; h >>= 1)
#pragma unroll
        for (int k = 0; k < h; k++) v[k] += __shfl_xor_sync(0xffffffffu, v[h + k], 2 * h);
    const double sum = v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
    if (!(lane & 1)) row[lane >> 1] += sum;
}

/*
 * Outside step specialised for a node with exactly two children of kinds (K0, K1) in
 * {(CUR, TIP), (CUR, STACK), (TIP, TIP)}: straight-line code, no filler factors.
 */
template <int C, int BD, int K0, int K1, bool PACK, bool CM, bool MARG, bool GM>
__device__ __forceinline__ void f4_outside2(const F4Args &a, const F4Op &op, const F4Child &c0, const F4Child &c1,
                                            bool from_slot, double *cur, const unsigned char *tile, const double *defs_s,
                                            const double *Pint, const double *Fint, const double *TP, const double *TF,
                                            int pstride, int tpstride, size_t T, size_t gtid, int tid,
                                            double &x0, double &x1, double *mgo, double *accG)
{
    double basev[4] = {1.0, 1.0, 1.0, 1.0};
    const bool has_base = op.code_row >= 0;
    if (has_base) f4_ld4(defs_s + f4_code<BD, PACK>(tile, op.code_row, tid) * 4, basev);
    const unsigned int sword_a = a.scratchS[(size_t)op.slot * T + gtid];
    int code0 = 0, code1 = 0, bc0 = 0, bc1 = 0;
    if (K0 == F4_KIND_TIP) code0 = f4_code<BD, PACK>(tile, c0.code_row, tid); else bc0 = (a.scratchS[(size_t)c0.slot * T + gtid] >> 6) & 1;
    if (K1 == F4_KIND_TIP) code1 = f4_code<BD, PACK>(tile, c1.code_row, tid); else bc1 = (a.scratchS[(size_t)c1.slot * T + gtid] >> 6) & 1;
    x0 = 0.0; x1 = 0.0;
    /* marginal mode: posterior state distribution of this node and of its tip children, summed over categories */
    double mg[4] = {0.0, 0.0, 0.0, 0.0}, mt0[4] = {0.0, 0.0, 0.0, 0.0}, mt1[4] = {0.0, 0.0, 0.0, 0.0};
    const int ptstride = a.Et * 16;
    /* (mode 3 walks the categories one at a time: its 16 outer products per edge leave no room for two in flight) */
#pragma unroll ((CM || GM) ? 1 : 2)
    for (int c = 0; c < C; c++) {
        /* loads of this category first */
        double l0[4], l1[4], fa[4];
        if (K0 != F4_KIND_TIP) {
            double4 v = f4_slab_ld(&a.scratch[((size_t)c0.slot * C + c) * T + gtid]);
            l0[0] = v.x; l0[1] = v.y; l0[2] = v.z; l0[3] = v.w;
        }
        if (K1 != F4_KIND_TIP) {
            double4 v = f4_slab_ld(&a.scratch[((size_t)c1.slot * C + c) * T + gtid]);
            l1[0] = v.x; l1[1] = v.y; l1[2] = v.z; l1[3] = v.w;
        }
        if (from_slot) {
            double4 v = f4_slab_ld(&a.scratch[((size_t)op.slot * C + c) * T + gtid]);
            fa[0] = v.x; fa[1] = v.y; fa[2] = v.z; fa[3] = v.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) fa[i] = cur[(c * 4 + i) * BD + tid];
        }
        if (has_base) {
#pragma unroll
            for (int i = 0; i < 4; i++) fa[i] *= basev[i];
        }
        const int sa = (sword_a >> (8 * c)) & 63;
        if (sa) {
            const double sc = __hiloint2double((1023 + PLF_SCALE_BITS * sa) << 20, 0);
#pragma unroll
            for (int i = 0; i < 4; i++) fa[i] *= sc;
        }
        double em0[4], y0[4], em1[4], y1[4];
        if (K0 == F4_KIND_TIP) {
            f4_ld4(TP + c * tpstride + (c0.mat * a.K + code0) * 4, em0);
            if (!MARG && !GM) f4_ld4(TF + c * tpstride + (c0.mat * a.K + code0) * 4, y0);
        } else {
            f4_mv<CM, 0>(Pint, c * pstride + c0.mat * 16, l0, em0);
            if (!MARG && !GM) f4_mv<CM, 1>(Fint, c * pstride + c0.mat * 16, l0, y0);
            if (bc0) {
#pragma unroll
                for (int i = 0; i < 4; i++) { em0[i] = l0[i]; if (!MARG && !GM && a.f_zero_rowsum) y0[i] = 0.0; }
            }
        }
        if (K1 == F4_KIND_TIP) {
            f4_ld4(TP + c * tpstride + (c1.mat * a.K + code1) * 4, em1);
            if (!MARG && !GM) f4_ld4(TF + c * tpstride + (c1.mat * a.K + code1) * 4, y1);
        } else {
            f4_mv<CM, 0>(Pint, c * pstride + c1.mat * 16, l1, em1);
            if (!MARG && !GM) f4_mv<CM, 1>(Fint, c * pstride + c1.mat * 16, l1, y1);
            if (bc1) {
#pragma unroll
                for (int i = 0; i < 4; i++) { em1[i] = l1[i]; if (!MARG && !GM && a.f_zero_rowsum) y1[i] = 0.0; }
            }
        }
        double fe0[4], fe1[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { fe0[i] = fa[i] * em1[i]; fe1[i] = fa[i] * em0[i]; }
        if (GM) {
            /* the child's inside vector: the slab line, or the definition row of a tip's character */
            if (K0 == F4_KIND_TIP) f4_ld4(defs_s + code0 * 4, l0);
            if (K1 == F4_KIND_TIP) f4_ld4(defs_s + code1 * 4, l1);
            f4_gm_add(accG + ((size_t)c * a.E + c0.edge) * 16, fe0, l0, tid & 31);
            f4_gm_add(accG + ((size_t)c * a.E + c1.edge) * 16, fe1, l1, tid & 31);
        } else if (!MARG) {
            double xv = fe0[0] * y0[0];
            xv = fma(fe0[1], y0[1], xv); xv = fma(fe0[2], y0[2], xv); xv = fma(fe0[3], y0[3], xv);
            x0 += xv;
            xv = fe1[0] * y1[0];
            xv = fma(fe1[1], y1[1], xv); xv = fma(fe1[2], y1[2], xv); xv = fma(fe1[3], y1[3], xv);
            x1 += xv;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) mg[i] = fma(fe0[i], em0[i], mg[i]);
            /* a tip's posterior is def .* (P^T fe); Fint holds P of the tip edges in this mode */
            if (K0 == F4_KIND_TIP) {
                double fb[4];
                f4_matvec_t(Fint + c * ptstride + c0.mat * 16, fe0, fb);
#pragma unroll
                for (int i = 0; i < 4; i++) mt0[i] += fb[i];
            }
            if (K1 == F4_KIND_TIP) {
                double fb[4];
                f4_matvec_t(Fint + c * ptstride + c1.mat * 16, fe1, fb);
#pragma unroll
                for (int i = 0; i < 4; i++) mt1[i] += fb[i];
            }
        }
        if (K0 != F4_KIND_TIP) {
            double fb[4];
            f4_mvt<CM>(Pint, c * pstride + c0.mat * 16, fe0, fb);
            if (K0 == F4_KIND_CUR) {
#pragma unroll
                for (int i = 0; i < 4; i++) cur[(c * 4 + i) * BD + tid] = fb[i];
            } else {
                f4_slab_st(&a.scratch[((size_t)c0.slot * C + c) * T + gtid], fb[0], fb[1], fb[2], fb[3]);
            }
        }
        if (K1 != F4_KIND_TIP) {
            double fb[4];
            f4_mvt<CM>(Pint, c * pstride + c1.mat * 16, fe1, fb);
            /* the child's inside vector is dead after this op: its slot carries fn down */
            f4_slab_st(&a.scratch[((size_t)c1.slot * C + c) * T + gtid], fb[0], fb[1], fb[2], fb[3]);
        }
    }
    if (MARG) {
#pragma unroll
        for (int i = 0; i < 4; i++) mgo[i] = mg[i];
        if (K0 == F4_KIND_TIP) {
            double d[4];
            f4_ld4(defs_s + code0 * 4, d);
#pragma unroll
            for (int i = 0; i < 4; i++) mgo[4 + i] = mt0[i] * d[i];
        }
        if (K1 == F4_KIND_TIP) {
            double d[4];
            f4_ld4(defs_s + code1 * 4, d);
#pragma unroll
            for (int i = 0; i < 4; i++) mgo[8 + i] = mt1[i] * d[i];
        }
    }
}

/* marginal mode: one node's four posterior values go to the per-site output or, summed over the warp's
 * sites (they carry the site weight already), to this warp's row of accumulators in global memory */
__device__ __forceinline__ void f4_marg_out(const F4Args &a, double *accM, int node, const double *m, bool valid,
                                            int64_t site, int lane)
{
    if (a.marg_site_out) {
        if (valid) {
#pragma unroll
            for (int i = 0; i < 4; i++) a.marg_site_out[((size_t)node * 4 + i) * a.S + site] = m[i];
        }
    } else {
        const double r01 = f4_warp_sum2(m[0], m[1], lane), r23 = f4_warp_sum2(m[2], m[3], lane);
        if (lane == 0) { accM[node * 4 + 0] += r01; accM[node * 4 + 2] += r23; }
        if (lane == 16) { accM[node * 4 + 1] += r01; accM[node * 4 + 3] += r23; }
    }
}


/* root of one site: likelihood of each category, combined over categories with their scale counts.
 * Kept free of data-dependent branches: with branches here nvcc 12.9 stops treating the op loops of the
 * constant-memory kernels as warp-uniform (tools/check_cm_uniform.sh). */
template <int C, int BD>
__device__ __forceinline__ void f4_root_site(const F4Args &a, const double *cur, int tid, int curf, const double *prior,
                                             const int *ktot, int *kcat, double &site_m, int &site_k, bool &have)
{
    constexpr int bd = BD;
    double vv[C];
#pragma unroll
        for (int c = 0; c < C; c++) {
            double r[4];
#pragma unroll
            for (int i = 0; i < 4; i++) r[i] = cur[(c * 4 + i) * bd + tid];
            double lh;
            if (a.root_mode == PLF_ROOT_NONE) lh = (r[0] + r[1]) + (r[2] + r[3]);
            else if (a.root_mode == PLF_ROOT_UNIFORM) lh = curf ? r[0] : ((r[0] + r[1]) + (r[2] + r[3])) * 0.25;
            else if (a.root_mode == PLF_ROOT_EQUILIBRIUM && curf) lh = r[0];
            else {
                lh = a.root_vec[0] * r[0];
                lh = fma(a.root_vec[1], r[1], lh);
                lh = fma(a.root_vec[2], r[2], lh);
                lh = fma(a.root_vec[3], r[3], lh);
            }
            vv[c] = prior[c] * lh;
            kcat[c] = (vv[c] > 0.0) ? ktot[c] : INT_MIN;
        }
        /* branch-free combination: largest exponent first, then every live category scaled onto it */
        int km = INT_MIN;
#pragma unroll
        for (int c = 0; c < C; c++) km = max(km, kcat[c]);
        have = km != INT_MIN;
        site_k = have ? km : 0;
        site_m = 0.0;
#pragma unroll
        for (int c = 0; c < C; c++) {
            const int dk = (kcat[c] == INT_MIN) ? 0 : kcat[c] - site_k;          /* <= 0 */
            const double sc = (dk < -3) ? 0.0 : __hiloint2double((1023 + PLF_SCALE_BITS * dk) << 20, 0);
            site_m += (kcat[c] == INT_MIN) ? 0.0 : vv[c] * sc;
        }
}

/* values of the kernel's frame that the out-of-line outside step needs */
struct F4Ctx {
    double *cur, *accE, *accM, *accG;
    const unsigned char *tile;
    const double *defs_s, *Pint, *Fint, *TP, *TF;
    const F4Child *chp;
    int pstride, tpstride, tid, lane, warp;
    size_t T, gtid;
    int64_t site;
    bool valid;
};

/*
 * Outside step for a node with any number of children (1..F4_MAXD) of any kind (non-CM kernels only).
 */
template <int C, int BD, bool PACK, bool CM, bool MARG, bool GM>
__device__ __forceinline__ void f4_outside_general(const F4Args &a, const F4Op &op, bool from_slot, const F4Ctx &k)
{
    constexpr int bd = BD;
    double *cur = k.cur, *accE = k.accE, *accM = k.accM, *accG = k.accG;
    const unsigned char *tile = k.tile;
    const double *defs_s = k.defs_s, *Pint = k.Pint, *Fint = k.Fint, *TP = k.TP, *TF = k.TF;
    const F4Child *chp = k.chp;
    const int pstride = k.pstride, tpstride = k.tpstride, tid = k.tid, lane = k.lane, warp = k.warp;
    const size_t T = k.T, gtid = k.gtid;
    const int64_t site = k.site;
    const bool valid = k.valid;
    double basev[4] = {1.0, 1.0, 1.0, 1.0};
    if (op.code_row >= 0) f4_ld4(defs_s + f4_code<BD, PACK>(tile, op.code_row, tid) * 4, basev);
    /* children descriptors and category-independent lookups */
    int kinds[F4_MAXD], mats[F4_MAXD], slots[F4_MAXD], edges[F4_MAXD], codes[F4_MAXD], bcs[F4_MAXD], nodes[F4_MAXD];
    double mg[4] = {0.0, 0.0, 0.0, 0.0}, mt[F4_MAXD][4];
    const int ptstride = a.Et * 16;
#pragma unroll
    for (int j = 0; j < F4_MAXD; j++) {
        kinds[j] = -1; mats[j] = 0; slots[j] = 0; edges[j] = 0; codes[j] = 0; bcs[j] = 0; nodes[j] = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) mt[j][i] = 0.0;
        if (j < op.nchild) {
            const F4Child ch = chp[op.first_child + j];
            kinds[j] = ch.kind; mats[j] = ch.mat; slots[j] = ch.slot; edges[j] = ch.edge; nodes[j] = ch.node;
            if (ch.kind == F4_KIND_TIP) codes[j] = f4_code<BD, PACK>(tile, ch.code_row, tid);
            else bcs[j] = (a.scratchS[(size_t)ch.slot * T + gtid] >> 6) & 1;
        }
    }
    double x[F4_MAXD] = {0.0, 0.0, 0.0};
    const unsigned int sword_a = a.scratchS[(size_t)op.slot * T + gtid];
#pragma unroll 1
    for (int c = 0; c < C; c++) {
        double fa[4];
        const size_t so_a = ((size_t)op.slot * C + c) * T + gtid;
        if (from_slot) {
            double4 f4v = f4_slab_ld(&a.scratch[so_a]);
            fa[0] = f4v.x; fa[1] = f4v.y; fa[2] = f4v.z; fa[3] = f4v.w;
        } else {
#pragma unroll
            for (int i = 0; i < 4; i++) fa[i] = cur[(c * 4 + i) * bd + tid];
        }
        const int sa = (sword_a >> (8 * c)) & 63;
#pragma unroll
        for (int i = 0; i < 4; i++) fa[i] *= basev[i];
        if (sa) {
            const double sc = __hiloint2double((1023 + PLF_SCALE_BITS * sa) << 20, 0);
#pragma unroll
            for (int i = 0; i < 4; i++) fa[i] *= sc;
        }
        double em[F4_MAXD][4], y[F4_MAXD][4];
#pragma unroll
        for (int j = 0; j < F4_MAXD; j++) {
#pragma unroll
            for (int i = 0; i < 4; i++) { em[j][i] = 1.0; y[j][i] = 0.0; }
            if (kinds[j] == F4_KIND_TIP) {
                f4_ld4(TP + c * tpstride + (mats[j] * a.K + codes[j]) * 4, em[j]);
                if (!MARG && !GM) f4_ld4(TF + c * tpstride + (mats[j] * a.K + codes[j]) * 4, y[j]);
            } else if (kinds[j] >= 0) {
                double4 l4 = f4_slab_ld(&a.scratch[((size_t)slots[j] * C + c) * T + gtid]);
                double lv[4] = {l4.x, l4.y, l4.z, l4.w};
                if (bcs[j]) {
#pragma unroll
                    for (int i = 0; i < 4; i++) em[j][i] = lv[i];
                } else {
                    f4_mv<CM, 0>(Pint, c * pstride + mats[j] * 16, lv, em[j]);
                }
                if (!MARG && !GM && !(bcs[j] && a.f_zero_rowsum)) f4_mv<CM, 1>(Fint, c * pstride + mats[j] * 16, lv, y[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < F4_MAXD; j++) {
            if (kinds[j] >= 0) {
                double fe[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    double f = fa[i];
#pragma unroll
                    for (int j2 = 0; j2 < F4_MAXD; j2++) if (j2 != j) f *= em[j2][i];
                    fe[i] = f;
                }
                if (GM) {
                    /* the child's inside vector, read again (its slot is rewritten below): fewer live registers */
                    double lb[4];
                    if (kinds[j] == F4_KIND_TIP) {
                        f4_ld4(defs_s + codes[j] * 4, lb);
                    } else {
                        const double4 l4 = f4_slab_ld(&a.scratch[((size_t)slots[j] * C + c) * T + gtid]);
                        lb[0] = l4.x; lb[1] = l4.y; lb[2] = l4.z; lb[3] = l4.w;
                    }
                    f4_gm_add(accG + ((size_t)c * a.E + edges[j]) * 16, fe, lb, lane);
                } else if (!MARG) {
                    double xv = fe[0] * y[j][0];
                    xv = fma(fe[1], y[j][1], xv);
                    xv = fma(fe[2], y[j][2], xv);
                    xv = fma(fe[3], y[j][3], xv);
                    x[j] += xv;
                } else {
                    if (j == 0) {
#pragma unroll
                        for (int i = 0; i < 4; i++) mg[i] = fma(fe[i], em[0][i], mg[i]);
                    }
                    if (kinds[j] == F4_KIND_TIP) {
                        double fb[4];
                        f4_matvec_t(Fint + c * ptstride + mats[j] * 16, fe, fb);
#pragma unroll
                        for (int i = 0; i < 4; i++) mt[j][i] += fb[i];
                    }
                }
                if (kinds[j] != F4_KIND_TIP) {
                    double fb[4];
                    f4_mvt<CM>(Pint, c * pstride + mats[j] * 16, fe, fb);
                    if (kinds[j] == F4_KIND_CUR) {
#pragma unroll
                        for (int i = 0; i < 4; i++) cur[(c * 4 + i) * bd + tid] = fb[i];
                    } else {
                        /* the child's inside vector is dead after this op: its slot carries fn down */
                        f4_slab_st(&a.scratch[((size_t)slots[j] * C + c) * T + gtid], fb[0], fb[1], fb[2], fb[3]);
                    }
                }
            }
        }
    }
    if (MARG) {
        f4_marg_out(a, accM, op.node, mg, valid, site, lane);
#pragma unroll
        for (int j = 0; j < F4_MAXD; j++) {
            if (kinds[j] == F4_KIND_TIP) {
                double d[4];
                f4_ld4(defs_s + codes[j] * 4, d);
#pragma unroll
                for (int i = 0; i < 4; i++) d[i] *= mt[j][i];
                f4_marg_out(a, accM, nodes[j], d, valid, site, lane);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < ((MARG || GM) ? 0 : F4_MAXD); j++) {
        if (kinds[j] >= 0) {
            const int e = edges[j];
            const bool me = !a.edge_mask || a.edge_mask[e];
            if (a.edge_site_out) {
                if (valid && me) a.edge_site_out[(size_t)e * a.S + site] = x[j];
            } else {
                double xs = f4_warp_sum(x[j]);
                if (lane == 0 && me) accE[warp * a.E + e] += xs;
            }
        }
    }
}

/*
 * C     : number of rate categories (1..4)
 * MODE  : 0 = log-likelihood only; 1 = log-likelihood + per-edge bilinear forms (deriv / dwell / trans);
 *         2 = log-likelihood + posterior marginals of every node;
 *         3 = log-likelihood + the matrices G_{e,c} = sum_s fe (x) L_b of every edge and category (plf_edge_expect_all):
 *             the outside pass of mode 2, with the outer products summed per warp into block_gmat
 * The dynamic shared memory layout below is mirrored on the host by f4_smem_bytes().
 */
/* STAGED: 2 = all tables in shared memory, 1 = all but TF (read through L1), 0 = none.
 * PACK: the tile's character codes are stored two per byte (needs K <= 16).
 * CM: internal-edge matrices in constant memory and the program in `prog` (see above); STAGED then
 *     only concerns the tip tables. */
template <int C, int MODE, int BD, int STAGED, bool PACK, bool CM>
__global__ void __launch_bounds__(BD) fused4_kernel(const F4Args a, const __grid_constant__ F4Prog prog)
{
    constexpr bool EDGE = MODE != 0;     /* an outside pass runs */
    constexpr bool MARG = MODE == 2;     /* ... and produces node marginals instead of per-edge forms */
    constexpr bool GM = MODE == 3;       /* ... or the per-edge outer-product matrices (no edge-form tables) */
    extern __shared__ __align__(16) unsigned char f4_smem[];
    const int tid = threadIdx.x;
    constexpr int bd = BD;
    const int lane = tid & 31, warp = tid >> 5;
    constexpr int nwarp = BD >> 5;
    const int64_t T = (int64_t)gridDim.x * bd;
    const int64_t gtid = (int64_t)blockIdx.x * bd + tid;

    /* pointers inside the argument struct are not assumed to be global memory by default */






    /* ---- carve shared memory ---- */
    size_t off = 0;
    F4Op *ops_s = reinterpret_cast<F4Op *>(f4_smem + off); off = f4_align16(off + (CM ? 0 : sizeof(F4Op) * a.nops));
    F4Child *chs_s = reinterpret_cast<F4Child *>(f4_smem + off); off = f4_align16(off + (CM ? 0 : sizeof(F4Child) * a.nchildren));
#define F4_OP(i) (CM ? prog.ops[i] : ops_s[i])
#define F4_CH(i) (CM ? prog.ch[i] : chs_s[i])
    double *cur = reinterpret_cast<double *>(f4_smem + off); off = f4_align16(off + sizeof(double) * 4 * C * bd);   /* [C][4][bd] */
    double *accE = reinterpret_cast<double *>(f4_smem + off); off = f4_align16(off + ((EDGE && !MARG && !GM) ? sizeof(double) * nwarp * a.E : 0));
    double *stack = reinterpret_cast<double *>(f4_smem + off); off = f4_align16(off + (EDGE ? 0 : sizeof(double) * 4 * C * bd * a.stack_depth));
    int *stackf = reinterpret_cast<int *>(f4_smem + off); off = f4_align16(off + (EDGE ? 0 : sizeof(int) * bd * a.stack_depth));
    unsigned char *tile = f4_smem + off; off = f4_align16(off + (size_t)(PACK ? (a.ncode_rows + 1) / 2 : a.ncode_rows) * bd);
    unsigned char *dconst = f4_smem + off; off = f4_align16(off + a.K);
    double *defs_s = reinterpret_cast<double *>(f4_smem + off); off = f4_align16(off + sizeof(double) * 4 * a.K);
    const double *Pint = a.Pint, *TP = a.TP, *Fint = a.Fint, *TF = a.TF;
    if (STAGED) {
        const size_t nP = CM ? 0 : (size_t)C * a.Ei * 16, nT = (size_t)C * a.Et * a.K * 4;
        const size_t nF = MARG ? (size_t)C * a.Et * 16 : nP;       /* marginal mode: P of the tip edges */
        double *sP = reinterpret_cast<double *>(f4_smem + off); off += sizeof(double) * nP;
        double *sT = reinterpret_cast<double *>(f4_smem + off); off += sizeof(double) * nT;
        double *sF = reinterpret_cast<double *>(f4_smem + off); off += (EDGE && !GM) ? sizeof(double) * nF : 0;
        double *sTF = reinterpret_cast<double *>(f4_smem + off); off += (EDGE && !MARG && !GM && STAGED == 2) ? sizeof(double) * nT : 0;
        /* (counts as int: a compile-time zero count would make the loop test an unsigned comparison with 0) */
        for (int i = tid; i < (int)nP; i += bd) sP[i] = a.Pint[i];
        for (int i = tid; i < ((EDGE && !GM) ? (int)nF : 0); i += bd) sF[i] = a.Fint[i];
        for (size_t i = tid; i < nT; i += bd) { sT[i] = a.TP[i]; if (EDGE && !MARG && !GM && STAGED == 2) sTF[i] = a.TF[i]; }
        Pint = sP; TP = sT; Fint = sF;
        if (STAGED == 2 && !MARG && !GM) TF = sTF;
    }
    if (!CM) {
        for (int i = tid; i < a.nops; i += bd) ops_s[i] = a.ops[i];
        for (int i = tid; i < a.nchildren; i += bd) chs_s[i] = a.children[i];
    }
    for (int i = tid; i < a.K; i += bd) dconst[i] = a.def_const[i];
    for (int i = tid; i < 4 * a.K; i += bd) defs_s[i] = a.defs[i];
    if (EDGE && !MARG && !GM) for (int i = tid; i < nwarp * a.E; i += bd) accE[i] = 0.0;
    double *accM = MARG ? a.block_marg + ((size_t)blockIdx.x * nwarp + warp) * ((size_t)a.N * 4) : nullptr;
    double *accG = GM ? a.block_gmat + ((size_t)blockIdx.x * nwarp + warp) * ((size_t)C * a.E * 16) : nullptr;
    __syncthreads();

    const int tpstride = a.Et * a.K * 4;     /* doubles per category in the tip tables */
    const int pstride = a.Ei * 16;
    double prior[C];
#pragma unroll
    for (int c = 0; c < C; c++) prior[c] = a.cat_prior[c];

    double ll_acc = 0.0;
    /* Every CTA owns one contiguous block of sites, the same number (a multiple of the warp size) for all of them, and
     * walks it in steps of bd; warps whose 32 sites lie beyond the block skip the step.  A launch whose sites are not
     * a whole number of waves (a shard of a strong-scaling run) then costs its share of sites per SM, not a whole
     * extra wave on some of the SMs. */
    const int64_t per_cta = (((a.s_end - a.s_begin) + gridDim.x - 1) / gridDim.x + 31) / 32 * 32;
    const int64_t blk0 = a.s_begin + (int64_t)blockIdx.x * per_cta;
    const int64_t blk1 = (blk0 + per_cta < a.s_end) ? blk0 + per_cta : a.s_end;

    for (int64_t s0 = blk0; s0 < blk1; s0 += bd) {
        const int64_t site_raw = s0 + tid;
        const bool valid = site_raw < blk1;
        /* (a vote, so that the compiler still sees warp-uniform control flow: the constant-memory kernels depend on it) */
        if (!__any_sync(0xffffffffu, valid)) continue;
        const int64_t site = valid ? site_raw : blk1 - 1;
        const double w = valid ? (a.site_w ? a.site_w[site] : 1.0) : 0.0;
        /* stage this tile's character codes: each thread only ever reads its own column */
        if (PACK) {
            for (int r = 0; r < a.ncode_rows; r += 2) {
                unsigned int lo = a.codes[(size_t)a.code_row_node[r] * a.S + site];
                unsigned int hi = (r + 1 < a.ncode_rows) ? a.codes[(size_t)a.code_row_node[r + 1] * a.S + site] : 0u;
                tile[(r >> 1) * bd + tid] = (unsigned char)(lo | (hi << 4));
            }
        } else {
            for (int r = 0; r < a.ncode_rows; r++)
                tile[r * bd + tid] = a.codes[(size_t)a.code_row_node[r] * a.S + site];
        }

        /* ---------------- inside pass (all categories together) ---------------- */
        int curf = 1, sp = 0;
        int ktot[C];
#pragma unroll
        for (int c = 0; c < C; c++) ktot[c] = 0;
#pragma unroll 1
        for (int o = 0; o < a.nops; o++) {
            const F4Op op = F4_OP(o);
            if (STAGED == 0 && !CM && o + 1 < a.nops) {
                const F4Op nx = F4_OP(o + 1);
                for (int j = 0; j < nx.nchild; j++)
                    f4_prefetch_tables<C, BD, PACK, false>(a, F4_CH(nx.first_child + j), tile, Pint, Fint, TP, TF, pstride, tpstride, tid, lane);
            }
            if (!EDGE && op.spill_before) {
                if (a.gstack) {
                    /* a few hundred bytes per thread that come back within the tile: they stay in L2 */
#pragma unroll
                    for (int c = 0; c < C; c++)
                        a.scratch[((size_t)sp * C + c) * T + gtid] =
                            make_double4(cur[(c * 4 + 0) * bd + tid], cur[(c * 4 + 1) * bd + tid],
                                         cur[(c * 4 + 2) * bd + tid], cur[(c * 4 + 3) * bd + tid]);
                    a.scratchS[(size_t)sp * T + gtid] = (unsigned int)curf;
                } else {
#pragma unroll
                    for (int c = 0; c < C; c++)
#pragma unroll
                        for (int i = 0; i < 4; i++) stack[((sp * C + c) * 4 + i) * bd + tid] = cur[(c * 4 + i) * bd + tid];
                    stackf[sp * bd + tid] = curf;
                }
                sp++;
            }
            double acc[C][4];
            int cst = 1;
            bool first = true;
            if (op.code_row >= 0) {
                const int code = f4_code<BD, PACK>(tile, op.code_row, tid);
                double b[4];
                f4_ld4(defs_s + code * 4, b);
#pragma unroll
                for (int c = 0; c < C; c++)
#pragma unroll
                    for (int i = 0; i < 4; i++) acc[c][i] = b[i];
                cst = dconst[code];
                first = false;
            }
#pragma unroll 1
            for (int j = 0; j < op.nchild; j++) {
                const F4Child ch = F4_CH(op.first_child + j);
                double em[C][4];
                int bc;
                if (ch.kind == F4_KIND_TIP) {
                    const int code = f4_code<BD, PACK>(tile, ch.code_row, tid);
                    bc = dconst[code];
                    const double *tp = TP + (ch.mat * a.K + code) * 4;
#pragma unroll
                    for (int c = 0; c < C; c++) f4_ld4(tp + c * tpstride, em[c]);
                } else {
                    double v[C][4];
                    if (ch.kind == F4_KIND_CUR) {
                        bc = curf;
#pragma unroll
                        for (int c = 0; c < C; c++)
#pragma unroll
                            for (int i = 0; i < 4; i++) v[c][i] = cur[(c * 4 + i) * bd + tid];
                    } else if (EDGE) {
                        const size_t so = ((size_t)ch.slot * C) * T + gtid;
                        bc = (a.scratchS[(size_t)ch.slot * T + gtid] >> 6) & 1;
#pragma unroll
                        for (int c = 0; c < C; c++) {
                            double4 l4 = f4_slab_ld(&a.scratch[so + (size_t)c * T]);
                            v[c][0] = l4.x; v[c][1] = l4.y; v[c][2] = l4.z; v[c][3] = l4.w;
                        }
                    } else {
                        sp--;
                        if (a.gstack) {
                            bc = (int)a.scratchS[(size_t)sp * T + gtid];
#pragma unroll
                            for (int c = 0; c < C; c++) {
                                const double4 l4 = a.scratch[((size_t)sp * C + c) * T + gtid];
                                v[c][0] = l4.x; v[c][1] = l4.y; v[c][2] = l4.z; v[c][3] = l4.w;
                            }
                        } else {
                            bc = stackf[sp * bd + tid];
#pragma unroll
                            for (int c = 0; c < C; c++)
#pragma unroll
                                for (int i = 0; i < 4; i++) v[c][i] = stack[((sp * C + c) * 4 + i) * bd + tid];
                        }
                    }
                    if (bc) {
#pragma unroll
                        for (int c = 0; c < C; c++)
#pragma unroll
                            for (int i = 0; i < 4; i++) em[c][i] = v[c][i];
                    } else {
#pragma unroll
                        for (int c = 0; c < C; c++) f4_mv<CM, 0>(Pint, ch.mat * 16 + c * pstride, v[c], em[c]);
                    }
                }
                if (first) {
#pragma unroll
                    for (int c = 0; c < C; c++)
#pragma unroll
                        for (int i = 0; i < 4; i++) acc[c][i] = em[c][i];
                    first = false;
                } else {
#pragma unroll
                    for (int c = 0; c < C; c++)
#pragma unroll
                        for (int i = 0; i < 4; i++) acc[c][i] *= em[c][i];
                }
                cst &= bc;
            }
            /* one rescale check per node is enough for out-degree <= 3 (each factor has max >= 2^-256 p_min) */
            unsigned int sword = 0;
#pragma unroll
            for (int c = 0; c < C; c++) {
                const int sloc = f4_rescale_up(acc[c]);
                ktot[c] -= sloc;
                sword |= (unsigned int)(sloc | (cst << 6)) << (8 * c);
#pragma unroll
                for (int i = 0; i < 4; i++) cur[(c * 4 + i) * bd + tid] = acc[c][i];
                if (EDGE) {
                    const size_t so = ((size_t)op.slot * C + c) * T + gtid;
                    f4_slab_st(&a.scratch[so], acc[c][0], acc[c][1], acc[c][2], acc[c][3]);
                }
            }
            if (EDGE) a.scratchS[(size_t)op.slot * T + gtid] = sword;
            curf = cst;
        }
        /* ---------------- root: site likelihood (model.c:282-350, arbplfll.c:149-169) ---------------- */
        double site_m = 0.0;
        int site_k = 0;
        bool have = false;
        int kcat[C];
        f4_root_site<C, BD>(a, cur, tid, curf, prior, ktot, kcat, site_m, site_k, have);
        {
            const double c_hi = 177.445678223346, c_lo = 5.936759843446527e-15;   /* 256 ln 2 */
            double ll = log(site_m);
            if (site_k != 0) { ll = fma((double)site_k, c_hi, ll); ll = fma((double)site_k, c_lo, ll); }
            if (valid) {
                if (a.site_ll) a.site_ll[site] = ll;
                if (w != 0.0) {
                    if (!have) atomicOr(a.error_flag, 1);
                    else ll_acc = fma(w, ll, ll_acc);
                }
            }
        }
        if (!EDGE) continue;

        /* ---------------- outside pass ---------------- */
        const bool per_site_out = MARG ? (a.marg_site_out != nullptr) : (a.edge_site_out != nullptr);
        const double inv_site = (have && w != 0.0) ? (per_site_out ? 1.0 : w) / site_m : 0.0;
        /* fn_root = root prior vector * prior_c * w / site_L, scaled so that fn .* L is O(1) */
#pragma unroll
        for (int c = 0; c < C; c++) {
            const int kc = kcat[c];
            const double sc0 = (kc != INT_MIN) ? scalbn(prior[c] * inv_site, PLF_SCALE_BITS * (kc - site_k)) : 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                double r = 1.0;
                if (a.root_mode == PLF_ROOT_UNIFORM) r = 0.25;
                else if (a.root_mode == PLF_ROOT_EQUILIBRIUM || a.root_mode == PLF_ROOT_CUSTOM) r = a.root_vec[i];
                cur[(c * 4 + i) * bd + tid] = r * sc0;
            }
        }
#pragma unroll 1
        for (int o = a.nops - 1; o >= 0; o--) {
            const F4Op op = F4_OP(o);
            /* fn_a comes from "cur" if this node was consumed from registers by its parent, else from its slot */
            const bool from_slot = (o != a.nops - 1) && F4_OP(o + 1).spill_before;
            /* the next node (o-1) reads these slab lines: start fetching them.  That includes the scale words of the
             * node and of its internal children and, when this op does not consume the node (spill_before), the fn its
             * parent left in its slot: they head the dependent chain of its step (the scale of fa, fa itself, the
             * constant-column flags), and without the prefetch each is a full L2 / DRAM round trip at its start. */
            if (o > 0) {
                const F4Op nx = F4_OP(o - 1);
                f4_prefetch(&a.scratchS[(size_t)nx.slot * T + gtid]);
                if (op.spill_before) {
#pragma unroll
                    for (int c = 0; c < C; c++) f4_prefetch(&a.scratch[((size_t)nx.slot * C + c) * T + gtid]);
                }
                for (int j = 0; j < nx.nchild; j++) {
                    const F4Child nc = F4_CH(nx.first_child + j);
                    if (nc.kind != F4_KIND_TIP) {
                        f4_prefetch(&a.scratchS[(size_t)nc.slot * T + gtid]);
#pragma unroll
                        for (int c = 0; c < C; c++) f4_prefetch(&a.scratch[((size_t)nc.slot * C + c) * T + gtid]);
                    }
                    if (STAGED == 0 && !CM)
                        f4_prefetch_tables<C, BD, PACK, !MARG && !GM>(a, nc, tile, Pint, Fint, TP, TF, pstride, tpstride, tid, lane);
                }
            }
            if (op.nchild == 2) {
                const F4Child c0 = F4_CH(op.first_child), c1 = F4_CH(op.first_child + 1);
                double x0, x1, mgo[12];
                if (c0.kind == F4_KIND_CUR && c1.kind == F4_KIND_TIP)
                    f4_outside2<C, BD, F4_KIND_CUR, F4_KIND_TIP, PACK, CM, MARG, GM>(a, op, c0, c1, from_slot, cur, tile, defs_s, Pint, Fint, TP, TF,
                                                                 pstride, tpstride, (size_t)T, (size_t)gtid, tid, x0, x1, mgo, accG);
                else if (c0.kind == F4_KIND_CUR)
                    f4_outside2<C, BD, F4_KIND_CUR, F4_KIND_STACK, PACK, CM, MARG, GM>(a, op, c0, c1, from_slot, cur, tile, defs_s, Pint, Fint, TP, TF,
                                                                   pstride, tpstride, (size_t)T, (size_t)gtid, tid, x0, x1, mgo, accG);
                else
                    f4_outside2<C, BD, F4_KIND_TIP, F4_KIND_TIP, PACK, CM, MARG, GM>(a, op, c0, c1, from_slot, cur, tile, defs_s, Pint, Fint, TP, TF,
                                                                 pstride, tpstride, (size_t)T, (size_t)gtid, tid, x0, x1, mgo, accG);
                if (MARG) {
                    f4_marg_out(a, accM, op.node, mgo, valid, site, lane);
                    if (c0.kind == F4_KIND_TIP) f4_marg_out(a, accM, c0.node, mgo + 4, valid, site, lane);
                    if (c1.kind == F4_KIND_TIP) f4_marg_out(a, accM, c1.node, mgo + 8, valid, site, lane);
                    continue;
                }
                if (GM) continue;
                const bool m0 = !a.edge_mask || a.edge_mask[c0.edge];
                const bool m1 = !a.edge_mask || a.edge_mask[c1.edge];
                if (a.edge_site_out) {
                    if (valid && m0) a.edge_site_out[(size_t)c0.edge * a.S + site] = x0;
                    if (valid && m1) a.edge_site_out[(size_t)c1.edge * a.S + site] = x1;
                } else {
                    /* the butterfly runs unconditionally: a shuffle under a condition the compiler cannot prove
                     * warp-uniform (the mask comes from memory) makes it treat the whole op loop as divergent */
                    const double r = f4_warp_sum2(m0 ? x0 : 0.0, m1 ? x1 : 0.0, lane);
                    if (lane == 0 && m0) accE[warp * a.E + c0.edge] += r;
                    if (lane == 16 && m1) accE[warp * a.E + c1.edge] += r;
                }
                continue;
            }
            if (!CM) {      /* the host selects a CM kernel only for programs made of two-children nodes */
                F4Ctx k;
                k.cur = cur; k.accE = accE; k.accM = accM; k.accG = accG; k.tile = tile; k.defs_s = defs_s; k.Pint = Pint; k.Fint = Fint; k.TP = TP; k.TF = TF;
                k.chp = CM ? prog.ch : chs_s;
                k.pstride = pstride; k.tpstride = tpstride; k.tid = tid; k.lane = lane; k.warp = warp;
                k.T = (size_t)T; k.gtid = (size_t)gtid; k.site = site; k.valid = valid;
                f4_outside_general<C, BD, PACK, CM, MARG, GM>(a, op, from_slot, k);
            }
        }
    }

    /* ---------------- CTA-level reductions ---------------- */
    {
        __shared__ double red[32];
        double xx = f4_warp_sum(ll_acc);
        if (lane == 0) red[warp] = xx;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int i = 0; i < nwarp; i++) s += red[i];
            a.block_ll[blockIdx.x] = s;
        }
        if (EDGE && !MARG && !GM && !a.edge_site_out) {
            for (int e = tid; e < a.E; e += bd) {
                double s = 0.0;
                for (int wv = 0; wv < nwarp; wv++) s += accE[wv * a.E + e];
                a.block_edge[(size_t)blockIdx.x * a.E + e] = s;
            }
        }
    }
}

