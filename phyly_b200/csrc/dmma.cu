/*
 * Pruning (inside) and outside passes for large state spaces (16 < n <= 64: amino-acid, codon)
 * on the FP64 tensor pipe, second generation.
 *
 * Reference loops being replaced: evaluate_site_lhood (evaluate_site_lhood.c:21-57) with
 * _prune_update_prob / _arb_mat_mul_stochastic (util.c:241-301, arb_mat_extras.c:54-113),
 * evaluate_site_forward (evaluate_site_forward.c:31-105) and evaluate_site_frechet
 * (evaluate_site_frechet.c:4-42) inside the site x category loops of arbplfll.c:139-170 and
 * arbplfderiv.c:274-357.
 *
 * Orientation.  The per-edge contraction em = P_e L_b is issued as mma.sync.m8n8k4.f64 with the
 * SITES as the M rows, the child's states as K and the parent's states as N:
 *
 *      em^T [8 sites x 8NB states] = L_b^T [8 sites x 8NB states] . P_e^T [8NB x 8NB]
 *
 * In the m8n8k4 fragment layout thread (g = lane/4, q = lane%4) of a warp holds, of an
 * accumulator block nb, the entries (site g, states 8nb+2q, 8nb+2q+1) -- and of an A block the
 * entry (site g, k-slot q).  With the k-slots of step kk mapped to the states
 * kappa(kk, q) = 8 (kk/2) + 2q + (kk%2), the accumulator registers of one contraction ARE the
 * A operand of the next one: a node's partial never leaves the registers of its warp on the way
 * to its parent, there is no shared-memory transposition and no block-wide barrier anywhere in
 * the data path.  A warp owns 8 site patterns for the whole tree walk; per-site bookkeeping
 * (scale exponent, constant-column flag, column maximum) is a 4-lane affair.
 *
 * The B operand (P_e^T, identical for every site) is packed once per model into the fragment
 * order (dm_pack_kernel) and streamed through a ring of shared-memory slots with bulk async
 * copies (cp.async.bulk + mbarrier): the warp that is last to finish a slot refills it with the
 * matrix R contractions ahead, so warps drift apart by up to R edges and the copy engine runs
 * ahead of the tensor pipe.  Tip children never enter a contraction: P_e def_k comes from a tip
 * table stored in the same per-thread order (NB 16-byte loads).  The tree is walked in the
 * post-order program of the fused 4-state kernel (Sethi-Ullman order): the newest partial stays
 * in registers, pending ones go to a small per-warp stack in global memory (L2 resident).
 *
 * The outside pass (dm_outside_kernel) runs the same program backwards.  For an internal-child
 * edge e = (a, b) it forms fe = fn_a . data_a . prod_{b' != b} em_b' in registers and contracts
 * it with two packed matrices: fn_b = P_e^T fe and z_b = F_e^T fe (F = rate Q P for derivatives,
 * a Frechet block for dwell / trans).  The edge value x_e = z_b . L_b is taken when the walk
 * reaches b, where L_b is rebuilt from the children's edge vectors the step loads anyway.
 *
 * Work per (site, internal-child edge): 2 (8NB)^2 flops on the padded state count per
 * contraction (one in the inside pass, two in the outside pass); HBM traffic in ll-only mode is
 * the character codes (1 byte per site and tip) -- partials never leave the SM.  In keep mode
 * every internal-child edge vector is also written once to a slab, in register order.
 */
#include <stdint.h>
#include <limits.h>
#include "dmma.h"

#define DM_TWO_P256 1.157920892373162e+77      /* 2^256  */
#define DM_TWO_M256 8.636168555094445e-78      /* 2^-256 */
#define DM_HI_M256 0x2FF00000                  /* high word of 2^-256 */
#define DM_HI_P256 0x4FF00000                  /* high word of 2^256  */

__device__ __forceinline__ void dm_dmma(double &d0, double &d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__device__ __forceinline__ unsigned dm_smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void dm_mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(dm_smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void dm_mbar_expect(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(dm_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void dm_mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "DM_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DM_DONE_%=;\n"
        "bra DM_WAIT_%=;\n"
        "DM_DONE_%=:\n"
        "}\n" ::"r"(dm_smem_addr(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void dm_bulk_load(void *dst, const void *src, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dm_smem_addr(dst)), "l"(src), "r"(bytes), "r"(dm_smem_addr(bar)) : "memory");
}

/* doubles per packed matrix: 2NB k-steps x ceil(NB/2) pairs of n-blocks x 32 lanes x 2 */
__host__ __device__ constexpr int dm_slot_doubles(int NB) { return 2 * NB * ((NB + 1) / 2) * 64; }

/*
 * Pack matrices into the B-fragment order.  dst[(m * 2NB + kk) * NBP + nbp][lane][j] with lane = 4g + q is
 *   transpose == 0:  M[out = 8 (2 nbp + j) + g][in = kappa(kk, q)]      (em = M L:      B = M^T)
 *   transpose == 1:  M[out' = kappa(kk, q)][in' = 8 (2 nbp + j) + g]    (fn = M^T fe:   B = M)
 * src_index[m] = position of the matrix in src ([C][E][n][n], the category offset is added here);
 * a negative index -(k+1) takes matrix k of src2 instead (the edge-form matrices of the outside pass).
 */
__global__ void dm_pack_kernel(const double *src, const double *src2, const int *src_index, const int *transpose, int nmat,
                               int C, int E, int n, int NB, double *dst)
{
    const int NBP = (NB + 1) / 2;
    const int per = dm_slot_doubles(NB);
    const size_t total = (size_t)C * nmat * per;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(i % per);
        const size_t mi = i / per;
        const int m = (int)(mi % nmat), c = (int)(mi / nmat);
        const int j = r & 1, lane = (r >> 1) & 31, rest = r >> 6;
        const int nbp = rest % NBP, kk = rest / NBP;
        const int g = lane >> 2, q = lane & 3;
        const int kap = 8 * (kk >> 1) + 2 * q + (kk & 1);
        const int col = 8 * (2 * nbp + j) + g;
        int idx = src_index[m];
        const double *M = src;
        if (idx < 0) { idx = -idx - 1; M = src2; }
        M += ((size_t)c * E + idx) * n * n;
        double v = 0.0;
        if (kap < n && col < n && 2 * nbp + j < NB) v = (transpose && transpose[m]) ? M[(size_t)kap * n + col] : M[(size_t)col * n + kap];
        dst[i] = v;
    }
}

/* tip tables in thread order: out[((c Et + te) K + k) 8NB + pos], pos = q 2NB + 2 nb + h <-> state 8nb + 2q + h.
 * mode as in tip_table_kernel (0: stochastic matrix, 1: zero row sums, 2: no shortcut);
 * M == NULL writes the definitions themselves (c and te ignored by the caller: C = Et = 1). */
__global__ void dm_tip_table_kernel(const double *M, const double *defs, const unsigned char *def_const,
                                    const int *edge_of_tip, int C, int E, int Et, int K, int n, int NB, int mode, double *out)
{
    const int W = 8 * NB;
    const size_t total = (size_t)C * Et * K * W;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int pos = (int)(idx % W);
    size_t r = idx / W;
    const int k = (int)(r % K); r /= K;
    const int te = (int)(r % Et), c = (int)(r / Et);
    const int q = pos / (2 * NB), rem = pos % (2 * NB);
    const int i = 8 * (rem >> 1) + 2 * q + (rem & 1);
    double v = 0.0;
    if (i < n) {
        const double *d = defs + (size_t)k * n;
        if (!M) v = d[i];
        else if (def_const[k] && mode == 0) v = d[0];
        else if (def_const[k] && mode == 1) v = 0.0;
        else {
            const double *row = M + (((size_t)c * E + edge_of_tip[te]) * n + i) * n;
            for (int j = 0; j < n; j++) v = fma(row[j], d[j], v);
        }
    }
    out[idx] = v;
}

/* four n-blocks (two packed pairs, chunk pc) of one contraction for the 8 sites of a warp:
 * em[i][h] = sum_k A[k] B[k][8 (4 pc + i) + ...]; every B fragment read from shared memory feeds 2 DMMAs */
template <int NB>
__device__ __forceinline__ void dm_gemm_chunk(const double (&A)[2 * NB], const double2 *sl, int pc, double (&em)[4][2])
{
    constexpr int NBP = (NB + 1) / 2;
#pragma unroll
    for (int i = 0; i < 4; i++) { em[i][0] = 0.0; em[i][1] = 0.0; }
#pragma unroll
    for (int kk = 0; kk < 2 * NB; kk++) {
#pragma unroll
        for (int p = 0; p < 2; p++) {
            const int nbp = 2 * pc + p;
            if (nbp < NBP) {
                const double2 b = sl[(kk * NBP + nbp) * 32];
                dm_dmma(em[2 * p][0], em[2 * p][1], A[kk], b.x);
                if (2 * nbp + 1 < NB) dm_dmma(em[2 * p + 1][0], em[2 * p + 1][1], A[kk], b.y);
            }
        }
    }
}

/* The ring of packed matrices.  Contraction number G of this CTA uses slot G % R in phase (G / R) & 1. */
template <int NB>
struct DmRing {
    static constexpr int SLOT = dm_slot_doubles(NB);
    double *slots;          /* [R][SLOT] */
    uint64_t *full;         /* [R] */
    int *done;              /* [R] warps that have finished the slot's current matrix */
    const double *src;      /* packed matrices [C][nmat][SLOT] */
    int nmat, C, R;
    int cat_inner;          /* 0: sequence number -> item -> category = item % C;  1: category = sequence % C */
    long long total;        /* contractions this CTA will run */

    __device__ __forceinline__ const double *source(long long G) const
    {
        const long long seq = G / nmat;
        const int c = cat_inner ? (int)(seq % C) : (int)(((long long)blockIdx.x + seq * gridDim.x) % C);
        return src + ((size_t)c * nmat + (size_t)(G % nmat)) * SLOT;
    }
    __device__ __forceinline__ void issue(long long G)
    {
        const int s = (int)(G % R);
        dm_mbar_expect(&full[s], SLOT * 8);
        dm_bulk_load(slots + (size_t)s * SLOT, source(G), SLOT * 8, &full[s]);
    }
    __device__ __forceinline__ const double2 *acquire(long long G, int lane)
    {
        const int s = (int)(G % R);
        dm_mbar_wait(&full[s], (unsigned)((G / R) & 1));
        return reinterpret_cast<const double2 *>(slots + (size_t)s * SLOT) + lane;
    }
    /* the warp is done with the matrix of contraction G; the last of the nact warps working on it refills the slot */
    __device__ __forceinline__ void release(long long G, int lane, int nact)
    {
        __syncwarp();
        if (lane == 0) {
            const int s = (int)(G % R);
            __threadfence_block();
            const int old = atomicAdd(&done[s], 1);
            if (old == nact - 1) {
                atomicExch(&done[s], 0);
                if (G + R < total) {
                    __threadfence_block();
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    issue(G + R);
                }
            }
        }
    }
    __device__ __forceinline__ void setup(unsigned char *smem, int tid)
    {
        slots = reinterpret_cast<double *>(smem);
        full = reinterpret_cast<uint64_t *>(smem + (size_t)R * SLOT * 8);
        done = reinterpret_cast<int *>(full + DM_MAX_R);
        if (tid == 0) {
            for (int r = 0; r < R; r++) { dm_mbar_init(&full[r], 1); done[r] = 0; }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            for (int r = 0; r < R && r < total; r++) issue(r);
        }
        __syncthreads();
    }
    __device__ __forceinline__ unsigned char *after() const { return reinterpret_cast<unsigned char *>(done + DM_MAX_R); }
};

/* the tree program in shared memory: ops {first_child, nchild, code_row, spill_before}, children {kind, mat, code_row, edge} */
struct DmProg {
    const int4 *ops, *ch;
    const unsigned char *def_const;
    unsigned char *after;
};
__device__ __forceinline__ DmProg dm_stage_program(const DmArgs &a, unsigned char *smem, int tid, int nthreads)
{
    DmProg p;
    int4 *o = reinterpret_cast<int4 *>(smem + ((16 - (reinterpret_cast<uintptr_t>(smem) & 15)) & 15));
    int4 *c = o + a.nops;
    for (int i = tid; i < a.nops; i += nthreads) o[i] = a.ops4[i];
    for (int i = tid; i < a.nchildren; i += nthreads) c[i] = a.ch4[i];
    __syncthreads();
    /* constant-row flags of the character definitions: read once per tip child, so keep them on chip too */
    unsigned char *dc = reinterpret_cast<unsigned char *>(c + a.nchildren);
    for (int i = tid; i < a.K; i += nthreads) dc[i] = a.def_const[i];
    __syncthreads();
    p.ops = o; p.ch = c; p.def_const = dc;
    p.after = dc + ((a.K + 15) & ~15);
    return p;
}
struct DmOpV { int first_child, nchild, code_row, spill_before; };
struct DmChV { int kind, mat, code_row, edge; };
__device__ __forceinline__ DmOpV dm_op(const DmProg &p, int o) { const int4 v = p.ops[o]; return DmOpV{v.x, v.y, v.z, v.w}; }
__device__ __forceinline__ DmChV dm_ch(const DmProg &p, int j) { const int4 v = p.ch[j]; return DmChV{v.x, v.y, v.z, v.w}; }

/* tile t of the chunk: 8-site groups [g0, g0 + cnt); the tiles of the last wave are smaller so that it is spread evenly */
__device__ __forceinline__ void dm_tile(const DmArgs &a, int t, int &g0, int &cnt)
{
    if (t < a.tiles_full) { g0 = t * DM_GROUPS; cnt = DM_GROUPS; }
    else { g0 = a.tiles_full * DM_GROUPS + (t - a.tiles_full) * a.tail_gs; cnt = min(a.tail_gs, a.ngroups - g0); }
}

/* pull the table row of a tip child (this thread's 16 NB bytes of it) into L1 ahead of its use */
__device__ __forceinline__ void dm_prefetch(const void *p)
{
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}

/* the warp's character codes of one tile: dst[row][8 sites] */
__device__ __forceinline__ void dm_stage_codes(const DmArgs &a, unsigned char *my_codes, int sw, int lane)
{
    __syncwarp();
    for (int r = lane; r < a.nrows; r += 32) {
        const unsigned char *src = a.codes + (size_t)a.code_row_node[r] * a.S + a.s0 + sw;
        unsigned char *dst = my_codes + r * 8;
        if (sw + 8 <= a.Sc && ((reinterpret_cast<uintptr_t>(src) & 7) == 0)) {
            *reinterpret_cast<uint2 *>(dst) = *reinterpret_cast<const uint2 *>(src);
        } else {
            /* ragged end of the chunk: sites beyond it repeat the chunk's last site (their results are not written) */
            for (int s = 0; s < 8; s++) dst[s] = src[(sw + s < a.Sc) ? s : (a.Sc - 1 - sw)];
        }
    }
    __syncwarp();
}

/* bring the maximum (high word m of a non-negative double) of a site's vector into [2^-256, 1):
 * returns the factor and subtracts the number of 2^256 steps from k */
__device__ __forceinline__ double dm_scale_up(int m, int &k)
{
    double sc = 1.0;
    if (m > 0) {
        while (m < DM_HI_M256) { m += 0x10000000; sc *= DM_TWO_P256; k -= 1; }
    }
    return sc;
}

template <int NB>
__device__ __forceinline__ int dm_site_max_hi(const double (&v)[2 * NB])
{
    int m = 0;
#pragma unroll
    for (int i = 0; i < 2 * NB; i++) m = max(m, __double2hiint(v[i]));
    m = max(m, __shfl_xor_sync(0xffffffffu, m, 1));
    m = max(m, __shfl_xor_sync(0xffffffffu, m, 2));
    return m;
}

/*
 * Inside pass.  grid = persistent CTAs (work item i = blockIdx.x + k gridDim.x -> tile i / C, category i % C),
 * NW = DM_GROUPS warps of one 8-site group each.
 */
template <int NB, int NW>
__global__ void __launch_bounds__(NW * 32, 1) dm_inside_kernel(const DmArgs a)
{
    extern __shared__ __align__(128) unsigned char dm_smem[];
    constexpr int NCH = ((NB + 1) / 2 + 1) / 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int W = 8 * NB;

    const long long nitems = (long long)a.ntiles * a.C;
    const long long my_items = (nitems > blockIdx.x) ? (nitems - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    DmRing<NB> ring;
    ring.src = a.Pf; ring.nmat = a.Ei; ring.C = a.C; ring.R = a.R; ring.cat_inner = 0;
    ring.total = my_items * a.Ei;
    ring.setup(dm_smem, tid);
    const DmProg prog = dm_stage_program(a, ring.after(), tid, NW * 32);
    unsigned char *my_codes = prog.after + (size_t)warp * a.nrows * 8;

    double2 *my_stack = a.stack + ((size_t)blockIdx.x * NW + warp) * a.stack_depth * (NB * 32);
    int *my_stack_meta = a.stack_meta + ((size_t)blockIdx.x * NW + warp) * a.stack_depth * 32;
    long long G = 0;

    for (long long it = 0; it < my_items; it++) {
        const long long item = (long long)blockIdx.x + it * gridDim.x;
        const int tile = (int)(item / a.C), c = (int)(item % a.C);
        int g0, nact;                                       /* warps with sites: one per 8-site group of the tile */
        dm_tile(a, tile, g0, nact);
        if (warp >= nact) {
            /* a short tile of the last wave: this warp has no sites; nothing after such a tile may overtake it */
            G += a.Ei;
            __syncthreads();
            continue;
        }
        const int gw = g0 + warp;                           /* this warp's 8-site group (within the chunk) */
        const int sw = gw * 8;
        dm_stage_codes(a, my_codes, sw, lane);

        const double *TPc = a.TPf + (size_t)c * a.Et * a.K * W + q * 2 * NB;
        double cur[2 * NB];
        int curk = 0, curc = 1, sp = 0;
#pragma unroll
        for (int i = 0; i < 2 * NB; i++) cur[i] = 0.0;

#pragma unroll 1
        for (int o = 0; o < a.nops; o++) {
            const DmOpV op = dm_op(prog, o);
            if (op.spill_before) {
                double2 *st = my_stack + (size_t)sp * (NB * 32) + lane;
#pragma unroll
                for (int nb = 0; nb < NB; nb++) __stcg(st + nb * 32, make_double2(cur[2 * nb], cur[2 * nb + 1]));
                my_stack_meta[sp * 32 + lane] = curk * 2 + curc;
                sp++;
            }
            double acc[2 * NB];
            int kacc = 0, cst = 1;
            if (op.code_row >= 0) {
                /* the node itself carries data (rare) */
                const int code = my_codes[op.code_row * 8 + g];
                const double2 *dp = reinterpret_cast<const double2 *>(a.defsf + (size_t)code * W + q * 2 * NB);
#pragma unroll
                for (int nb = 0; nb < NB; nb++) { const double2 v = __ldg(dp + nb); acc[2 * nb] = v.x; acc[2 * nb + 1] = v.y; }
                cst = prog.def_const[code];
            } else {
#pragma unroll
                for (int i = 0; i < 2 * NB; i++) acc[i] = 1.0;
            }
#pragma unroll 1
            for (int j = 0; j < op.nchild; j++) {
                const DmChV ch = dm_ch(prog, op.first_child + j);
                int bc;
                if (ch.kind == F4_KIND_TIP) {
                    const int code = my_codes[ch.code_row * 8 + g];
                    bc = prog.def_const[code];
                    const double2 *tp = reinterpret_cast<const double2 *>(TPc + ((size_t)ch.mat * a.K + code) * W);
#pragma unroll
                    for (int nb = 0; nb < NB; nb++) { const double2 v = __ldg(tp + nb); acc[2 * nb] *= v.x; acc[2 * nb + 1] *= v.y; }
                } else {
                    int kb;
                    if (ch.kind == F4_KIND_STACK) {
                        sp--;
                        const double2 *st = my_stack + (size_t)sp * (NB * 32) + lane;
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v = __ldcg(st + nb * 32); cur[2 * nb] = v.x; cur[2 * nb + 1] = v.y; }
                        const int meta = my_stack_meta[sp * 32 + lane];
                        kb = meta >> 1; bc = meta & 1;
                    } else {
                        kb = curk; bc = curc;
                    }
                    /* a constant column maps to itself under a stochastic matrix (arb_mat_extras.c:84-91) */
                    const double v0 = __shfl_sync(0xffffffffu, cur[0], lane & ~3);
                    const double2 *sl = ring.acquire(G, lane);
                    double2 *slab = nullptr;
                    if (a.slab) {
                        const size_t cell = ((size_t)c * a.Ei + ch.mat) * a.ngroups + (size_t)gw;
                        slab = a.slab + cell * (NB * 32) + lane;
                        if (gw < a.ngroups) a.slab_meta[cell * 32 + lane] = kb * 2 + bc;
                    }
#pragma unroll
                    for (int pc = 0; pc < NCH; pc++) {
                        double em[4][2];
                        dm_gemm_chunk<NB>(cur, sl, pc, em);
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const int nb = 4 * pc + i;
                            if (nb < NB) {
                                if (bc) {
                                    em[i][0] = (8 * nb + 2 * q < a.n) ? v0 : 0.0;
                                    em[i][1] = (8 * nb + 2 * q + 1 < a.n) ? v0 : 0.0;
                                }
                                if (slab && gw < a.ngroups) __stcs(slab + nb * 32, make_double2(em[i][0], em[i][1]));
                                acc[2 * nb] *= em[i][0]; acc[2 * nb + 1] *= em[i][1];
                            }
                        }
                    }
                    ring.release(G, lane, nact);
                    G++;
                    kacc += kb;
                }
                /* per-site rescale after every second factor (non-negative doubles order like their high words) */
                const bool resc = (j & 1) || j == op.nchild - 1;
                cst &= bc;
                if (resc) {
                    const double sc = dm_scale_up(dm_site_max_hi<NB>(acc), kacc);
                    if (sc != 1.0) {
#pragma unroll
                        for (int i = 0; i < 2 * NB; i++) acc[i] *= sc;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 2 * NB; i++) cur[i] = acc[i];
            curk = kacc; curc = cst;
        }
        /* root_prior_expectation (model.c:282-350) */
        const double2 *rp = reinterpret_cast<const double2 *>(a.rootf + q * 2 * NB);
        double lh = 0.0;
#pragma unroll
        for (int nb = 0; nb < NB; nb++) { const double2 rv = __ldg(rp + nb); lh = fma(rv.x, cur[2 * nb], lh); lh = fma(rv.y, cur[2 * nb + 1], lh); }
        lh += __shfl_xor_sync(0xffffffffu, lh, 1);
        lh += __shfl_xor_sync(0xffffffffu, lh, 2);
        const double v0 = __shfl_sync(0xffffffffu, cur[0], lane & ~3);
        if (curc && a.root_const_ok) lh = v0;
        const int site = sw + g;
        if (site < a.Sc && q == 0) {
            a.cat_lh[(size_t)c * a.Sc + site] = lh;
            a.cat_k[(size_t)c * a.Sc + site] = curk;
        }
        if (nact < NW) __syncthreads();
    }
}

/* edge vector of a child at the 8 sites of this warp: block nb of em (tip table or slab), its exponent and constant flag */
struct DmChildRef {
    const double2 *p;       /* + nb * stride */
    int stride;
    int k, bc;
};

template <int NB>
__device__ __forceinline__ DmChildRef dm_child_ref(const DmArgs &a, const DmProg &prog, const DmChV &ch, int c, int gw, int lane, int g, int q,
                                                   const unsigned char *my_codes)
{
    DmChildRef ref;
    const int W = 8 * NB;
    if (ch.kind == F4_KIND_TIP) {
        const int code = my_codes[ch.code_row * 8 + g];
        ref.p = reinterpret_cast<const double2 *>(a.TPf + (((size_t)c * a.Et + ch.mat) * a.K + code) * W + q * 2 * NB);
        ref.stride = 1;
        ref.k = 0; ref.bc = prog.def_const[code];
    } else {
        /* groups beyond the chunk read the chunk's last group (their results are not written) */
        const size_t cell = ((size_t)c * a.Ei + ch.mat) * a.ngroups + (size_t)min(gw, a.ngroups - 1);
        ref.p = a.slab + cell * (NB * 32) + lane;
        ref.stride = 32;
        const int meta = a.slab_meta[cell * 32 + lane];
        ref.k = meta >> 1; ref.bc = meta & 1;
    }
    return ref;
}

/* bring a non-negative site vector into [2^-256, 2^256] both ways */
template <int NB>
__device__ __forceinline__ void dm_rescale_both(double (&v)[2 * NB], int &k)
{
    int m = dm_site_max_hi<NB>(v);
    if (m <= 0) return;
    double sc = 1.0;
    while (m < DM_HI_M256) { m += 0x10000000; sc *= DM_TWO_P256; k -= 1; }
    while (m >= DM_HI_P256) { m -= 0x10000000; sc *= DM_TWO_M256; k += 1; }
    if (sc != 1.0) {
#pragma unroll
        for (int i = 0; i < 2 * NB; i++) v[i] *= sc;
    }
}

__device__ __forceinline__ double dm_scale256(double x, int k)
{
    /* x 2^(256 k) without overflowing the exponent argument */
    return scalbn(x, 256 * max(-16, min(16, k)));
}

/*
 * Outside pass: the program backwards.  grid = persistent CTAs over tiles, the categories are looped inside so
 * that each (edge, site) output cell is accumulated by one thread.  Needs the slab of a keep-mode inside pass and
 * the combined site likelihoods (site_m, site_k).
 *
 * Per-warp stack entry: [fn | z][NB][32] double2 and int4 meta [32] {exponent, high word of max fn, csr edge, -}.
 */
template <int NB, int NW>
__global__ void __launch_bounds__(NW * 32, 1) dm_outside_kernel(const DmArgs a)
{
    extern __shared__ __align__(128) unsigned char dm_smem[];
    constexpr int NCH = ((NB + 1) / 2 + 1) / 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int W = 8 * NB;

    const long long my_items = (a.ntiles > (int)blockIdx.x) ? (a.ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    DmRing<NB> ring;
    ring.src = a.Of; ring.nmat = 2 * a.Ei; ring.C = a.C; ring.R = a.R; ring.cat_inner = 1;
    ring.total = my_items * a.C * 2 * a.Ei;
    ring.setup(dm_smem, tid);
    const DmProg prog = dm_stage_program(a, ring.after(), tid, NW * 32);
    unsigned char *my_codes = prog.after + (size_t)warp * a.nrows * 8;

    double2 *my_stack = a.stack + ((size_t)blockIdx.x * NW + warp) * a.stack_depth * (2 * NB * 32);
    int4 *my_stack_meta = reinterpret_cast<int4 *>(a.stack_meta) + ((size_t)blockIdx.x * NW + warp) * a.stack_depth * 32;
    long long G = 0;

    for (long long it = 0; it < my_items; it++) {
        const int tile = (int)(blockIdx.x + it * gridDim.x);
        int g0, nact;
        dm_tile(a, tile, g0, nact);
        if (warp >= nact) {
            G += (long long)a.C * 2 * a.Ei;
            __syncthreads();
            continue;
        }
        const int gw = g0 + warp;
        const int sw = gw * 8;
        dm_stage_codes(a, my_codes, sw, lane);
        const int site = sw + g;
        const bool valid = site < a.Sc;
        const double sm = valid ? a.site_m[site] : 0.0;
        const int sk = valid ? a.site_k[site] : 0;

#pragma unroll 1
        for (int c = 0; c < a.C; c++) {
            const double *TFc = a.TFf + (size_t)c * a.Et * a.K * W + q * 2 * NB;
            int sp = 0;
            double fn[2 * NB];
            /* arbplfmarginal.c:184-191 / arbplfderiv.c:300-310: categories (and sites) of zero likelihood contribute nothing */
            double coef = 0.0;
            if (valid) {
                const double prior = a.cat_prior[c];
                if (prior * a.cat_lh[(size_t)c * a.Sc + sw + g] > 0.0 && sm > 0.0) coef = prior / sm;
            }
            int kf = -sk;
            const double2 *rp = reinterpret_cast<const double2 *>(a.rootf + q * 2 * NB);
#pragma unroll
            for (int nb = 0; nb < NB; nb++) { const double2 rv = __ldg(rp + nb); fn[2 * nb] = rv.x * coef; fn[2 * nb + 1] = rv.y * coef; }
            bool fn_in_regs = true;               /* the root's fn was formed above */
#pragma unroll 1
            for (int o = a.nops - 1; o >= 0; o--) {
                const DmOpV op = dm_op(prog, o);
                const bool popped = (o != a.nops - 1);
                const double2 *zp = nullptr;
                int in_edge = -1, kz = 0;
                if (popped) {
                    /* (fn, z) of this node: z always comes from the stack entry; fn only when the node is not the last
                     * internal child of the op handled just before (then it is still in registers, unscaled) */
                    sp--;
                    const double2 *st = my_stack + (size_t)sp * (2 * NB * 32) + lane;
                    const int4 meta = my_stack_meta[sp * 32 + lane];
                    in_edge = meta.z; kz = meta.x;          /* z keeps the exponent it was computed with */
                    kf = meta.x;
                    int m = meta.y;
                    double sc = 1.0;
                    if (m > 0) {
                        while (m < DM_HI_M256) { m += 0x10000000; sc *= DM_TWO_P256; kf -= 1; }
                        while (m >= DM_HI_P256) { m -= 0x10000000; sc *= DM_TWO_M256; kf += 1; }
                    }
                    if (fn_in_regs) {
                        if (sc != 1.0) {
#pragma unroll
                            for (int i = 0; i < 2 * NB; i++) fn[i] *= sc;
                        }
                    } else {
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v = __ldcg(st + nb * 32); fn[2 * nb] = v.x * sc; fn[2 * nb + 1] = v.y * sc; }
                    }
                    zp = st + NB * 32;
                }
                fn_in_regs = false;

                /* contraction of fe with (P_e, F_e) of an internal child: fn_b into `dst_fn` (registers, when the child is
                 * the next op's node) or into the stack entry, z_b always into the stack entry */
                auto contract_and_push = [&](const double (&fe)[2 * NB], int kfe, int edge, bool keep_fn) {
                    double2 *st = my_stack + (size_t)sp * (2 * NB * 32) + lane;
                    int m = 0;
#pragma unroll 1
                    for (int which = 0; which < 2; which++) {
                        const double2 *sl = ring.acquire(G, lane);
#pragma unroll
                        for (int pc = 0; pc < NCH; pc++) {
                            double em[4][2];
                            dm_gemm_chunk<NB>(fe, sl, pc, em);
#pragma unroll
                            for (int i = 0; i < 4; i++) {
                                const int nb = 4 * pc + i;
                                if (nb < NB) {
                                    if (which == 0) {
                                        m = max(m, max(__double2hiint(em[i][0]), __double2hiint(em[i][1])));
                                        if (keep_fn) { fn[2 * nb] = em[i][0]; fn[2 * nb + 1] = em[i][1]; }
                                        else __stcg(st + nb * 32, make_double2(em[i][0], em[i][1]));
                                    } else {
                                        __stcg(st + (NB + nb) * 32, make_double2(em[i][0], em[i][1]));
                                    }
                                }
                            }
                        }
                        ring.release(G, lane, nact);
                        G++;
                    }
                    m = max(m, __shfl_xor_sync(0xffffffffu, m, 1));
                    m = max(m, __shfl_xor_sync(0xffffffffu, m, 2));
                    my_stack_meta[sp * 32 + lane] = make_int4(kfe, m, edge, 0);
                    sp++;
                };
                auto emit = [&](double x, int edge, int k) {
                    x += __shfl_xor_sync(0xffffffffu, x, 1);
                    x += __shfl_xor_sync(0xffffffffu, x, 2);
                    if (valid && q == 0 && (!a.edge_mask || a.edge_mask[edge])) {
                        double *dst = a.edge_out + (size_t)edge * a.Sc + sw + g;
                        /* the first category writes, the others add: no read-modify-write (a dependent global load) for C = 1 */
                        if (c == 0) *dst = dm_scale256(x, k);
                        else if (x != 0.0) *dst += dm_scale256(x, k);
                    }
                };
                /* the slab rows the next op (o - 1) will read come from HBM: ask for them one op ahead */
                if (o > 0) {
                    const DmOpV opn = dm_op(prog, o - 1);
                    for (int j = 0; j < opn.nchild; j++) {
                        const DmChV chn = dm_ch(prog, opn.first_child + j);
                        if (chn.kind == F4_KIND_TIP) continue;
                        const size_t cell = ((size_t)c * a.Ei + chn.mat) * a.ngroups + (size_t)min(gw, a.ngroups - 1);
                        const double2 *pp = a.slab + cell * (NB * 32) + lane;
#pragma unroll
                        for (int nb = 0; nb < NB; nb += 2) asm volatile("prefetch.global.L2 [%0];" ::"l"(pp + nb * 32));
                    }
                }

                if (op.nchild == 2 && op.code_row < 0) {
                    /* ---- two children, no data at the node: every vector is loaded once ---- */
                    const DmChV c0 = dm_ch(prog, op.first_child), c1 = dm_ch(prog, op.first_child + 1);
                    const DmChildRef r0 = dm_child_ref<NB>(a, prog, c0, c, gw, lane, g, q, my_codes);
                    const DmChildRef r1 = dm_child_ref<NB>(a, prog, c1, c, gw, lane, g, q, my_codes);
                    const bool int0 = c0.kind != F4_KIND_TIP, int1 = c1.kind != F4_KIND_TIP;
                    const double2 *tf0 = nullptr, *tf1 = nullptr;
                    if (!int0) tf0 = reinterpret_cast<const double2 *>(TFc + ((size_t)c0.mat * a.K + my_codes[c0.code_row * 8 + g]) * W);
                    if (!int1) tf1 = reinterpret_cast<const double2 *>(TFc + ((size_t)c1.mat * a.K + my_codes[c1.code_row * 8 + g]) * W);
                    double fe[2 * NB];
                    double xa = 0.0, x0 = 0.0, x1 = 0.0;
                    /* fe <- fn . em0 (the outside vector of child 1) when child 1 is internal, else fn . em1 (child 0's) */
#pragma unroll
                    for (int nb = 0; nb < NB; nb++) {
                        const double2 v0 = r0.p[nb * r0.stride], v1 = r1.p[nb * r1.stride];
                        if (popped) {
                            const double2 zz = __ldcg(zp + nb * 32);
                            xa = fma(zz.x, v0.x * v1.x, xa); xa = fma(zz.y, v0.y * v1.y, xa);
                        }
                        const double f0x = fn[2 * nb] * v1.x, f0y = fn[2 * nb + 1] * v1.y;     /* child 0: fn . em1 */
                        const double f1x = fn[2 * nb] * v0.x, f1y = fn[2 * nb + 1] * v0.y;     /* child 1: fn . em0 */
                        if (!int0) { const double2 t = __ldg(tf0 + nb); x0 = fma(t.x, f0x, x0); x0 = fma(t.y, f0y, x0); }
                        if (!int1) { const double2 t = __ldg(tf1 + nb); x1 = fma(t.x, f1x, x1); x1 = fma(t.y, f1y, x1); }
                        if (int1) { fe[2 * nb] = f1x; fe[2 * nb + 1] = f1y; }
                        else { fe[2 * nb] = f0x; fe[2 * nb + 1] = f0y; }
                    }
                    if (popped) {
                        if (a.f_zero_rowsum && (r0.bc & r1.bc)) xa = 0.0;
                        emit(xa, in_edge, kz + r0.k + r1.k);
                    }
                    if (!int0) emit(x0, c0.edge, kf + r1.k);
                    if (!int1) emit(x1, c1.edge, kf + r0.k);
                    if (int1) {
                        /* both internal: child 1 first (it goes to the stack), then child 0 with em1 loaded again */
                        int kfe = kf + r0.k;
                        dm_rescale_both<NB>(fe, kfe);
                        contract_and_push(fe, kfe, c1.edge, false);
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v1 = r1.p[nb * r1.stride]; fe[2 * nb] = fn[2 * nb] * v1.x; fe[2 * nb + 1] = fn[2 * nb + 1] * v1.y; }
                    }
                    if (int0) {
                        int kfe = kf + r1.k;
                        dm_rescale_both<NB>(fe, kfe);
                        contract_and_push(fe, kfe, c0.edge, true);
                        fn_in_regs = true;
                    }
                    continue;
                }

                /* ---- general shape ---- */
                if (popped) {
                    /* L_a from the children's edge vectors, then x_e = z . L_a (evaluate_site_frechet.c:18-39) */
                    double La[2 * NB];
                    int kL = 0, cstL = 1;
                    if (op.code_row >= 0) {
                        const int code = my_codes[op.code_row * 8 + g];
                        const double2 *dp = reinterpret_cast<const double2 *>(a.defsf + (size_t)code * W + q * 2 * NB);
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v = __ldg(dp + nb); La[2 * nb] = v.x; La[2 * nb + 1] = v.y; }
                        cstL = prog.def_const[code];
                    } else {
#pragma unroll
                        for (int i = 0; i < 2 * NB; i++) La[i] = 1.0;
                    }
#pragma unroll 1
                    for (int j = 0; j < op.nchild; j++) {
                        const DmChildRef ref = dm_child_ref<NB>(a, prog, dm_ch(prog, op.first_child + j), c, gw, lane, g, q, my_codes);
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v = ref.p[nb * ref.stride]; La[2 * nb] *= v.x; La[2 * nb + 1] *= v.y; }
                        kL += ref.k; cstL &= ref.bc;
                        if ((j & 1) || j == op.nchild - 1) {
                            const double sc2 = dm_scale_up(dm_site_max_hi<NB>(La), kL);
                            if (sc2 != 1.0) {
#pragma unroll
                                for (int i = 0; i < 2 * NB; i++) La[i] *= sc2;
                            }
                        }
                    }
                    double x = 0.0;
#pragma unroll
                    for (int nb = 0; nb < NB; nb++) { const double2 v = __ldcg(zp + nb * 32); x = fma(v.x, La[2 * nb], x); x = fma(v.y, La[2 * nb + 1], x); }
                    if (a.f_zero_rowsum && cstL) x = 0.0;
                    emit(x, in_edge, kz + kL);
                }
                /* fn_a . data_a */
                if (op.code_row >= 0) {
                    const int code = my_codes[op.code_row * 8 + g];
                    const double2 *dp = reinterpret_cast<const double2 *>(a.defsf + (size_t)code * W + q * 2 * NB);
#pragma unroll
                    for (int nb = 0; nb < NB; nb++) { const double2 v = __ldg(dp + nb); fn[2 * nb] *= v.x; fn[2 * nb + 1] *= v.y; }
                }
                /* children: tips in any order, internal ones from the last to the first so that the stack unwinds in
                 * the reverse of the inside pass */
#pragma unroll 1
                for (int j = op.nchild - 1; j >= 0; j--) {
                    const DmChV ch = dm_ch(prog, op.first_child + j);
                    double fe[2 * NB];
                    int kfe = kf;
#pragma unroll
                    for (int i = 0; i < 2 * NB; i++) fe[i] = fn[i];
                    int nmul = 0;
#pragma unroll 1
                    for (int j2 = 0; j2 < op.nchild; j2++) {
                        if (j2 == j) continue;
                        const DmChildRef ref = dm_child_ref<NB>(a, prog, dm_ch(prog, op.first_child + j2), c, gw, lane, g, q, my_codes);
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v = ref.p[nb * ref.stride]; fe[2 * nb] *= v.x; fe[2 * nb + 1] *= v.y; }
                        kfe += ref.k;
                        if ((++nmul & 1) == 0) dm_rescale_both<NB>(fe, kfe);
                    }
                    dm_rescale_both<NB>(fe, kfe);
                    if (ch.kind == F4_KIND_TIP) {
                        const int code = my_codes[ch.code_row * 8 + g];
                        const double2 *tf = reinterpret_cast<const double2 *>(TFc + ((size_t)ch.mat * a.K + code) * W);
                        double x = 0.0;
#pragma unroll
                        for (int nb = 0; nb < NB; nb++) { const double2 v = __ldg(tf + nb); x = fma(v.x, fe[2 * nb], x); x = fma(v.y, fe[2 * nb + 1], x); }
                        emit(x, ch.edge, kfe);
                    } else {
                        contract_and_push(fe, kfe, ch.edge, false);
                    }
                }
            }
        }
        if (nact < NW) __syncthreads();
    }
}

/* ------------------------------------------------------------------ */
/* host side                                                           */
/* ------------------------------------------------------------------ */

int dm_blocks_for(int n)
{
    if (n > 16 && n <= 24) return 3;
    if (n > 24 && n <= 32) return 4;
    if (n > 32 && n <= 64) return 8;
    return 0;
}

size_t dm_slot_doubles_host(int NB) { return (size_t)dm_slot_doubles(NB); }

size_t dm_smem_bytes(int NB, int R, int nrows, int nops, int nchildren)
{
    return (size_t)R * dm_slot_doubles(NB) * 8 + DM_MAX_R * 8 + DM_MAX_R * 4 + 16 + (size_t)(nops + nchildren) * 16 +
           (size_t)DM_GROUPS * nrows * 8 + 16 + 272;          /* + the constant-row flags (K <= 256) */
}

void dm_tiling(int ngroups, int items_per_tile, int grid, int *tiles_full, int *tail_gs, int *ntiles)
{
    const long long cap = (long long)grid * DM_GROUPS;
    const long long waves = ((long long)ngroups * items_per_tile) / cap;
    int tf = (int)(waves * grid / items_per_tile);
    if (tf > ngroups / DM_GROUPS) tf = ngroups / DM_GROUPS;
    const int rest = ngroups - tf * DM_GROUPS;
    *tiles_full = tf;
    if (rest == 0) { *tail_gs = DM_GROUPS; *ntiles = tf; return; }
    const int tiles_tail = grid / items_per_tile > 0 ? grid / items_per_tile : 1;
    int gs = (rest + tiles_tail - 1) / tiles_tail;
    if (gs > DM_GROUPS) gs = DM_GROUPS;
    *tail_gs = gs;
    *ntiles = tf + (rest + gs - 1) / gs;
}

cudaError_t dm_pack(const double *src, const double *src2, const int *src_index, const int *transpose, int nmat,
                    int C, int E, int n, int NB, double *dst, cudaStream_t st)
{
    const size_t total = (size_t)C * nmat * dm_slot_doubles(NB);
    if (!total) return cudaSuccess;
    const unsigned blocks = (unsigned)((total + 255) / 256 > 65535 ? 65535 : (total + 255) / 256);
    dm_pack_kernel<<<blocks, 256, 0, st>>>(src, src2, src_index, transpose, nmat, C, E, n, NB, dst);
    return cudaGetLastError();
}

cudaError_t dm_tip_table(const double *M, const double *defs, const unsigned char *def_const, const int *edge_of_tip,
                         int C, int E, int Et, int K, int n, int NB, int mode, double *out, cudaStream_t st)
{
    const size_t total = (size_t)C * Et * K * 8 * NB;
    if (!total) return cudaSuccess;
    dm_tip_table_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(M, defs, def_const, edge_of_tip, C, E, Et, K, n, NB, mode, out);
    return cudaGetLastError();
}

template <int NB>
static cudaError_t dm_launch_t(const DmArgs &a, int grid, bool outside, cudaStream_t st)
{
    constexpr int NW = DM_GROUPS;
    const size_t smem = dm_smem_bytes(NB, a.R, a.nrows, a.nops, a.nchildren);
    cudaError_t r;
    if (outside) {
        r = cudaFuncSetAttribute(dm_outside_kernel<NB, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (r != cudaSuccess) return r;
        dm_outside_kernel<NB, NW><<<grid, NW * 32, smem, st>>>(a);
    } else {
        r = cudaFuncSetAttribute(dm_inside_kernel<NB, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (r != cudaSuccess) return r;
        dm_inside_kernel<NB, NW><<<grid, NW * 32, smem, st>>>(a);
    }
    return cudaGetLastError();
}

static cudaError_t dm_launch(const DmArgs &a, int NB, int grid, bool outside, cudaStream_t st)
{
    switch (NB) {
    case 3: return dm_launch_t<3>(a, grid, outside, st);
    case 4: return dm_launch_t<4>(a, grid, outside, st);
    case 8: return dm_launch_t<8>(a, grid, outside, st);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t dm_launch_inside(const DmArgs &a, int NB, int grid, cudaStream_t st) { return dm_launch(a, NB, grid, false, st); }
cudaError_t dm_launch_outside(const DmArgs &a, int NB, int grid, cudaStream_t st) { return dm_launch(a, NB, grid, true, st); }
