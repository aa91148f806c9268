/*
 * Host interface of the FP64 tensor-pipe kernels for large state spaces (dmma.cu):
 * amino-acid (20 states) and codon (61 states) models, 16 < n <= 64.
 *
 * Reference loops being replaced: evaluate_site_lhood (evaluate_site_lhood.c:21-57),
 * evaluate_site_forward (evaluate_site_forward.c:31-105) and evaluate_site_frechet
 * (evaluate_site_frechet.c:4-42) inside the site x category loops of arbplfll.c:139-170 and
 * arbplfderiv.c:274-357.
 */
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>
#include "f4prog.h"

#define DM_MAX_R 8        /* slots of the matrix ring */
#define DM_GROUPS 16      /* 8-site groups per full tile, one warp each */
#define DM_TILE (8 * DM_GROUPS)

struct DmArgs {
    int n, C, K;
    int nops;
    int nchildren;
    const int4 *ops4;                /* [nops] {first_child, nchild, code_row, spill_before} */
    const int4 *ch4;                 /* [nchildren] {kind, mat, code_row, csr edge} */
    int Ei, Et;                      /* internal-child (GEMM) edges, tip edges */
    int nrows;                       /* rows of the code tile (nodes that may carry data) */
    const int *code_row_node;        /* [nrows] */
    const unsigned char *codes;      /* [N][S] node major */
    int64_t S, s0;                   /* all sites; first site of this chunk */
    int Sc;                          /* sites of this chunk */
    const unsigned char *def_const;  /* [K] */
    const double *defsf;             /* [K][8NB] definitions in thread order (zero padded) */
    const double *Pf;                /* [C][Ei][slot] packed P_e^T, consumption order of the inside pass */
    const double *TPf;               /* [C][Et][K][8NB] tip table P_e def_k in thread order */
    const double *rootf;             /* [8NB] root prior weights in thread order (zero padded) */
    int root_const_ok;               /* uniform / equilibrium prior: a constant column has expectation = its value */
    double *cat_lh; int *cat_k;      /* [C][Sc] */
    int ntiles;                      /* tiles of the chunk: tiles_full of DM_GROUPS 8-site groups, the rest of tail_gs groups */
    int tiles_full, tail_gs;
    int R;                           /* ring slots in use (2..DM_MAX_R) */
    int stack_depth;                 /* entries of the per-warp stacks */
    double2 *stack;                  /* inside: [ctas][groups][depth][NB][32]; outside: [ctas][groups][depth][2][NB][32] */
    int *stack_meta;                 /* inside: [ctas][groups][depth][32];     outside: [ctas][groups][depth][32][4] */
    /* keep mode (an outside pass follows): the edge vectors em_e = P_e L_b of the internal-child edges */
    double2 *slab;                   /* [C][Ei][ngroups][NB][32] or NULL */
    int *slab_meta;                  /* [C][Ei][ngroups][32]: exponent of the child * 2 + constant flag */
    int ngroups;                     /* 8-site groups in the chunk */
    /* outside pass */
    const double *Of;                /* [C][2 Ei][slot]: (P_e, F_e) of the internal-child edges, consumption order */
    const double *TFf;               /* [C][Et][K][8NB] tip table F_e def_k in thread order */
    const double *cat_prior;         /* [C] */
    const double *site_m;            /* [Sc] mantissa of the site likelihood */
    const int *site_k;               /* [Sc] its exponent in units of 2^256 */
    const unsigned char *edge_mask;  /* [E] or NULL */
    int f_zero_rowsum;               /* F has zero row sums: a constant column gives exactly 0 (util.c:338-344) */
    double *edge_out;                /* [E][Sc], zeroed by the caller, accumulated over categories here */
};

/* number of 8-state blocks the kernels are instantiated for, 0 = unsupported state count */
int dm_blocks_for(int n);
size_t dm_slot_doubles_host(int NB);
/* dynamic shared memory of a launch with R ring slots */
size_t dm_smem_bytes(int NB, int R, int nrows, int nops, int nchildren);
/* tiles of a chunk of ngroups 8-site groups for a persistent grid: full tiles while whole waves can be filled, then
 * smaller tiles that spread the remainder evenly over the CTAs (items_per_tile = categories for the inside pass) */
void dm_tiling(int ngroups, int items_per_tile, int grid, int *tiles_full, int *tail_gs, int *ntiles);

/* pack nmat matrices per category into the B-fragment order (see dmma.cu) */
cudaError_t dm_pack(const double *src, const double *src2, const int *src_index, const int *transpose, int nmat,
                    int C, int E, int n, int NB, double *dst, cudaStream_t st);
/* tip tables / definitions in thread order; M == NULL writes the definitions themselves */
cudaError_t dm_tip_table(const double *M, const double *defs, const unsigned char *def_const, const int *edge_of_tip,
                         int C, int E, int Et, int K, int n, int NB, int mode, double *out, cudaStream_t st);
cudaError_t dm_launch_inside(const DmArgs &a, int NB, int grid, cudaStream_t st);
cudaError_t dm_launch_outside(const DmArgs &a, int NB, int grid, cudaStream_t st);
