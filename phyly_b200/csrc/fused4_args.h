/*
 * Argument blocks of the fused 4-state kernels (fused4.cuh) and the entry points of the translation unit that
 * instantiates them (fused4_kernels.cu); included by the host side (plf_engine.cu).
 */
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>
#include "f4prog.h"

struct F4Args {
    int nops, nchildren;
    const F4Op *ops;
    const F4Child *children;
    int E, K, Ei, Et;                /* edges, characters, internal-child edges, tip edges */
    int64_t S;
    int ncode_rows;
    const int *code_row_node;        /* [ncode_rows] node whose codes fill the row */
    const unsigned char *codes;      /* [N][S] */
    const double *defs;              /* [K][4] */
    const unsigned char *def_const;  /* [K] */
    const double *Pint;              /* [C][Ei][16] */
    const double *TP;                /* [C][Et][K][4] */
    const double *Fint;              /* [C][Ei][16] or NULL; marginal mode: P of the tip edges, [C][Et][16] */
    const double *TF;                /* [C][Et][K][4] or NULL */
    int f_zero_rowsum;
    const double *cat_prior;
    int root_mode;
    double root_vec[4];
    const double *site_w;            /* [S] or NULL */
    const unsigned char *edge_mask;  /* [E] or NULL */
    int stack_depth;                 /* ll-only mode: shared-memory stack entries (0 when the stack is global) */
    int gstack;                      /* ll-only mode: pending partials go to scratch / scratchS (L2-resident) */
    int nslots;
    double4 *scratch;                /* [nslots][C][T] */
    unsigned int *scratchS;          /* [nslots][T]: byte c = rescale count | const flag << 6 */
    double *site_ll;                 /* [S] or NULL */
    double *edge_site_out;           /* [E][S] or NULL */
    int64_t s_begin, s_end;          /* this launch covers sites [s_begin, s_end) (a chunk of the data) */
    int N;                           /* nodes */
    double *marg_site_out;           /* marginal mode: [N][4][S] or NULL */
    double *block_marg;              /* marginal mode: [grid * warps][N][4], zeroed by the host, accumulated here */
    double *block_ll;                /* [grid] */
    double *block_edge;              /* [grid][E] */
    int *error_flag;
    double *block_gmat;              /* mode 3: [grid * warps][C][E][16], zeroed by the host, accumulated here */
    int nch;                         /* folded cherries (F4_KIND_CHERRY children; modes 0 and 1), tables by code pair p: */
    const double *chEm;              /* [C][nch][K*K][4]: the vector the parent multiplies in (staged in shared memory) */
    const unsigned int *chW;         /* [nch][K*K]: scale word, the layout of scratchS (staged in shared memory) */
    const double *chOut;             /* mode 1: [C][nch][K*K][16]: chEm, y, z_a, z_b (f4_tables_kernel), read through L1 */
};

/*
 * Constant-memory variant (CM): the compact matrices of the internal-child edges live in __constant__
 * memory and the tree program travels as a kernel parameter.  Everything the op loop decodes is then
 * warp-uniform by construction (loop counters -> constant bank), so the compiler keeps it in uniform
 * registers and the 4x4 matrices enter the DFMAs as uniform operands (LDCU) instead of costing one
 * shared-memory wavefront per 16 bytes -- the kernel is bound by the LSU pipe, not by fp64 issue.
 */
#define F4_CM_MAXD 4064      /* doubles per matrix set: C * Ei * 16 <= 4064 (2 sets = 65024 of the 65536 bytes) */
#define F4_CM_MAXOPS 128
#define F4_CM_MAXCH 256

struct F4Prog {
    F4Op ops[F4_CM_MAXOPS];
    F4Child ch[F4_CM_MAXCH];
};

__host__ __device__ inline size_t f4_align16(size_t x) { return (x + 15) & ~(size_t)15; }

typedef void (*f4_kernel_t)(const F4Args, const F4Prog);

/* kernel instantiation for (block size, staging level, packed codes, constant-memory matrices, categories, mode):
 * mode 0 = ll only, 1 = ll + edge forms, 2 = ll + marginals, 3 = ll + per-edge outer-product matrices (the 256- and
 * 128-thread configurations of mode 2); NULL when the combination is not instantiated */
f4_kernel_t f4_get_kernel(int bd, int staged, bool pack, bool cm, int C, int mode);
/* copy the compact matrices of the internal-child edges into the constant bank (device to device, in-stream) */
cudaError_t f4_upload_const(const double *Pint, const double *Fint, size_t bytes, cudaStream_t st);
