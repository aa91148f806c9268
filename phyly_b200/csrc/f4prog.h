/*
 * The post-order tree program shared by the fused 4-state kernels (fused4.cuh) and the FP64
 * tensor-pipe kernels (dmma.cu).  Built on the host by build_program (plf_engine.cu) from the
 * csr_graph of the reference (csr_graph.c:47-151) with Sethi-Ullman child ordering.
 */
#pragma once

#define F4_MAXD 3          /* max out-degree handled by the fused kernel */
#define F4_KIND_TIP 0
#define F4_KIND_CUR 1
#define F4_KIND_STACK 2
#define F4_KIND_CHERRY 3     /* a node whose two children are tips, folded into per-code-pair tables (ll / edge forms) */

struct F4Op {
    int node;
    int first_child;
    int nchild;
    int slot;            /* scratch slot of this node's inside vector */
    int code_row;        /* row of the codes tile if the node carries data, else -1 */
    int spill_before;    /* the register-resident partial is not consumed by this op */
};

struct F4Child {
    int kind;
    int slot;            /* scratch slot if internal, else -1 */
    int mat;             /* internal child: index into the compact internal-edge matrices;
                            tip child: index into the compact tip tables; cherry: index of its tables */
    int code_row;        /* tip child: row of the codes tile; cherry: row of its first tip */
    int edge;            /* csr idx (output position) */
    int node;            /* the child node (output position of its marginal) */
    int code_row_b;      /* cherry: row of its second tip */
    int tip_edge;        /* cherry: csr idx of the edge to its first tip (the second's is tip_edge + 1) */
};

