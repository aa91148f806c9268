/*
 * plf.h -- device seam of the B200 phylogenetic likelihood engine (C ABI).
 *
 * This is the boundary "host C calls CUDA through a thin C-ABI layer".  It
 * replaces, for the hot path, the reference's in-process workspaces:
 *
 *   plf_set_tree      <- csr_graph_t + navigation_t built by _validate_edges
 *                        (parsemodel.c:210-368, csr_graph.h:17-51, model.c:23-45)
 *   plf_set_model     <- cross_site_ws_update_with_edge_rates
 *                        (cross_site_ws.c:199-242; transition matrices :150-168)
 *   plf_set_data      <- pmat_t / pmat_update_base_node_vectors
 *                        (model.h:41-48, model.c:181-199)
 *   plf_ll            <- _nd_accum_update of arbplfll.c:110-177
 *                        (evaluate_site_lhood.c:6-63 inside the site x category loop)
 *   plf_deriv         <- _nd_accum_update of arbplfderiv.c:210-371
 *   plf_marginal      <- _nd_accum_update of arbplfmarginal.c:111-264
 *   plf_edge_expect   <- _update_site of arbplfdwell.c:201-312 / arbplftrans.c:222-346
 *                        with the Frechet matrices of util.c:500-548
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from plf_last_error().  Nothing aborts the host process.
 *   - all pointers are HOST pointers owned by the caller unless the name ends
 *     in _dev.  Arrays are C-contiguous.
 *   - edges are always in CSR order ("csr idx", csr_graph.c:28-46): position
 *     of the edge in indices[]; node labels are the user's.
 *   - there is no CPU implementation behind this interface: if no CUDA device
 *     is usable plf_create fails.
 *   - a handle is not thread safe; use one handle per host thread / per GPU.
 */
/*
 * Threading and sharing: an engine handle is to be used from one host thread at a time; different
 * handles (also on the same device) may be used from different threads -- the one device-wide resource,
 * the constant bank that holds the matrices of the small-tree kernels, is serialised inside the library.
 * Queries are synchronous: when a plf_* query returns, its host outputs are final.
 */
#ifndef PLF_H
#define PLF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct plf_engine plf_engine;

/* root prior modes, model.h (enum root_prior_mode) */
enum { PLF_ROOT_NONE = 0, PLF_ROOT_UNIFORM = 1, PLF_ROOT_EQUILIBRIUM = 2, PLF_ROOT_CUSTOM = 3 };
/* edge expectation kinds */
enum { PLF_KIND_DWELL = 0, PLF_KIND_TRANS = 1 };
/* kernel path selection (PLF_PATH_AUTO picks the fused 4-state kernel when it applies) */
enum { PLF_PATH_AUTO = 0, PLF_PATH_GENERIC = 1, PLF_PATH_FUSED4 = 2 };

int  plf_create(plf_engine **out, int device);
void plf_destroy(plf_engine *e);
const char *plf_last_error(const plf_engine *e);

/* Force a kernel path (tests / benchmarks); default PLF_PATH_AUTO. */
int plf_set_path(plf_engine *e, int path);

/*
 * Tree in the reference's CSR form.  preorder is the BFS level order from the
 * root (csr_graph_get_tree_topo_sort); preorder[0] is the root.
 */
int plf_set_tree(plf_engine *e, int node_count,
                 const int *indptr /*[N+1]*/, const int *indices /*[E]*/,
                 const int *preorder /*[N]*/);

/*
 * Model.  Q is the *scaled* rate matrix (divisor applied, diagonal = -row sum),
 * row major, given as a double-double pair (q_lo may be NULL).  Transition
 * matrices exp(cat_rates[c]*edge_rates[e]*Q) are computed on the device.
 * root_vec: custom prior (PLF_ROOT_CUSTOM) or equilibrium (PLF_ROOT_EQUILIBRIUM);
 * ignored otherwise.
 */
int plf_set_model(plf_engine *e, int state_count, int category_count,
                  const double *q_hi /*[n*n]*/, const double *q_lo /*[n*n] or NULL*/,
                  const double *edge_rates /*[E] csr order*/,
                  const double *cat_rates /*[C]*/, const double *cat_prior /*[C]*/,
                  int root_mode, const double *root_vec /*[n] or NULL*/);

/* Creates the CUDA context of a device ahead of the first plf_create (no engine, no message; 0 or -1): a process that
 * answers one document (the arbplf-* executables, runjson.c:117-157) calls it from a second thread while it reads and
 * parses its input. */
int plf_warmup(int device);

/* Change only the edge rate coefficients (csr order); recomputes matrices lazily. */
int plf_set_edge_rates(plf_engine *e, const double *edge_rates /*[E]*/);

/*
 * Data as character codes: codes[site][node] indexes rows of defs[K][n]
 * (parsemodel.c:514-628).  code_bytes is 1 (uint8), 4 (int32) or
 * PLF_CODES_PACKED4: two codes per byte (def_count <= 16, the nucleotide case),
 * rows of (N + 1) / 2 bytes, node 2j in the low and node 2j + 1 in the high
 * nibble of byte j -- half the host-to-device traffic of uint8 codes.  A dense
 * probability_array is passed by first de-duplicating its rows into defs.
 * The copy to the device happens inside this call (pinned staging).
 */
#define PLF_CODES_PACKED4 0
int plf_set_data(plf_engine *e, int64_t site_count, int def_count,
                 const double *defs /*[K][n]*/, const void *codes /*[S][N]*/, int code_bytes);

/*
 * The same, without waiting for the copy: the codes (and, if given, the site
 * weights) travel in chunks on a second stream and the next query starts on
 * the first chunk while the later ones are still in flight (4-state fused
 * path; other paths simply wait).  `codes` and `site_weights` must stay valid
 * and unchanged until the next query or plf_synchronize returns; use pinned
 * host memory, otherwise the copy is staged and nothing overlaps.
 */
int plf_set_data_async(plf_engine *e, int64_t site_count, int def_count,
                       const double *defs /*[K][n]*/, const void *codes /*[S][N]*/, int code_bytes,
                       const double *site_weights /*[S] or NULL*/);

/*
 * Site-pattern compression (the reference leaves it to its input generators, examples/BEAST.GTRG/mknuc.py:57-66):
 * identical rows of codes[S][N] are merged.  Patterns come out in order of first occurrence: codes_out[P][N] (room for
 * S rows), counts_out[P] their multiplicities (the site weights of the compressed alignment), site_to_pattern[S] the
 * pattern of every site (scatter-back map when the site axis is kept).  Outputs other than n_patterns may be NULL.
 * Hash + full row comparison on the device; integer results, identical to the oracle's.
 */
int plf_compress_patterns(plf_engine *e, int64_t site_count, int node_count, const void *codes, int code_bytes,
                          int64_t *n_patterns, void *codes_out, int64_t *counts_out, int64_t *site_to_pattern);

/* Per-site weights used by the *_sum outputs (NULL = all ones).  reduction.c:24-118. */
int plf_set_site_weights(plf_engine *e, const double *w /*[S] or NULL*/);

/* log-likelihood.  site_ll[S] and/or sum = sum_s w_s ll_s; either may be NULL. */
int plf_ll(plf_engine *e, double *site_ll, double *sum);

/*
 * d log L / d edge_rate for the edges with edge_mask[idx] != 0 (NULL = all).
 * site_deriv is [S][E] (csr edge order), sum_deriv[E] = sum_s w_s d[s][e].
 * Any output may be NULL.  Unrequested edges are returned as 0.
 */
int plf_deriv(plf_engine *e, const unsigned char *edge_mask,
              double *site_ll, double *sum_ll, double *site_deriv, double *sum_deriv);

/*
 * Certified mode: enclosures site_lo[s] <= log L_s <= site_hi[s] computed with directed rounding (interval arithmetic
 * on the pruning recursion and on the matrix exponentials; csrc/certified.cuh), in place of the reference's Arb balls
 * (util.c:12-50, arbplfll.c:206-224).  Rigorous for inputs within the stated relative uncertainties: delta_rate on
 * rate_c * t_e and on an equilibrium root prior (the host's gamma quantiles / linear solve are accurate to 1e-14, not
 * certified; 4e-15 is the documented default), delta_q on the scaled rate matrix and the derived category priors
 * (2^-60).  sum_lo / sum_hi enclose sum_s w_s log L_s.  Any output may be NULL.
 */
int plf_ll_certified(plf_engine *e, double delta_rate, double delta_q, double *site_lo, double *site_hi,
                     double *sum_lo, double *sum_hi);

/*
 * Certified mode for plf_deriv: site_lo[s][e] <= d log L_s / d edge_rate_e <= site_hi[s][e] (csr edge order) for the
 * edges with edge_mask[idx] != 0 (NULL = all); unrequested edges are 0 in both bounds.  sum_lo / sum_hi [E] enclose
 * sum_s w_s d[s][e]; they are summed on the device in a fixed order (the same bits on every call), a negative weight
 * swapping the bounds it multiplies.  Any output may be NULL.  The input uncertainties are those of plf_ll_certified.
 * Rate matrix derivatives r_c Q P_e come from R = P - 1 P_0 (R 1 = 0, so Q P = Q R and R(y)^2 = R(2y)): R is enclosed
 * where the scaled Taylor series is, then squared, so a long branch keeps its relative width (csrc/certified.cuh).
 * Certified: the bounds contain the exact derivative of the model given to the engine within those uncertainties.
 * Not certified: the host's inputs beyond them; and after plf_comm_init the sums cover this engine's sites only (no
 * directed-rounding all-reduce).  A site of non-zero weight whose likelihood enclosure reaches 0 makes the sums an
 * error ("a site with non-zero weight has zero likelihood"); its per-site bounds are -inf / +inf.  At most 75 states
 * ("state count ... is too large for the certified kernels" otherwise).
 */
int plf_deriv_certified(plf_engine *e, double delta_rate, double delta_q, const unsigned char *edge_mask /*[E] or NULL*/,
                        double *site_lo /*[S][E]*/, double *site_hi /*[S][E]*/, double *sum_lo /*[E]*/, double *sum_hi /*[E]*/);

/*
 * Certified mode for plf_marginal and plf_edge_expect: enclosures of exactly what those return, with the input
 * uncertainties, the errors, the 75-state limit, the fixed-order device sums and the sums after plf_comm_init (this
 * engine's sites only) of plf_deriv_certified.  Any output may be NULL.
 *   plf_marginal_certified: site_lo[s][v][i] <= marg <= site_hi[s][v][i] for every node v (root and leaves included)
 *     and state i; sum_lo / sum_hi [N][n] enclose sum_s w_s marg.  A state that a node's data excludes is 0.0 in both
 *     bounds.
 *   plf_edge_expect_certified: the same for the edge expectations of direction L = l_hi + l_lo (l_lo may be NULL) and
 *     kind PLF_KIND_DWELL or PLF_KIND_TRANS (any other kind is an error); unrequested edges (edge_mask) are 0.0 in
 *     both bounds.  L may have entries of both signs (F is linear in L: F(L+) - F(L-), the second only when L has a
 *     negative entry); each entry is taken within the relative delta_q, as a TRANS direction holds entries of Q.
 * The Frechet matrices F = the top-right block of exp([[A, L], [0, A]]), A = r_c t_e Q, are enclosed by the Taylor
 * series of the shifted block matrix, whose terms are non-negative for L >= 0 (csrc/certified.cuh).
 */
int plf_marginal_certified(plf_engine *e, double delta_rate, double delta_q, double *site_lo /*[S][N][n]*/,
                           double *site_hi /*[S][N][n]*/, double *sum_lo /*[N][n]*/, double *sum_hi /*[N][n]*/);
int plf_edge_expect_certified(plf_engine *e, double delta_rate, double delta_q, int kind,
                              const double *l_hi /*[n*n]*/, const double *l_lo /*[n*n] or NULL*/,
                              const unsigned char *edge_mask /*[E] or NULL*/,
                              double *site_lo /*[S][E]*/, double *site_hi /*[S][E]*/, double *sum_lo /*[E]*/, double *sum_hi /*[E]*/);

/*
 * Second order (arbplfhess.c:502-829): sum_ll = sum_s w_s log L_s, sum_deriv[E] its gradient and sum_hess[E][E] its
 * Hessian with respect to the edge rate coefficients (csr edge order, full symmetric matrix).  sum_ll and sum_deriv
 * may be NULL.  A rate category with a non-zero rate and zero likelihood at a weighted site is an error
 * ("infeasible", arbplfhess.c:640-660).
 */
int plf_hess(plf_engine *e, double *sum_ll, double *sum_deriv /*[E]*/, double *sum_hess /*[E][E]*/);

/* posterior marginals: site_marg [S][N][n], sum_marg [N][n] = sum_s w_s marg. */
int plf_marginal(plf_engine *e, double *site_marg, double *sum_marg);

/*
 * Posterior edge expectations from Frechet matrices with direction L (n x n,
 * double-double pair, l_lo may be NULL):
 *   PLF_KIND_DWELL: sum_c prior_c fe^T F L_b / L_site
 *   PLF_KIND_TRANS: sum_c prior_c rate_c t_e fe^T F L_b / L_site
 */
int plf_edge_expect(plf_engine *e, int kind,
                    const double *l_hi /*[n*n]*/, const double *l_lo,
                    const unsigned char *edge_mask,
                    double *site_out /*[S][E]*/, double *sum_out /*[E]*/);

/*
 * All Frechet directions of plf_edge_expect at once, summed over the sites with the site weights (edges in csr order,
 * no edge mask, no per-site output):
 *   dwell[e][i][j] = what plf_edge_expect(PLF_KIND_DWELL, L = E_ij) returns in sum_out[e]
 *   trans[e][i][j] = what plf_edge_expect(PLF_KIND_TRANS, L = E_ij) returns in sum_out[e]
 * so plf_edge_expect(kind, L)[e] == sum_ij L_ij X_kind[e][i][j] for every L; sum_ll = sum_s w_s log L_s.  Any output
 * may be NULL.  As in plf_edge_expect, a rate category of zero likelihood at a site adds nothing there (which only
 * shows in the off-diagonal dwell entries of a category of rate 0).  One pass over the sites: the edge form is bilinear in the outside and inside vectors, so the pass sums
 * G_{e,c} = sum_s w_s prior_c fe L_b^T / L_s and the directions come from the adjoint Frechet derivative at A^T.
 *
 * Gradient of the log-likelihood with respect to the rate matrix:
 *   d sum_ll / d Q_ij = sum_e trans[e][i][j]
 * where Q is the scaled matrix given to plf_set_model with its n^2 entries treated as independent, and the category
 * rates, category priors and root prior are held fixed.  The dependence of an equilibrium root prior on Q is not
 * included; the caller applies the chain rule for the rate divisor, the diagonal and the equilibrium.
 *
 * Errors as for the other queries (no configuration; a site of zero likelihood with non-zero weight).  After
 * plf_comm_init the sums are all-reduced like every other *_sum output.
 */
int plf_edge_expect_all(plf_engine *e, double *sum_ll, double *dwell /*[E][n][n]*/, double *trans /*[E][n][n]*/);

/* Copies of device-computed matrices, for tests: P[C][E][n][n] (row major). */
int plf_get_transition_matrices(plf_engine *e, double *p_out);
/* rate_c * Q * P, the matrices used by plf_deriv */
int plf_get_derivative_matrices(plf_engine *e, double *d_out);
/* Frechet matrices for a direction L (unscaled: the top-right block of util.c:500-548) */
int plf_get_frechet_matrices(plf_engine *e, const double *l_hi, const double *l_lo, double *f_out);

/*
 * Timing / accounting of the most recent query (CUDA events on the engine's
 * stream): milliseconds for the matrix kernels (expm etc.) and the per-site
 * kernels, and the number of kernel launches since the last reset.
 */
int plf_last_timing(plf_engine *e, float *ms_matrices, float *ms_sites);
/* duration of the dominant per-site kernel alone (the fused 4-state kernel), 0 if it did not run */
int plf_last_kernel_ms(plf_engine *e, float *ms_kernel);
int64_t plf_launch_count(plf_engine *e, int reset);
/* which instantiation ran as the dominant per-site kernel of the most recent query, spelled as the profiler spells it
 * (e.g. "fused4_kernel<4,1,512,2,1,1>": categories, mode, block size, staging, packed codes, constant-memory matrices;
 * the fused kernel's configuration is picked by timing, so this is the only way to know) */
const char *plf_last_kernel_name(const plf_engine *e);

/*
 * Multi-GPU: one engine per rank, sites sharded by the caller.  After
 * plf_comm_init the *_sum outputs are all-reduced (ncclAllReduce, sum, fp64) in
 * stream, right after the block reduction.  id is an ncclUniqueId (128 bytes).
 */
int plf_comm_unique_id(char id[128]);
int plf_comm_init(plf_engine *e, int nranks, int rank, const char id[128]);
/* paused != 0: the *_sum outputs stay local (this rank's sites only) until resumed; for cross-checks of the collective */
int plf_comm_pause(plf_engine *e, int paused);

/* The CUDA stream the engine launches on (cudaStream_t as void*), for event timing. */
void *plf_stream(plf_engine *e);
int plf_synchronize(plf_engine *e);

#ifdef __cplusplus
}
#endif
#endif
