/*
 * arbplf.h -- reference-facing C ABI of the B200 engine: one JSON document in,
 * one JSON document out.
 *
 * Each function replaces the string-level entry point that the reference
 * builds from its json_t-level driver through json_induced_string_hom
 * (runjson.h:28-33, runjson.c:10-77) and that its executables
 * (src/arbplf-ll.c:4-15 ...) and Python module (src/arbplf.c:208-250,521-534)
 * call:
 *
 *   arbplf_ll        <- arbplf_ll_run        (arbplfll.h:10,  arbplfll.c:291-323)
 *   arbplf_deriv     <- arbplf_deriv_run     (arbplfderiv.h:10, arbplfderiv.c:490-531)
 *   arbplf_marginal  <- arbplf_marginal_run  (arbplfmarginal.c:404-446)
 *   arbplf_dwell     <- arbplf_dwell_run     (arbplfdwell.c:570-610)
 *   arbplf_trans     <- arbplf_trans_run     (arbplftrans.c:612-660)
 *   arbplf_em_update <- arbplf_em_update_run (arbplfem.c:540-588): two trans-type passes
 *                       (exit rates on the diagonal / rates off the diagonal) and their ratio
 *
 * Contract (same as runjson.c:10-66): the returned string is malloc'd and
 * owned by the caller (free()); on failure NULL is returned, *retcode is
 * non-zero and a message has been written to stderr.  The input is borrowed.
 * The functions are not re-entrant (one shared engine handle per process).
 *
 * The second-order programs of the reference (hess, inv-hess, newton-*) are
 * outside this build's hot path; their entry points exist so that a binding
 * can link, and fail with retcode -1.
 */
#ifndef ARBPLF_B200_H
#define ARBPLF_B200_H

#ifdef __cplusplus
extern "C" {
#endif

char *arbplf_ll(const char *json_in, int *retcode);
char *arbplf_deriv(const char *json_in, int *retcode);
char *arbplf_marginal(const char *json_in, int *retcode);
char *arbplf_dwell(const char *json_in, int *retcode);
char *arbplf_trans(const char *json_in, int *retcode);
char *arbplf_em_update(const char *json_in, int *retcode);

/* arbplf-ll answered with an enclosure {"lower": table, "upper": table} (certified mode, directed rounding) */
char *arbplf_ll_certified(const char *json_in, int *retcode);
/* arbplf-deriv answered the same way (both tables in the format of arbplf-deriv) */
char *arbplf_deriv_certified(const char *json_in, int *retcode);
/* arbplf-marginal, arbplf-dwell and arbplf-trans answered the same way (each in its program's table format); site
 * aggregation is the engine's weighted sum, node, state, edge and transition aggregation are done with directed rounding
 * on the host or folded into the Frechet direction as the uncertified programs fold them (signed weights allowed) */
char *arbplf_marginal_certified(const char *json_in, int *retcode);
char *arbplf_dwell_certified(const char *json_in, int *retcode);
char *arbplf_trans_certified(const char *json_in, int *retcode);

char *arbplf_hess(const char *json_in, int *retcode);
char *arbplf_inv_hess(const char *json_in, int *retcode);
char *arbplf_newton_delta(const char *json_in, int *retcode);
char *arbplf_newton_update(const char *json_in, int *retcode);
char *arbplf_newton_refine(const char *json_in, int *retcode);

/* run_string_script of runjson.c:117-147: stdin -> f -> stdout, returns the exit status */
int arbplf_run_stdio(char *(*f)(const char *, int *));

/*
 * Site-independent part of a model, without touching the device: parses
 * {"model_and_data": ...} and returns what cross_site_ws_update computes
 * before the matrix exponentials (cross_site_ws.c:199-232) as JSON:
 * {"state_count", "category_count", "cat_rates", "cat_prior", "rate_divisor_expect",
 *  "equilibrium", "q_hi", "q_lo", "edge_rates_csr", "root_mode", "root_vec",
 *  "indptr", "indices", "preorder", "order", "definition_count", "codes_sum", "codes_weighted_sum"}
 * (the last two: sums over the site data as read, codes in row-major order, modulo 2^64, as strings).
 * Used by tools that drive the device seam (plf.h) with binary site data.
 */
char *arbplf_model_summary(const char *json_in, int *retcode);

/* Wall-clock seconds of the phases of the most recent arbplf_* call: JSON parse + schema validation, derived model
 * quantities + upload, device compute + reductions, output formatting (bench.py reports them as json_e2e). */
void arbplf_last_timing(double out[4]);

/* GPU ordinal used by the JSON entry points (default 0, or env ARBPLF_DEVICE). */
void arbplf_set_device(int device);

#ifdef __cplusplus
}
#endif
#endif
