"""
CPU check of the brute-force reference of plf_edge_expect_all (tests/edge_expect_all_ref.py): summed over the edges,
its trans matrices are the gradient of the log-likelihood with respect to the entries of the scaled rate matrix, with
category rates, category priors and the root prior held fixed (include/plf.h).  Compared with central finite
differences of the oracle's log-likelihood, everything in 320-bit arithmetic.  The data has no missing characters:
a perturbed entry breaks the zero row sums of Q, and with them the shortcut the likelihood takes for constant columns
(P 1 = 1), which the gradient of the matrix function does not see.
"""
import dataclasses

import numpy as np
from mpmath import mpf

from oracle import arbplf_oracle as O
from tests import helpers as H
from tests import edge_expect_all_ref as R


def _total_ll(m, cs, be, base, Q):
    """sum_s log L_s with the transition matrices recomputed from the scaled matrix Q."""
    P = np.empty(cs.P.shape, dtype=object)
    for c in range(cs.C):
        for e in range(cs.E):
            s = cs.rates[c] * cs.edge_rates[e]
            P[c, e] = be.asarray(np.eye(m.n)) if s == 0 else be.expm(Q * s)
    tot, _ = O._site_likelihoods(m, dataclasses.replace(cs, Q=Q, P=P), be, base)
    return sum(be.log(x) for x in tot)


def test_trans_summed_over_edges_is_the_rate_matrix_gradient():
    prob = H.random_problem(301, ntips=4, n=3, S=3, ncat=2, root="equilibrium_distribution", missing=0.0)
    m = O.parse_model(prob["model_and_data"])
    be = O.get_backend("mp")
    sites = list(range(m.site_count))
    _, Xt, cs = R.per_site_edge_expect_all(m, be, sites)
    grad = Xt.sum(axis=(0, 1))                      # sum over sites and edges: [n, n]
    base = O._base_vectors(m, be, sites)
    h = mpf(10) ** -30
    n = m.n
    for i in range(n):
        for j in range(n):
            Qp, Qm = cs.Q.copy(), cs.Q.copy()
            Qp[i, j] += h
            Qm[i, j] -= h
            fd = (_total_ll(m, cs, be, base, Qp) - _total_ll(m, cs, be, base, Qm)) / (2 * h)
            assert abs(fd - grad[i, j]) <= mpf(10) ** -25 * max(abs(x) for x in grad.flatten()), (i, j, fd, grad[i, j])
