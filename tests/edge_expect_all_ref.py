"""
Brute-force reference for plf_edge_expect_all: the oracle's edge expectations (its Frechet matrices and the
accumulation of _edge_expectations) looped over the n^2 elementary directions E_ij.  It does not use the adjoint identity
the engine relies on, so it checks that identity too.  Results are cached as tests/golden/edge_expect_all/<name>.npz
(generated on first use; the cache is committed so that GPU runs do not spend minutes in mpmath).
"""
import os

import numpy as np

from oracle import arbplf_oracle as O
from tests import helpers as H

CACHE = os.path.join(H.GOLDEN, "edge_expect_all")


def _edge_expectations(m, cs, be, base, F):
    """The oracle's _edge_expectations for dwell and trans at once, with the rule of plf_edge_expect for a category of
    zero likelihood at a site (arbplfem.c:322): it contributes nothing.  That only matters where the direction is
    off-diagonal and the category has rate 0 (the invariable category at a variable site)."""
    t = m.tree
    S = base.shape[0]
    site_L = be.zeros(S)
    xd = be.zeros(S, t.edge_count)
    xt = be.zeros(S, t.edge_count)
    for c in range(cs.C):
        lh, node, nconst, edge = O.site_lhood(m, cs, be, base, c, keep_edges=True)
        fn, fe = O.site_forward(m, cs, be, base, c, edge)
        site_L = site_L + cs.prior[c] * lh
        live = np.array([bool(x != 0) for x in lh])
        for idx in range(t.edge_count):
            x = (O._matvec(F[c, idx], node[t.indices[idx]]) * fe[idx]).sum(axis=1)
            x = np.where(live, x * cs.prior[c], be.num(0))
            xd[:, idx] = xd[:, idx] + x
            xt[:, idx] = xt[:, idx] + x * (cs.rates[c] * cs.edge_rates[idx])
    return xd / site_L[:, None], xt / site_L[:, None]


def per_site_edge_expect_all(m, be, sites):
    """Per-site dwell and trans matrices [S', E, n, n] (csr edge order): entry [s, e, i, j] is the edge expectation
    (per_site_edge_expect) of site s and edge e for the direction E_ij."""
    t = m.tree
    n, E = m.n, t.edge_count
    cs = O.cross_site(m, be)
    base = O._base_vectors(m, be, sites)
    req = [True] * E
    dt = np.float64 if be.name == "fp64" else object
    Xd = np.empty((len(sites), E, n, n), dtype=dt)
    Xt = np.empty((len(sites), E, n, n), dtype=dt)
    for i in range(n):
        for j in range(n):
            L = be.zeros(n, n)
            L[i, j] = be.num(1)
            Xd[:, :, i, j], Xt[:, :, i, j] = _edge_expectations(m, cs, be, base, O.frechet_matrices(cs, be, L, req))
    return Xd, Xt, cs


def reference(name, prob, mode="mp"):
    """{"ll": [S], "Xd": [S, E, n, n], "Xt": [S, E, n, n]} for every site of prob, in fp64."""
    path = os.path.join(CACHE, name + ".npz")
    if os.path.exists(path):
        z = np.load(path)
        return {k: z[k] for k in z.files}
    m = O.parse_model(prob["model_and_data"])
    be = O.get_backend(mode)
    sites = list(range(m.site_count))
    ll, _, _ = O.per_site_ll_and_deriv(m, be, sites, want_deriv=False)
    Xd, Xt, _ = per_site_edge_expect_all(m, be, sites)
    out = {"ll": H._fl(ll), "Xd": H._fl(Xd), "Xt": H._fl(Xt)}
    os.makedirs(CACHE, exist_ok=True)
    np.savez_compressed(path, **out)
    return out
