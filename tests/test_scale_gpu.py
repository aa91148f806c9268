"""
Parity at BASELINE.json's sizes (SURVEY.md section 8d), where the 320-bit oracle is too slow:
  cfg2  1M sites x 64 taxa, GTR+Gamma4: fused kernel vs the C restatement (itself pinned on the
        320-bit oracle, tests/test_oracle_c.py) on ALL sites, plus linearity in the site weights;
  cfg3  HKY85+I marginals on 128 taxa: posterior marginals sum to 1 at every (site, node);
  cfg4  61-state codon model: tensor-pipe kernels vs the C restatement (16 taxa, and 256 taxa x 100k sites),
        matrices vs scipy expm;
  cfg5  dwell / trans on the cfg2 model: dwell over all states is exactly the edge (1 per site),
        fused path vs generic path (independent kernels) for a weighted trans direction.
"""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _bench():
    import bench
    return bench


def _problem(sites, taxa=64):
    b = _bench()

    class A:
        pass
    args = A()
    args.taxa = taxa
    args.sites = sites
    return b, b.build_problem(args, 0, 0)


def test_cfg2_full_size_against_c_port():
    from oracle import c_port
    b, pb = _problem(1000000)
    eng = pb["eng"]
    defs = np.array(b.DEFS, dtype=np.float64)
    eng.set_data(defs, pb["codes"])
    rng = np.random.default_rng(7)
    w = 1.0 + rng.poisson(3.0, pb["S"]).astype(np.float64)        # SURVEY 8d: weights ~ 1 + Poisson(3)
    eng.set_site_weights(w)
    r = eng.deriv(per_site=False)
    s = pb["summary"]
    D = eng.derivative_matrices()
    P = eng.transition_matrices()
    _, sum_ll, sum_d = c_port.ll_deriv(s["indptr"], s["indices"], s["preorder"], P, D, np.array(s["cat_prior"]),
                                       s["root_mode"], np.array(s["root_vec"]), pb["codes"], defs, w=w,
                                       want_site_ll=False)
    assert abs(r["sum_ll"] - sum_ll) <= 1e-11 * abs(sum_ll)
    scale = np.abs(sum_d).max()
    assert np.all(np.abs(r["sum_deriv"] - sum_d) <= 1e-11 * np.abs(sum_d) + 1e-12 * scale)
    # linearity in the weights: two halves add up to the whole
    w1 = w.copy(); w1[pb["S"] // 2:] = 0
    w2 = w - w1
    eng.set_site_weights(w1); r1 = eng.deriv(per_site=False)
    eng.set_site_weights(w2); r2 = eng.deriv(per_site=False)
    assert abs(r1["sum_ll"] + r2["sum_ll"] - r["sum_ll"]) <= 1e-12 * abs(r["sum_ll"])
    assert np.all(np.abs(r1["sum_deriv"] + r2["sum_deriv"] - r["sum_deriv"]) <= 1e-11 * np.abs(r["sum_deriv"]) + 1e-12 * scale)
    # per-site log-likelihoods of a subsample against the C port
    site_ll, _ = eng.ll(per_site=True)
    idx = rng.choice(pb["S"], 5000, replace=False)
    ref_ll, _, _ = c_port.ll_deriv(s["indptr"], s["indices"], s["preorder"], P, None, np.array(s["cat_prior"]),
                                   s["root_mode"], np.array(s["root_vec"]), pb["codes"][idx], defs, want_deriv=False)
    np.testing.assert_allclose(site_ll[idx], ref_ll, rtol=1e-11, atol=2e-15)
    eng.close()


def test_cfg5_dwell_is_one_and_paths_agree():
    from phyly_b200 import engine as E
    b, pb = _problem(60000)
    eng = pb["eng"]
    defs = np.array(b.DEFS, dtype=np.float64)
    eng.set_data(defs, pb["codes"])
    n = 4
    # dwell with all states: the chain is always somewhere -> exactly 1 per (site, edge)
    so, tot = eng.edge_expect(E.KIND_DWELL, np.eye(n), per_site=False)
    np.testing.assert_allclose(tot, pb["S"], rtol=1e-12)
    # a weighted trans direction through both kernel families
    q = np.array(pb["summary"]["q_hi"]).reshape(n, n)
    L = q * (1.0 + np.arange(16).reshape(4, 4) % 3)
    np.fill_diagonal(L, 0.0)
    eng.set_path(E.PATH_FUSED4)
    _, t_f = eng.edge_expect(E.KIND_TRANS, L, per_site=False)
    eng.set_path(E.PATH_GENERIC)
    _, t_g = eng.edge_expect(E.KIND_TRANS, L, per_site=False)
    np.testing.assert_allclose(t_f, t_g, rtol=1e-11)
    # per-site dwell / trans of a subsample of the 64-taxon alignment against the numpy oracle (fp64 back end)
    from oracle import arbplf_oracle as O
    rng = np.random.default_rng(17)
    idx = np.sort(rng.choice(pb["S"], 48, replace=False))
    md = dict(pb["doc"]["model_and_data"])
    md["character_data"] = pb["codes"][idx].tolist()
    m = O.parse_model(md)
    be = O.get_backend("fp64")
    Ld = np.diag([1.0, 0.0, 0.5, 0.0])
    want_d, _ = O.per_site_edge_expect(m, be, list(range(idx.size)), Ld, trans=False)
    want_t, _ = O.per_site_edge_expect(m, be, list(range(idx.size)), L, trans=True)
    for path in (E.PATH_FUSED4, E.PATH_GENERIC):
        eng.set_path(path)
        so_d, _ = eng.edge_expect(E.KIND_DWELL, Ld)
        so_t, _ = eng.edge_expect(E.KIND_TRANS, L)
        np.testing.assert_allclose(so_d[idx], np.asarray(want_d, dtype=np.float64), rtol=1e-10, atol=1e-14)
        np.testing.assert_allclose(so_t[idx], np.asarray(want_t, dtype=np.float64), rtol=1e-10, atol=1e-14)
    eng.close()


def _hky_doc(taxa, kappa=2.0, pi=(0.3, 0.2, 0.25, 0.25)):
    b = _bench()
    edges, N = b.yule_tree(taxa, seed=11)
    rng = np.random.default_rng(12)
    Q = [[0.0] * 4 for _ in range(4)]
    for i in range(4):
        for j in range(4):
            if i != j:
                ts = (i, j) in ((0, 2), (2, 0), (1, 3), (3, 1))
                Q[i][j] = pi[j] * (kappa if ts else 1.0)
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.05, len(edges))],
          "rate_matrix": Q, "root_prior": list(pi), "rate_divisor": "equilibrium_exit_rate",
          "rate_mixture": {"rates": [0.0, 2.0], "prior": [0.5, 0.5]},
          "character_definitions": b.DEFS, "character_data": [[4] * N]}
    return {"model_and_data": md}, N


def test_cfg3_marginals_sum_to_one():
    import phyly_b200.arbplf as A
    from phyly_b200.engine import Engine
    b = _bench()
    doc, N = _hky_doc(128)
    s = json.loads(A.arbplf_model_summary(json.dumps(doc)))
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(4, 4), np.array(s["q_lo"]).reshape(4, 4), s["edge_rates_csr"],
                  s["cat_rates"], s["cat_prior"], s["root_mode"], s["root_vec"])
    P = eng.transition_matrices()
    S = 4096
    codes = np.empty((S, N), dtype=np.uint8)
    b.simulate_codes(s, P, S, seed=13, out=codes)
    eng.set_data(np.array(b.DEFS, dtype=np.float64), codes)
    sm, tot = eng.marginal()
    np.testing.assert_allclose(sm.sum(axis=2), 1.0, rtol=0, atol=1e-12)
    # observed leaves are certain
    leaf = [a for a in range(N) if s["indptr"][a] == s["indptr"][a + 1]][0]
    obs = codes[:, leaf] < 4
    assert np.allclose(sm[obs, leaf, :].max(axis=1), 1.0, atol=1e-12)
    np.testing.assert_allclose(tot, sm.sum(axis=0), rtol=1e-11, atol=1e-9)
    # the fused kernel (used above) against the independent generic kernels, per site
    from phyly_b200 import engine as E
    eng.set_path(E.PATH_GENERIC)
    sm_g, tot_g = eng.marginal()
    np.testing.assert_allclose(sm, sm_g, rtol=1e-11, atol=1e-14)
    np.testing.assert_allclose(tot, tot_g, rtol=1e-11, atol=1e-9)
    # a subsample of the 128-taxon columns against the numpy oracle (fp64 back end; same node numbering)
    from oracle import arbplf_oracle as O
    idx = np.sort(np.random.default_rng(18).choice(S, 64, replace=False))
    md = dict(doc["model_and_data"])
    md["character_data"] = codes[idx].tolist()
    m = O.parse_model(md)
    want = np.asarray(O.per_site_marginal(m, O.get_backend("fp64"), list(range(idx.size))), dtype=np.float64)
    np.testing.assert_allclose(sm[idx], want, rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(sm_g[idx], want, rtol=1e-10, atol=1e-14)
    eng.close()


def _codon_model(**kw):
    """GY94-style 61-state rate matrix with F3x4 frequencies (SURVEY 8d cfg4); bench.py owns the definition."""
    return _bench().codon_model(**kw)


def test_cfg4_codon_generic_path_against_c_port():
    import scipy.linalg
    import phyly_b200.arbplf as A
    from oracle import c_port
    from phyly_b200.engine import Engine
    b = _bench()
    Q, pi = _codon_model()
    n = Q.shape[0]
    assert n == 61
    edges, N = b.yule_tree(16, seed=21)
    rng = np.random.default_rng(22)
    defs = np.vstack([np.eye(n), np.ones((1, n))])
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.1, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "character_definitions": defs.tolist(), "character_data": [[n] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    np.testing.assert_allclose(s["equilibrium"], pi, rtol=1e-12)
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    qh = np.array(s["q_hi"]).reshape(n, n)
    eng.set_model(qh, np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"], s["cat_prior"],
                  s["root_mode"], s["root_vec"])
    P = eng.transition_matrices()
    D = eng.derivative_matrices()
    for e in range(0, N - 1, 7):
        Pw = scipy.linalg.expm(qh * s["edge_rates_csr"][e])
        np.testing.assert_allclose(P[0, e], Pw, rtol=1e-10, atol=1e-15)
        np.testing.assert_allclose(D[0, e], qh @ Pw, rtol=1e-9, atol=1e-13)
    # data: random codons at the leaves (5 % missing), internal nodes unobserved
    S = 300
    codes = np.full((S, N), n, dtype=np.uint8)
    for a in range(N):
        if s["indptr"][a] == s["indptr"][a + 1]:
            col = rng.integers(0, n, S)
            col[rng.random(S) < 0.05] = n
            codes[:, a] = col
    eng.set_data(defs, codes)
    w = rng.random(S) + 0.5
    eng.set_site_weights(w)
    r = eng.deriv(per_site=False)
    site_ll, _ = eng.ll()
    ref_ll, sum_ll, sum_d = c_port.ll_deriv(s["indptr"], s["indices"], s["preorder"], P, D, np.array(s["cat_prior"]),
                                            s["root_mode"], np.array(s["root_vec"]), codes, defs, w=w)
    np.testing.assert_allclose(site_ll, ref_ll, rtol=1e-11)
    assert abs(r["sum_ll"] - sum_ll) <= 1e-11 * abs(sum_ll)
    np.testing.assert_allclose(r["sum_deriv"], sum_d, rtol=1e-11, atol=1e-12 * np.abs(sum_d).max())
    # the same through the tile / scalar kernels (forced generic path)
    from phyly_b200 import engine as E
    eng.set_path(E.PATH_GENERIC)
    rg = eng.deriv(per_site=False)
    np.testing.assert_allclose(rg["sum_deriv"], sum_d, rtol=1e-11, atol=1e-12 * np.abs(sum_d).max())
    eng.close()


def test_cfg4_full_size_against_c_port():
    """BASELINE cfg4 at its full size: 61-state codon model, 256 taxa x 100 000 sites (deep-tree rescaling inside the
    tensor-pipe kernels, ragged tiles, the evenly spread last wave).  Per-site ll of a fixed 1000-site subsample and
    the derivative sums over that subsample against the C restatement at 1e-11; all sites through linearity."""
    import phyly_b200.arbplf as A
    from oracle import c_port
    from phyly_b200.engine import Engine
    b = _bench()
    Q, pi = _codon_model()
    n = Q.shape[0]
    taxa, S = 256, 100000
    edges, N = b.yule_tree(taxa, seed=21)
    rng = np.random.default_rng(23)
    defs = np.vstack([np.eye(n), np.ones((1, n))])
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.05, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "character_definitions": defs.tolist(), "character_data": [[n] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(n, n), np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    P = eng.transition_matrices()
    D = eng.derivative_matrices()
    # columns evolved down the tree (realistic, deep underflow): 25 000 simulated, repeated with fresh missing data
    base = np.full((S // 4, N), n, dtype=np.uint8)
    b.simulate_codes(s, P, S // 4, seed=24, out=base, pi=np.array(s["equilibrium"]), missing=0.0)
    codes = np.tile(base, (4, 1))
    leaves = np.array([a for a in range(N) if s["indptr"][a] == s["indptr"][a + 1]])
    sub = codes[:, leaves]
    sub[rng.random(sub.shape) < 0.02] = n
    codes[:, leaves] = sub
    eng.set_data(defs, codes)
    idx = np.sort(rng.choice(S, 1000, replace=False))
    w = np.zeros(S)
    w[idx] = 1.0 + rng.poisson(3.0, idx.size)
    eng.set_site_weights(w)
    r = eng.deriv(per_site=False)
    site_ll, tot = eng.ll()
    assert np.mean(site_ll < -256 * np.log(2.0)) > 0.1      # many sites below 2^-256: the per-site rescaling is exercised
    ref_ll, sum_ll, sum_d = c_port.ll_deriv(s["indptr"], s["indices"], s["preorder"], P, D, np.array(s["cat_prior"]),
                                            s["root_mode"], np.array(s["root_vec"]), codes[idx], defs, w=w[idx])
    np.testing.assert_allclose(site_ll[idx], ref_ll, rtol=1e-11)
    assert abs(r["sum_ll"] - sum_ll) <= 1e-11 * abs(sum_ll)
    assert abs(tot - sum_ll) <= 1e-11 * abs(sum_ll)
    np.testing.assert_allclose(r["sum_deriv"], sum_d, rtol=1e-11, atol=1e-12 * np.abs(sum_d).max())
    # every site: the two halves of a random split add up to the whole (ll and derivative sums)
    wa = 1.0 + rng.poisson(2.0, S).astype(np.float64)
    w1 = wa * (rng.random(S) < 0.5)
    eng.set_site_weights(wa); ra = eng.deriv(per_site=False)
    eng.set_site_weights(w1); r1 = eng.deriv(per_site=False)
    eng.set_site_weights(wa - w1); r2 = eng.deriv(per_site=False)
    assert abs(r1["sum_ll"] + r2["sum_ll"] - ra["sum_ll"]) <= 1e-12 * abs(ra["sum_ll"])
    scale = np.abs(ra["sum_deriv"]).max()
    assert np.all(np.abs(r1["sum_deriv"] + r2["sum_deriv"] - ra["sum_deriv"]) <= 1e-11 * np.abs(ra["sum_deriv"]) + 1e-12 * scale)
    assert abs(np.dot(wa, site_ll) - ra["sum_ll"]) <= 1e-12 * abs(ra["sum_ll"])
    eng.close()


def test_amino_acid_sized_model_against_c_port():
    """A 20-state reversible model (3 state blocks in the tensor-pipe kernels of dmma.cu): ll, ll+deriv and
    marginals on a 40-taxon tree against the C restatement / the independent scalar kernels."""
    import phyly_b200.arbplf as A
    from oracle import c_port
    from phyly_b200.engine import Engine
    b = _bench()
    rng = np.random.default_rng(77)
    n = 20
    pi = rng.dirichlet(np.ones(n) * 4)
    R = rng.random((n, n)) + 0.05
    R = (R + R.T) / 2
    Q = R * pi[None, :]
    np.fill_diagonal(Q, 0.0)
    edges, N = b.yule_tree(40, seed=5)
    defs = np.vstack([np.eye(n), np.ones((1, n))])
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.15, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "rate_mixture": {"rates": [0.3, 1.7], "prior": [0.4, 0.6]},
          "character_definitions": defs.tolist(), "character_data": [[n] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(n, n), np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    P = eng.transition_matrices()
    D = eng.derivative_matrices()
    S = 1000 + 37                                   # ragged last tile
    codes = np.full((S, N), n, dtype=np.uint8)
    for a in range(N):
        if s["indptr"][a] == s["indptr"][a + 1]:
            col = rng.integers(0, n, S)
            col[rng.random(S) < 0.05] = n
            codes[:, a] = col
    eng.set_data(defs, codes)
    w = rng.random(S) + 0.5
    eng.set_site_weights(w)
    r = eng.deriv(per_site=False)
    site_ll, _ = eng.ll()
    ref_ll, sum_ll, sum_d = c_port.ll_deriv(s["indptr"], s["indices"], s["preorder"], P, D, np.array(s["cat_prior"]),
                                            s["root_mode"], np.array(s["root_vec"]), codes, defs, w=w)
    np.testing.assert_allclose(site_ll, ref_ll, rtol=1e-11)
    assert abs(r["sum_ll"] - sum_ll) <= 1e-11 * abs(sum_ll)
    np.testing.assert_allclose(r["sum_deriv"], sum_d, rtol=1e-11, atol=1e-12 * np.abs(sum_d).max())
    # marginals: tile kernels against the scalar generic kernels (PLF_NO_TILE is read per query)
    sm, tot = eng.marginal()
    np.testing.assert_allclose(sm.sum(axis=2), 1.0, rtol=0, atol=1e-12)
    os.environ["PLF_NO_TILE"] = "1"
    try:
        sm_g, tot_g = eng.marginal()
        r_g = eng.deriv(per_site=False)
    finally:
        del os.environ["PLF_NO_TILE"]
    np.testing.assert_allclose(sm, sm_g, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(r["sum_deriv"], r_g["sum_deriv"], rtol=1e-11, atol=1e-12 * np.abs(sum_d).max())
    eng.close()


def test_async_upload_matches_synchronous_upload():
    """plf_set_data_async (chunked upload overlapped with the fused kernel) gives the sums of plf_set_data:
    several chunks with a ragged tail, per-site outputs, and a change of which nodes carry data between two
    uploads (the cached tree program is then stale and the query repeats itself)."""
    b, pb = _problem(400001)
    eng = pb["eng"]
    defs = np.array(b.DEFS, dtype=np.float64)
    codes = pb["codes"]
    rng = np.random.default_rng(11)
    w = 1.0 + rng.poisson(3.0, pb["S"]).astype(np.float64)
    eng.set_data(defs, codes)
    eng.set_site_weights(w)
    want = eng.deriv(per_site=True, per_site_ll=True)
    want_ll = eng.ll(per_site=False)[1]
    for _ in range(2):
        eng.set_data_async(defs, codes, w)
        got = eng.deriv(per_site=True, per_site_ll=True)
        assert abs(got["sum_ll"] - want["sum_ll"]) <= 1e-13 * abs(want["sum_ll"])
        assert np.allclose(got["sum_deriv"], want["sum_deriv"], rtol=1e-12, atol=1e-12 * np.abs(want["sum_deriv"]).max())
        assert np.array_equal(got["site_ll"], want["site_ll"])
        assert np.array_equal(got["site_deriv"], want["site_deriv"])
    eng.set_data_async(defs, codes, w)
    assert abs(eng.ll(per_site=False)[1] - want_ll) <= 1e-13 * abs(want_ll)
    # wipe the data of one leaf: the program built for the previous upload no longer applies
    codes2 = codes.copy()
    leaf = int(np.flatnonzero((codes != 4).any(axis=0))[0])
    codes2[:, leaf] = 4
    eng.set_data(defs, codes2)
    eng.set_site_weights(w)
    want2 = eng.deriv(per_site=False)
    eng.set_data(defs, codes)
    eng.set_site_weights(w)
    eng.deriv(per_site=False)
    eng.set_data_async(defs, codes2, w)
    got2 = eng.deriv(per_site=False)
    assert abs(got2["sum_ll"] - want2["sum_ll"]) <= 1e-13 * abs(want2["sum_ll"])
    assert np.allclose(got2["sum_deriv"], want2["sum_deriv"], rtol=1e-12, atol=1e-12 * np.abs(want2["sum_deriv"]).max())
    # an upload in flight followed by a query on the generic path (marginals) simply waits for it
    eng.set_data_async(defs, codes, w)
    tot = eng.marginal(per_site=False)[1]
    assert np.allclose(tot.sum(axis=1), w.sum(), rtol=1e-11)


# What each forced index of PLF_F4_CONFIG_MARG / PLF_F4_CONFIG / PLF_F4_CONFIG_LL selects in
# test_every_fused_configuration_agrees, per problem (taxa): the template arguments of fused4_kernel<...> for the
# (marginal, edge forms, ll) query, None where no configuration fits.  The indices are positions in the candidate
# tables of plf_engine.cu that tools/cfg_sweep.py and the recorded profiles refer to.  Recorded on an NVIDIA B200.
FORCED_KERNELS = {
    24: [
        ("4,2,384,1,1,0", "4,1,512,2,1,1", "4,0,512,2,1,1"),
        ("4,2,384,1,0,0", "4,1,512,2,0,1", "4,0,512,2,1,0"),
        ("4,2,256,1,0,0", "4,1,384,2,0,1", "4,0,512,2,0,1"),
        ("4,2,384,0,1,0", "4,1,384,2,1,0", "4,0,384,2,1,0"),
        ("4,2,384,0,0,0", "4,1,384,1,0,0", "4,0,384,2,1,0"),
        ("4,2,256,0,0,0", "4,1,512,1,0,0", "4,0,384,1,0,0"),
        ("4,2,128,0,0,0", "4,1,256,2,0,0", "4,0,256,2,0,0"),
        (None, "4,1,512,0,1,0", "4,0,256,2,0,0"),
        (None, "4,1,384,0,1,0", "4,0,512,0,1,0"),
        (None, "4,1,384,0,0,0", "4,0,384,0,1,0"),
        (None, "4,1,256,0,0,0", "4,0,384,0,0,0"),
        (None, "4,1,128,0,0,0", "4,0,256,0,0,0"),
        (None, None, "4,0,128,0,0,0"),
        (None, None, "4,0,128,0,0,0"),
        (None, None, None),
        (None, None, None),
    ],
    160: [
        (None, None, None),
        (None, None, None),
        (None, None, None),
        ("4,2,384,0,1,0", None, None),
        ("4,2,384,0,0,0", None, None),
        ("4,2,256,0,0,0", None, None),
        ("4,2,128,0,0,0", None, None),
        (None, "4,1,512,0,1,0", None),
        (None, "4,1,384,0,1,0", "4,0,512,0,1,0"),
        (None, "4,1,384,0,0,0", "4,0,384,0,1,0"),
        (None, "4,1,256,0,0,0", "4,0,384,0,0,0"),
        (None, "4,1,128,0,0,0", "4,0,256,0,0,0"),
        (None, None, "4,0,128,0,0,0"),
        (None, None, "4,0,128,0,0,0"),
        (None, None, None),
        (None, None, None),
    ],
}


def test_every_fused_configuration_agrees(monkeypatch):
    """Each candidate configuration of the fused kernel (block size, staged / unstaged tables with prefetch,
    packed codes, constant-memory matrices, shared / global stack) is forced in turn on one problem and must
    reproduce the sums of the default choice; the same for a tree too large for the constant-memory kernels.
    Each index must also still select the kernel it selected when FORCED_KERNELS was recorded."""
    from phyly_b200.engine import EngineError
    for taxa, sites in ((24, 30000), (160, 6000)):
        b, pb = _problem(sites, taxa)
        eng = pb["eng"]
        defs = np.array(b.DEFS, dtype=np.float64)
        eng.set_data(defs, pb["codes"])
        rng = np.random.default_rng(5)
        w = 1.0 + rng.poisson(2.0, pb["S"]).astype(np.float64)
        eng.set_site_weights(w)
        monkeypatch.delenv("PLF_F4_CONFIG", raising=False)
        monkeypatch.delenv("PLF_F4_CONFIG_LL", raising=False)
        monkeypatch.delenv("PLF_F4_CONFIG_MARG", raising=False)
        want = eng.deriv(per_site=False)
        want_ll = eng.ll(per_site=False)[1]
        want_mg = eng.marginal(per_site=False)[1]
        scale = np.abs(want["sum_deriv"]).max()
        ran_edge = ran_ll = ran_mg = 0
        for i in range(16):
            want_k = ["fused4_kernel<%s>" % k if k else None for k in FORCED_KERNELS[taxa][i]]
            monkeypatch.setenv("PLF_F4_CONFIG", str(i))
            monkeypatch.setenv("PLF_F4_CONFIG_LL", str(i))
            monkeypatch.setenv("PLF_F4_CONFIG_MARG", str(i))
            try:
                got_mg = eng.marginal(per_site=False)[1]
            except EngineError as ex:
                assert "no configuration fits" in str(ex) and want_k[0] is None, (taxa, i, ex)
            else:
                ran_mg += 1
                assert eng.last_kernel_name() == want_k[0], (taxa, i)
                assert np.allclose(got_mg, want_mg, rtol=1e-11, atol=1e-12 * np.abs(want_mg).max()), (taxa, i)
            try:
                got = eng.deriv(per_site=False)
            except EngineError as ex:
                assert "no configuration fits" in str(ex) and want_k[1] is None, (taxa, i, ex)
            else:
                ran_edge += 1
                assert eng.last_kernel_name() == want_k[1], (taxa, i)
                assert abs(got["sum_ll"] - want["sum_ll"]) <= 1e-12 * abs(want["sum_ll"]), (taxa, i)
                assert np.all(np.abs(got["sum_deriv"] - want["sum_deriv"]) <= 1e-11 * np.abs(want["sum_deriv"]) + 1e-12 * scale), (taxa, i)
            try:
                got_ll = eng.ll(per_site=False)[1]
            except EngineError as ex:
                assert "no configuration fits" in str(ex) and want_k[2] is None, (taxa, i, ex)
            else:
                ran_ll += 1
                assert eng.last_kernel_name() == want_k[2], (taxa, i)
                assert abs(got_ll - want_ll) <= 1e-12 * abs(want_ll), (taxa, i)
        assert ran_edge >= 3 and ran_ll >= 3 and ran_mg >= 2, (taxa, ran_edge, ran_ll, ran_mg)
        eng.close()
