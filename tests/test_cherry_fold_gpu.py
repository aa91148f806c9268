"""
Folded cherries on the fused 4-state path (plf_engine.cu: build_program, f4_tables_kernel; fused4.cuh): ll and edge-form
queries on trees whose cherries fold into per-code-pair tables meet the 320-bit oracle, give the bits of the unfolded
program (run by padding the character count past the fold budget) where they are meant to, and leave the marginal and
edge-matrix queries on their kernels.
"""
import numpy as np
import pytest

from oracle import arbplf_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

RTOL = 1e-11
CANCEL = 2e-14          # floors of tests/test_engine_gpu.py
LL_ATOL = 2e-15
K_PAD = 40              # character count at which no cherry of these trees fits the fold budget


def _assert_close(got, want, what, rtol=RTOL, atol=0.0):
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = np.abs(got - want)
    bad = ~(err <= rtol * np.abs(want) + atol)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError("%s: %d mismatches, first at %s: got %r want %r" % (what, bad.sum(), i, got[i], want[i]))


def _rescale_cherry_problem():
    """Root -> (cherry of two tips on edges of rate 1e-80, cherry): where the two tips differ, every entry of the first
    cherry's inside vector is below 2^-256, so the cherry is rescaled."""
    n = 4
    rng = np.random.default_rng(40)
    Q = rng.random((n, n)) + 0.05
    np.fill_diagonal(Q, 0.0)
    codes = [(0, 1, 2, 2), (2, 3, 0, 1), (1, 1, 3, 0), (0, 4, 1, 1), (3, 0, 4, 4), (2, 2, 2, 2), (1, 3, 0, 3)]
    data = [[4, 4, 4, c[0], c[1], c[2], c[3]] for c in codes]
    md = {
        "edges": [[0, 1], [0, 2], [1, 3], [1, 4], [2, 5], [2, 6]],
        "edge_rate_coefficients": [0.1, 0.2, 1e-80, 1e-80, 0.3, 0.15],
        "rate_matrix": [[float(x) for x in row] for row in Q],
        "rate_divisor": "equilibrium_exit_rate",
        "root_prior": [0.1, 0.2, 0.3, 0.4],
        "gamma_rate_mixture": {"gamma_shape": 0.7, "gamma_categories": 2},
        "character_definitions": [[1.0 if i == k else 0.0 for i in range(n)] for k in range(n)] + [[1.0] * n],
        "character_data": data,
    }
    return {"model_and_data": md}


PROBLEMS = [
    ("cherry1", H.random_problem(41, ntips=9, n=4, S=13, ncat=4, mixture="gamma", missing=0.2)),
    ("cherry2", H.random_problem(42, ntips=14, n=4, S=11, ncat=1)),
    ("cherry3", H.random_problem(43, ntips=10, n=4, S=9, ncat=3, max_degree=3, root_degree=3)),
    ("cherry4", H.random_problem(44, ntips=11, n=4, S=10, ncat=2, internal_data=True, root="uniform_distribution")),
    ("cherry5", H.random_problem(45, ntips=3, n=4, S=8, ncat=2)),
    ("cherry6", H.random_problem(46, ntips=2, n=4, S=6, ncat=2, root="equilibrium_distribution")),
    ("cherry7", H.random_problem(47, ntips=4, n=4, S=12, ncat=4, mixture="gamma", root_degree=2)),
    ("cherry_rescale", _rescale_cherry_problem()),
]
IDS = [p[0] for p in PROBLEMS]


def _folded_tip_edges(m):
    """csr positions of the edges to the tips of the cherries the engine folds (build_program's rule)"""
    t = m.tree
    N = t.node_count
    deg = [t.indptr[a + 1] - t.indptr[a] for a in range(N)]
    parent = [-1] * N
    for a in range(N):
        for j in range(t.indptr[a], t.indptr[a + 1]):
            parent[t.indices[j]] = a
    dense = m.dense_pmat()
    data = [bool(np.any(dense[:, a, :] != 1.0)) for a in range(N)]
    out = []
    for b in range(N):
        p = parent[b]
        if p < 0 or deg[b] != 2 or deg[p] != 2 or data[b] or data[p]:
            continue
        kids = t.indices[t.indptr[b]:t.indptr[b + 1]]
        if all(deg[k] == 0 for k in kids):
            out += [t.indptr[b], t.indptr[b] + 1]
    return np.array(out, dtype=int)


def _engine(m, K=None):
    from phyly_b200 import engine as E
    eng = E.Engine(0)
    cs = H.fill_engine(eng, m)
    if K:
        defs, codes = H.dedupe_rows(m.dense_pmat())
        extra = np.random.default_rng(7).random((K - defs.shape[0], m.n)) + 0.05
        eng.set_data(np.vstack([defs, extra]), codes.astype(np.int32))
    eng.set_path(E.PATH_FUSED4)
    return eng, cs


def _binary(m):
    t = m.tree
    return all(t.indptr[a + 1] - t.indptr[a] in (0, 2) for a in range(t.node_count))


def test_the_problems_have_folded_cherries():
    folded = {name: len(_folded_tip_edges(O.parse_model(p["model_and_data"]))) // 2 for name, p in PROBLEMS}
    assert folded["cherry5"] == 1 and folded["cherry6"] == 0 and folded["cherry_rescale"] == 2, folded
    assert all(folded[k] > 0 for k in ("cherry1", "cherry2", "cherry3", "cherry7")), folded


@pytest.mark.parametrize("config", [None, 0])
@pytest.mark.parametrize("name,prob", PROBLEMS, ids=IDS)
def test_folded_program_meets_the_oracle(name, prob, config, monkeypatch):
    """ll, per-site and summed derivatives with and without an edge mask, dwell and trans; config 0 forces the
    constant-memory kernels (binary trees)"""
    m = O.parse_model(prob["model_and_data"])
    ref = H.seam_reference(name, prob)
    if config is not None:
        if not _binary(m):
            pytest.skip("the constant-memory kernels take binary trees")
        monkeypatch.setenv("PLF_F4_CONFIG", str(config))
        monkeypatch.setenv("PLF_F4_CONFIG_LL", str(config))
    from phyly_b200 import engine as E
    ll_w, D_w = ref["ll"], ref["D"]
    S, E_ = D_w.shape
    eng, cs = _engine(m)
    site_ll, tot = eng.ll()
    _assert_close(site_ll, ll_w, name + " ll", atol=LL_ATOL)
    r = eng.deriv(per_site=True, per_site_ll=True)
    _assert_close(r["site_ll"], ll_w, name + " deriv-ll", atol=LL_ATOL)
    _assert_close(r["site_deriv"], D_w, name + " deriv", atol=CANCEL * ref["Dabs"] + 1e-300)
    assert np.all(r["site_deriv"][D_w == 0.0] == 0.0)
    w = np.random.default_rng(1).integers(0, 4, S).astype(np.float64) + 0.5
    eng.set_site_weights(w)
    want = (w[:, None] * D_w).sum(axis=0)
    mag = np.abs(w[:, None] * D_w).sum(axis=0).max()
    r2 = eng.deriv(per_site=False)
    _assert_close(r2["sum_deriv"], want, name + " sum deriv", atol=1e-13 * mag)
    assert H.close(r2["sum_ll"], float((w * ll_w).sum()), 1e-11, 1e-13)
    for start in (0, 1):
        mask = np.zeros(E_, dtype=np.uint8)
        mask[start::2] = 1
        r3 = eng.deriv(edge_mask=mask, per_site=False)
        _assert_close(r3["sum_deriv"][mask == 1], want[mask == 1], name + " masked sums", atol=1e-13 * mag)
        assert np.all(r3["sum_deriv"][mask == 0] == 0.0)
        r4 = eng.deriv(edge_mask=mask, per_site=True)
        _assert_close(r4["site_deriv"][:, mask == 1], D_w[:, mask == 1], name + " masked deriv",
                      atol=CANCEL * ref["Dabs"][:, mask == 1] + 1e-300)
    eng.set_site_weights(np.ones(S))
    Ld, Lt, Lt_hi, Lt_lo, Lg = H.frechet_directions(m, cs)
    so, tot = eng.edge_expect(E.KIND_DWELL, Ld)
    _assert_close(so, ref["Xd"], name + " dwell", atol=1e-300)
    _assert_close(tot, ref["Xd"].sum(axis=0), name + " dwell sums", atol=1e-13 * S)
    so, tot = eng.edge_expect(E.KIND_TRANS, Lt_hi, Lt_lo)
    _assert_close(so, ref["Xt"], name + " trans", atol=1e-300)
    eng.close()


@pytest.mark.parametrize("name,prob", PROBLEMS, ids=IDS)
def test_unfolded_program_gives_the_same_bits(name, prob, monkeypatch):
    """Past the fold budget the engine runs the unfolded program: with the same kernel configuration the
    log-likelihoods and every derivative but those of folded cherries' tip edges have the same bits."""
    monkeypatch.setenv("PLF_F4_CONFIG", "4")          # 384 threads, no packed codes, no constant memory: both programs
    monkeypatch.setenv("PLF_F4_CONFIG_LL", "5")
    m = O.parse_model(prob["model_and_data"])
    tips = _folded_tip_edges(m)
    out = []
    for K in (None, K_PAD):
        eng, _ = _engine(m, K)
        ll_site, ll_sum = eng.ll()
        r = eng.deriv(per_site=True, per_site_ll=True)
        r2 = eng.deriv(per_site=False)
        out.append((ll_site, ll_sum, r["site_ll"], r["site_deriv"], r2["sum_ll"], r2["sum_deriv"]))
        eng.close()
    (a_site, a_sum, a_dll, a_d, a_dsum_ll, a_dsum), (b_site, b_sum, b_dll, b_d, b_dsum_ll, b_dsum) = out
    assert np.array_equal(a_site, b_site) and a_sum == b_sum
    assert np.array_equal(a_dll, b_dll) and a_dsum_ll == b_dsum_ll
    keep = np.ones(a_d.shape[1], dtype=bool)
    keep[tips] = False
    assert np.array_equal(a_d[:, keep], b_d[:, keep]) and np.array_equal(a_dsum[keep], b_dsum[keep])
    np.testing.assert_allclose(a_d[:, tips], b_d[:, tips], rtol=0, atol=1e-13 * np.abs(b_d).max())
    np.testing.assert_allclose(a_dsum[tips], b_dsum[tips], rtol=0, atol=1e-13 * np.abs(b_dsum).max())


def test_marginal_and_edge_matrix_queries_keep_their_kernels():
    name, prob = PROBLEMS[0]
    m = O.parse_model(prob["model_and_data"])
    ref = H.seam_reference(name, prob)
    eng, _ = _engine(m)
    C = int(ref["C"])
    sm, _ = eng.marginal()
    assert eng.last_kernel_name().startswith("fused4_kernel<%d,2," % C), eng.last_kernel_name()
    _assert_close(sm, ref["marg"], name + " marginal", atol=1e-300)
    eng.edge_expect_all()
    assert eng.last_kernel_name().startswith("fused4_kernel<%d,3," % C), eng.last_kernel_name()
    eng.ll()
    assert eng.last_kernel_name().startswith("fused4_kernel<%d,0," % C), eng.last_kernel_name()
    eng.close()
