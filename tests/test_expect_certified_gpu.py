"""
Certified posterior marginals and edge expectations (plf_marginal_certified, plf_edge_expect_certified,
arbplf-{marginal,dwell,trans}-certified): enclosures [lower, upper] of what plf_marginal and plf_edge_expect return.

1. Every marginal, dwell and trans golden lies inside its enclosure, with a width below 1e-10 of its value plus 1e-12
   of the table's largest entry.  States a leaf's data excludes are literal 0.0 in both marginal tables.
2. Random problems (mixtures with a rate-0 category, constant-column children, soft and internal data, 20 states, every
   root mode, degree 3, long branches, a zero edge rate, a reducible rate matrix) against the 320-bit oracle.
3. Aggregations of both signs: site weights (summed on the device), node and state weights of marginals, signed dwell
   state and trans aggregations (directions with negative entries), edge reductions.
4. Engine level: the edge mask, repeatability, errors, and the 61-state and cfg2-sized problems against fp64.
"""
import copy
import json
import os
import subprocess

import numpy as np
import pytest

from tests import helpers as H
from tests.test_deriv_certified_gpu import _check_enclosure, _engine_for, _fp64_inside, _run

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
PROGRAMS = ("marginal", "dwell", "trans")
GOLDENS = [(c["name"], c["program"]) for c in H.manifest() if c["program"] in PROGRAMS]


def test_goldens_are_all_covered():
    assert sorted(GOLDENS) == sorted([
        ("fels_marginal", "marginal"), ("beast_anc_marginal", "marginal"), ("jc_long_marginal", "marginal"),
        ("fels_dwell_adenine", "dwell"), ("fels_dwell_pyrimidines", "dwell"), ("mj_rewards", "dwell"),
        ("jc_long_dwell", "dwell"),
        ("fels_trans_all", "trans"), ("fels_trans_AC", "trans"), ("fels_trans_tv", "trans"), ("fels_trans_tv2", "trans"),
        ("mj_jumps", "trans"), ("mj_jumps_reordered", "trans"), ("mj_marginal_rate", "trans"),
        ("mj_marginal_rate_pedantic", "trans"), ("jc_long_trans", "trans")])


@pytest.mark.parametrize("name,program", GOLDENS, ids=[g[0] for g in GOLDENS])
def test_golden_inside_a_tight_enclosure(name, program):
    doc = H.golden_in(name)
    got = _run(program + "_certified", doc)
    _check_enclosure(got, H.golden_out(name), name)
    if program == "marginal":
        _check_excluded_states_are_zero(doc, got, name)


def _check_excluded_states_are_zero(doc, got, what):
    """a state that a leaf's data excludes has the marginal 0.0 exactly, in both tables (per-site, per-node tables)"""
    md = doc["model_and_data"]
    if "character_data" not in md or any(doc.get(k, {}).get("aggregation") for k in ("site_reduction", "node_reduction",
                                                                                        "state_reduction")):
        return
    defs, data = md["character_definitions"], md["character_data"]
    excluded = {(s, a, j) for s, row in enumerate(data) for a, code in enumerate(row)
                for j, x in enumerate(defs[code]) if x == 0}
    seen = 0
    for a, b in zip(got["lower"]["data"], got["upper"]["data"]):
        if tuple(a[:3]) in excluded:
            assert repr(a[-1]) == "0.0" and repr(b[-1]) == "0.0", (what, a, b)
            seen += 1
    assert seen > 0, what


RANDOM = [
    ("n4_c1", dict(seed=61, ntips=8, n=4, S=9, ncat=1)),
    ("n4_gamma4_missing", dict(seed=62, ntips=10, n=4, S=14, ncat=4, mixture="gamma", missing=0.3)),
    ("median_inv", dict(seed=63, ntips=6, n=4, S=8, ncat=4, mixture="median_inv")),
    ("n5_soft_internal", dict(seed=64, ntips=6, n=5, S=7, ncat=2, soft=True, internal_data=True)),
    ("n20_equilibrium", dict(seed=65, ntips=4, n=20, S=5, ncat=1, root="equilibrium_distribution")),
    ("root_uniform", dict(seed=66, ntips=7, n=4, S=8, ncat=2, root="uniform_distribution")),
    ("root_equilibrium", dict(seed=67, ntips=7, n=4, S=8, ncat=2, root="equilibrium_distribution", internal_data=True)),
    ("root_none", dict(seed=68, ntips=7, n=3, S=8, ncat=2, root=None, divisor=2.5)),
    ("degree3", dict(seed=69, ntips=9, n=4, S=8, ncat=2, max_degree=3, root_degree=3)),
    ("long_branches", dict(seed=70, ntips=6, n=4, S=8, ncat=2, mixture="gamma", edge_scale=12.0)),
    ("zero_edge", dict(seed=71, ntips=7, n=4, S=8, ncat=2)),
]
AGGREGATED = ["n4_gamma4_missing", "median_inv", "long_branches"]


def _random_doc(name):
    doc = {"model_and_data": copy.deepcopy(H.random_problem(**dict(RANDOM)[name])["model_and_data"])}
    if name == "long_branches":
        assert max(doc["model_and_data"]["edge_rate_coefficients"]) >= 10.0
    if name == "zero_edge":
        doc["model_and_data"]["edge_rate_coefficients"][2] = 0.0
    return doc


def _selection(doc, program):
    """The cells checked per site: two states (dwell), two transitions (trans); the 320-bit oracle needs minutes per
    20-state Frechet direction"""
    n = len(doc["model_and_data"]["rate_matrix"])
    if program == "dwell":
        return {"state_reduction": {"selection": [3, 17] if n == 20 else [0, n - 1]}}
    if program == "trans":
        return {"trans_reduction": {"selection": [[0, 1], [19, 7]] if n == 20 else [[0, 1], [n - 1, 0]]}}
    return {}


def _random_case(name, program):
    """one site, every node / edge: the site with the most missing leaves (constant-column children), else site 0"""
    doc = _random_doc(name)
    data = doc["model_and_data"].get("character_data")
    n = len(doc["model_and_data"]["rate_matrix"])
    site = 0 if data is None else max(range(len(data)), key=lambda s: (sum(c == n for c in data[s]), -s))
    return dict(doc, site_reduction={"selection": [site]}, **_selection(doc, program))


def _aggregated_cases(name):
    """(cache name, program, document): site weights of both signs (summed on the device), node / state / transition /
    edge weights of both signs"""
    doc = _random_doc(name)
    S, N = len(doc["model_and_data"]["character_data"]), len(doc["model_and_data"]["edges"]) + 1
    site_w = {"site_reduction": {"aggregation": [((-1) ** i) * (0.5 + i % 3) for i in range(S)]}}
    edge_w = {"edge_reduction": {"selection": [N - 2, 0, 2, 0], "aggregation": [0.5, -1.0, 2.0, -0.25]}}
    site_sum = {"site_reduction": {"aggregation": "sum"}}
    node_state = {"node_reduction": {"selection": [N - 1, 0, 2, 0], "aggregation": [0.5, -1.0, 2.0, -0.25]},
                  "state_reduction": {"aggregation": [1.0, -0.5, 0.25, 2.0]}}
    dwell_w = {"state_reduction": {"aggregation": [1.0, -0.5, 0.25, -2.0]}}
    trans_w = {"trans_reduction": {"selection": [[0, 1], [2, 3], [3, 0], [1, 0]], "aggregation": [1.0, -2.0, 0.5, -0.25]}}
    red = [("marginal", "site_w", site_w),
           ("marginal", "node_state_w_site_w", dict(node_state, **site_w)),
           ("dwell", "state_w_site_w", dict(dwell_w, **site_w)),
           ("dwell", "edge_w_site_sum", dict(_selection(doc, "dwell"), **edge_w, **site_sum)),
           ("trans", "trans_w_site_w", dict(trans_w, **site_w)),
           ("trans", "edge_w_site_sum", dict(_selection(doc, "trans"), **edge_w, **site_sum))]
    return [("ec_%s_%s_%s" % (name, program, tag), program, dict(doc, **r)) for program, tag, r in red]


def oracle_cases():
    """every (cache name, program, document) whose 320-bit output this module reads from tests/golden/json_cases"""
    cases = [("ec_%s_%s" % (name, program), program, _random_case(name, program)) for name, _ in RANDOM for program in PROGRAMS]
    for name in AGGREGATED:
        cases += _aggregated_cases(name)
    return cases


@pytest.mark.parametrize("name,program", [(name, program) for name, _ in RANDOM for program in PROGRAMS],
                         ids=["%s-%s" % (name, program) for name, _ in RANDOM for program in PROGRAMS])
def test_random_problems_against_the_oracle(name, program):
    doc = _random_case(name, program)
    got = _run(program + "_certified", doc)
    _check_enclosure(got, H.expected_json("ec_%s_%s" % (name, program), program, doc), (name, program))
    if program == "marginal":
        _check_excluded_states_are_zero(doc, got, name)


@pytest.mark.parametrize("program", PROGRAMS)
def test_reducible_rate_matrix(program):
    # tests/helpers.py reduction_cases: n = 2, absorbing state, no unique equilibrium, an edge of rate 0
    name, prog, path = [c for c in H.reduction_cases() if c[0] == "absorbing_path_" + program][0]
    _check_enclosure(_run(program + "_certified", path), H.expected_json(name, prog, path), name)


@pytest.mark.parametrize("name", AGGREGATED)
def test_aggregations_enclose_the_oracle(name):
    for cache, program, doc in _aggregated_cases(name):
        want = H.expected_json(cache, program, doc)
        got = _run(program + "_certified", doc)
        assert got["lower"]["columns"] == want["columns"] == got["upper"]["columns"], cache
        assert len(got["lower"]["data"]) == len(want["data"]), cache
        for a, b, w in zip(got["lower"]["data"], got["upper"]["data"], want["data"]):
            assert a[:-1] == w[:-1] == b[:-1], cache
            assert a[-1] <= w[-1] <= b[-1], (cache, a, w, b)


def _directions(n):
    """a dwell direction and a signed trans-like direction (negative entries take the L- branch)"""
    Ld = np.diag(np.linspace(0.25, 1.0, n))
    Lt = np.zeros((n, n))
    for i in range(n):
        for j in range(n):
            if i != j:
                Lt[i, j] = (1 + (i + 2 * j) % 3) * (1.0 if (i + j) % 2 else -0.5)
    return Ld, Lt


KEYS = ("site_lo", "site_hi", "sum_lo", "sum_hi")


def test_edge_mask_repeatability_and_kernel_names():
    from phyly_b200.engine import KIND_DWELL, KIND_TRANS
    eng = _engine_for(dict(seed=72, ntips=9, n=4, S=40, ncat=3, mixture="gamma", missing=0.2))
    E = eng.E
    w = np.linspace(-1.0, 2.0, eng.S)
    eng.set_site_weights(w)
    Ld, Lt = _directions(4)
    mask = np.zeros(E, dtype=np.uint8)
    mask[::2] = 1
    for kind, L in ((KIND_DWELL, Ld), (KIND_TRANS, Lt)):
        full = eng.edge_expect_certified(kind, L)
        assert "cert_frechet_kernel" in eng.last_kernel_name() and "cert_outside_kernel" in eng.last_kernel_name()
        part = eng.edge_expect_certified(kind, L, edge_mask=mask)
        for k in KEYS:
            x, y = full[k], part[k]
            assert np.all(x[..., mask == 1] == y[..., mask == 1]), k
            z = y[..., mask == 0]
            assert np.all(z == 0.0) and not np.any(np.signbit(z)), k
        again = eng.edge_expect_certified(kind, L)
        for k in KEYS:
            assert full[k].tobytes() == again[k].tobytes(), k
        sums = eng.edge_expect_certified(kind, L, per_site=False)
        assert sums["site_lo"] is None
        assert sums["sum_lo"].tobytes() == full["sum_lo"].tobytes() and sums["sum_hi"].tobytes() == full["sum_hi"].tobytes()
        _, tot = eng.edge_expect(kind, L, per_site=False)
        _sums_inside(tot, full, w, "edge sums")
    full = eng.marginal_certified()
    assert "cert_outside_kernel" in eng.last_kernel_name() and "cert_frechet_kernel" not in eng.last_kernel_name()
    again = eng.marginal_certified()
    for k in KEYS:
        assert full[k].tobytes() == again[k].tobytes(), k
    sums = eng.marginal_certified(per_site=False)
    assert sums["sum_lo"].tobytes() == full["sum_lo"].tobytes() and sums["sum_hi"].tobytes() == full["sum_hi"].tobytes()
    _, tot = eng.marginal(per_site=False)
    _sums_inside(tot, full, w, "marginal sums")
    eng.close()


def test_errors():
    from phyly_b200.engine import Engine, EngineError, KIND_DWELL, KIND_TRANS
    eng = _engine_for(dict(seed=73, ntips=5, n=4, S=6, ncat=1))
    Ld, _ = _directions(4)
    for dr, dq in ((-1.0, 0.0), (float("nan"), 0.0), (1.0, 0.0), (4e-15, -1.0), (4e-15, float("nan")), (4e-15, 0.5)):
        with pytest.raises(EngineError, match="bad input uncertainties"):
            eng.marginal_certified(delta_rate=dr, delta_q=dq)
        with pytest.raises(EngineError, match="bad input uncertainties"):
            eng.edge_expect_certified(KIND_DWELL, Ld, delta_rate=dr, delta_q=dq)
    for kind in (-1, 2, 7):
        with pytest.raises(EngineError, match="invalid kind"):
            eng.edge_expect_certified(kind, Ld)
    eng.close()
    # a site of zero likelihood: the root is observed in the state the root prior excludes
    doc = {"model_and_data": {"edges": [[0, 1]], "edge_rate_coefficients": [0.5], "rate_matrix": [[0, 1], [0, 0]],
                              "root_prior": [1, 0], "probability_array": [[[1, 0], [1, 1]], [[0, 1], [1, 1]]]}}
    from oracle import arbplf_oracle as O
    eng = Engine(0)
    H.fill_engine(eng, O.parse_model(doc["model_and_data"]))
    L = np.eye(2)
    for call in (lambda: eng.marginal_certified(per_site=False), lambda: eng.edge_expect_certified(KIND_DWELL, L, per_site=False),
                 lambda: eng.edge_expect_certified(KIND_TRANS, L, per_site=False)):
        with pytest.raises(EngineError, match="a site with non-zero weight has zero likelihood"):
            call()
    eng.set_site_weights(np.array([1.0, 0.0]))          # weight 0 on the site of zero likelihood: no error
    r = eng.marginal_certified()
    assert np.all(r["site_lo"][1] == -np.inf) and np.all(r["site_hi"][1] == np.inf)
    assert np.all(np.isfinite(r["site_lo"][0])) and np.all(np.isfinite(r["sum_lo"])) and np.all(np.isfinite(r["sum_hi"]))
    for kind in (KIND_DWELL, KIND_TRANS):
        r = eng.edge_expect_certified(kind, L)
        assert r["site_lo"][1, 0] == -np.inf and r["site_hi"][1, 0] == np.inf
        assert np.isfinite(r["sum_lo"][0]) and np.isfinite(r["sum_hi"][0])
        assert r["site_lo"][0, 0] <= r["sum_lo"][0] + 1e-300 and r["sum_hi"][0] <= r["site_hi"][0, 0]
    eng.close()
    for program in PROGRAMS:
        with pytest.raises(RuntimeError):
            _run(program + "_certified", dict(doc, site_reduction={"aggregation": "sum"}))


def _sums_inside(tot, c, w, what):
    """The sums against fp64.  An interval sum is as wide as the weighted per-site widths it adds up: the width bar is
    those widths (+1 %)."""
    per_site = np.tensordot(np.abs(w), c["site_hi"] - c["site_lo"], axes=1)
    _fp64_inside(tot, c["sum_lo"], c["sum_hi"], what, width_floor=1e-12 * np.abs(tot).max() + 1.01 * per_site)


def _check_engine_against_fp64(eng, w, what):
    from phyly_b200.engine import KIND_DWELL, KIND_TRANS
    eng.set_site_weights(w)
    c = eng.marginal_certified()
    _, tot = eng.marginal(per_site=False)
    _sums_inside(tot, c, w, what + " marginal sums")
    eng.set_site_weights(None)
    sm, _ = eng.marginal(per_site=True)
    _fp64_inside(sm, c["site_lo"], c["site_hi"], what + " marginal per site")
    Ld, Lt = _directions(eng.n)
    for kind, L in ((KIND_DWELL, Ld), (KIND_TRANS, Lt)):
        eng.set_site_weights(w)
        c = eng.edge_expect_certified(kind, L)
        _, tot = eng.edge_expect(kind, L, per_site=False)
        _sums_inside(tot, c, w, "%s kind %d sums" % (what, kind))
        eng.set_site_weights(None)
        so, _ = eng.edge_expect(kind, L, per_site=True)
        _fp64_inside(so, c["site_lo"], c["site_hi"], "%s kind %d per site" % (what, kind))


def test_61_states_against_fp64():
    import bench
    from phyly_b200.engine import Engine
    import phyly_b200.arbplf as A
    Q, _ = bench.codon_model()
    n = Q.shape[0]
    edges, N = bench.yule_tree(5, seed=31)
    rng = np.random.default_rng(32)
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.3, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "gamma_rate_mixture": {"gamma_shape": 0.8, "gamma_categories": 2},
          "character_definitions": np.vstack([np.eye(n), np.ones((1, n))]).tolist(), "character_data": [[n] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(n, n), np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    S = 7
    codes = np.full((S, N), n, dtype=np.uint8)
    for a in range(N):
        if s["indptr"][a] == s["indptr"][a + 1]:
            codes[:, a] = rng.integers(0, n + 1, S)
    eng.set_data(np.vstack([np.eye(n), np.ones((1, n))]), codes)
    _check_engine_against_fp64(eng, rng.random(S) - 0.3, "61 states")
    eng.close()


def test_cfg2_sized_problem_against_fp64():
    import bench

    class Args:
        taxa = 64
        sites = 200000
    pb = bench.build_problem(Args(), 0, 0)
    eng = pb["eng"]
    eng.set_data(np.array(bench.DEFS, dtype=np.float64), pb["codes"])
    rng = np.random.default_rng(9)
    _check_engine_against_fp64(eng, 1.0 + rng.poisson(3.0, pb["S"]).astype(np.float64), "cfg2")
    eng.close()


@pytest.mark.parametrize("program,golden", [("marginal", "fels_marginal"), ("dwell", "fels_dwell_adenine"),
                                            ("trans", "fels_trans_AC")])
def test_cli_executable(program, golden):
    exe = os.path.join(ROOT, "phyly_b200", "bin", "arbplf-%s-certified" % program)
    p = subprocess.run([exe], input=json.dumps(H.golden_in(golden)), capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    _check_enclosure(json.loads(p.stdout), H.golden_out(golden), golden)
