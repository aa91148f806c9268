"""
Certified derivatives (plf_deriv_certified, arbplf-deriv-certified): enclosures [lower, upper] of d log L / d t_e.

1. Every arbplf-deriv golden lies inside its enclosure, and every non-zero golden has a width below 1e-10 of its value,
   so its sign is certified -- the long-branch cases included, which an enclosure of Q P formed from [Plo, Phi] loses.
   Structural zeros are literal 0.0 in both tables.
2. Random problems (mixtures, soft and internal data, 20 states, every root mode, degree 3, long branches, a zero edge
   rate, a reducible rate matrix) against the 320-bit oracle, per site and edge and aggregated.
3. Engine level: the edge mask, repeatability, errors, and the 61-state and cfg2-sized problems against fp64 plf_deriv.
"""
import copy
import json
import math
import os
import subprocess

import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DERIV_GOLDENS = [c["name"] for c in H.manifest() if c["program"] == "deriv"]


def _run(program, doc):
    import phyly_b200.arbplf as A
    return json.loads(getattr(A, "arbplf_" + program)(json.dumps(doc)))


def _check_enclosure(got, want, what, rtol=1e-10, floor=1e-12):
    """containment in every cell; width <= rtol |value| + floor * (largest |entry| of the table)"""
    lo, hi = got["lower"], got["upper"]
    assert lo["columns"] == want["columns"] == hi["columns"], what
    assert len(lo["data"]) == len(want["data"]) == len(hi["data"]), what
    scale = max([abs(r[-1]) for r in want["data"]] + [0.0])
    for a, b, w in zip(lo["data"], hi["data"], want["data"]):
        assert a[:-1] == w[:-1] == b[:-1], (what, a, w, b)
        assert a[-1] <= w[-1] <= b[-1], (what, a, w, b)
        assert b[-1] - a[-1] <= rtol * abs(w[-1]) + floor * scale, (what, a, w, b)


def test_deriv_goldens_are_all_covered():
    assert sorted(DERIV_GOLDENS) == sorted(["fels_deriv", "bpp_deriv", "jc_long_deriv", "jc29_same_deriv", "jc29_diff_deriv",
                                            "jc30_same_deriv", "jc30_diff_deriv", "jc600_same_deriv"])


@pytest.mark.parametrize("name", DERIV_GOLDENS)
def test_golden_inside_a_tight_enclosure(name):
    got = _run("deriv_certified", H.golden_in(name))
    want = H.golden_out(name)
    lo, hi = got["lower"], got["upper"]
    assert lo["columns"] == want["columns"] == hi["columns"]
    assert len(lo["data"]) == len(want["data"]) == len(hi["data"])
    scale = max(abs(r[-1]) for r in want["data"])
    for a, b, w in zip(lo["data"], hi["data"], want["data"]):
        assert a[:-1] == w[:-1] == b[:-1]
        assert a[-1] <= w[-1] <= b[-1], (name, a, w, b)
        if w[-1] != 0.0:
            assert b[-1] - a[-1] <= 1e-10 * abs(w[-1]), (name, a, w, b)
            assert (a[-1] > 0.0) == (w[-1] > 0.0) and (b[-1] > 0.0) == (w[-1] > 0.0), (name, a, w, b)
        elif name == "jc600_same_deriv":
            assert -1e-300 <= a[-1] and b[-1] <= 1e-300, (a, b)      # an underflow, not a structural zero
        else:
            # site 2 of jc_long_deriv cancels to 0 (uniform root, JC columns of D sum to zero): the width of the form is
            # that of its terms, ~2.5e-12 relative on this 20-unit branch (2^5 squarings of R)
            assert b[-1] - a[-1] <= 1e-11 * scale, (name, a, w, b)
    # structural zeros: data-free site of fels_deriv, site 3 of jc_long_deriv (both ends missing)
    zero_sites = {"fels_deriv": [0], "jc_long_deriv": [3]}.get(name, [])
    for a, b in zip(lo["data"], hi["data"]):
        if a[0] in zero_sites:
            assert repr(a[-1]) == "0.0" and repr(b[-1]) == "0.0", (name, a, b)


def test_long_branches_certify_the_sign():
    """jc29_same_deriv is -6.4e-17: Q expm(29 Q) formed directly has the wrong sign; the enclosure excludes 0."""
    got = _run("deriv_certified", H.golden_in("jc29_same_deriv"))
    assert got["upper"]["data"][0][-1] < 0.0
    got = _run("deriv_certified", H.golden_in("jc_long_deriv"))
    assert got["lower"]["data"][0][-1] > 0.0 and got["upper"]["data"][1][-1] < 0.0


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
]
# the relative width of R(x) doubles with each of its s = log2(rate * t) squarings: on branches of t = 4..38 (s up to 7)
# a form that cancels within its site keeps the width of its terms, up to 2e-11 of the table's largest entry
FLOOR = {"long_branches": 1e-10}


def _random_doc(name, kw):
    doc = {"model_and_data": copy.deepcopy(H.random_problem(**kw)["model_and_data"])}
    if name == "long_branches":
        assert max(doc["model_and_data"]["edge_rate_coefficients"]) >= 10.0
    return doc


@pytest.mark.parametrize("name,kw", RANDOM, ids=[r[0] for r in RANDOM])
def test_random_problems_against_the_oracle(name, kw):
    doc = _random_doc(name, kw)
    want = H.expected_json("dc_" + name, "deriv", doc)
    _check_enclosure(_run("deriv_certified", doc), want, name, floor=FLOOR.get(name, 1e-12))


def test_zero_edge_rate_and_reducible_rate_matrix():
    doc = _random_doc("zero_edge", dict(seed=71, ntips=7, n=4, S=8, ncat=2))
    doc["model_and_data"]["edge_rate_coefficients"][2] = 0.0
    _check_enclosure(_run("deriv_certified", doc), H.expected_json("dc_zero_edge", "deriv", doc), "zero edge")
    # tests/helpers.py reduction_cases: n = 2, absorbing state, no unique equilibrium, an edge of rate 0
    name, program, path = [c for c in H.reduction_cases() if c[0] == "absorbing_path_deriv"][0]
    _check_enclosure(_run("deriv_certified", path), H.expected_json(name, program, path), name)


@pytest.mark.parametrize("name", ["n4_gamma4_missing", "median_inv", "long_branches"])
def test_aggregations_enclose_the_oracle(name):
    kw = dict(RANDOM)[name]
    doc = _random_doc(name, kw)
    want = H.expected_json("dc_" + name, "deriv", doc)
    S = len(doc["model_and_data"]["character_data"])
    E = len(doc["model_and_data"]["edges"])
    # site weights of both signs: the engine's directed-rounding sums
    wts = [((-1) ** i) * (0.5 + i % 3) for i in range(S)]
    got = _run("deriv_certified", dict(doc, site_reduction={"selection": list(range(S)), "aggregation": wts}))
    assert [r[0] for r in got["lower"]["data"]] == list(range(E))
    for e in range(E):
        tot = math.fsum(wts[s] * r[-1] for s in range(S) for r in want["data"] if r[0] == s and r[1] == e)
        assert got["lower"]["data"][e][-1] <= tot <= got["upper"]["data"][e][-1], (name, e, tot)
    # edge reductions: sum, and signed weights on a selection with a duplicate, per site and with the site sum
    ew = [0.5, -1.0, 2.0, -0.25]
    sel = [E - 1, 0, 2, 0]
    for tag, red in (("edge_sum", {"edge_reduction": {"aggregation": "sum"}}),
                     ("edge_w", {"edge_reduction": {"selection": sel, "aggregation": ew}}),
                     ("edge_w_site_sum", {"edge_reduction": {"selection": sel, "aggregation": ew},
                                          "site_reduction": {"aggregation": "sum"}})):
        d = dict(doc, **red)
        agg = H.expected_json("dc_%s_%s" % (name, tag), "deriv", d)
        got = _run("deriv_certified", d)
        assert got["lower"]["columns"] == agg["columns"]
        for a, b, w in zip(got["lower"]["data"], got["upper"]["data"], agg["data"]):
            assert a[:-1] == w[:-1] == b[:-1]
            assert a[-1] <= w[-1] <= b[-1], (name, red, a, w, b)


def _engine_for(kw):
    from oracle import arbplf_oracle as O
    from phyly_b200.engine import Engine
    prob = H.random_problem(**kw)
    eng = Engine(0)
    H.fill_engine(eng, O.parse_model(prob["model_and_data"]))
    return eng


def test_edge_mask_repeatability_and_kernel_name():
    eng = _engine_for(dict(seed=72, ntips=9, n=4, S=40, ncat=3, mixture="gamma", missing=0.2))
    E = eng.E
    w = np.linspace(-1.0, 2.0, eng.S)
    eng.set_site_weights(w)
    full = eng.deriv_certified()
    assert "cert_outside_kernel" in eng.last_kernel_name()
    mask = np.zeros(E, dtype=np.uint8)
    mask[::2] = 1
    part = eng.deriv_certified(edge_mask=mask)
    for k in ("site_lo", "site_hi", "sum_lo", "sum_hi"):
        x, y = full[k], part[k]
        assert np.all(x[..., mask == 1] == y[..., mask == 1]), k
        z = y[..., mask == 0]
        assert np.all(z == 0.0) and not np.any(np.signbit(z)), k
    again = eng.deriv_certified()
    for k in ("site_lo", "site_hi", "sum_lo", "sum_hi"):
        assert full[k].tobytes() == again[k].tobytes(), k
    # no per-site output: the same sums
    sums = eng.deriv_certified(per_site=False)
    assert sums["sum_lo"].tobytes() == full["sum_lo"].tobytes() and sums["sum_hi"].tobytes() == full["sum_hi"].tobytes()
    # the fp64 derivative lies inside (its per-site output skips the sites of weight 0: taken without weights)
    r = eng.deriv(per_site=False)
    _sums_inside(r, full, w, "sums")
    eng.set_site_weights(None)
    r = eng.deriv(per_site=True)
    _fp64_inside(r["site_deriv"], full["site_lo"], full["site_hi"], "per site")
    eng.close()


def test_errors():
    from phyly_b200.engine import Engine, EngineError
    eng = _engine_for(dict(seed=73, ntips=5, n=4, S=6, ncat=1))
    for dr, dq in ((-1.0, 0.0), (float("nan"), 0.0), (1.0, 0.0), (4e-15, -1.0), (4e-15, float("nan")), (4e-15, 0.5)):
        with pytest.raises(EngineError, match="bad input uncertainties"):
            eng.deriv_certified(delta_rate=dr, delta_q=dq)
    eng.close()
    # a site of zero likelihood: the root is observed in the state the root prior excludes
    doc = {"model_and_data": {"edges": [[0, 1]], "edge_rate_coefficients": [0.5], "rate_matrix": [[0, 1], [0, 0]],
                              "root_prior": [1, 0], "probability_array": [[[1, 0], [1, 1]], [[0, 1], [1, 1]]]}}
    from oracle import arbplf_oracle as O
    eng = Engine(0)
    H.fill_engine(eng, O.parse_model(doc["model_and_data"]))
    with pytest.raises(EngineError, match="a site with non-zero weight has zero likelihood"):
        eng.deriv_certified(per_site=False)
    with pytest.raises(EngineError, match="a site with non-zero weight has zero likelihood"):
        eng.ll_certified()
    eng.set_site_weights(np.array([1.0, 0.0]))          # weight 0 on the site of zero likelihood: no error
    r = eng.deriv_certified()
    assert r["site_lo"][1, 0] == -np.inf and r["site_hi"][1, 0] == np.inf
    assert r["site_lo"][0, 0] == 0.0 == r["site_hi"][0, 0]
    assert r["sum_lo"][0] == 0.0 == r["sum_hi"][0]
    eng.close()
    with pytest.raises(RuntimeError):
        _run("deriv_certified", dict(doc, site_reduction={"aggregation": "sum"}))


def _fp64_inside(v, lo, hi, what, width_floor=None):
    floor = 1e-12 * np.abs(v).max()
    assert np.all(lo - 1e-11 * np.abs(v) - floor <= v), what
    assert np.all(v <= hi + 1e-11 * np.abs(v) + floor), what
    if width_floor is None:
        width_floor = floor
    assert np.all(hi - lo <= 1e-10 * np.abs(v) + width_floor), (what, np.max(hi - lo - 1e-10 * np.abs(v) - width_floor))


def _sums_inside(r, c, w, what):
    """The sums against fp64 plf_deriv.  An interval sum is as wide as the weighted per-site widths it adds up, which
    over many sites exceeds 1e-10 of a gradient that cancels between sites: the width bar is those widths (+1 %)."""
    per_site = np.abs(w) @ (c["site_hi"] - c["site_lo"])
    _fp64_inside(r["sum_deriv"], c["sum_lo"], c["sum_hi"], what, width_floor=1e-12 * np.abs(r["sum_deriv"]).max() + 1.01 * per_site)


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
    w = rng.random(S) - 0.3
    eng.set_site_weights(w)
    r = eng.deriv(per_site=True)
    c = eng.deriv_certified()
    _fp64_inside(r["site_deriv"], c["site_lo"], c["site_hi"], "61 states per site")
    _sums_inside(r, c, w, "61 states sums")
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
    w = 1.0 + rng.poisson(3.0, pb["S"]).astype(np.float64)
    eng.set_site_weights(w)
    r = eng.deriv(per_site=True)
    c = eng.deriv_certified()
    _fp64_inside(r["site_deriv"], c["site_lo"], c["site_hi"], "cfg2 per site")
    _sums_inside(r, c, w, "cfg2 sums")
    eng.close()


def test_cli_executable():
    exe = os.path.join(ROOT, "phyly_b200", "bin", "arbplf-deriv-certified")
    p = subprocess.run([exe], input=json.dumps(H.golden_in("fels_deriv")), capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    out = json.loads(p.stdout)
    want = H.golden_out("fels_deriv")
    for a, b, w in zip(out["lower"]["data"], out["upper"]["data"], want["data"]):
        assert a[:-1] == w[:-1] and a[-1] <= w[-1] <= b[-1]
