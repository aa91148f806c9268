"""
Which kernels each query shape runs (plf_engine.cu: choose_path), pinned by plf_last_kernel_name or the error text,
and the upload-in-flight rule of that choice: only the single-window fused path overlaps an asynchronous upload.
"""
import numpy as np
import pytest

from oracle import arbplf_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

# random_problem arguments, and the number of character definitions to pad the data to (257: 4-byte device codes)
SHAPES = {
    "n3": (dict(seed=31, ntips=8, n=3, S=64, ncat=2), None),
    "n4c4": (dict(seed=32, ntips=8, n=4, S=64, ncat=4, mixture="gamma"), None),
    "n4c5": (dict(seed=33, ntips=8, n=4, S=64, ncat=5, mixture="median_inv"), None),
    "n4deg4": (dict(seed=34, ntips=9, n=4, S=64, ncat=2, max_degree=4, root_degree=4), None),
    "n4k257": (dict(seed=35, ntips=8, n=4, S=64, ncat=2), 257),
    "n20": (dict(seed=36, ntips=8, n=20, S=64, ncat=2), None),
    "n20k300": (dict(seed=37, ntips=8, n=20, S=64, ncat=2), 300),
    "n61": (dict(seed=38, ntips=6, n=61, S=32, ncat=1), None),
}
QUERIES = {
    "ll": lambda eng, n: eng.ll(per_site=False),
    "deriv": lambda eng, n: eng.deriv(per_site=False),
    "marginal": lambda eng, n: eng.marginal(per_site=False),
    "hess": lambda eng, n: eng.hess(),
    "dwell": lambda eng, n: eng.edge_expect(0, np.eye(n), per_site=False),       # KIND_DWELL
    "edge_expect_all": lambda eng, n: eng.edge_expect_all(),
}
PATHS = ("auto", "generic", "fused4")
CASES = [(s, False) for s in SHAPES] + [("n20", True), ("n61", True)]      # (shape, PLF_NO_TILE set)


def observe(shape):
    """{path: [kernel name or "error: <text>" per query]}"""
    from phyly_b200 import engine as E
    kw, K = SHAPES[shape]
    m = O.parse_model(H.random_problem(**kw)["model_and_data"])
    eng = E.Engine(0)
    H.fill_engine(eng, m)
    if K:
        defs, codes = H.dedupe_rows(m.dense_pmat())
        extra = np.random.default_rng(kw["seed"]).random((K - defs.shape[0], m.n)) + 0.05
        eng.set_data(np.vstack([defs, extra]), codes.astype(np.int32))
    out = {}
    for name, path in zip(PATHS, (E.PATH_AUTO, E.PATH_GENERIC, E.PATH_FUSED4)):
        eng.set_path(path)
        out[name] = []
        for run in QUERIES.values():
            try:
                run(eng, m.n)
                out[name].append(eng.last_kernel_name())
            except E.EngineError as exc:
                out[name].append("error: %s" % exc)
    eng.close()
    return out


G = "generic_inside_kernel / generic_outside_kernel"
T = "tile_inside_kernel / tile_outside_kernel"
X = "error: the fused 4-state path does not apply to this query"
# Recorded on an NVIDIA B200: per path, the outcome of each query in the order of QUERIES.
EXPECTED = {
    ("n3", False): {"auto": [G] * 6, "generic": [G] * 6, "fused4": [X] * 6},
    ("n4c4", False): {"auto": ["fused4_kernel<4,0,512,2,1,0>", "fused4_kernel<4,1,384,2,1,0>", "fused4_kernel<4,2,384,1,1,0>", G, "fused4_kernel<4,1,384,2,1,0>", "fused4_kernel<4,3,384,1,1,0>"],
                      "generic": [G] * 6,
                      "fused4": ["fused4_kernel<4,0,512,2,1,0>", "fused4_kernel<4,1,384,2,1,0>", "fused4_kernel<4,2,384,1,1,0>", X, "fused4_kernel<4,1,384,2,1,0>", "fused4_kernel<4,3,384,1,1,0>"]},
    ("n4c5", False): {"auto": ["fused4_kernel<1,0,512,2,1,0> (x2 category windows)", "fused4_kernel<1,1,384,2,1,0> (x2 category windows)", "fused4_kernel<1,2,384,1,1,0> (x2 category windows)", G, "fused4_kernel<1,1,384,2,1,0> (x2 category windows)", G],
                      "generic": [G] * 6,
                      "fused4": ["fused4_kernel<1,0,512,2,1,0> (x2 category windows)", "fused4_kernel<1,1,384,2,1,0> (x2 category windows)", "fused4_kernel<1,2,384,1,1,0> (x2 category windows)", X, "fused4_kernel<1,1,384,2,1,0> (x2 category windows)", X]},
    ("n4deg4", False): {"auto": [G] * 6, "generic": [G] * 6, "fused4": [X] * 6},
    ("n4k257", False): {"auto": [G] * 6, "generic": [G] * 6, "fused4": [X] * 6},
    ("n20", False): {"auto": ["dm_inside_kernel<3,16,1>", "dm_inside_kernel<3,16,1> + dm_outside_kernel<3,16,1>", T, G, "dm_inside_kernel<3,16,1> + dm_outside_kernel<3,16,1>", G],
                     "generic": [T, T, T, G, T, G], "fused4": [X] * 6},
    ("n20k300", False): {"auto": [T, T, T, G, T, G], "generic": [T, T, T, G, T, G], "fused4": [X] * 6},
    ("n61", False): {"auto": ["dm_inside_kernel<8,16,1>", "dm_inside_kernel<8,16,1> + dm_outside_kernel<8,16,1>", T, G, "dm_inside_kernel<8,16,1> + dm_outside_kernel<8,16,1>", G],
                     "generic": [T, T, T, G, T, G], "fused4": [X] * 6},
    ("n20", True): {"auto": ["dm_inside_kernel<3,16,1>", "dm_inside_kernel<3,16,1> + dm_outside_kernel<3,16,1>", G, G, "dm_inside_kernel<3,16,1> + dm_outside_kernel<3,16,1>", G],
                    "generic": [G] * 6, "fused4": [X] * 6},
    ("n61", True): {"auto": ["dm_inside_kernel<8,16,1>", "dm_inside_kernel<8,16,1> + dm_outside_kernel<8,16,1>", G, G, "dm_inside_kernel<8,16,1> + dm_outside_kernel<8,16,1>", G],
                    "generic": [G] * 6, "fused4": [X] * 6},
}


@pytest.mark.parametrize("shape,no_tile", CASES, ids=["%s%s" % (s, "-no_tile" if t else "") for s, t in CASES])
def test_path_choice(shape, no_tile, monkeypatch):
    if no_tile:
        monkeypatch.setenv("PLF_NO_TILE", "1")
    got, want = observe(shape), EXPECTED[(shape, no_tile)]
    bad = ["%s %s: got %r, want %r" % (p, q, g, w) for p in PATHS for q, g, w in zip(QUERIES, got[p], want[p]) if g != w]
    assert not bad, "\n".join(bad)


def test_async_upload_on_category_windows_sees_new_internal_data():
    """More than 4 categories (category windows) with an upload in flight that makes an internal node carry data: the
    query must run on a program built for the new data, as after a synchronous upload of the same codes."""
    from phyly_b200.engine import Engine
    m = O.parse_model(H.random_problem(39, ntips=10, n=4, S=300, ncat=5, mixture="median_inv")["model_and_data"])
    eng = Engine(0)
    H.fill_engine(eng, m)                  # no internal node carries data
    defs, codes = H.dedupe_rows(m.dense_pmat())
    deg = np.diff(m.tree.indptr)
    codes2 = codes.copy()                  # the first non-root internal node gets the data of the first leaf
    codes2[:, [v for v in np.flatnonzero(deg) if v != m.tree.root][0]] = codes[:, np.flatnonzero(deg == 0)[0]]
    eng.set_data(defs, codes2)
    want = eng.deriv(per_site=False)
    eng.set_data(defs, codes)
    eng.deriv(per_site=False)
    eng.set_data_async(defs, codes2)
    got = eng.deriv(per_site=False)
    assert eng.last_kernel_name().endswith("(x2 category windows)"), eng.last_kernel_name()
    assert abs(got["sum_ll"] - want["sum_ll"]) <= 1e-13 * abs(want["sum_ll"]), (got["sum_ll"], want["sum_ll"])
    assert np.allclose(got["sum_deriv"], want["sum_deriv"], rtol=1e-12, atol=1e-12 * np.abs(want["sum_deriv"]).max())
    eng.close()
