"""
GPU tests of plf_edge_expect_all (include/plf.h): every Frechet direction of the edge expectations in one pass, and
the gradient of the log-likelihood with respect to the rate matrix.

The entries are checked against the brute-force reference of tests/edge_expect_all_ref.py (the oracle looped over the
n^2 elementary directions, 320-bit except at 20 states), on the fused 4-state path (mode 3 of fused4_kernel) and on
the generic path; then against the existing one-direction query, deriv(), finite differences of ll() and the EM update.
"""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import arbplf_oracle as O
from tests import helpers as H
from tests import edge_expect_all_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

RTOL = 1e-11
CANCEL = 2e-14        # the floor of tests/test_engine_gpu.py for sums of signed terms

# (name, problem, oracle mode)
CASES = [
    ("n4c1", H.random_problem(201, ntips=6, n=4, S=6, ncat=1), "mp"),
    ("n4c2_deg3", H.random_problem(202, ntips=7, n=4, S=6, ncat=2, max_degree=3, root_degree=3,
                                   root="uniform_distribution", missing=0.3), "mp"),
    ("n4c3_soft", H.random_problem(203, ntips=6, n=4, S=5, ncat=3, soft=True, internal_data=True,
                                   root="equilibrium_distribution"), "mp"),
    ("n4c4_internal", H.random_problem(204, ntips=7, n=4, S=6, ncat=4, mixture="gamma", internal_data=True,
                                       missing=0.3), "mp"),
    ("jc_long", H.golden_in("jc_long_ll"), "mp"),
    ("n3", H.random_problem(205, ntips=5, n=3, S=5, ncat=2, root=None, divisor=2.5, missing=0.3), "mp"),
    ("n20", H.random_problem(206, ntips=4, n=20, S=4, ncat=1, root="equilibrium_distribution"), "fp64"),
    ("g4i", H.random_problem(207, ntips=6, n=4, S=5, ncat=5, mixture="median_inv"), "mp"),
]
IDS = [c[0] for c in CASES]


def _engine():
    from phyly_b200.engine import Engine
    return Engine(0)


def _assert_close(got, want, what, rtol=RTOL, atol=1e-300):
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = np.abs(got - want)
    bad = ~(err <= rtol * np.abs(want) + atol)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError("%s: %d mismatches, first at %s: got %r want %r (rel %.3e)" % (
            what, bad.sum(), i, got[i], want[i], err[i] / max(abs(want[i]), 1e-300)))


def _paths(m, C):
    from phyly_b200 import engine as E
    p = [E.PATH_GENERIC]
    if m.n == 4 and C <= 4:
        p.append(E.PATH_FUSED4)
    return p


def _setup(prob):
    eng = _engine()
    m = O.parse_model(prob["model_and_data"])
    cs = H.fill_engine(eng, m)
    return eng, m, cs


@pytest.mark.parametrize("name,prob,mode", CASES, ids=IDS)
def test_entries_against_brute_force_oracle(name, prob, mode):
    from phyly_b200 import engine as E
    ref = R.reference(name, prob, mode)
    m = O.parse_model(prob["model_and_data"])
    S = m.site_count
    w = np.random.default_rng(5).random(S) + 0.25
    want_d = np.einsum("s,seij->eij", w, ref["Xd"])
    want_t = np.einsum("s,seij->eij", w, ref["Xt"])
    C = None
    for path in _paths(m, 5 if name == "g4i" else 4):
        eng, m, cs = _setup(prob)
        C = cs.C
        eng.set_site_weights(w)
        eng.set_path(path)
        r = eng.edge_expect_all()
        what = "%s path%d" % (name, path)
        _assert_close(r["dwell"], want_d, what + " dwell")
        _assert_close(r["trans"], want_t, what + " trans")
        assert H.close(r["sum_ll"], float((w * ref["ll"]).sum()), 1e-11, 1e-13), (what, r["sum_ll"])
        np.testing.assert_array_equal(r["q_grad"], r["trans"].sum(axis=0))
        if path == E.PATH_FUSED4:
            assert eng.last_kernel_name().startswith("fused4_kernel<%d,3," % C), eng.last_kernel_name()
        else:
            assert eng.last_kernel_name() == "generic_inside_kernel / generic_outside_kernel", eng.last_kernel_name()
        eng.close()
    if name == "g4i":
        # five categories: the matrices need the whole site likelihood, so no category windows on the fused path
        eng, m, cs = _setup(prob)
        eng.set_path(E.PATH_FUSED4)
        with pytest.raises(E.EngineError):
            eng.edge_expect_all()
        eng.set_path(E.PATH_AUTO)
        eng.edge_expect_all()
        assert eng.last_kernel_name().startswith("generic_inside_kernel"), eng.last_kernel_name()
        eng.close()


def _check_linearity(eng, X, n, what, rng, extra=()):
    """sum_ij L_ij X[e][i][j] against edge_expect(kind, L) for the test directions and random non-negative L."""
    from phyly_b200 import engine as E
    dirs = list(extra) + [(k, rng.random((n, n)), None) for k in (E.KIND_DWELL, E.KIND_TRANS)]
    for kind, L_hi, L_lo in dirs:
        _, want = eng.edge_expect(kind, L_hi, L_lo, per_site=False)
        L = L_hi + (0.0 if L_lo is None else L_lo)
        got = np.einsum("ij,eij->e", L, X[kind])
        _assert_close(got, want, "%s kind %d" % (what, kind))


@pytest.mark.parametrize("name,prob,mode", CASES, ids=IDS)
def test_linear_in_the_direction(name, prob, mode):
    from phyly_b200 import engine as E
    m = O.parse_model(prob["model_and_data"])
    for path in _paths(m, 5 if name == "g4i" else 4):
        eng, m, cs = _setup(prob)
        eng.set_site_weights(np.random.default_rng(6).random(m.site_count) + 0.25)
        eng.set_path(path)
        r = eng.edge_expect_all()
        Ld, Lt, Lt_hi, Lt_lo, Lg = H.frechet_directions(m, cs)
        _check_linearity(eng, {E.KIND_DWELL: r["dwell"], E.KIND_TRANS: r["trans"]}, m.n, "%s path%d" % (name, path),
                         np.random.default_rng(7), extra=[(E.KIND_DWELL, Ld, None), (E.KIND_TRANS, Lt_hi, Lt_lo)])
        eng.close()


def test_linear_in_the_direction_on_a_large_problem():
    """The 64-taxon GTR+Gamma4 model of bench.py at 2e5 sites: both paths against edge_expect, and against each other."""
    import bench
    from phyly_b200 import engine as E

    class A:
        taxa, sites = 64, 200000
    pb = bench.build_problem(A, 0, 0)
    eng = pb["eng"]
    defs = np.array(bench.DEFS, dtype=np.float64)
    eng.set_data(defs, pb["codes"])
    w = 1.0 + np.random.default_rng(3).poisson(2.0, pb["S"]).astype(np.float64)
    eng.set_site_weights(w)
    out = {}
    for path in (E.PATH_FUSED4, E.PATH_GENERIC):
        eng.set_path(path)
        r = eng.edge_expect_all()
        out[path] = r
        _check_linearity(eng, {E.KIND_DWELL: r["dwell"], E.KIND_TRANS: r["trans"]}, 4, "bench path%d" % path,
                         np.random.default_rng(8), extra=[(E.KIND_DWELL, np.eye(4), None)])
    assert eng.last_kernel_name().startswith("generic"), eng.last_kernel_name()
    for k in ("dwell", "trans"):
        _assert_close(out[E.PATH_FUSED4][k], out[E.PATH_GENERIC][k], "bench fused vs generic " + k)
    assert H.close(out[E.PATH_FUSED4]["sum_ll"], out[E.PATH_GENERIC]["sum_ll"], 1e-12), (
        out[E.PATH_FUSED4]["sum_ll"], out[E.PATH_GENERIC]["sum_ll"])
    eng.close()


@pytest.mark.parametrize("name,prob,mode", CASES, ids=IDS)
def test_trans_contracted_with_q_is_the_edge_derivative(name, prob, mode):
    m = O.parse_model(prob["model_and_data"])
    for path in _paths(m, 5 if name == "g4i" else 4):
        eng, m, cs = _setup(prob)
        params, _ = H.model_params(m)
        Q = params["q_hi"] + params["q_lo"]
        t = params["edge_rates"]
        eng.set_path(path)
        r = eng.edge_expect_all()
        d = eng.deriv(per_site=False)["sum_deriv"]
        live = t > 0
        got = np.einsum("ij,eij->e", Q, r["trans"])[live] / t[live]
        terms = np.einsum("ij,eij->e", np.abs(Q), r["trans"])[live] / t[live]
        _assert_close(got, d[live], "%s path%d" % (name, path), atol=CANCEL * terms + 1e-300)
        eng.close()


# no constant columns (missing characters): a perturbed entry breaks the zero row sums of Q, and ll() keeps the
# shortcut P 1 = 1 for such columns, which the gradient of the matrix function does not see
FD_PROBLEMS = {
    "n4c3_soft": CASES[2][1],
    "n4c3": H.random_problem(208, ntips=7, n=4, S=8, ncat=3, missing=0.0, root="equilibrium_distribution"),
    "n3c2": H.random_problem(209, ntips=5, n=3, S=6, ncat=2, missing=0.0, root=None, divisor=2.5),
}


@pytest.mark.parametrize("name", sorted(FD_PROBLEMS))
def test_q_grad_matches_finite_differences(name):
    eng, m, cs = _setup(FD_PROBLEMS[name])
    params, _ = H.model_params(m)
    g = eng.edge_expect_all()["q_grad"]
    n = m.n
    fd = np.zeros((n, n))
    for i in range(n):
        for j in range(n):
            h = 1e-6 * max(abs(params["q_hi"][i, j]), 0.1)
            vals = []
            for sgn in (1.0, -1.0):
                p = dict(params)
                p["q_hi"] = params["q_hi"].copy()
                p["q_hi"][i, j] += sgn * h
                eng.set_model(**p)
                vals.append(eng.ll(per_site=False)[1])
            fd[i, j] = (vals[0] - vals[1]) / (2 * h)
    eng.set_model(**params)
    assert np.max(np.abs(fd - g)) <= 1e-6 * np.max(np.abs(g)), (fd, g)
    eng.close()


@pytest.mark.parametrize("name", ["fels_em_full", "fels_em_leaf", "fels_em_none"])
def test_em_update_from_one_call(name):
    prob = H.golden_in(name)
    want = H.golden_out(name)
    eng, m, cs = _setup(prob)
    params, _ = H.model_params(m)
    Q = params["q_hi"] + params["q_lo"]
    t = params["edge_rates"]
    tr = eng.edge_expect_all()["trans"]
    off = ~np.eye(m.n, dtype=bool)
    exits = np.einsum("i,eii->e", -np.diag(Q), tr)
    jumps = np.einsum("ij,eij->e", np.where(off, Q, 0.0), tr)
    ratio = np.where(jumps != 0.0, t * jumps / np.where(exits != 0.0, exits, 1.0), 0.0)
    tree = m.tree
    for e, v in want["data"]:
        assert H.close(ratio[tree.order[e]], v, 1e-11, 1e-300), (name, e, ratio[tree.order[e]], v)
    eng.close()


def test_repeated_calls_give_the_same_bits():
    import bench
    from phyly_b200 import engine as E

    class A:
        taxa, sites = 24, 100000
    pb = bench.build_problem(A, 0, 0)
    eng = pb["eng"]
    eng.set_data(np.array(bench.DEFS, dtype=np.float64), pb["codes"])
    eng.set_path(E.PATH_FUSED4)
    eng.edge_expect_all()                                 # tunes the fused kernel
    r1, r2 = eng.edge_expect_all(), eng.edge_expect_all()
    name = eng.last_kernel_name()
    assert name.startswith("fused4_kernel<4,3,"), name
    for k in ("dwell", "trans"):
        assert r1[k].tobytes() == r2[k].tobytes(), k
    assert r1["sum_ll"] == r2["sum_ll"]
    eng.close()


@pytest.mark.parametrize("name", ["n4c2_deg3", "n4c4_internal", "n3"])
def test_mixed_sign_weights(name):
    case = [c for c in CASES if c[0] == name][0]
    ref = R.reference(name, case[1], case[2])
    m = O.parse_model(case[1]["model_and_data"])
    w = np.random.default_rng(9).random(m.site_count) * 4.0 - 2.0
    for key, X in (("dwell", ref["Xd"]), ("trans", ref["Xt"])):
        want = np.einsum("s,seij->eij", w, X)
        mag = np.einsum("s,seij->eij", np.abs(w), X)
        for path in _paths(m, 4):
            eng, m, cs = _setup(case[1])
            eng.set_site_weights(w)
            eng.set_path(path)
            _assert_close(eng.edge_expect_all()[key], want, "%s path%d %s" % (name, path, key), atol=2e-14 * mag)
            eng.close()


def test_weighted_zero_likelihood_site_is_an_error():
    from phyly_b200 import engine as E
    prob = CASES[0][1]
    m = O.parse_model(prob["model_and_data"])
    defs, codes = H.dedupe_rows(m.dense_pmat())
    defs = np.vstack([defs, np.zeros((1, m.n))])          # a character no state can explain
    codes = codes.copy()
    codes[2, m.tree.indices[0]] = defs.shape[0] - 1
    for path in _paths(m, 1):
        eng, m, cs = _setup(prob)
        eng.set_data(defs, codes)
        eng.set_path(path)
        with pytest.raises(E.EngineError, match="zero likelihood"):
            eng.edge_expect_all()
        w = np.ones(m.site_count)
        w[2] = 0.0
        eng.set_site_weights(w)
        r = eng.edge_expect_all()
        assert np.all(np.isfinite(r["trans"])) and np.isfinite(r["sum_ll"])
        eng.close()


WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
import bench
from phyly_b200 import engine as E
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
class A: pass
args = A(); args.taxa = 64; args.sites = 40000
pb = bench.build_problem(args, local, 0)             # every rank builds the SAME problem (rank 0's seed)
eng = pb["eng"]; S = pb["S"]; defs = np.array(bench.DEFS, dtype=np.float64)
codes = pb["codes"]
w = 1.0 + np.random.default_rng(3).poisson(2.0, S).astype(np.float64)
def query(e):
    r = e.edge_expect_all()
    return np.concatenate([[r["sum_ll"]], r["dwell"].ravel(), r["trans"].ravel()])
eng.set_data(defs, codes); eng.set_site_weights(w)
want = query(eng)
lo, hi = rank * S // world, (rank + 1) * S // world
uid = [E.comm_unique_id() if rank == 0 else None]
dist.broadcast_object_list(uid, src=0)
eng.comm_init(world, rank, uid[0])
eng.set_data(defs, np.ascontiguousarray(codes[lo:hi])); eng.set_site_weights(w[lo:hi])
got = query(eng)
peers = [None] * world
dist.all_gather_object(peers, got.tobytes())
same = all(p == peers[0] for p in peers)
ok = same and bool(np.all(np.abs(got - want) <= 1e-11 * np.abs(want) + 1e-300))
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print("MULTIGPU_RESULT", int(flag.item()), float(np.abs(got - want).max()))
dist.destroy_process_group()
'''


def test_two_rank_allreduce_matches_single_gpu(tmp_path):
    """The all-reduced [sum_ll | G] (8065 doubles at 64 taxa and 4 categories: the peer-memory path) gives every rank
    the matrices of a one-GPU run, with the same bits on every rank."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT})
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("MULTIGPU_RESULT")]
    assert lines and lines[0].split()[1] == "1", r.stdout[-2000:] + r.stderr[-2000:]
