"""Development check of the FP64 tensor-pipe kernels (dmma.cu): the default path against the forced generic path
(tile / scalar kernels) on small codon and amino-acid problems, then cfg4 timings (61 states, 256 taxa x 100k sites).
usage: python tools/dm_check.py [taxa sites]"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
import phyly_b200.arbplf as A
from phyly_b200 import engine as E
from phyly_b200.engine import Engine
from tests.test_scale_gpu import _codon_model


def make(n, Q, taxa, S, seed, mixture=None, missing=0.05, rate=0.1):
    edges, N = bench.yule_tree(taxa, seed=seed)
    rng = np.random.default_rng(seed + 1)
    defs = np.vstack([np.eye(n), np.ones((1, n))])
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(rate, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "character_definitions": defs.tolist(), "character_data": [[n] * N]}
    if mixture:
        md["rate_mixture"] = mixture
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(n, n), np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    codes = np.full((S, N), n, dtype=np.uint8)
    for a in range(N):
        if s["indptr"][a] == s["indptr"][a + 1]:
            col = rng.integers(0, n, S)
            col[rng.random(S) < missing] = n
            codes[:, a] = col
    eng.set_data(defs, codes)
    return eng, s, N


def compare(name, eng):
    eng.set_path(E.PATH_AUTO)
    r = eng.deriv(per_site=True, per_site_ll=True)
    ll = eng.ll(per_site=True)[0]
    eng.set_path(E.PATH_GENERIC)
    g = eng.deriv(per_site=True, per_site_ll=True)
    eng.set_path(E.PATH_AUTO)
    e_ll = np.max(np.abs(r["site_ll"] - g["site_ll"]) / np.abs(g["site_ll"]))
    e_ll2 = np.max(np.abs(ll - g["site_ll"]) / np.abs(g["site_ll"]))
    scale = np.abs(g["site_deriv"]).max()
    e_d = np.max(np.abs(r["site_deriv"] - g["site_deriv"]) / (np.abs(g["site_deriv"]) + 1e-6 * scale))
    e_s = np.max(np.abs(r["sum_deriv"] - g["sum_deriv"]) / np.abs(g["sum_deriv"]).max())
    print(json.dumps({"check": name, "err_ll": e_ll, "err_ll_only": e_ll2, "err_site_deriv": e_d, "err_sum_deriv": e_s}), flush=True)
    return max(e_ll, e_ll2, e_d, e_s)


if __name__ == "__main__":
    Q, pi = _codon_model()
    worst = 0.0
    if len(sys.argv) <= 3:
        eng, s, N = make(61, Q, 16, 300, 21)
        worst = max(worst, compare("codon 16x300", eng)); eng.close()
        eng, s, N = make(61, Q, 70, 1037, 31)
        worst = max(worst, compare("codon 70x1037", eng)); eng.close()
        rng = np.random.default_rng(77)
        n = 20
        p = rng.dirichlet(np.ones(n) * 4)
        R = rng.random((n, n)) + 0.05
        R = (R + R.T) / 2
        Qa = R * p[None, :]
        np.fill_diagonal(Qa, 0.0)
        eng, s, N = make(20, Qa, 40, 1037, 5, mixture={"rates": [0.3, 1.7], "prior": [0.4, 0.6]})
        worst = max(worst, compare("aa 40x1037 C=2", eng)); eng.close()
        n = 30
        p = rng.dirichlet(np.ones(n) * 4)
        R = rng.random((n, n)) + 0.05
        R = (R + R.T) / 2
        Qb = R * p[None, :]
        np.fill_diagonal(Qb, 0.0)
        eng, s, N = make(30, Qb, 33, 555, 6, mixture={"rates": [0.2, 1.0, 2.5], "prior": [0.3, 0.4, 0.3]})
        worst = max(worst, compare("n=30 33x555 C=3", eng)); eng.close()
        print(json.dumps({"worst": worst}), flush=True)
    taxa = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    S = int(sys.argv[2]) if len(sys.argv) > 2 else 100000
    eng, s, N = make(61, Q, taxa, S, 21, missing=0.0, rate=0.05)
    Eg = N - 1
    n = 61
    walls = []
    for it in range(6):
        t0 = time.perf_counter()
        _, tot = eng.ll(per_site=False)
        walls.append((time.perf_counter() - t0) * 1e3)
        ms_mat, ms_sites = eng.last_timing()
        ms_k = eng.last_kernel_ms()
    print(json.dumps({"ll_wall_ms_per_call": walls}), flush=True)
    flops = float(S) * (taxa - 2) * 2 * n * n
    print(json.dumps({"what": "cfg4 ll", "taxa": taxa, "sites": S, "ms_matrices": ms_mat, "ms_sites": ms_sites, "ms_kernels": ms_k,
                      "updates_per_s": S * Eg / (ms_sites * 1e-3), "tflops_gemm_edges": flops / (ms_k * 1e-3) / 1e12, "sum_ll": tot}), flush=True)
    for it in range(3):
        r = eng.deriv(per_site=False)
        ms_mat, ms_sites = eng.last_timing()
        ms_k = eng.last_kernel_ms()
    print(json.dumps({"what": "cfg4 ll+deriv", "ms_matrices": ms_mat, "ms_sites": ms_sites, "ms_kernels": ms_k,
                      "updates_per_s": S * Eg / (ms_sites * 1e-3), "tflops_gemm_edges": 3 * flops / (ms_k * 1e-3) / 1e12,
                      "sum_ll": r["sum_ll"], "d0": float(r["sum_deriv"][0])}), flush=True)
    eng.set_path(E.PATH_GENERIC)
    if S <= 20000:
        g = eng.deriv(per_site=False)
        print(json.dumps({"what": "generic path", "sum_ll": g["sum_ll"], "err_ll": abs(g["sum_ll"] - r["sum_ll"]) / abs(g["sum_ll"]),
                          "err_d": float(np.max(np.abs(g["sum_deriv"] - r["sum_deriv"]) / np.abs(g["sum_deriv"]).max()))}), flush=True)
