"""Cost of the certified derivative: plf_deriv_certified beside plf_deriv and plf_ll_certified (site sums only, data
resident, wall time of the synchronous call), on cfg2 (64 taxa, GTR+Gamma4) at 1e5 and 1e6 sites and on cfg4 (61-state
codon model, 256 taxa) at 1e4 sites.  Prints the GPU and its power limit first, then one JSON line per size."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
import phyly_b200.arbplf as A
from phyly_b200.engine import Engine


def timed(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return min(ts)


def measure(what, eng):
    out = {"what": what, "sites": eng.S, "states": eng.n, "categories": eng.C, "edges": eng.E}
    out["deriv_ms"] = timed(lambda: eng.deriv(per_site=False))
    out["ll_certified_ms"] = timed(lambda: eng.ll_certified())
    out["deriv_certified_ms"] = timed(lambda: eng.deriv_certified(per_site=False))
    r = eng.deriv(per_site=False)
    c = eng.deriv_certified(per_site=False)
    v = r["sum_deriv"]
    out["inside"] = bool(np.all((c["sum_lo"] <= v + 1e-11 * np.abs(v)) & (v - 1e-11 * np.abs(v) <= c["sum_hi"])))
    out["max_rel_width"] = float(np.max((c["sum_hi"] - c["sum_lo"]) / np.maximum(np.abs(v), 1e-300)))
    print(json.dumps(out), flush=True)


def cfg2(sites):
    class Args:
        taxa = 64
    Args.sites = sites
    pb = bench.build_problem(Args(), 0, 0)
    eng = pb["eng"]
    eng.set_data(np.array(bench.DEFS, dtype=np.float64), pb["codes"])
    measure("cfg2 GTR+G4, 64 taxa", eng)
    eng.close()


def cfg4(sites, taxa=256):
    Q, _ = bench.codon_model()
    n = Q.shape[0]
    edges, N = bench.yule_tree(taxa, seed=21)
    rng = np.random.default_rng(22)
    defs = np.vstack([np.eye(n), np.ones((1, n))])
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.05, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "character_definitions": defs.tolist(), "character_data": [[n] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(0)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(n, n), np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    codes = np.full((sites, N), n, dtype=np.uint8)
    for a in range(N):
        if s["indptr"][a] == s["indptr"][a + 1]:
            codes[:, a] = rng.integers(0, n, sites)
    eng.set_data(defs, codes)
    measure("cfg4 GY94 61 states, %d taxa" % taxa, eng)
    eng.close()


if __name__ == "__main__":
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    cfg2(100000)
    cfg2(1000000)
    cfg4(10000)
