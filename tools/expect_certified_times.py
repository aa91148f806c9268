"""Cost of the certified marginals and edge expectations: plf_marginal_certified and plf_edge_expect_certified (one
dwell and one signed trans direction) beside fp64 plf_marginal and one-direction plf_edge_expect (site sums only, data
resident, wall time of the synchronous call), on cfg2 (64 taxa, GTR+Gamma4) at 1e5 and 1e6 sites.  Prints the GPU and
its power limit first, then one JSON line per size."""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from phyly_b200.engine import KIND_DWELL, KIND_TRANS


def timed(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return min(ts)


def inside(v, c):
    return bool(np.all((c["sum_lo"] <= v + 1e-11 * np.abs(v)) & (v - 1e-11 * np.abs(v) <= c["sum_hi"])))


def measure(what, eng):
    out = {"what": what, "sites": eng.S, "states": eng.n, "categories": eng.C, "edges": eng.E}
    n = eng.n
    Ld = np.diag(np.linspace(0.25, 1.0, n))
    Lt = np.array([[0.0 if i == j else (1 + (i + 2 * j) % 3) * (1.0 if (i + j) % 2 else -0.5) for j in range(n)] for i in range(n)])
    out["marginal_ms"] = timed(lambda: eng.marginal(per_site=False))
    out["marginal_certified_ms"] = timed(lambda: eng.marginal_certified(per_site=False))
    out["dwell_ms"] = timed(lambda: eng.edge_expect(KIND_DWELL, Ld, per_site=False))
    out["dwell_certified_ms"] = timed(lambda: eng.edge_expect_certified(KIND_DWELL, Ld, per_site=False))
    out["trans_ms"] = timed(lambda: eng.edge_expect(KIND_TRANS, Lt, per_site=False))
    out["trans_certified_ms"] = timed(lambda: eng.edge_expect_certified(KIND_TRANS, Lt, per_site=False))
    ok = inside(eng.marginal(per_site=False)[1], eng.marginal_certified(per_site=False))
    ok &= inside(eng.edge_expect(KIND_DWELL, Ld, per_site=False)[1], eng.edge_expect_certified(KIND_DWELL, Ld, per_site=False))
    ok &= inside(eng.edge_expect(KIND_TRANS, Lt, per_site=False)[1], eng.edge_expect_certified(KIND_TRANS, Lt, per_site=False))
    out["inside"] = ok
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


if __name__ == "__main__":
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    cfg2(100000)
    cfg2(1000000)
