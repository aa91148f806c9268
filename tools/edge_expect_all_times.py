"""
Timing of plf_edge_expect_all on the cfg2 problem (GTR+G4, 64 taxa x 1M sites, data resident), next to one
plf_edge_expect(TRANS) pass and one plf_deriv pass: the kernel time of the fused kernel and the call time (host clock
around the synchronous query), median of --reps calls after warm-up and tuning.  Prints the card and its power limit
read in the same run, and one JSON line.

  python tools/edge_expect_all_times.py [--sites 1000000] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import bench  # noqa: E402
from phyly_b200 import engine as E  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return r.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()

    class A:
        taxa, sites = 64, args.sites
    pb = bench.build_problem(A, 0, 0)
    eng = pb["eng"]
    eng.set_data_ptr(np.array(bench.DEFS, dtype=np.float64), pb["codes_t"].data_ptr(), pb["S"], 1)
    Lt = np.ones((4, 4)) - np.eye(4)
    queries = {
        "edge_expect_all": lambda: eng.edge_expect_all(),
        "edge_expect_trans": lambda: eng.edge_expect(E.KIND_TRANS, Lt, per_site=False),
        "deriv": lambda: eng.deriv(per_site=False),
    }
    out = {"card": card(), "taxa": 64, "sites": pb["S"], "reps": args.reps}
    names = {}
    for name, fn in queries.items():
        for _ in range(3):          # warm-up; the first call of a kind tunes the fused kernel
            fn()
        call, kern = [], []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            call.append((time.perf_counter() - t0) * 1e3)
            kern.append(eng.last_kernel_ms())
        out[name + "_call_ms"] = float(np.median(call))
        out[name + "_kernel_ms"] = float(np.median(kern))
        names[name] = eng.last_kernel_name()
        print("%-18s call %8.3f ms  kernel %8.3f ms  (%s)" % (name, out[name + "_call_ms"], out[name + "_kernel_ms"],
                                                             names[name]))
    out["kernels"] = names
    out["all_over_two_trans_calls"] = out["edge_expect_all_call_ms"] / (2 * out["edge_expect_trans_call_ms"])
    out["all_over_deriv_calls"] = out["edge_expect_all_call_ms"] / out["deriv_call_ms"]
    print("card: %s" % out["card"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
