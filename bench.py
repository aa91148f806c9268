#!/usr/bin/env python
"""
bench.py -- headline benchmark of the B200 phylogenetic likelihood engine.

Metric (BASELINE.json): site-edge-category updates/s for ll + deriv.  One update
= one (site pattern, edge, rate category) triple processed once
(evaluate_site_lhood.c:54 in the reference); updates per evaluation = S*E*C.

Workload at N=1 (BASELINE.json configs[1], "cfg2"): GTR+Gamma4 model of
examples/BEAST.GTRG on a synthetic 64-taxon tree x 1,000,000 site patterns,
arbplf-ll + arbplf-deriv with the site axis summed.  A "step" is one full
evaluation: edge rates change -> E*C matrix exponentials (+ Q.P) -> tip tables
-> fused pruning + outside pass over all sites -> reduction (-> ncclAllReduce
when N > 1) -> (1+E) doubles back on the host.

  value : inputs (codes, weights) already resident in HBM.
  e2e   : the same evaluation through the C ABI with HOST buffers: the step
          also copies the alignment codes and the site weights from pinned
          host memory to the device and reads the results back.

With --impl reference the same metric is measured for the reference's CPU
algorithm: the C restatement in oracle/c (the Arb reference itself cannot be
built in this image), all host threads, on a bounded sample of the same
workload.

N > 1: one process per GPU (torchrun); the SAME alignment is sharded over the
ranks in contiguous blocks of sites (strong scaling, BASELINE.json configs[1]:
"sharded 1/2/4/8"), results are summed with one in-stream ncclAllReduce; a
weak-scaling measurement (a whole alignment per GPU) is reported beside it.

At N = 1 the line also carries "cfg4" (61-state codon model on the FP64 tensor
pipe), "cfg3" (HKY85+I marginals and the Hessian query) and "json_e2e" (the cfg2
document through the arbplf-deriv drop-in).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# examples/BEAST.GTRG/in.json (model part)
PI = [0.26121198857732775, 0.24655436448599188, 0.33909428971935046, 0.1531393572173299]
RATE_MATRIX = [[0.0 if i == j else PI[j] for j in range(4)] for i in range(4)]
DEFS = [[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1], [1, 1, 1, 1]]

# SURVEY.md section 8(d): algorithmic HBM bytes per update of the streamed formulation
BYTES_PER_UPDATE_LL_DERIV = 79.4
BYTES_PER_UPDATE_LL = 31.9


def yule_tree(taxa, seed):
    """Random binary tree, edges parent -> child listed in random user order (SURVEY 8d)."""
    rng = np.random.default_rng(seed)
    children = {0: []}
    leaves = [0]
    nxt = 1
    while len(leaves) < taxa:
        a = leaves.pop(int(rng.integers(len(leaves))))
        children[a] = [nxt, nxt + 1]
        for k in (nxt, nxt + 1):
            children[k] = []
            leaves.append(k)
        nxt += 2
    N = nxt
    perm = rng.permutation(N)
    edges = [[int(perm[a]), int(perm[b])] for a in children for b in children[a]]
    order = rng.permutation(len(edges))
    return [edges[i] for i in order], N


def model_document(taxa):
    edges, N = yule_tree(taxa, seed=1)
    rng = np.random.default_rng(2)
    rates = rng.exponential(0.05, len(edges))
    md = {
        "edges": edges,
        "edge_rate_coefficients": [float(x) for x in rates],
        "rate_matrix": RATE_MATRIX,
        "root_prior": PI,
        "rate_divisor": "equilibrium_exit_rate",
        "normalized_median_gamma_rate_mixture": {"gamma_categories": 4, "gamma_shape": 0.5},
        "character_definitions": DEFS,
        "character_data": [[4] * N],
    }
    return {"model_and_data": md}, N


def simulate_codes(summary, P, S, seed, out, pi=None, missing=0.01):
    """Simulate S columns down the tree under the model; leaves observed (1% missing), internal nodes unobserved.
    Any state count: the code of state i is i, the missing-data code is n."""
    rng = np.random.default_rng(seed)
    indptr, indices, preorder = summary["indptr"], summary["indices"], summary["preorder"]
    N = len(preorder)
    C, n = P.shape[0], P.shape[-1]
    cum = np.cumsum(P, axis=3)
    cat = rng.integers(0, C, S)
    state = np.empty((N, S), dtype=np.int16)
    root = preorder[0]
    state[root] = np.searchsorted(np.cumsum(PI if pi is None else pi), rng.random(S)).clip(0, n - 1)
    for a in preorder:
        for idx in range(indptr[a], indptr[a + 1]):
            b = indices[idx]
            rows = cum[cat, idx, state[a].astype(np.int64)]          # [S,n]
            u = rng.random(S)
            state[b] = (u[:, None] > rows).sum(axis=1).clip(0, n - 1)
    for a in range(N):
        if indptr[a] == indptr[a + 1]:
            col = state[a].astype(np.uint8)
            miss = rng.random(S) < missing
            col[miss] = n
            out[:, a] = col
        else:
            out[:, a] = n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []          # (arrival time, text)
        self.windows = []        # timed regions [t0, t1] (time.perf_counter)

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # samples that arrived inside a timed region; a region shorter than the sampling period may hold none,
        # then every sample taken while the GPU was under load (warm-up to the last timed step) is used
        inside = [ln for t, ln in self.lines if any(a <= t <= b + 0.02 for a, b in self.windows)]
        window = "timed regions"
        if not inside and self.windows:
            lo, hi = self.windows[0][0] - 1.0, self.windows[-1][1] + 0.02
            inside = [ln for t, ln in self.lines if lo <= t <= hi]
            window = "warm-up + timed regions (timed regions shorter than the sampling period)"
        sm, mx, reasons = [], None, set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "window": window, "reasons": sorted(reasons)}


def load_json(path):
    try:
        with open(path) as f:
            return json.load(f)
    except Exception:
        return None


def dist_setup(n_gpus):
    """torch.distributed over NCCL (one process per GPU), gloo for host objects."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group(backend="cpu:gloo,cuda:nccl", rank=rank, world_size=world)
    return rank, world, local


def bind_near_gpu(local):
    """Multi-rank runs: keep this process (and the pinned buffers it is about to allocate, which land on the NUMA node of
    the allocating thread) on the CPUs next to its GPU, as sysfs lists them.  Returns the cpulist string or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/local_cpulist" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        text = open(path).read().strip()
        cpus = set()
        for part in text.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return text
    except Exception:
        return None


def host_matrices(summary):
    """P and rate*Q*P on the host (scipy), used only to simulate data and by the CPU reference arm."""
    import scipy.linalg
    n, C = summary["state_count"], summary["category_count"]
    Q = np.array(summary["q_hi"]).reshape(n, n)
    t = np.array(summary["edge_rates_csr"])
    r = np.array(summary["cat_rates"])
    P = np.empty((C, len(t), n, n))
    D = np.empty_like(P)
    for c in range(C):
        for e in range(len(t)):
            P[c, e] = scipy.linalg.expm(Q * (r[c] * t[e]))
            D[c, e] = r[c] * (Q @ P[c, e])
    return P, D


def build_problem(args, local, rank, use_engine=True):
    """Host-side setup through the product's own C host layer (no oracle involved).  Every rank simulates the same
    alignment of args.sites columns (seed 3); sharding happens in run_ours."""
    import phyly_b200.arbplf as A
    doc, N = model_document(args.taxa)
    summary = json.loads(A.arbplf_model_summary(json.dumps(doc)))
    n, C = summary["state_count"], summary["category_count"]
    edge_rates = np.array(summary["edge_rates_csr"])
    S = args.sites
    P, D = host_matrices(summary)
    eng = None
    if use_engine:
        import torch
        from phyly_b200.engine import Engine
        eng = Engine(local)
        eng.set_tree(summary["indptr"], summary["indices"], summary["preorder"])
        q_hi = np.array(summary["q_hi"]).reshape(n, n)
        q_lo = np.array(summary["q_lo"]).reshape(n, n)
        eng.set_model(q_hi, q_lo, edge_rates, summary["cat_rates"], summary["cat_prior"], summary["root_mode"],
                      summary["root_vec"])
        codes_t = torch.empty((S, N), dtype=torch.uint8, pin_memory=True)
        codes = codes_t.numpy()
        w_t = torch.ones(S, dtype=torch.float64, pin_memory=True)
    else:
        codes_t, w_t = None, None
        codes = np.empty((S, N), dtype=np.uint8)
    simulate_codes(summary, P, S, seed=3, out=codes)
    codes4_t = None
    if use_engine:
        # the same alignment as PLF_CODES_PACKED4 rows (include/plf.h): what the end-to-end step uploads
        from phyly_b200.engine import pack4
        codes4_t = torch.empty((S, (N + 1) // 2), dtype=torch.uint8, pin_memory=True)
        pack4(codes, out=codes4_t.numpy())
    return dict(eng=eng, summary=summary, N=N, E=N - 1, n=n, C=C, S=S, codes_t=codes_t, codes=codes, w_t=w_t,
                codes4_t=codes4_t, edge_rates=edge_rates, P=P, D=D, doc=doc)


def codon_model(kappa=2.0, omega=0.5, seed=4):
    """GY94-style 61-state rate matrix with F3x4 frequencies (SURVEY 8d cfg4)."""
    rng = np.random.default_rng(seed)
    code = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
    codons = [(a, b_, c) for a in range(4) for b_ in range(4) for c in range(4)]
    aa = {cd: code[16 * cd[0] + 4 * cd[1] + cd[2]] for cd in codons}
    sense = [cd for cd in codons if aa[cd] != "*"]
    f = rng.dirichlet(np.ones(4) * 5, size=3)
    pi = np.array([f[0][cd[0]] * f[1][cd[1]] * f[2][cd[2]] for cd in sense])
    pi /= pi.sum()
    n = len(sense)
    Q = np.zeros((n, n))
    transitions = {(0, 1), (1, 0), (2, 3), (3, 2)}       # T<->C, A<->G
    for i, ci in enumerate(sense):
        for j, cj in enumerate(sense):
            diff = [k for k in range(3) if ci[k] != cj[k]]
            if len(diff) != 1:
                continue
            k = diff[0]
            r = pi[j]
            if (ci[k], cj[k]) in transitions:
                r *= kappa
            if aa[ci] != aa[cj]:
                r *= omega
            Q[i, j] = r
    return Q, pi


def bench_cfg4(local, peaks_fp64, taxa=256, sites=100000, steps=10):
    """BASELINE.json configs[3] (cfg4): 61-state GY94 codon model, 256 taxa x 100 000 codon sites, ll and ll + deriv on
    the FP64 tensor-pipe kernels (dmma.cu).  Timed on the device, data resident."""
    import torch
    import phyly_b200.arbplf as A
    from phyly_b200.engine import Engine
    Q, pi = codon_model()
    n = Q.shape[0]
    edges, N = yule_tree(taxa, seed=21)
    rng = np.random.default_rng(22)
    defs = np.vstack([np.eye(n), np.ones((1, n))])
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.05, len(edges))],
          "rate_matrix": Q.tolist(), "root_prior": "equilibrium_distribution", "rate_divisor": "equilibrium_exit_rate",
          "character_definitions": defs.tolist(), "character_data": [[n] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(local)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(n, n), np.array(s["q_lo"]).reshape(n, n), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    P = eng.transition_matrices()
    base = np.full((sites // 4, N), n, dtype=np.uint8)
    simulate_codes(s, P, sites // 4, seed=24, out=base, pi=np.array(s["equilibrium"]))
    codes = np.tile(base, (4, 1))
    eng.set_data(defs, codes)
    S, E = codes.shape[0], N - 1
    Ei = sum(1 for b in s["indices"] if s["indptr"][b] != s["indptr"][b + 1])
    stream = torch.cuda.ExternalStream(eng.stream(), device=local)
    out = {"workload": "cfg4: GY94 61-state codon model (kappa 2, omega 0.5, F3x4) x %d-taxon Yule tree x %d codon sites, "
                       "C = 1, data resident" % (taxa, S), "taxa": taxa, "sites": S, "states": n, "edges": E,
           "flop_convention": "2 n^2 flops per contraction on the true state count n = 61 (the kernels work on 64 padded states) "
                              "plus n per edge for the Hadamard products: ll = Ei (2 n^2) + E n per site (SURVEY 8d: 1.92e11 per "
                              "evaluation); ll+deriv = 3 Ei (2 n^2) + 4 E n (two more contractions per internal-child edge in "
                              "the outside pass: P^T fe and F^T fe)",
           "peak_tflops": peaks_fp64.get("dmma_m8n8k4_tflops"), "peak_source": "profiles/fp64_peak.json (tools/fp64_peak.cu, this GPU model)"}
    for kind in ("ll", "ll_deriv"):
        fn = (lambda: eng.ll(per_site=False)) if kind == "ll" else (lambda: eng.deriv(per_site=False))
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        km = []
        walls = []
        e0.record(stream)
        for _ in range(steps):
            tw = time.perf_counter()
            r = fn()
            walls.append((time.perf_counter() - tw) * 1e3)
            km.append(eng.last_kernel_ms())
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        k_ms = float(np.mean(km))
        flops = float(S) * ((1 if kind == "ll" else 3) * Ei * 2.0 * n * n + (1 if kind == "ll" else 4) * E * n)
        tf = flops / (k_ms * 1e-3) / 1e12
        out[kind] = {"ms_per_step": ms, "kernels_ms": k_ms, "host_wall_ms_per_call": [round(x, 3) for x in walls], "updates_per_s": float(S) * E / (ms * 1e-3),
                     "kernel": eng.last_kernel_name(), "flops_per_step": flops,
                     "roofline": {"bound": "tensor", "achieved": tf, "peak": out["peak_tflops"], "unit": "TFLOP/s",
                                  "frac": tf / out["peak_tflops"] if out["peak_tflops"] else None},
                     "sum_ll": (r[1] if kind == "ll" else r["sum_ll"])}
    eng.close()
    return out


def bench_cfg3(local, taxa=128, sites=500000, hess_sites=500000, steps=5):
    """BASELINE.json configs[2] (cfg3): HKY85+I (kappa 2, invariant category), 128 taxa x 500 000 sites: posterior
    marginals summed over sites, and the second-order query (gradient + Hessian of the log likelihood, E x E) that
    arbplf-hess / newton-update need (the Hessian kernel is O(E^2) per site; one timed evaluation after one warm-up)."""
    import torch
    import phyly_b200.arbplf as A
    from phyly_b200.engine import Engine
    edges, N = yule_tree(taxa, seed=11)
    rng = np.random.default_rng(12)
    pi = (0.3, 0.2, 0.25, 0.25)
    Q = [[0.0] * 4 for _ in range(4)]
    for i in range(4):
        for j in range(4):
            if i != j:
                Q[i][j] = pi[j] * (2.0 if (i, j) in ((0, 2), (2, 0), (1, 3), (3, 1)) else 1.0)
    md = {"edges": edges, "edge_rate_coefficients": [float(x) for x in rng.exponential(0.05, len(edges))],
          "rate_matrix": Q, "root_prior": list(pi), "rate_divisor": "equilibrium_exit_rate",
          "rate_mixture": {"rates": [0.0, 2.0], "prior": [0.5, 0.5]},
          "character_definitions": DEFS, "character_data": [[4] * N]}
    s = json.loads(A.arbplf_model_summary(json.dumps({"model_and_data": md})))
    eng = Engine(local)
    eng.set_tree(s["indptr"], s["indices"], s["preorder"])
    eng.set_model(np.array(s["q_hi"]).reshape(4, 4), np.array(s["q_lo"]).reshape(4, 4), s["edge_rates_csr"], s["cat_rates"],
                  s["cat_prior"], s["root_mode"], s["root_vec"])
    P = eng.transition_matrices()
    codes = np.empty((sites, N), dtype=np.uint8)
    simulate_codes(s, P, sites, seed=13, out=codes)
    defs = np.array(DEFS, dtype=np.float64)
    E = N - 1
    stream = torch.cuda.ExternalStream(eng.stream(), device=local)

    def timed(fn, n, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(n):
            r = fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, r

    out = {"workload": "cfg3: HKY85 (kappa 2) + invariant category x %d-taxon Yule tree x %d sites, C = 2, data resident" % (taxa, sites),
           "taxa": taxa, "sites": sites, "edges": E}
    eng.set_data(defs, codes)
    ms, r = timed(lambda: eng.marginal(per_site=False), steps)
    out["marginal_site_sum"] = {"ms_per_step": ms, "updates_per_s": float(sites) * E * 2 / (ms * 1e-3), "kernel": eng.last_kernel_name()}
    ms, r = timed(lambda: eng.deriv(per_site=False), steps)
    out["ll_deriv"] = {"ms_per_step": ms, "updates_per_s": float(sites) * E * 2 / (ms * 1e-3), "kernel": eng.last_kernel_name()}
    eng.set_data(defs, codes[:hess_sites])
    ms, r = timed(lambda: eng.hess(), 1, warm=1)
    H = r[2]
    out["hess"] = {"sites": hess_sites, "ms_per_step": ms, "ms_per_1000_sites": ms / hess_sites * 1000.0,
                   "extrapolated_ms_at_full_size": ms / hess_sites * sites,
                   "pair_updates_per_s": float(hess_sites) * 2 * E * (E + 1) / 2 / (ms * 1e-3),
                   "kernel": "generic_inside / generic_outside / generic_hess_kernel / gram_rows_kernel (scalar fp64, thread = site)",
                   "hessian_is_symmetric": bool(np.array_equal(H, H.T)), "sum_ll": r[0],
                   "note": "one tangent sweep per edge, O(E^2) per (site, category); the reference re-walks two root paths per pair, O(E^2 depth)"}
    eng.close()
    return out


def json_document_bytes(doc, codes):
    """The arbplf JSON document of the workload with its character_data, built without a Python-level loop."""
    S, N = codes.shape
    row = np.empty((S, 2 * N + 2), dtype=np.uint8)
    row[:, 0] = ord("[")
    row[:, 1:2 * N:2] = codes + ord("0")
    row[:, 2:2 * N:2] = ord(",")
    row[:, 2 * N] = ord("]")
    row[:, 2 * N + 1] = ord(",")
    data = row.tobytes()[:-1]
    md = dict(doc["model_and_data"])
    md["character_data"] = "@@DATA@@"
    top = {"model_and_data": md, "site_reduction": {"aggregation": "sum"}}
    head, tail = json.dumps(top).split('"@@DATA@@"')
    return head.encode() + b"[" + data + b"]" + tail.encode()


def bench_json_e2e(pb, max_sites):
    """The drop-in path at size: the cfg2 document (character_data for every site) through arbplf_deriv of the C ABI in
    this process and through the arbplf-deriv executable (stdin -> stdout), with the host layer's own phase timings."""
    import ctypes as c
    from phyly_b200 import _lib
    S = min(pb["S"], max_sites)
    t0 = time.perf_counter()
    text = json_document_bytes(pb["doc"], pb["codes"][:S])
    t_build = time.perf_counter() - t0
    lib = _lib.load()
    lib.arbplf_deriv.restype = c.c_void_p
    lib.arbplf_deriv.argtypes = [c.c_char_p, c.POINTER(c.c_int)]
    lib.arbplf_last_timing.argtypes = [c.POINTER(c.c_double)]
    libc = c.CDLL(None)
    libc.free.argtypes = [c.c_void_p]
    out = {"sites": S, "document_bytes": len(text), "build_document_s": t_build}
    # call 1: cold process state (engine creation, kernel tuning); call 2: the same document with the reader's data cache
    # switched off (every call reads and uploads the alignment); "repeat_call": the same document once more with the
    # cache on, after one call that made the alignment resident -- what an optimiser's loop over one alignment pays
    labels = ["in_process_call_1", "in_process_call_2", None, "repeat_call"]
    for rep in range(4):
        if rep == 1:
            os.environ["ARBPLF_NO_DATA_CACHE"] = "1"
        else:
            os.environ.pop("ARBPLF_NO_DATA_CACHE", None)
        rc = c.c_int(0)
        t0 = time.perf_counter()
        res = lib.arbplf_deriv(text, c.byref(rc))
        wall = time.perf_counter() - t0
        if not res or rc.value != 0:
            return {"error": "arbplf_deriv failed with retcode %d" % rc.value}
        first = c.string_at(res)[:200].decode()
        libc.free(res)
        ph = (c.c_double * 4)()
        lib.arbplf_last_timing(ph)
        if labels[rep]:
            out[labels[rep]] = {"wall_s": wall, "parse_s": ph[0], "model_and_upload_s": ph[1], "compute_s": ph[2],
                                "emit_s": ph[3], "updates_per_s": float(S) * pb["E"] * pb["C"] / wall}
    out["output_head"] = first[:120]
    # the site axis kept: arbplf_ll without a site reduction writes one row per site pattern
    tail = b', "site_reduction": {"aggregation": "sum"}}'
    if text.endswith(tail):
        lib.arbplf_ll.restype = c.c_void_p
        lib.arbplf_ll.argtypes = [c.c_char_p, c.POINTER(c.c_int)]
        per_site = text[:-len(tail)] + b"}"
        rc = c.c_int(0)
        t0 = time.perf_counter()
        res = lib.arbplf_ll(per_site, c.byref(rc))
        wall = time.perf_counter() - t0
        if res and rc.value == 0:
            nbytes = len(c.string_at(res))
            libc.free(res)
            ph = (c.c_double * 4)()
            lib.arbplf_last_timing(ph)
            out["per_site_ll_call"] = {"wall_s": wall, "parse_s": ph[0], "model_and_upload_s": ph[1], "compute_s": ph[2],
                                       "emit_s": ph[3], "output_bytes": nbytes}
    exe = os.path.join(ROOT, "phyly_b200", "bin", "arbplf-deriv")
    if os.path.exists(exe):
        t0 = time.perf_counter()
        pr = subprocess.run([exe], input=text, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        out["cli"] = {"wall_s": time.perf_counter() - t0, "retcode": pr.returncode,
                      "note": "process start, CUDA context and first-query kernel tuning included"}
    return out


def dump_outputs(path, m):
    """The last timed step of each cfg2 loop as a caller of include/plf.h receives it (all ranks' sums when N > 1): ll + deriv
    with resident inputs (the headline), the same query end to end, and ll alone.  The inputs are seeded, so two builds of
    the project can be compared array for array."""
    os.makedirs(path, exist_ok=True)
    arrays = {"sum_ll": [m["res"]["sum_ll"]], "sum_deriv": m["res"]["sum_deriv"],
              "e2e_sum_ll": [m["res2"]["sum_ll"]], "e2e_sum_deriv": m["res2"]["sum_deriv"],
              "ll_only_sum_ll": [m["res3"][1]]}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from phyly_b200 import engine as E
    rank, world, local = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    numa = bind_near_gpu(local) if world > 1 and not os.environ.get("PLF_BENCH_NO_BIND") else None
    pb = build_problem(args, local, rank)
    eng = pb["eng"]
    S_total, Eg, C, N = pb["S"], pb["E"], pb["C"], pb["N"]
    defs = np.array(DEFS, dtype=np.float64)
    if world > 1:
        uid = [E.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(world, rank, uid[0])
    stream = torch.cuda.ExternalStream(eng.stream(), device=local)
    sync_upload = bool(os.environ.get("PLF_BENCH_SYNC_UPLOAD"))
    packed = not os.environ.get("PLF_BENCH_UNPACKED")        # end-to-end step uploads 4-bit codes (two per byte)
    row_bytes = (N + 1) // 2 if packed else N

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(lo, hi, steps, want_e2e, want_ll):
        """Times the step on the site patterns [lo, hi) of the alignment: resident, end to end, ll only."""
        S = hi - lo
        codes_ptr = pb["codes_t"].data_ptr() + lo * N
        e2e_ptr = pb["codes4_t"].data_ptr() + lo * row_bytes if packed else codes_ptr
        e2e_cb = E.CODES_PACKED4 if packed else 1
        w_ptr = pb["w_t"].data_ptr() + 8 * lo
        w_np = pb["w_t"].numpy()[lo:hi]

        def step_resident():
            eng.set_edge_rates(pb["edge_rates"])          # invalidates P, Q.P and the tip tables
            return eng.deriv(per_site=False)

        def step_e2e():
            if sync_upload:
                eng.set_data_ptr(defs, e2e_ptr, S, e2e_cb)
                eng.set_site_weights(w_np)
            else:       # chunked upload overlapped with the kernel
                eng.set_data_async_ptr(defs, e2e_ptr, S, w_ptr, e2e_cb)
            eng.set_edge_rates(pb["edge_rates"])
            return eng.deriv(per_site=False)

        def step_ll():
            eng.set_edge_rates(pb["edge_rates"])
            return eng.ll(per_site=False)

        eng.set_data_ptr(defs, codes_ptr, S, 1)
        eng.set_site_weights(w_np)
        for _ in range(args.warmup):
            res = step_resident()
        barrier()
        eng.launch_count(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kern_ms, mat_ms, site_ms = [], [], []
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            res = step_resident()
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        # the engine's own event timings (kernel, matrices) from a few extra steps: reading them costs host time
        # between the steps, which the timed loop should not carry
        for _ in range(min(steps, 10)):
            step_resident()
            kern_ms.append(eng.last_kernel_ms())
            tm = eng.last_timing()
            mat_ms.append(tm[0]); site_ms.append(tm[1])
        barrier()
        out = dict(S=S, steps=steps, ms=e0.elapsed_time(e1), wall=wall, t0=t0, launches=eng.launch_count(), res=res,
                   kern_ms=float(np.mean(kern_ms)), mat_ms=float(np.mean(mat_ms)), site_ms=float(np.mean(site_ms)),
                   kernel=eng.last_kernel_name())
        if want_e2e:
            e2e_steps = steps
            for _ in range(min(args.warmup, 3)):
                step_e2e()
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t1 = time.perf_counter()
            f0.record(stream)
            for _ in range(e2e_steps):
                res2 = step_e2e()
            f1.record(stream)
            barrier()
            out.update(e2e_steps=e2e_steps, ms_e2e=f0.elapsed_time(f1), t1=t1, t1_end=time.perf_counter(), res2=res2)
        if want_ll:
            ll_steps = steps
            for _ in range(3):
                step_ll()
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ll_kern = []
            g0.record(stream)
            for _ in range(ll_steps):
                res3 = step_ll()
                ll_kern.append(eng.last_kernel_ms())
            g1.record(stream)
            barrier()
            out.update(ll_steps=ll_steps, ms_ll=g0.elapsed_time(g1), ll_kern=float(np.mean(ll_kern)), ll_kernel=eng.last_kernel_name(),
                       res3=res3)
        return out

    def max_over_ranks(vals):
        if world == 1:
            return [float(v) for v in vals]
        tt = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return [float(x) for x in tt]

    # ---- headline: the SAME alignment sharded over the ranks (strong scaling; at N = 1 the whole of it) ----
    lo, hi = rank * S_total // world, (rank + 1) * S_total // world
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    m = measure(lo, hi, args.steps, True, True)
    if rank == 0:
        sampler.mark(m["t0"], m["t0"] + m["wall"])
        sampler.mark(m["t1"], m["t1_end"])
    clocks = sampler.stop() if rank == 0 else None
    ms, ms_e2e, ms_ll = max_over_ranks([m["ms"], m["ms_e2e"], m["ms_ll"]])
    # ---- the collective checked against its inputs: local sums gathered over gloo vs the all-reduced vector ----
    allreduce_check = None
    if world > 1:
        eng.comm_pause(True)
        loc = eng.deriv(per_site=False)
        eng.comm_pause(False)
        glob = eng.deriv(per_site=False)
        mine = np.concatenate([[loc["sum_ll"]], loc["sum_deriv"]])
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        want = np.sum(np.stack(gathered), axis=0)
        got = np.concatenate([[glob["sum_ll"]], glob["sum_deriv"]])
        err = float(np.max(np.abs(got - want) / np.maximum(np.abs(want), 1e-300)))
        allreduce_check = {"values": int(got.size), "max_rel_diff_vs_sum_of_local": err, "ok": bool(err <= 1e-13),
                           "sum_ll_all_ranks": float(got[0]), "local_sum_ll": [float(g[0]) for g in gathered]}
        assert allreduce_check["ok"], allreduce_check
    # ---- weak scaling beside it (N > 1 only): every rank owns a whole alignment of args.sites patterns ----
    weak = None
    if world > 1:
        mw = measure(0, S_total, args.steps, True, False)
        ms_w, ms_w_e2e = max_over_ranks([mw["ms"], mw["ms_e2e"]])
        weak = {"scaling": "weak", "sites_per_gpu": S_total, "steps": mw["steps"], "ms_per_step": ms_w / mw["steps"],
                "value": float(S_total) * Eg * C * world * mw["steps"] / (ms_w * 1e-3), "unit": "updates/s",
                "kernel_ms": mw["kern_ms"],
                "e2e": {"value": float(S_total) * Eg * C * world * mw["e2e_steps"] / (ms_w_e2e * 1e-3), "unit": "updates/s",
                        "ms_per_step": ms_w_e2e / mw["e2e_steps"], "steps": mw["e2e_steps"],
                        "h2d_bytes_per_step": int(S_total * row_bytes + 8 * S_total + 8 * Eg),
                        "note": "every rank uploads a whole alignment every step; bytes are per GPU"}}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, m)
    S = m["S"]
    updates_per_step = float(S_total) * Eg * C
    value = updates_per_step * args.steps / (ms * 1e-3)
    e2e_value = updates_per_step * m["e2e_steps"] / (ms_e2e * 1e-3)
    peaks = load_json(os.path.join(ROOT, "MEASURED_PEAKS.json"))
    hbm_peak = peaks["hbm_gbs"] if peaks and "hbm_gbs" in peaks else 6650.0
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    fp64 = load_json(os.path.join(ROOT, "profiles", "fp64_peak.json")) or {}
    traffic_db = (load_json(os.path.join(ROOT, "profiles", "ncu_traffic.json")) or {}).get("kernels", {})
    k_ms = m["kern_ms"]
    # ---- roofline of the dominant kernel (rank 0's shard of S sites) ----
    summary = pb["summary"]
    n_int_edges = sum(1 for b in summary["indices"] if summary["indptr"][b] != summary["indptr"][b + 1])
    n_tip_edges = Eg - n_int_edges
    n_internal = n_int_edges + 1
    tr = traffic_db.get(m["kernel"])
    traffic = tr["dram_bytes_per_launch"] * (float(S) / tr["sites"]) if tr else None
    # bytes the kernel is written to move (fused4.cuh): every internal node's partial goes once to the slab and comes back
    # once (double4 + 1 byte per category), the codes of the tips once, weights in, site log-likelihoods out
    own_bytes = float(S) * (2.0 * 33.0 * n_internal * C + (n_tip_edges) + 8 + 8)
    streamed_bytes = BYTES_PER_UPDATE_LL_DERIV * float(S) * Eg * C
    compulsory = float(S) * (n_tip_edges + 8)
    moved = traffic if traffic else own_bytes
    flops = float(S) * C * (n_int_edges * (36 + 108) + n_tip_edges * (4 + 14))
    roofline = {
        "bound": "hbm", "kernel": m["kernel"],
        "achieved": moved / (k_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
        "frac": moved / (k_ms * 1e-3) / 1e9 / hbm_peak,
        "traffic": traffic,
        "bytes_basis": ("DRAM bytes per launch measured by ncu for exactly this instantiation (profiles/ncu_traffic.json), scaled "
                        "to this launch's sites" if traffic else "the kernel's own byte model (no ncu capture of this instantiation)"),
        "peak_source": peak_src,
        "own_model_bytes_per_launch": own_bytes,
        "frac_own_model": own_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak,
        "streamed_model_bytes_per_launch": streamed_bytes,
        "frac_streamed_model": streamed_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak,
        "compulsory_bytes_per_launch": compulsory,
        "compulsory_bound_ms": compulsory / (hbm_peak * 1e9) * 1e3,
        "note": ("frac = bytes this kernel really moves / its time / measured HBM copy peak.  frac_streamed_model is SURVEY "
                 "8(d)'s figure for a formulation that streams every partial (79.4 B/update), which this kernel does not follow "
                 "(its value above 1 only says the kernel moves fewer bytes than that); compulsory = tip codes + weights, the "
                 "bound of a traversal that kept every partial on chip"),
        "fp64": {"achieved_tflops": flops / (k_ms * 1e-3) / 1e12, "peak_tflops": fp64.get("dfma_tflops"),
                 "frac": (flops / (k_ms * 1e-3) / 1e12) / fp64["dfma_tflops"] if fp64.get("dfma_tflops") else None,
                 "flops_per_launch": flops},
        "kernel_ms": k_ms,
    }
    step_ms = ms / args.steps
    line = {
        "metric": "site-edge-category updates/s (ll+deriv)", "value": value, "unit": "updates/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg2: GTR+Gamma4 (examples/BEAST.GTRG model) x %d-taxon Yule tree x %d site patterns in total, "
                               "sharded over the GPUs, arbplf-ll + arbplf-deriv, site axis summed" % (args.taxa, S_total),
                   "sites_total": S_total, "sites_per_gpu": S, "taxa": args.taxa, "edges": Eg, "categories": C, "states": pb["n"],
                   "sharding": "contiguous blocks of sites, one ncclAllReduce of %d doubles per step" % (1 + Eg),
                   "cache": "inputs and scratch (%.0f MB per GPU) exceed the 126 MB L2; no explicit flush" % (S * N / 1e6 + 600)},
        "step_breakdown_ms": {"matrices_and_tables": m["mat_ms"], "fused_kernel": k_ms,
                              "reduction_allreduce_readback": max(0.0, m["site_ms"] - k_ms),
                              "host_gaps": max(0.0, step_ms - m["mat_ms"] - m["site_ms"]),
                              "note": "CUDA events of rank 0 inside the step; host_gaps = step time not covered by them"},
        "e2e": {"value": e2e_value, "unit": "updates/s", "h2d_bytes_per_step": int(S * row_bytes + 8 * S + 8 * Eg),
                "d2h_bytes_per_step": int(8 * (1 + Eg)), "steps": m["e2e_steps"], "ms_per_step": ms_e2e / m["e2e_steps"],
                "api": ("plf_set_data + plf_set_site_weights" if sync_upload else "plf_set_data_async") + " + plf_set_edge_rates + plf_deriv (include/plf.h), pinned host buffers, codes as "
                       + ("PLF_CODES_PACKED4 (two per byte)" if packed else "uint8") + "; bytes are per GPU"},
        "gpu_launches": int(m["launches"]),
        "clocks": clocks,
        "roofline": roofline,
        "ll_only": {"metric": "site-edge-category updates/s (ll)", "value": updates_per_step * m["ll_steps"] / (ms_ll * 1e-3),
                    "unit": "updates/s", "steps": m["ll_steps"], "ms_per_step": ms_ll / m["ll_steps"],
                    "kernel_ms": m["ll_kern"], "kernel": m["ll_kernel"],
                    "compulsory_bound_ms": compulsory / (hbm_peak * 1e9) * 1e3,
                    "frac_streamed_model": (BYTES_PER_UPDATE_LL * float(S) * Eg * C / (m["ll_kern"] * 1e-3) / 1e9) / hbm_peak,
                    "note": "supplementary; no slab, partials never leave the SM: HBM traffic is the tip codes, the kernel is bound by issue / LSU, not DRAM"},
        "result_check": {"sum_ll": m["res"]["sum_ll"], "sum_ll_e2e": m["res2"]["sum_ll"], "wall_s": m["wall"]},
    }
    if allreduce_check:
        line["allreduce_check"] = allreduce_check
    if world > 1:
        line["host_binding"] = {"rank0_cpulist": numa, "note": "each rank pinned to the CPUs sysfs lists next to its GPU before its "
                                "pinned buffers are allocated (null: sysfs entry not available, no binding)"}
    if weak:
        line["weak"] = weak
    if world == 1 and not args.no_extras:
        eng.close()
        try:
            line["cfg4"] = bench_cfg4(local, fp64)
        except Exception as ex:       # a supplementary measurement must not lose the headline
            line["cfg4"] = {"error": repr(ex)}
        try:
            line["cfg3"] = bench_cfg3(local)
        except Exception as ex:
            line["cfg3"] = {"error": repr(ex)}
        try:
            line["json_e2e"] = bench_json_e2e(pb, args.json_sites)
        except Exception as ex:
            line["json_e2e"] = {"error": repr(ex)}
    # last: its OpenMP team keeps spinning on the host cores for a while after the parallel region
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(pb, target_seconds=args.cpu_seconds)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def cpu_port_problem(pb):
    """Inputs of the C restatement taken from the engine (matrices) and the workload (codes)."""
    return dict(P=pb["P"], D=pb["D"], prior=np.array(pb["summary"]["cat_prior"]),
                root_mode=pb["summary"]["root_mode"], root_vec=np.array(pb["summary"]["root_vec"]))


def host_threads():
    """All host cores this process may use.  Not omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to
    its workers, which would silently turn the reference arm into a one-thread run for N > 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_baseline(pb, target_seconds=15.0, sample=None):
    """Time oracle/c (the 'port' of the reference algorithm) on a bounded sample, all host threads."""
    from oracle import c_port
    cp = cpu_port_problem(pb)
    s = pb["summary"]
    threads = host_threads()
    defs = np.array(DEFS, dtype=np.float64)

    def run(nsites):
        t0 = time.perf_counter()
        c_port.ll_deriv(s["indptr"], s["indices"], s["preorder"], cp["P"], cp["D"], cp["prior"], cp["root_mode"],
                        cp["root_vec"], pb["codes"][:nsites], defs, w=None, nthreads=threads, want_site_ll=False)
        return time.perf_counter() - t0
    if sample is None:
        pilot = min(pb["S"], 4000 * threads)
        run(min(pilot, 1000))
        dt = run(pilot)
        sample = int(min(pb["S"], max(pilot, pilot * target_seconds / max(dt, 1e-6))))
    dt = run(sample)
    return {"value": sample * pb["E"] * pb["C"] / dt, "unit": "updates/s", "cores": threads, "kind": "port",
            "sample": "%d of %d site patterns, ll+deriv, oracle/c/plf_oracle.c (OpenMP, fp64), %.2f s" % (sample, pb["S"], dt),
            "seconds": dt, "sample_sites": sample}


def build_problem_reference(args):
    """The same workload set up WITHOUT the product: model quantities and matrices from the oracle (fp64 back end), so that
    the reference arm never maps libarbplf_b200.so."""
    from oracle import arbplf_oracle as O
    doc, N = model_document(args.taxa)
    be = O.get_backend("fp64")
    m = O.parse_model(doc["model_and_data"])
    cs = O.cross_site(m, be)
    t = m.tree
    summary = {"indptr": list(t.indptr), "indices": list(t.indices), "preorder": list(t.preorder),
               "cat_prior": [float(x) for x in cs.prior], "root_mode": int(m.root_mode),
               "root_vec": [float(x) for x in O.root_prior_vector(m, cs, be)]}
    P = np.asarray(cs.P, dtype=np.float64)
    D = np.empty_like(P)
    Q = np.asarray(cs.Q, dtype=np.float64)
    for c in range(cs.C):
        for e in range(cs.E):
            D[c, e] = float(cs.rates[c]) * (Q @ P[c, e])
    S = args.sites
    codes = np.empty((S, N), dtype=np.uint8)
    simulate_codes(summary, P, S, seed=3, out=codes)
    return dict(eng=None, summary=summary, N=N, E=N - 1, n=m.n, C=cs.C, S=S, codes=codes, P=P, D=D, doc=doc)


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (C restatement; Arb cannot be built here) on host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pb = build_problem_reference(args)
    from oracle import c_port
    threads = host_threads()
    # size each step so that the whole run ends within a few minutes
    first = cpu_baseline(pb, target_seconds=2.0)
    rate = first["value"] / (pb["E"] * pb["C"])               # sites per second
    budget = 120.0 / max(1, args.steps + args.warmup)
    sample = int(min(pb["S"], max(1000, rate * min(budget, 15.0))))
    for _ in range(args.warmup):
        cpu_baseline(pb, sample=sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = cpu_baseline(pb, sample=sample)
    dt = time.perf_counter() - t0
    value = sample * pb["E"] * pb["C"] * args.steps / dt
    cb = {"value": value, "unit": "updates/s", "cores": threads, "kind": "port",
          "sample": "%d of %d site patterns per step, ll+deriv, oracle/c/plf_oracle.c (OpenMP, fp64)" % (sample, pb["S"])}
    Eg, C = pb["E"], pb["C"]
    line = {
        "impl": "reference", "metric": "site-edge-category updates/s (ll+deriv)", "value": value, "unit": "updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        # the same keys and workload string as the product arm (the GPUs only shard it; this arm has none)
        "config": {"workload": "cfg2: GTR+Gamma4 (examples/BEAST.GTRG model) x %d-taxon Yule tree x %d site patterns in total, "
                               "sharded over the GPUs, arbplf-ll + arbplf-deriv, site axis summed" % (args.taxa, pb["S"]),
                   "sites_total": pb["S"], "taxa": args.taxa, "edges": Eg, "categories": C, "states": pb["n"],
                   "sample": "each step evaluates %d of the %d site patterns (bounded sample), all host threads" % (sample, pb["S"]),
                   "note": "the Arb reference cannot be compiled in this image (no arb/flint/gmp/jansson headers); "
                           "this is its algorithm restated in C (oracle/c), fp64, one OpenMP thread per host core; "
                           "set up from the oracle alone, the product library is not loaded"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def emit(line):
    """Print the one JSON line on the real stdout (libraries such as NCCL write banners to fd 1)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)          # anything else that writes to fd 1 goes to stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sites", type=int, default=1000000)
    ap.add_argument("--taxa", type=int, default=64)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg4 and JSON drop-in measurements (N = 1)")
    ap.add_argument("--json-sites", type=int, default=1000000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each cfg2 loop returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a site sample and keeps no outputs")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
