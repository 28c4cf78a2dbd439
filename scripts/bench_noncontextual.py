"""Throughput of NoncontextualOp.solve (brute-force ground-state search, kernel sym_nc_min) on one GPU.

Times solve() with CUDA events after a warm-up call on the noncontextual parts of the HOOH STO-3G Hamiltonian (24 q,
both strategies) and on synthetic noncontextual operators with f = 28, 32, 36 free generators, ~500 terms and 3
cliques, and reports assignments/s. A NumPy direct evaluation (one sign per assignment and term) of an f = 20
instance is timed in the same run for comparison. The card name and power limit are read in the same run.

    python scripts/bench_noncontextual.py --out <dir>      # writes <dir>/bench_noncontextual.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)


def synthetic(f, n_terms=500, N=3, seed=0):
    """f independent Z generators on qubits 0..f-1 and N anticommuting clique representatives on two more qubits
    (X, Y, Z X); every term is a random Z string times no representative or one of them."""
    from symmer_b200 import NoncontextualOp
    rng = np.random.default_rng(seed)
    n = f + 2
    reps = np.zeros((N, 2 * n), dtype=bool)
    reps[0, f] = True
    reps[1, [f, n + f]] = True
    reps[2, [f + 1, n + f]] = True
    symp = np.zeros((n_terms, 2 * n), dtype=bool)
    symp[:, n:n + f] = rng.random((n_terms, f)) < 0.5
    clique = rng.integers(-1, N, size=n_terms)
    clique[:N] = np.arange(N)
    symp[clique >= 0] ^= reps[clique[clique >= 0]]
    return NoncontextualOp(symp, rng.normal(size=n_terms))


def time_solve(nc, reps):
    import torch
    nc.solve()                                      # warm-up: module load, workspace
    times = []
    for _ in range(reps):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        nc.solve()
        end.record()
        end.synchronize()
        times.append(start.elapsed_time(end) / 1e3)
    return times


def numpy_direct(f, n_assignments):
    """Direct evaluation of E(m) for the first n_assignments m of a synthetic f-generator instance."""
    nc = synthetic(f, seed=1)
    J = np.zeros(nc.n_terms, dtype=np.uint64)
    for q in range(nc._J.shape[1]):
        J |= nc._J[:, q].astype(np.uint64) << np.uint64(q)
    v = nc.coeff_vec.real * nc._signs
    cl = nc._clique
    t0 = time.perf_counter()
    best = np.inf
    for m0 in range(0, n_assignments, 4096):
        m = np.arange(m0, m0 + 4096, dtype=np.uint64)
        terms = (1.0 - 2.0 * (np.bitwise_count(m[:, None] & J[None, :]) & 1)) * v[None, :]
        w2 = sum(terms[:, cl == i].sum(axis=1) ** 2 for i in range(3))
        best = min(best, float(np.min(terms[:, cl < 0].sum(axis=1) - np.sqrt(w2))))
    dt = time.perf_counter() - t0
    return {"f": f, "terms": int(nc.n_terms), "assignments_timed": n_assignments, "seconds": dt,
            "ns_per_assignment_term": dt / (n_assignments * nc.n_terms) * 1e9,
            "assignments_per_s": n_assignments / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_noncontextual.py needs a CUDA device")
    from symmer_b200 import NoncontextualOp, PauliwordOp
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    result = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "cases": []}
    d = np.load(os.path.join(ROOT, "tests", "golden", "hamiltonians", "HOOH_STO3G.npz"))
    n = int(d["n_qubits"][0])
    H = PauliwordOp(np.unpackbits(d["symp"], axis=1)[:, :2 * n].astype(bool), d["coeff"])
    cases = [(f"HOOH {s}", lambda s=s: NoncontextualOp.from_hamiltonian(H, strategy=s))
             for s in ("diag", "SingleSweep_magnitude")]
    cases += [(f"synthetic f={f}", lambda f=f: synthetic(f)) for f in (28, 32, 36)]
    for name, make in cases:
        t0 = time.perf_counter()
        nc = make()
        build = time.perf_counter() - t0
        f = nc.symmetry_generators.n_terms
        times = time_solve(nc, args.reps)
        best = min(times)
        row = {"case": name, "terms": int(nc.n_terms), "cliques": int(nc.clique_operator.n_terms), "f": f,
               "construct_s": build, "solve_s": times, "assignments_per_s": float(2 ** f / best),
               "energy": float(nc.energy)}
        result["cases"].append(row)
        print(json.dumps(row), flush=True)
    result["numpy_direct"] = numpy_direct(20, 1 << 16)
    print(json.dumps(result["numpy_direct"]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_noncontextual.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"gpu": result["gpu"], "nvidia_smi": result["nvidia_smi"]}))


if __name__ == "__main__":
    main()
