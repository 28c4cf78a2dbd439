#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: PauliwordOp multiply + cleanup (cross-terms/s).

    python bench.py --gpus N --steps K --warmup W            # this engine (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port)
    python bench.py --steps K --dump-outputs DIR             # also save a sample of the last timed step's result

Workload (config C5 of BASELINE.json, weak-scaled): 1000-qubit product of a 12 500*N-term operator A
(each rank holds one 12 500-row block, seeds 100+rank) with a 10 000-term operator B (seed 7),
i.e. 1.25e8 cross terms per GPU; at N = 8 this is exactly C5 (1e5 x 1e4 terms, 1e9 cross terms).
Inputs are generated on the host with the reference's own generator (PauliwordOp.random).
A step = one full product + cleanup through the public API (symmer_b200.PauliwordOp.__mul__ on one GPU,
symmer_b200.dist.sharded_product on several). Prints ONE JSON line on rank 0.

Besides the contract keys the line carries, on one GPU: `secondary_dedup` (the duplicate-heavy variant of
SURVEY.md section 8d: operands from the span of 28 generators), `e2e_host_result` (config C1 with the
result arrays landing on the host), `c5_streamed` (all of C5 on one GPU, generated in 8 hash partitions
that are consumed one after the other), `secondary` (commute-pair checks/s) and `cpu_baseline`; on every
GPU count: `check`, the verification of the timed product's output (it fails the run when it fails).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_QUBITS = 1000
ROWS_A_PER_GPU = 12500
ROWS_B = 10000
ROW_BYTES = 16 * ((N_QUBITS + 63) // 64) + 16          # R of SURVEY.md §8d: packed row + coefficient = 272 B
# bounded CPU sample (BASELINE.md §3): the first 125 rows of A against three 1000-row chunks of B, timed chunk by
# chunk (the bool tensor of a chunk is 250 MB; the full size needs 250 GB) and extrapolated per cross term
CPU_ROWS_A = 125
CPU_CHUNK_B = 1000
CPU_CHUNKS = 3
SPAN_GENERATORS = 28
C1_TERMS = 500
DUMP_TERMS = 4096                                     # --dump-outputs: 4096 sampled rows x 2000 bits as float32 = 33 MB
DUMP_SEED = 20240


def make_operator(n_terms, seed):
    from oracle import pauli_oracle as po           # only the input generator (same draws as the reference)
    return po.random_operator(N_QUBITS, n_terms, seed=seed)


def span_operator(gens, n_rows, rng):
    """n_rows random GF(2) combinations of the generator rows, random complex coefficients."""
    pick = rng.random((n_rows, gens.shape[0])) < 0.5
    symp = (pick.astype(np.uint8) @ gens.astype(np.uint8)) % 2
    return symp.astype(bool), rng.standard_normal(n_rows) + 1j * rng.standard_normal(n_rows)


def cpu_sample_inputs():
    a_s, a_c = make_operator(ROWS_A_PER_GPU, 100)
    b_s, b_c = make_operator(ROWS_B, 7)
    return a_s[:CPU_ROWS_A], a_c[:CPU_ROWS_A], b_s, b_c


def cpu_sample_text():
    return (f"per step {CPU_CHUNKS} chunks of ({CPU_ROWS_A} rows of A) x ({CPU_CHUNK_B} rows of B) of the same operators = "
            f"{CPU_CHUNKS * CPU_ROWS_A * CPU_CHUNK_B} cross terms, each chunk multiplied and cleaned on its own and the time "
            f"extrapolated linearly per cross term (BASELINE.md section 3; the full size needs a 250 GB bool tensor on the "
            f"reference's path)")


def time_cpu_reference(steps, warmup):
    """The reference's NumPy algorithm (oracle port, single core like the reference) on the bounded sample."""
    from oracle import pauli_oracle as po
    a_s, a_c, b_s, b_c = cpu_sample_inputs()
    T = CPU_CHUNKS * a_s.shape[0] * CPU_CHUNK_B

    def one_step(k):
        for ch in range(CPU_CHUNKS):
            lo = ((k * CPU_CHUNKS + ch) * CPU_CHUNK_B) % (ROWS_B - CPU_CHUNK_B + 1)
            po.multiply(a_s, a_c, b_s[lo:lo + CPU_CHUNK_B], b_c[lo:lo + CPU_CHUNK_B])

    for k in range(warmup):
        one_step(k)
    t0 = time.perf_counter()
    for k in range(steps):
        one_step(warmup + k)
    dt = (time.perf_counter() - t0) / max(1, steps)
    return T / dt, dt, T


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    value, dt, T = time_cpu_reference(steps, warmup)
    sample = cpu_sample_text()
    line = {
        "impl": "reference", "metric": "cross-terms/s (multiply+cleanup)", "value": value, "unit": "cross-terms/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64+c128", "data": "synthetic",
        "config": {"workload": "C5/8 per GPU: 1000 q, 12500x10000-term product + cleanup (bounded CPU sample, extrapolated "
                               "per cross term)",
                   "n_qubits": N_QUBITS, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "cross-terms/s", "cores": 1, "kind": "port", "sample": sample,
                         "host_cpu_count": os.cpu_count(),
                         "note": "oracle port of the reference's NumPy path (single-threaded like the reference: broadcast XOR, "
                                 "sequential first-occurrence hash loop, np.add.at); the reference itself cannot be installed "
                                 "on the GPU box (qiskit / openfermion / ray / quimb wheels absent)"},
        "e2e": {"value": value, "unit": "cross-terms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False).name
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm)}


def pinned_pair(symp, coeff):
    """Page-locked host copies of an operator's arrays, as NumPy views (what a caller would hand to PauliwordOp)."""
    import torch
    ts = torch.from_numpy(np.ascontiguousarray(symp)).pin_memory()
    tc = torch.from_numpy(np.ascontiguousarray(coeff)).pin_memory()
    return ts.numpy(), tc.numpy(), int(ts.numel() * ts.element_size() + tc.numel() * tc.element_size())


def dump_outputs(out_dir, xz, c, prefix=""):
    """Save the result operator of a timed step as its caller sees it (PauliwordOp.symp_matrix and .coeff_vec) so
    that two builds can be compared output for output. The result has 1.25e8 terms per GPU (34 GB), so the rows
    are a fixed, seeded sample of DUMP_TERMS term positions; n_terms and the coefficient sums cover all of it.
    Files: <prefix><name>.npy, float32 (0/1 Pauli bits) or float64, 33 MB in all."""
    import torch

    from symmer_b200 import ops
    n_terms = int(xz.shape[0])
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n_terms, size=min(n_terms, DUMP_TERMS), replace=False))
    sel = torch.from_numpy(idx).to(xz.device)
    symp = ops.to_host(ops.unpack(xz[sel].contiguous(), N_QUBITS))
    coeff = c[sel].cpu().numpy()
    total = complex(c.sum().item())
    arrays = {
        "n_terms": np.array([n_terms], dtype=np.float64),
        "coeff_vec_sum": np.array([total.real, total.imag, c.abs().sum().item()], dtype=np.float64),
        "term_index": idx.astype(np.float64),
        "symp_matrix": symp.astype(np.float32),
        "coeff_vec_real": coeff.real.astype(np.float64),
        "coeff_vec_imag": coeff.imag.astype(np.float64),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from symmer_b200 import PauliwordOp, ops
    from symmer_b200 import dist as sdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = ops.device()
    tuning = {}
    for kv in filter(None, os.environ.get("SYMMER_TUNING", "").split(",")):   # A/B knobs, e.g. "10=0,7=32"
        k, v = kv.split("=")
        tuning[int(k)] = int(v)
        ops.set_tuning(int(k), int(v))
    tile_mode = tuning.get(6, 1) != 0                              # ordered-tile mode (default) vs sorted-hash order
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    quick = os.environ.get("SYMMER_BENCH_QUICK") == "1"           # profiling runs (ncu): the two timed arms + check only

    # ---------------------------------------------------------------- inputs (host, reference generator)
    a_s, a_c = make_operator(ROWS_A_PER_GPU, 100 + rank)
    b_s, b_c = make_operator(ROWS_B, 7)
    a_np, ac_np, a_bytes = pinned_pair(a_s, a_c)
    b_np, bc_np, b_bytes = pinned_pair(b_s, b_c)
    h2d_bytes = a_bytes + b_bytes
    T_local = ROWS_A_PER_GPU * ROWS_B
    T_total = T_local * world
    cache = {}

    def product(A, B):
        """The public call: PauliwordOp.__mul__ on one GPU, the sharded product on several."""
        if world == 1:
            R = A * B
            return R.device_rows, R.device_coeffs, None
        return sdist.sharded_product(A.device_rows, A.device_coeffs, B.device_rows, B.device_coeffs, 1e-15,
                                     method=os.environ.get("SYMMER_DIST_METHOD", "owner"),
                                     block_sizes=[ROWS_A_PER_GPU] * world, cache=cache)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def timed(fn, n, keep_last=False):
        """n steps, each bracketed by CUDA events on the launching stream; L2 flushed between steps.
        With keep_last, returns (times, output of the last step)."""
        ms, last = [], None
        for i in range(n):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
            if keep_last and i == n - 1:
                last = out
            del out
        return (ms, last) if keep_last else ms

    # ---------------------------------------------------------------- device-resident arm (`value`)
    A_op, B_op = PauliwordOp(a_np, ac_np), PauliwordOp(b_np, bc_np)
    state = {}

    def step_resident():
        xz, c, info = product(A_op, B_op)
        state["U"] = xz.shape[0]
        return xz, c

    clocks = ClockSampler(local_rank)
    clocks.start()
    warmup = max(3, args.warmup)
    for _ in range(warmup):
        timed(step_resident, 1)
    barrier()
    ops.emit_events = []
    ops.emit_kernel_events = []
    launches0 = ops.launch_count()
    t_wall0 = time.perf_counter()
    ms_steps, last_out = timed(step_resident, args.steps, keep_last=True)
    barrier()
    wall = time.perf_counter() - t_wall0
    launches = ops.launch_count() - launches0
    emit_ms = [s.elapsed_time(e) for s, e in ops.emit_events]
    kern_ms = [s.elapsed_time(e) for s, e in ops.emit_kernel_events]
    ops.emit_events = None
    ops.emit_kernel_events = None
    step_ms = float(np.mean(ms_steps))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last_out, prefix=f"rank{rank}_" if world > 1 else "")
    del last_out

    # ---------------------------------------------------------------- end-to-end arm (`e2e`): host buffers in, result summary out
    def step_e2e():
        A, B = PauliwordOp(a_np, ac_np), PauliwordOp(b_np, bc_np)     # page-locked host arrays -> device, pack
        xz, c, _ = product(A, B)
        summary = torch.stack([torch.sum(c), torch.tensor(complex(xz.shape[0]), device=dev, dtype=torch.complex128)])
        return summary.cpu()                                        # device->host read of the step's result summary

    timed(step_e2e, 1)
    barrier()
    e2e_ms = float(np.mean(timed(step_e2e, 1 if quick else max(1, min(args.steps, 10)))))
    barrier()
    clock_info = clocks.stop()

    # ---------------------------------------------------------------- check: the product that was timed, verified on the device
    xz, c, info = product(A_op, B_op)
    U_local = int(xz.shape[0])
    chk = {"survivors_equal_cross_terms": None, "sampled_rows_equal_xor_of_operands": None, "abs_coefficient_checksum": None}
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    n_samp = 1_000_000
    if world == 1:
        a_x, a_cc, b_x, b_cc = A_op.device_rows, A_op.device_coeffs, B_op.device_rows, B_op.device_coeffs
        blocks = [(0, ROWS_A_PER_GPU, 0, ROWS_B)]
    else:
        (a_x, a_cc, _), (b_x, b_cc, _), blocks = info["a_part"], info["b_part"], info["blocks"]
        # every row this rank emitted must be owned by it (GF(2)-linear owner class of the row), so parts are disjoint
        own = ops.owner_classes(xz[:: max(1, U_local // 4_000_000)].contiguous(), sdist.log2_exact(world))
        chk["rows_owned_by_this_rank"] = bool((own == rank).all().item())
    # collision-free workload: every cross term survives, in block-major (q, p) order
    t_blocks = sum((p1 - p0) * (q1 - q0) for p0, p1, q0, q1 in blocks)
    chk["survivors_equal_cross_terms"] = U_local == t_blocks
    if chk["survivors_equal_cross_terms"]:
        ok_rows, mag_ref, off = True, 0.0, 0
        for p0, p1, q0, q1 in blocks:
            m, nq = p1 - p0, q1 - q0
            if m * nq == 0:
                continue
            ns = max(1, n_samp * m * nq // t_blocks)
            ts = torch.randint(0, m * nq, (ns,), device=dev, generator=g)
            ok_rows &= bool(torch.equal(xz[off + ts], a_x[p0 + ts % m] ^ b_x[q0 + ts // m]))
            mag_ref += float(a_cc[p0:p1].abs().sum().item()) * float(b_cc[q0:q1].abs().sum().item())
            off += m * nq
        chk["sampled_rows_equal_xor_of_operands"] = ok_rows
        mag = float(c.abs().sum().item())
        chk["abs_coefficient_checksum"] = abs(mag - mag_ref) <= 1e-9 * mag_ref
    chk_ok = all(v is True for v in chk.values())
    del xz, c, info
    if world > 1:
        t = torch.tensor([1.0 if chk_ok else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        chk_all = bool(t.item() == 1.0)
    else:
        chk_all = chk_ok
    chk["all_ranks_ok"] = chk_all
    chk["what"] = ("collision-free workload: survivors == cross terms, 1e6 sampled output rows == A[p]^B[q] at their "
                   "first-occurrence position, sum|c| == sum|a| * sum|b|" +
                   ("; sampled output rows carry this rank's owner class (parts are disjoint)" if world > 1 else ""))

    # ---------------------------------------------------------------- one-GPU extras
    extras = {}
    if world == 1 and not quick:
        del A_op, B_op
        torch.cuda.empty_cache()
        extras = one_gpu_extras(torch, ops, sdist, PauliwordOp, dev, timed, flush)

    # ---------------------------------------------------------------- max over ranks
    if world > 1:
        t = torch.tensor([step_ms, e2e_ms, float(np.mean(emit_ms)) if emit_ms else 0.0,
                          float(np.mean(kern_ms)) if kern_ms else 0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        step_ms, e2e_ms, emit_mean, kern_mean = [float(x) for x in t.cpu()]
        u = torch.tensor([state["U"]], dtype=torch.int64, device=dev)
        dist.all_reduce(u)
        U_total = int(u.item())
    else:
        emit_mean = float(np.mean(emit_ms)) if emit_ms else 0.0
        kern_mean = float(np.mean(kern_ms)) if kern_ms else 0.0
        U_total = state["U"]

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        U_local = state["U"]
        row_only = 16 * ((N_QUBITS + 63) // 64)
        # tile_emit_kernel writes row + coefficient (272 B per survivor); in the sorted-hash path emit_kernel
        # writes the 256 B row and the coefficient leaves in compact_kernel
        emit_bytes = U_local * (ROW_BYTES if tile_mode else row_only)
        achieved = emit_bytes / (kern_mean * 1e-3) / 1e9 if kern_mean > 0 else None
        phase_gbs = U_local * ROW_BYTES / (emit_mean * 1e-3) / 1e9 if emit_mean > 0 else None
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "tile_emit_traffic.json" if tile_mode else "emit_traffic.json")
        if os.path.exists(tpath):
            traffic = float(json.load(open(tpath))["dram_bytes_per_row"]) * U_local
        path_bytes = T_local * (2 * ROW_BYTES + (U_local / T_local) * ROW_BYTES)   # SURVEY §8d model: 816 B/ct at U=T
        out_bound_ms = U_local * ROW_BYTES / (peak * 1e9) * 1e3
        line = {
            "metric": "cross-terms/s (multiply+cleanup)", "value": T_total / (step_ms * 1e-3), "unit": "cross-terms/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64+c128", "data": "synthetic",
            "config": {"workload": "C5/8 per GPU: 1000 q, (12500 x n_gpus)-term A times 10000-term B, product + cleanup; "
                                   "n_gpus=8 is BASELINE config C5 (1e9 cross terms)",
                       "n_qubits": N_QUBITS, "rows_a_per_gpu": ROWS_A_PER_GPU, "rows_b": ROWS_B,
                       "cross_terms_total": T_total, "unique_terms_total": U_total,
                       "api": ("symmer_b200.PauliwordOp.__mul__" if world == 1 else
                               "symmer_b200.dist.sharded_product (device rows of PauliwordOp operands)"),
                       "parallelism": ("term-block sharded A all-gathered once; exchange-free hash partition (GF(2)-linear owner "
                                       "classes): every rank generates and dedups exactly the cross terms it owns") if world > 1 else "1 GPU",
                       "l2": "explicit 256 MB flush write between timed steps; per-step working set ~35 GB >> L2",
                       "output_materialised": True},
            "e2e": {"value": T_total / (e2e_ms * 1e-3), "unit": "cross-terms/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 32, "ms_per_step": e2e_ms,
                    "result_location": "device",
                    "note": "PauliwordOp(bool[M,2n], complex128[M]) built from page-locked host arrays every step (H2D + pack), "
                            "product + cleanup; the 34 GB result operator stays device-resident, as it does for a user of the API — "
                            "only its term count and coefficient checksum (32 B) are read back. Copying the rows back would add "
                            ">= 0.6 s of PCIe time per step; `e2e_host_result` is the end-to-end number with the result arrays on the host."},
            "gpu_launches": int(launches),
            "clocks": clock_info,
            "roofline": {"bound": "hbm", "kernel": ("tile_emit_kernel (rows + coefficients of the survivors in cross-term order: "
                                                    "272 B per survivor, one launch per block)") if tile_mode else
                                                   "emit_kernel (row emission of the survivors: 256 B per row, one launch per step)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                         "kernel_ms": kern_mean, "kernel_share_of_step": kern_mean / step_ms if step_ms else None,
                         "emit_phase_ms": emit_mean, "emit_phase_gbs": phase_gbs,
                         "emit_phase_note": ("tile_emit_kernel + fix-up of group sums" if tile_mode else
                                             "compact_kernel + emit_kernel") + ": 272 B (row + coefficient) per survivor",
                         "tuning": tuning,
                         "step_output_write_bound_ms": out_bound_ms,
                         "step_frac_of_output_write_bound": out_bound_ms / step_ms if step_ms else None,
                         "step_note": "whole step against the irreducible HBM write of its output (survivors x 272 B at the measured "
                                      "peak); the rest of the step is the class-local duplicate detection, which reads two L2-resident "
                                      "sketch tables and writes nothing per unique row",
                         "path_model_bytes_per_step": path_bytes,
                         "path_achieved_gbs": path_bytes / (step_ms * 1e-3) / 1e9,
                         "path_frac": path_bytes / (step_ms * 1e-3) / 1e9 / peak,
                         "path_note": "SURVEY section 8d model (816 B per cross term: write, re-read, write survivors) for an "
                                      "implementation that never materialises the cross terms: not a utilisation figure"},
            "cpu_baseline": extras.get("cpu_baseline"),
            "check": chk,
            "secondary_dedup": extras.get("secondary_dedup"),
            "e2e_host_result": extras.get("e2e_host_result"),
            "c5_streamed": extras.get("c5_streamed"),
            "secondary": extras.get("commute"),
            "wall_s_timed_region": wall,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not chk_all:
        raise SystemExit("bench.py: the output check failed: " + json.dumps(chk))


def one_gpu_extras(torch, ops, sdist, PauliwordOp, dev, timed, flush):
    from oracle import pauli_oracle as po
    out = {}
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0

    # ---- secondary_dedup: the duplicate-heavy product of SURVEY §8d (operands from the span of 28 generators)
    rng = np.random.default_rng(11)
    gens = rng.random((SPAN_GENERATORS, 2 * N_QUBITS)) < 0.3
    sa_s, sa_c = span_operator(gens, ROWS_A_PER_GPU, rng)
    sb_s, sb_c = span_operator(gens, ROWS_B, rng)
    SA, SB = PauliwordOp(sa_s, sa_c), PauliwordOp(sb_s, sb_c)
    st = {}

    def step_span():
        R = SA * SB
        st["U"] = R.n_terms
        return R

    timed(step_span, 2)
    ms = float(np.mean(timed(step_span, 5)))
    T = ROWS_A_PER_GPU * ROWS_B
    U = st["U"]
    model = T * (2 * ROW_BYTES + (U / T) * ROW_BYTES)
    # every output row must be a distinct row: the GF(2)-linear sketches of the output, sorted, have no equal neighbours
    # unless two different rows share a sketch (probability ~ U^2 / 2^65)
    R = SA * SB
    sk, _ = ops.sort_pairs(ops.sketch(R.device_rows), torch.zeros(R.n_terms, dtype=torch.int32, device=dev))
    distinct = bool((sk[1:] != sk[:-1]).all().item())
    del R, sk
    out["secondary_dedup"] = {
        "metric": "cross-terms/s (multiply+cleanup), duplicate-heavy operands", "value": T / (ms * 1e-3), "unit": "cross-terms/s",
        "ms_per_step": ms, "cross_terms": T, "unique_terms": U,
        "workload": f"1000 q, {ROWS_A_PER_GPU} x {ROWS_B} terms drawn from the span of {SPAN_GENERATORS} generators (SURVEY section 8d "
                    f"high-collision variant): {T - U} cross terms are merged into earlier ones (np.add.at order)",
        "model_bytes_per_step": model, "model_gbs": model / (ms * 1e-3) / 1e9, "model_frac_of_hbm_peak": model / (ms * 1e-3) / 1e9 / peak,
        "output_write_bound_ms": U * ROW_BYTES / (peak * 1e9) * 1e3,
        "output_rows_distinct": distinct,
        "kernels": "class_dedup_kernel (candidates grouped in shared memory), group_kernel (exact row compare, phases, sums: "
                   "512 B of operand rows per candidate, from L2), tile_emit_kernel",
        "parity": "tests/test_gpu_class_dedup.py::test_span_operands_high_collision (oracle, reduced size, -m gpu)"}
    del SA, SB
    torch.cuda.empty_cache()

    # ---- e2e_host_result: config C1 (square of a 1000-qubit, 500-term operator) with the result arrays on the host
    p_s, p_c = make_operator(C1_TERMS, 1)
    t_cpu0 = time.perf_counter()
    ref_s, ref_c = po.multiply(p_s, p_c, p_s, p_c)
    cpu_c1 = time.perf_counter() - t_cpu0
    reps, lat = 20, []
    S = None
    for it in range(reps + 3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P = PauliwordOp(p_s, p_c)
        S = P * P
        s_host, c_host = S.symp_matrix, S.coeff_vec          # device -> host: the reference's result arrays
        dt = time.perf_counter() - t0
        if it >= 3:
            lat.append(dt)
    ok, why = po.compare_term_sets(s_host, c_host, ref_s, ref_c, scale=float(np.abs(p_c).max() ** 2))
    c1_T = C1_TERMS * C1_TERMS
    c1_ms = float(np.median(lat)) * 1e3
    out["e2e_host_result"] = {
        "metric": "cross-terms/s (multiply+cleanup), host arrays in, host arrays out", "value": c1_T / (c1_ms * 1e-3),
        "unit": "cross-terms/s", "ms_per_step": c1_ms,
        "workload": "config C1 (README laptop benchmark): P = PauliwordOp.random(1000, 500), P * P = 250000 cross terms + cleanup",
        "api": "P = PauliwordOp(symp_matrix, coeff_vec); S = P * P; S.symp_matrix, S.coeff_vec",
        "h2d_bytes_per_step": int(p_s.size + p_c.size * 16), "d2h_bytes_per_step": int(s_host.size + c_host.size * 16),
        "survivors": int(len(c_host)), "parity_vs_oracle": "ok" if ok else why,
        "cpu_baseline": {"value": c1_T / cpu_c1, "unit": "cross-terms/s", "cores": 1, "kind": "port", "seconds": cpu_c1,
                         "sample": "the whole of config C1, one pass"}}
    assert ok, why
    del S, P

    # ---- c5_streamed: ALL of config C5 (1e5 x 1e4 terms, 1e9 cross terms, 272 GB of output) on one GPU, generated in 8 hash
    # partitions that are consumed one after the other (never resident as a whole)
    blocks = [make_operator(ROWS_A_PER_GPU, 100 + r) for r in range(8)]
    A = PauliwordOp(np.vstack([b[0] for b in blocks]), np.hstack([b[1] for b in blocks]))
    b_s, b_c = make_operator(ROWS_B, 7)
    B = PauliwordOp(b_s, b_c)
    del blocks

    def consumer(part, xz, c):
        return torch.stack([torch.sum(c), torch.tensor(complex(xz.shape[0]), device=dev, dtype=torch.complex128)])

    def step_stream():
        parts = sdist.streamed_product(A.device_rows, A.device_coeffs, B.device_rows, B.device_coeffs, 3, consumer)
        return torch.stack(parts).cpu()

    timed(step_stream, 1)
    ms_stream = timed(step_stream, 3)
    res = step_stream()
    n_terms = int(sum(complex(x).real for x in res[:, 1]))
    T5 = 8 * ROWS_A_PER_GPU * ROWS_B
    out["c5_streamed"] = {
        "metric": "cross-terms/s (multiply+cleanup)", "value": T5 / (float(np.mean(ms_stream)) * 1e-3), "unit": "cross-terms/s",
        "ms_per_pass": float(np.mean(ms_stream)), "cross_terms": T5, "unique_terms": n_terms, "n_gpus": 1, "scaling": "strong (all of C5)",
        "api": "symmer_b200.dist.streamed_product(A, B, log2_parts=3, consumer)",
        "note": "BASELINE config C5 itself on ONE GPU: the 272 GB result never exists as a whole; it is produced in 8 hash partitions "
                "(GF(2)-linear owner classes, so every partition is final when it is handed over) of 34 GB each, each consumed on the "
                "device (term count + coefficient checksum, 32 B per partition read back) and dropped"}
    assert n_terms == T5, (n_terms, T5)
    del A, B
    ops.release_workspace()
    torch.cuda.empty_cache()

    # ---- secondary metric of BASELINE.json: commute-pair checks/s
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)
    W2 = 2 * ((N_QUBITS + 63) // 64)
    big = torch.randint(-2 ** 63, 2 ** 63 - 1, (65536, W2), dtype=torch.int64, device=dev, generator=gen)
    blk = big[:16384].contiguous()
    ops.commute(blk, big)
    torch.cuda.synchronize()
    cms = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        adj = ops.commute(blk, big)
        e1.record()
        torch.cuda.synchronize()
        cms.append(e0.elapsed_time(e1))
        del adj
    pairs = 16384 * 65536
    del big, blk
    out["commute"] = {"metric": "commute-pair checks/s", "value": pairs / (min(cms) * 1e-3), "unit": "pairs/s",
                      "workload": "16384 x 65536 block of a 1024-bit-wide (1000-qubit layout) adjacency matrix, random rows",
                      "kernel": "commute_mma_ws_kernel (tcgen05 kind::i8, TMEM accumulators, warp-specialised expander / issuer warps)",
                      "int8_tops": pairs * 2 * 2048 / (min(cms) * 1e-3) / 1e12,
                      "note": "K = 2048 unpacked bits per pair; nominal dense int8 peak 4500 TOP/s"}

    # ---- cpu_baseline: the reference's algorithm on this box's host cores, bounded sample of the same workload
    cpu_value, cpu_dt, cpu_T = time_cpu_reference(steps=3, warmup=1)
    out["cpu_baseline"] = {"value": cpu_value, "unit": "cross-terms/s", "cores": 1, "kind": "port", "host_cpu_count": os.cpu_count(),
                           "sample": cpu_sample_text() + f"; {cpu_dt:.2f} s per step, NumPy single core like the reference"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--check", action="store_true", help="(always on) verify the timed product's output; the run fails if it does not hold")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of the last timed step's result to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the result of this engine's timed product; the reference arm has none")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)      # fail before any GPU work if DIR cannot be created
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
