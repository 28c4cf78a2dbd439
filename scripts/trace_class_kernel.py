"""Kernel times of the bench step (C5/8 product: 12 500 x 10 000 terms, 1000 q, PauliwordOp.__mul__) from a
torch.profiler (CUPTI) trace of warmed steps, L2 flushed before each; the class kernel is the line to watch.

    python scripts/trace_class_kernel.py OUT_DIR [STEPS] [span]

`span`: the operands of bench.py's secondary_dedup instead (both from the span of 28 generators, duplicate-heavy).

Writes OUT_DIR/class_kernel_trace.json (device ms per step and kernel, sorted; per step, the start and end of the class
kernel launches and of tile_emit_kernel relative to the step's first kernel, which shows whether they overlap) and the
chrome trace beside it. Run it on its own: tracing slows the host, so the step times of bench.py are taken without it."""
import json
import os
import sys

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
from oracle import pauli_oracle as po  # noqa: E402
from symmer_b200 import PauliwordOp, ops  # noqa: E402


def span_operator(gens, n_rows, rng):
    """bench.py's generator: n_rows random GF(2) combinations of the generator rows, random complex coefficients."""
    pick = rng.random((n_rows, gens.shape[0])) < 0.5
    symp = (pick.astype(np.uint8) @ gens.astype(np.uint8)) % 2
    return symp.astype(bool), rng.standard_normal(n_rows) + 1j * rng.standard_normal(n_rows)


def main():
    out_dir = sys.argv[1]
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    os.makedirs(out_dir, exist_ok=True)
    dev = ops.device()
    if len(sys.argv) > 3 and sys.argv[3] == "span":
        rng = np.random.default_rng(11)
        gens = rng.random((28, 2000)) < 0.3
        (a_s, a_c), (b_s, b_c) = [span_operator(gens, rows, rng) for rows in (12500, 10000)]
    else:
        a_s, a_c = po.random_operator(1000, 12500, seed=100)
        b_s, b_c = po.random_operator(1000, 10000, seed=7)
    A, B = PauliwordOp(a_s, a_c), PauliwordOp(b_s, b_c)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        R = A * B
        del R
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            flush.fill_(1)
            R = A * B
            torch.cuda.synchronize()
            del R
    trace = os.path.join(out_dir, "class_kernel.pt.trace.json")
    prof.export_chrome_trace(trace)
    events = sorted((e for e in json.load(open(trace))["traceEvents"] if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    per_kernel, timeline = {}, []
    for e in events:
        name = e["name"]
        if "fill" in name.lower() and "symb" not in name:          # the L2 flush: a step starts after it
            timeline.append({"t0": None, "kernels": []})
            continue
        per_kernel.setdefault(name, []).append(e["dur"] / 1e3)
        if timeline:
            step = timeline[-1]
            if step["t0"] is None:
                step["t0"] = e["ts"]
            if "class_dedup" in name or "tile_emit" in name:
                step["kernels"].append({"name": name.split("(")[0].replace("void symb::", ""),
                                        "start_ms": round((e["ts"] - step["t0"]) / 1e3, 4),
                                        "end_ms": round((e["ts"] + e["dur"] - step["t0"]) / 1e3, 4)})
    rows = sorted(((sum(v) / steps, len(v) / steps, k) for k, v in per_kernel.items()), reverse=True)
    result = {
        "gpu": torch.cuda.get_device_name(0), "steps": steps,
        "kernel_ms_per_step": sum(r[0] for r in rows),
        "kernels": [{"ms_per_step": ms, "launches_per_step": n, "name": k} for ms, n, k in rows],
        "class_kernel_ms": [float(np.round(d, 4)) for k, v in per_kernel.items() if "class_dedup" in k for d in v],
        "timeline": [step["kernels"] for step in timeline],
    }
    with open(os.path.join(out_dir, "class_kernel_trace.json"), "w") as f:
        json.dump(result, f, indent=1)
    for ms, n, k in rows[:8]:
        print(f"{ms:8.3f} ms  x{n:g}  {k[:110]}")
    print("class kernel per step (ms):", result["class_kernel_ms"])
    for k in result["timeline"][-1]:
        print(f"{k['start_ms']:8.3f} -> {k['end_ms']:8.3f} ms  {k['name']}")


if __name__ == "__main__":
    main()
