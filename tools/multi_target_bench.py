"""Throughput of multi-target runs against single-target runs on the same program and total batch.

    python tools/multi_target_bench.py [--out FILE] [--steps 200] [--quick]

1. Fused Adam loop, evals/s (samples x Adam steps per second, CUDA events around whole cpf_adam_run calls after a
   warm-up of every shape): cpf_adam_run_multi with the batch spread over many targets, against cpf_adam_run on one
   target with the runtime-pair Heisenberg kernel (CPF_HEIS_ANY=1, the kernel family the multi-target path uses) and
   with the compile-time-layer kernel the single-target path picks by default.  Shapes: the C3 template (4q chain,
   K = 40, 10^5 samples over 256 targets) and a 3-qubit one (3q chain, K = 12, 10^5 samples over 256 targets).
2. synthesize_many on 64 three-qubit Haar-random targets x 1000 samples, wall time against a loop of 64
   Synthesize.static() calls with the same options (host clock around work that ends in a device synchronise).

Prints one JSON object (and writes it to --out) with the card name and power limit read in the same run.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy.stats import unitary_group  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the numbers are still measured; say that the card could not be read
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def adam_rate(anz, targets, B, steps, mode, reps=3):
    """evals/s of one configuration; mode 'multi' | 'any' (single target, runtime-pair kernel) | 'default'."""
    from cpflow_b200.engine import Loss, MultiLoss, Penalty
    from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.001476, pf.segments, pf.period)
    init = anz.program.initial_angles(0, B)
    idx = np.arange(B) % len(targets)
    ml, one = MultiLoss("hs", targets), Loss("hs", targets[0])
    if mode == "any":
        os.environ["CPF_HEIS_ANY"] = "1"
    try:
        def run(n):
            st = anz.program.adam_state(init.clone())
            if mode == "multi":
                anz.program.adam_run_multi(st, ml, idx, pen, 0.1, n)
            else:
                anz.program.adam_run(st, one, pen, 0.1, n)
            return st
        run(steps)                                           # warm-up: module load, pool growth, this shape
        torch.cuda.synchronize()
        times = []
        for _ in range(reps):
            st = anz.program.adam_state(init.clone())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if mode == "multi":
                anz.program.adam_run_multi(st, ml, idx, pen, 0.1, steps)
            else:
                anz.program.adam_run(st, one, pen, 0.1, steps)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
    finally:
        os.environ.pop("CPF_HEIS_ANY", None)
    return {"evals_per_s": B * steps / min(times), "spread": (max(times) - min(times)) / min(times)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--quick", action="store_true", help="small sizes (a run-through, not a measurement)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "multi_target_bench needs a CUDA device"
    import cpflow_b200 as cp
    from cpflow_b200 import ansatz as A
    from cpflow_b200.gates import u_toff4
    from cpflow_b200.topology import chain_layer, fill_layers
    B = 2000 if a.quick else 100000
    res = {"card": card(), "steps": a.steps, "adam": {}}
    for name, n, K in (("4q chain K=40", 4, 40), ("3q chain K=12", 3, 12)):
        anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), K), "xyz")
        tg = np.stack([u_toff4 if n == 4 else np.eye(8)] + [unitary_group.rvs(2 ** n, random_state=s)
                                                             for s in range(255)])
        row = {"batch": B, "targets": 256}
        for mode in ("multi", "any", "default"):
            row[mode] = adam_rate(anz, tg, B, a.steps, mode)
        row["multi_over_any"] = row["multi"]["evals_per_s"] / row["any"]["evals_per_s"]
        row["multi_over_default"] = row["multi"]["evals_per_s"] / row["default"]["evals_per_s"]
        res["adam"][name] = row
        print(name, json.dumps(row), flush=True)

    T, S = (4, 100) if a.quick else (64, 1000)
    targets = np.stack([unitary_group.rvs(8, random_state=1000 + t) for t in range(T)])
    opts = cp.StaticOptions(num_cp_gates=12, accepted_num_cz_gates=20, num_samples=S)
    layer = chain_layer(3)
    with contextlib.redirect_stdout(io.StringIO()):
        cp.synthesize_many(layer, targets[:2], cp.StaticOptions(num_cp_gates=12, accepted_num_cz_gates=20,
                                                                num_samples=50))   # warm-up
        cp.Synthesize(layer, target_unitary=targets[0]).static(
            cp.StaticOptions(num_cp_gates=12, accepted_num_cz_gates=20, num_samples=50), save_results=False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        many = cp.synthesize_many(layer, targets, opts)
        torch.cuda.synchronize()
        t_many = time.perf_counter() - t0
        t0 = time.perf_counter()
        loop = [cp.Synthesize(layer, target_unitary=targets[t]).static(opts, save_results=False) for t in range(T)]
        torch.cuda.synchronize()
        t_loop = time.perf_counter() - t0
    res["synthesize"] = {"targets": T, "samples": S, "options": "3q chain, K=12, accepted_num_cz_gates=20, defaults",
                         "synthesize_many_s": t_many, "static_loop_s": t_loop, "speedup": t_loop / t_many,
                         "decompositions_many": sum(len(r.decompositions) for r in many),
                         "decompositions_loop": sum(len(r.decompositions) for r in loop)}
    print(json.dumps(res["synthesize"]), flush=True)
    out = json.dumps(res, indent=1)
    print(out)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
