"""Isometry-loss throughput on one GPU: fused Adam evals/s (samples x steps / time) of the isometry kernel on 6-7
qubits (chain, K = 60, complex64) for k = 2, 8, 32 input columns, beside the state-preparation rate of the same
template measured in the same run, and the 5-qubit isometry rate (the HS kernels) beside HS.

    python tools/isometry_bench.py [--samples 10000] [--steps 200] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cpflow_b200.ansatz import Ansatz  # noqa: E402
from cpflow_b200.engine import Loss, Penalty  # noqa: E402
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function  # noqa: E402
from cpflow_b200.topology import chain_layer, fill_layers  # noqa: E402


def rate(anz, loss, samples, steps, reps=3):
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.00055, pf.segments, pf.period)
    a0 = anz.program.initial_angles(0, samples)
    st = anz.program.adam_state(a0.clone())
    anz.program.adam_run(st, loss, pen, 0.1, 5)                        # warm-up (module load, scratch pool)
    best = 0.0
    for _ in range(reps):
        st = anz.program.adam_state(a0.clone())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        anz.program.adam_run(st, loss, pen, 0.1, steps)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, samples * steps / (e0.elapsed_time(e1) * 1e-3))
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=10000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [f"GPU: {smi[0] if smi else 'unknown'}  (name, power limit, max SM clock)",
             f"fused Adam, complex64, chain, K = 60, {args.samples} samples x {args.steps} steps, best of 3", ""]
    rng = np.random.default_rng(0)
    for n in (6, 7):
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        st_rate = rate(anz, Loss("state", psi / np.linalg.norm(psi)), args.samples, args.steps)
        lines.append(f"n = {n}  state preparation        {st_rate / 1e6:8.3f} M evals/s")
        for k in (2, 8, 32):
            a = n - int(np.log2(k))
            anc = list(range(a))                                          # ancillas on the most significant qubits
            W = np.linalg.qr(rng.normal(size=(2 ** n, k)) + 1j * rng.normal(size=(2 ** n, k)))[0]
            r = rate(anz, Loss("isometry", W, ancillas=anc), args.samples, args.steps)
            lines.append(f"n = {n}  isometry k = {k:2d}          {r / 1e6:8.3f} M evals/s   k x rate / state = "
                         f"{k * r / st_rate:5.2f}")
    anz = Ansatz(5, "cp", fill_layers(chain_layer(5), 60))
    V = np.linalg.qr(rng.normal(size=(32, 32)) + 1j * rng.normal(size=(32, 32)))[0]
    hs = rate(anz, Loss("hs", V), args.samples, args.steps)
    iso = rate(anz, Loss("isometry", V[:, :8], ancillas=[0, 1]), args.samples, args.steps)
    lines.append(f"n = 5  HS                       {hs / 1e6:8.3f} M evals/s")
    lines.append(f"n = 5  isometry k = 8 (HS path) {iso / 1e6:8.3f} M evals/s   ratio {iso / hs:5.3f}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
