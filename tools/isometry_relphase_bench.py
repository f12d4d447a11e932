"""Relative-phase isometry throughput on one GPU: fused Adam evals/s (samples x steps / time) of the relative-phase
isometry kernel (chain, K = 60, complex64)
  - on 6, 7 and 8 qubits for k = 2, 8 and 32 input columns, beside the isometry kind with the same ancilla mask;
  - on 3, 4 and 5 qubits with no ancillas and a permutation target, beside the relphase kind (full-unitary
    state-adjoint kernel) on the same template.
The two kinds of a row are timed alternately, best of 3 each.

    python tools/isometry_relphase_bench.py [--samples 10000] [--steps 200] [--out FILE]
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


def rates(anz, losses, samples, steps, reps=3):
    """best evals/s of each loss, the losses timed in turn within each repetition"""
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.00055, pf.segments, pf.period)
    a0 = anz.program.initial_angles(0, samples)
    for loss in losses:                                                  # warm-up (module load, scratch pool)
        anz.program.adam_run(anz.program.adam_state(a0.clone()), loss, pen, 0.1, 5)
    best = [0.0] * len(losses)
    for _ in range(reps):
        for i, loss in enumerate(losses):
            st = anz.program.adam_state(a0.clone())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            anz.program.adam_run(st, loss, pen, 0.1, steps)
            e1.record()
            torch.cuda.synchronize()
            best[i] = max(best[i], samples * steps / (e0.elapsed_time(e1) * 1e-3))
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
    for n in (6, 7, 8):
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        for k in (2, 8, 32):
            anc = list(range(n - int(np.log2(k))))                       # ancillas on the most significant qubits
            W = np.linalg.qr(rng.normal(size=(2 ** n, k)) + 1j * rng.normal(size=(2 ** n, k)))[0]
            rel, iso = rates(anz, [Loss("isometry_relphase", W, ancillas=anc), Loss("isometry", W, ancillas=anc)],
                             args.samples, args.steps)
            lines.append(f"n = {n}  k = {k:2d}  isometry_relphase {rel / 1e6:8.3f} M evals/s   isometry "
                         f"{iso / 1e6:8.3f} M evals/s   ratio {rel / iso:5.3f}")
    for n in (3, 4, 5):
        N = 2 ** n
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        V = np.zeros((N, N), complex)
        V[rng.permutation(N), np.arange(N)] = 1
        rel, rp = rates(anz, [Loss("isometry_relphase", V, ancillas=[]), Loss("relphase", V)], args.samples,
                        args.steps)
        lines.append(f"n = {n}  k = {N:2d}  isometry_relphase {rel / 1e6:8.3f} M evals/s   relphase "
                     f"{rp / 1e6:8.3f} M evals/s   ratio {rel / rp:5.3f}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
