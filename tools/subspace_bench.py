"""Subspace-loss throughput on one GPU: fused Adam evals/s (samples x steps / time), chain, K = 60, complex64.
  - On 6, 7 and 8 qubits with k = 2, 4, 8 and 32 Haar-random input states: 'subspace' beside 'isometry', and
    'subspace_relphase' beside 'isometry_relphase', with the same k (the isometry kinds' ancillas are the first
    n - log2 k qubits); then the same 'subspace' objective as a torch callable on the host-driven loop (TorchLoss),
    in sample-steps/s.
  - On 3, 4 and 5 qubits with k = 4: 'subspace' (the HS kernels on V = (N/k) B A^dag) beside 'hs' on the same
    template, and 'subspace_relphase' beside 'isometry_relphase'.
The fused kinds of a row are timed alternately, best of 3 each.

    python tools/subspace_bench.py [--samples 10000] [--steps 200] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from isometry_relphase_bench import rates  # noqa: E402
from cpflow_b200.ansatz import Ansatz  # noqa: E402
from cpflow_b200.engine import Loss, Penalty, TorchLoss  # noqa: E402
from cpflow_b200.optimization import run_adam_batch, torch_loss_chunk  # noqa: E402
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function  # noqa: E402
from cpflow_b200.topology import chain_layer, fill_layers  # noqa: E402

# host-loop samples per n (U [B,N,N] complex64 at 128-256 MiB, as tools/callable_loss_bench.py) and timed steps
TORCH_SAMPLES = {6: 4096, 7: 2048, 8: 256}
TORCH_STEPS = 10


def haar(N, k, rng):
    return np.linalg.qr(rng.normal(size=(N, k)) + 1j * rng.normal(size=(N, k)))[0]


def subspace_callable(A, B):
    k = A.shape[1]
    return lambda u: 1 - torch.abs((B.conj() * (u @ A)).sum()) ** 2 / k ** 2


def torch_rate(anz, A, B, samples, steps):
    """best sample-steps/s of the host-driven loop on the 'subspace' objective written as a torch function"""
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.00055, pf.segments, pf.period)
    At = torch.as_tensor(A).to("cuda", torch.complex64)
    Bt = torch.as_tensor(B).to("cuda", torch.complex64)
    loss = TorchLoss(subspace_callable(At, Bt))
    prog = anz.program
    a0 = prog.initial_angles(0, samples)
    chunk = torch_loss_chunk(prog, torch.float32)
    run_adam_batch(prog, loss, pen, a0, 0.1, 2, chunk=chunk)             # warm-up (modules, vmap, scratch pool)
    best = 0.0
    for _ in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_adam_batch(prog, loss, pen, a0, 0.1, steps, chunk=chunk)
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
    if not torch.cuda.is_available():
        raise SystemExit("subspace_bench.py measures on a GPU and found none")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [f"GPU: {smi[0] if smi else 'unknown'}  (name, power limit, max SM clock)",
             f"fused Adam, complex64, chain, K = 60, {args.samples} samples x {args.steps} steps, best of 3 (M evals/s);",
             f"host loop (TorchLoss, same objective as 'subspace'): {TORCH_STEPS} steps, best of 2 (M sample-steps/s)",
             ""]
    rng = np.random.default_rng(0)
    for n in (6, 7, 8):
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        for k in (2, 4, 8, 32):
            A, B = haar(2 ** n, k, rng), haar(2 ** n, k, rng)
            anc = list(range(n - int(np.log2(k))))
            sub, iso, subr, isor = rates(anz, [Loss("subspace", B, inputs=A), Loss("isometry", B, ancillas=anc),
                                               Loss("subspace_relphase", B, inputs=A),
                                               Loss("isometry_relphase", B, ancillas=anc)], args.samples, args.steps)
            tl = torch_rate(anz, A, B, TORCH_SAMPLES[n], TORCH_STEPS)
            lines.append(f"n = {n}  k = {k:2d}  subspace {sub / 1e6:7.3f}  isometry {iso / 1e6:7.3f}  ratio "
                         f"{sub / iso:5.3f}   subspace_relphase {subr / 1e6:7.3f}  isometry_relphase {isor / 1e6:7.3f}"
                         f"  ratio {subr / isor:5.3f}   TorchLoss {tl / 1e6:7.4f}  subspace / TorchLoss "
                         f"{sub / tl:6.1f}")
            print(lines[-1], flush=True)
    for n in (3, 4, 5):
        k = 4
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        A, B = haar(2 ** n, k, rng), haar(2 ** n, k, rng)
        V = haar(2 ** n, 2 ** n, rng)
        anc = list(range(n - 2))
        sub, hs, subr, isor = rates(anz, [Loss("subspace", B, inputs=A), Loss("hs", V),
                                          Loss("subspace_relphase", B, inputs=A),
                                          Loss("isometry_relphase", B, ancillas=anc)], args.samples, args.steps)
        lines.append(f"n = {n}  k = {k:2d}  subspace {sub / 1e6:7.3f}  hs       {hs / 1e6:7.3f}  ratio {sub / hs:5.3f}"
                     f"   subspace_relphase {subr / 1e6:7.3f}  isometry_relphase {isor / 1e6:7.3f}  ratio "
                     f"{subr / isor:5.3f}")
        print(lines[-1], flush=True)
    text = "\n".join(lines)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
