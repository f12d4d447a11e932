"""Callable (TorchLoss) losses on 6-8 qubits on one GPU: the host-driven Adam loop with an HS callable against a
Haar-random target (chain template, K = 60, complex64).  Per n it prints

  - host-loop Adam steps/s and sample-steps/s (`run_adam_batch`, end to end, best of 3);
  - the split of one step between cpf_unitary, the torch value and autograd cotangent, cpf_adjoint_from_cotangent
    and cpf_adam_step (CUDA events around each stage of the same loop, averaged over the timed steps);
  - the adjoint's rate in column evaluations/s (samples x N / adjoint time), beside the fused state-preparation rate
    of the same template (one column's forward and backward sweep per evaluation), and their ratio.

    python tools/callable_loss_bench.py [--steps 50] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import torch
from scipy.stats import unitary_group

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from isometry_bench import rate  # noqa: E402
from cpflow_b200.ansatz import Ansatz  # noqa: E402
from cpflow_b200.engine import Loss, Penalty, TorchLoss  # noqa: E402
from cpflow_b200.optimization import run_adam_batch  # noqa: E402
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function  # noqa: E402
from cpflow_b200.topology import chain_layer, fill_layers  # noqa: E402

# samples per n: a multi-start batch of the size static() runs, with U [B,N,N] complex64 at 128-256 MiB
SAMPLES = {6: 4096, 7: 2048, 8: 256}


def hs_callable(V):
    N = V.shape[0]
    return lambda u: 1 - torch.abs((u * V.conj()).sum()) ** 2 / N ** 2


def split(prog, loss, pen, a0, steps):
    """Mean ms per step of each stage of run_adam_batch's TorchLoss loop, from CUDA events."""
    st = prog.adam_state(a0.clone())
    names = ["cpf_unitary", "torch value + cotangent", "cpf_adjoint_from_cotangent", "cpf_adam_step"]
    tot = [0.0] * 4
    for it in range(steps + 2):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        U = prog.unitary(st.angles)
        ev[1].record()
        values, cot = loss.value_and_cotangent(U)
        ev[2].record()
        grad = prog.adjoint_from_cotangent(st.angles, cot)
        ev[3].record()
        prog.adam_step(st, values.to(st.angles.dtype).contiguous(), grad, pen, 0.1)
        ev[4].record()
        torch.cuda.synchronize()
        if it >= 2:                                                       # two warm-up steps
            for i in range(4):
                tot[i] += ev[i].elapsed_time(ev[i + 1])
    return dict(zip(names, [t / steps for t in tot]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("callable_loss_bench.py measures on a GPU and found none")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = [f"GPU: {smi[0] if smi else 'unknown'}  (name, power limit, max SM clock)",
             f"TorchLoss HS callable vs a Haar-random target, complex64, chain, K = 60, {args.steps} timed steps", ""]
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.00055, pf.segments, pf.period)
    for n in (6, 7, 8):
        B, N = SAMPLES[n], 2 ** n
        first = len(lines)
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        prog = anz.program
        V = torch.as_tensor(unitary_group.rvs(N, random_state=n)).to("cuda", torch.complex64)
        loss = TorchLoss(hs_callable(V))
        a0 = prog.initial_angles(0, B)
        run_adam_batch(prog, loss, pen, a0, 0.1, 3)                      # warm-up (modules, vmap, scratch pool)
        best = float("inf")
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_adam_batch(prog, loss, pen, a0, 0.1, args.steps)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) * 1e-3)
        sp = split(prog, loss, pen, a0, args.steps)
        psi = V[:, 0].cpu().numpy()
        st_rate = rate(anz, Loss("state", psi), 10000, 200)
        adj_rate = B * N / (sp["cpf_adjoint_from_cotangent"] * 1e-3)
        lines.append(f"n = {n}  B = {B}  P = {prog.n_params}")
        lines.append(f"  host loop            {args.steps / best:9.1f} steps/s   {B * args.steps / best / 1e3:9.1f} k "
                     f"sample-steps/s")
        step_ms = sum(sp.values())
        for k, v in sp.items():
            lines.append(f"  {k:28s} {v:8.3f} ms/step  ({100 * v / step_ms:5.1f} %)")
        lines.append(f"  adjoint              {adj_rate / 1e6:9.3f} M column evals/s")
        lines.append(f"  fused state prep     {st_rate / 1e6:9.3f} M evals/s (10000 samples x 200 steps)   "
                     f"adjoint / state = {adj_rate / st_rate:5.3f}; one sample's adjoint = "
                     f"{st_rate / (adj_rate / N):6.1f} state evaluations")
        lines.append("")
        print("\n".join(lines[first:]), flush=True)
    text = "\n".join(lines)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
