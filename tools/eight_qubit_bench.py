"""8-qubit throughput on one GPU: fused Adam evals/s (samples x steps / time) of state preparation on the 7- and
8-qubit chain templates (K = 60, complex64), and of the isometry kernel on 8 qubits for k = 2, 8, 32 input columns
on the same 8-qubit template.

    python tools/eight_qubit_bench.py [--samples 10000] [--steps 200] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from isometry_bench import rate  # noqa: E402
from cpflow_b200.ansatz import Ansatz  # noqa: E402
from cpflow_b200.engine import Loss  # noqa: E402
from cpflow_b200.topology import chain_layer, fill_layers  # noqa: E402


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
    st_rate = {}
    for n in (7, 8):
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 60))
        psi = rng.normal(size=2 ** n) + 1j * rng.normal(size=2 ** n)
        st_rate[n] = rate(anz, Loss("state", psi / np.linalg.norm(psi)), args.samples, args.steps)
        lines.append(f"n = {n}  state preparation        {st_rate[n] / 1e6:8.3f} M evals/s")
    lines.append(f"        n = 8 / n = 7 state rate  {st_rate[8] / st_rate[7]:8.3f}")
    for k in (2, 8, 32):
        anc = list(range(8 - int(np.log2(k))))                             # ancillas on the most significant qubits
        W = np.linalg.qr(rng.normal(size=(256, k)) + 1j * rng.normal(size=(256, k)))[0]
        r = rate(anz, Loss("isometry", W, ancillas=anc), args.samples, args.steps)
        lines.append(f"n = 8  isometry k = {k:2d}          {r / 1e6:8.3f} M evals/s   k x rate / state = "
                     f"{k * r / st_rate[8]:5.2f}")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
