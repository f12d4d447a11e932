"""Measured parity maxima of the CUDA engine against the CPU oracle (run on the GPU box):

    python tools/parity_report.py > profiles/parity_r2.txt
    python tools/parity_report.py --steps > profiles/adam_steps_r2.txt

Same measurement functions as tests/test_gpu_parity.py (tests/parity_lib.py); the tests assert the contract's
tolerances (1e-5 complex64, 1e-12 complex128), this prints what was actually measured per configuration."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import parity_lib as P  # noqa: E402
from cpflow_b200.gates import u_toff4  # noqa: E402
from cpflow_b200.topology import chain_layer  # noqa: E402


def main():
    print("# loss / reg: max |x - oracle| / max |oracle| over 37 samples; grad: max over samples of |g - g_o| / |g_o|")
    print(f"# device: {torch.cuda.get_device_name(0)}")
    print(f"{'config':44s} {'dtype':5s} {'kind':8s} {'engine':6s} {'loss':>9s} {'reg':>9s} {'grad':>9s} {'unitary':>9s}")
    worst = {torch.float32: 0.0, torch.float64: 0.0}
    for n, layer, K, rg in P.CONFIGS:
        for dt in (torch.float32, torch.float64):
            m = P.measure_loss_grad(n, layer, K, rg, dt)
            anz, _, _ = P.setup(n, layer, K, rg)
            for kind in ("hs", "relphase", "state"):
                e = m[kind]
                eng = anz.program.launch_plan(37, loss_kind={"hs": 0, "state": 1, "relphase": 2}[kind], dtype=dt)["engine"]
                name = f"n={n} K={K} {rg} {layer}"
                print(f"{name[:44]:44s} {'c64' if dt == torch.float32 else 'c128':5s} {kind:8s} "
                      f"{'heis' if eng == 1 else 'adj':6s} {e['loss']:9.2e} {e['reg']:9.2e} {e['grad']:9.2e} {m['unitary']:9.2e}")
                worst[dt] = max(worst[dt], e["loss"], e["reg"], e["grad"])
    print(f"# worst complex64: {worst[torch.float32]:.3e} (contract 1e-5)   worst complex128: {worst[torch.float64]:.3e} (contract 1e-12)")
    print("#\n# fused Adam loop vs the oracle loop, C3 shape (n=4, K=40, 32 samples, complex128, T=150): max abs errors")
    for lname, layer in (("chain", chain_layer(4)), ("star", P.STAR4)):
        for freeze in (False, True):
            m = P.measure_adam_loop(4, layer, 40, u_toff4, B=32, T=150, freeze=freeze)
            print(f"{lname:6s} freeze={int(freeze)} " + " ".join(f"{k}={v:.2e}" if isinstance(v, float) else f"{k}={v}"
                                                                 for k, v in m.items()))
    m = P.measure_adam_loop(4, chain_layer(4), 40, u_toff4, B=32, T=10, dt=torch.float32)
    print("chain  complex64 T=10 " + " ".join(f"{k}={v:.2e}" if isinstance(v, float) else f"{k}={v}" for k, v in m.items()))


def steps():
    """Per-step maxima of tests/test_gpu_adam_steps.py: for every case and checkpoint k the largest error over the
    samples and its ratio to the bound the test asserts (<= 1 passes; parity_lib.measure_adam_steps)."""
    import subprocess
    from cpflow_b200 import _lib
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,driver_version,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# device: {torch.cuda.get_device_name(0)}; nvidia-smi: {smi}")
    print(f"# torch {torch.__version__} (CUDA {torch.version.cuda}); library {os.path.relpath(_lib.LIB_PATH, ROOT)}, cpf_version "
          f"{_lib.load().cpf_version()}")
    print("# m, v: max over samples of the norm-wise error; theta: max entry error; loss: max |regloss / reg - oracle|;"
          " *_r: ratio to the asserted bound")
    import test_gpu_adam_steps as S
    for name, dt in S.CASES:
        got = P.measure_adam_steps(name, dt)
        print(f"{name} {'c64' if dt == torch.float32 else 'c128'}: engine={got['engine']} "
              f"words={got['words_per_sample']} chain_identical={got['chain_identical']} "
              f"f32_breakpoint_entries={got['breakpoint_fixes']}")
        for r in got["rows"]:
            print(f"  k={r['k']:5d} m={r['m']:9.2e} m_r={r['m_ratio']:7.3f} v={r['v']:9.2e} v_r={r['v_ratio']:7.3f} "
                  f"theta={r['theta']:9.2e} theta_r={r['theta_ratio']:7.3f} loss={r['loss']:9.2e} "
                  f"loss_r={r['loss_ratio']:7.3f} improved={r['improved']:3d} best_ok={int(r['best_ok'])} "
                  f"frozen_ok={int(r['frozen_unchanged'])}")


if __name__ == "__main__":
    steps() if "--steps" in sys.argv[1:] else main()
