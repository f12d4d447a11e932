"""One-step consistency of the fused Adam loop (cpf_adam_run, cpf_adam_run_multi) along 2000-step runs, on every kernel
path the loop dispatches to: at checkpoints k the state the kernel hands from step k to step k + 1 (angles, moments,
best parameters and losses) is checked against the float64 oracle's gradient at the kernel's own theta_k and optax's
update (tests/parity_lib.py: measure_adam_steps, which states the bounds and their derivation).  The checkpointed chain
of launches must be bit-identical to one uninterrupted launch, so the checked steps are steps of the real run.

Inputs cover the threefry batch of static(), CP angles over [-3 pi, 5 pi) (every branch of the penalty's modulus), the
penalty's breakpoints and, on the packed float path, angles beyond the fast sin / cos reduction.  Measured maxima:
tools/parity_report.py --steps (profiles/adam_steps_r1.txt)."""
import numpy as np
import pytest
import torch

import parity_lib as P

pytestmark = pytest.mark.gpu

F32, F64 = torch.float32, torch.float64
CASES = [("heis_chain4", F32), ("heis_chain4", F64), ("heis_chain4_freeze", F32), ("heis_any_kite4", F32),
         ("heis_any_mt_chain3", F32), ("heis_any_mt_chain3", F64), ("layer_relphase_chain4", F32),
         ("layer_state_chain5", F32), ("interp_state_chain6", F32), ("interp_mt_state_chain4", F32),
         ("interp_mt_state_chain4", F64), ("interp_mt_state_chain6", F32), ("interp_mt_state_chain6", F64),
         ("interp_mt_relphase_chain4", F32), ("interp_mt_relphase_chain4", F64)]
# launch_plan's words_per_sample of the 4q chain, K = 40 on the compile-time layer; the runtime-pair kernel
# (HeisSweepAny) stages one more layer of rows and needs 860
HEIS_CHAIN4_WORDS, HEIS_ANY_CHAIN4_WORDS = 844, 860


def _check_path(name, dt, got):
    """What launch_plan can show of the path a case ran on (measure_adam_steps clears inherited dispatch switches and
    sets only the case's own).  For engine 0 launch_plan exposes nothing more: LayerSweep (4q chain full unitary, 5q
    chain single column) against the interpreter (6 qubits) follows from the compiled layer tables
    (inst_layer_*.cu), with CPF_NO_LAYERED unset.  For the multi-target cases launch_plan reports the single-target
    dispatch: engine 1 says the HS run is staged for the Heisenberg kernels, whose only multi-target instantiations are
    HeisSweepAnyMT; engine 0 sends a multi-target run to InterpSweepMT."""
    n, layer, K, kind, nt, B, freeze, env, path = P.adam_steps_case(name)
    assert got["engine"] == (0 if path == "state_adjoint" else 1), got
    assert (got["engine"] == 1) == (kind == "hs")
    if name.startswith("heis_chain4"):
        assert got["words_per_sample"] == HEIS_CHAIN4_WORDS, got
    # with the case's switches in effect, the dispatcher sends every template to HeisSweepAny (heis_any_kite4) or
    # keeps the compile-time layers (every other case)
    want = HEIS_ANY_CHAIN4_WORDS if path == "heis_any" and not nt else HEIS_CHAIN4_WORDS
    assert got["chain4_probe_words"] == want, got


@pytest.mark.parametrize("name,dt", CASES, ids=[f"{c}-{'c64' if d == F32 else 'c128'}" for c, d in CASES])
def test_adam_steps_match_the_oracle(name, dt):
    got = P.measure_adam_steps(name, dt)
    _check_path(name, dt, got)
    assert got["chain_identical"], "checkpointed chain of launches differs from one 2000-step launch"
    for row in got["rows"]:
        k = row["k"]
        assert row["m_ratio"] <= 1.0, (k, row)
        assert row["v_ratio"] <= 1.0, (k, row)
        assert row["theta_ratio"] <= 1.0, (k, row)
        assert row["loss_ratio"] <= 1.0, (k, row)
        assert row["frozen_unchanged"], (k, row)
        assert row["best_ok"], (k, row)
    # the improving branch of best tracking is exercised
    assert any(row["improved"] for row in got["rows"] if row["k"] > 0)


def test_step_inputs_reach_every_modulus_branch():
    """The inputs put CP angles in every range penalty_eval_fast reduces differently: [0, p), [p, 2p), (-p, 0) and the
    rest, and on the breakpoints (needs no device work beyond the initial batch)."""
    n, layer, K = 4, P.chain_layer(4), 40
    anz, _, _ = P.setup(n, layer, K, "xyz")
    a = P.adam_steps_inputs(anz, 32, F32, big=True).numpy()
    cp = a[:, np.asarray(anz.cp_mask, dtype=bool)]
    p = np.float32(2 * np.pi)
    assert ((cp >= 0) & (cp < p)).any() and ((cp >= p) & (cp < 2 * p)).any()
    assert ((cp < 0) & (cp > -p)).any() and ((cp <= -p) | (cp >= 2 * p)).any()
    assert (cp == np.float32(-1e-8)).any() and np.float32(-1e-8) + p == p    # the f32 rounding the oracle fix covers
    assert np.abs(a).max() > 192000
