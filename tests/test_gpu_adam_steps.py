"""One-step consistency of the Adam loop along 2000-step runs, on every path it dispatches to: the fused loop
(cpf_adam_run, cpf_adam_run_multi) on the Heisenberg-picture kernels, the state-adjoint kernels and the isometry kernels,
and the host-driven loop of callable losses (cpf_adam_step).  At checkpoints k the state handed from step k to step
k + 1 (angles, moments, best parameters and losses) is checked against the float64 reference's gradient at the
kernel's own theta_k and optax's update (tests/parity_lib.py: measure_adam_steps, which states the bounds and their
derivation).  The checkpointed chain of launches must be bit-identical to one uninterrupted launch, so the checked
steps are steps of the real run; the optimiser state starts as NaN, so every entry a fresh run must write is checked.

Inputs cover the threefry batch of static(), CP angles over [-3 pi, 5 pi) (every branch of the penalty's modulus), the
penalty's breakpoints and, on the packed float path, angles beyond the fast sin / cos reduction.  Measured maxima:
tools/parity_report.py --steps (profiles/adam_steps_r2.txt)."""
import numpy as np
import pytest
import torch

import parity_lib as P

pytestmark = pytest.mark.gpu

F32, F64 = torch.float32, torch.float64
BOTH = (F32, F64)
_CASE_DTYPES = [
    ("heis_chain4", BOTH), ("heis_chain4_freeze", (F32,)), ("heis_chain4_xz", (F32,)), ("heis_star4_zyx", (F32,)),
    ("heis_any_kite4", (F32,)), ("heis_any_mt_chain3", BOTH), ("iso_as_hs_chain4", (F32,)), ("adj_hs_chain5", (F64,)),
    ("layer_relphase_chain4", (F32,)), ("layer_state_chain5", (F32,)), ("interp_state_chain6", (F32,)),
    ("interp_state_chain7", BOTH), ("interp_state_chain8", BOTH), ("interp_mt_state_chain4", BOTH),
    ("interp_mt_state_chain6", BOTH), ("interp_mt_state_chain8", (F32,)), ("interp_mt_relphase_chain4", BOTH),
    ("iso_chain6_k8", BOTH), ("iso_chain8_k32", BOTH), ("iso_chain8_k32_freeze", BOTH), ("isorel_chain3", BOTH),
    ("isorel_chain5_k2", BOTH), ("isorel_chain7_k8_freeze", BOTH), ("isorel_chain8_k32", (F32,)),
    ("host_hs_chain6", BOTH), ("host_hs_chain6_k120", (F64,)), ("host_state_chain8_freeze", BOTH)]
CASES = [(c, d) for c, dts in _CASE_DTYPES for d in dts]
# launch_plan's words_per_sample of the 4q chain, K = 40 on the compile-time layer; the runtime-pair kernel
# (HeisSweepAny) stages one more layer of rows and needs 860
HEIS_CHAIN4_WORDS, HEIS_ANY_CHAIN4_WORDS = 844, 860


def _register_bits(c):
    """Register bits of iso_kernel's sweep (iso_impl.cuh: iso_rb, iso_phase_rb)."""
    if c.n == 8:
        return 3
    return 1 if c.kind == "isometry_relphase" and c.n in (4, 5) else 2


def _check_path(name, dt, got):
    """What launch_plan can show of the path a case ran on (measure_adam_steps clears inherited dispatch switches and
    sets only the case's own).  Engine 1 is the Heisenberg-picture kernels: HS on block-structured templates, and the
    isometry loss on <= 5 qubits as HS on its padded target.  Engine 0 is everything else: for the state-adjoint cases
    LayerSweep (4q chain full unitary, 5q chain single column) against the interpreter (6-8 qubits) follows from the
    compiled layer tables (inst_layer_*.cu), with CPF_NO_LAYERED unset; HS runs there only under CPF_ENGINE=adjoint.
    The isometry kernel reports k lane groups of 2^(n - RB) threads per sample.  For the host loop the plan
    is that of cpf_adjoint_from_cotangent's launch item.  For the multi-target cases launch_plan reports the
    single-target dispatch: engine 1 says the HS run is staged for the Heisenberg kernels, whose only multi-target
    instantiations are HeisSweepAnyMT; engine 0 sends a multi-target run to InterpSweepMT."""
    c = P.adam_steps_case(name)
    assert got["engine"] == (1 if c.path in ("heis", "heis_any", "iso_as_hs") else 0), got
    if c.path == "state_adjoint":
        assert (c.kind == "hs") == (c.env.get("CPF_ENGINE") == "adjoint"), got
    if c.path == "iso":
        k = 2 ** (c.n - len(c.anc))
        assert got["threads_per_sample"] == k << (c.n - _register_bits(c)), got
    if c.path == "host":
        assert got["cot_columns"] == (16 if name == "host_hs_chain6_k120" and dt == F64 else 32), got
    if name.startswith("heis_chain4") and c.rg == "xyz":
        assert got["words_per_sample"] == HEIS_CHAIN4_WORDS, got
    # with the case's switches in effect, the dispatcher sends every template to HeisSweepAny (heis_any_kite4) or
    # keeps the compile-time layers (every other case but adj_hs_chain5, which keeps HS off the Heisenberg kernels)
    want = HEIS_ANY_CHAIN4_WORDS if c.path == "heis_any" and not c.nt else HEIS_CHAIN4_WORDS
    if "CPF_ENGINE" not in c.env:
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
