"""The plan of a loss call, host side: on every kernel route, a bad workspace or penalty is refused before any device
work, and the query entry points refuse what a loss call would refuse.  Every library call below fails validation
first: its device pointers are fake and never dereferenced, so a call that reached the device would fail here with
CPF_ERR_CUDA (no device) instead of the refusal asserted."""
import ctypes as C

import numpy as np
import pytest

from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.topology import chain_layer, fill_layers

B = 40
WS = 1 << 20          # a fake, 256-byte aligned device address for the caller-owned workspace


def _chain(n, K=8):
    return Ansatz(n, "cp", fill_layers(chain_layer(n), K)).program


def _err():
    return L.load().cpf_last_error().decode()


# (name, n, loss kind, ancilla mask, number of targets (0: one target), dtype, environment, Heisenberg-picture kernel)
ROUTES = [
    ("hs_heis_f32", 4, L.LOSS_HS, 0, 0, L.F32, {}, 1),
    ("hs_heis_f64", 4, L.LOSS_HS, 0, 0, L.F64, {}, 1),
    ("hs_adjoint_f32", 4, L.LOSS_HS, 0, 0, L.F32, {"CPF_ENGINE": "adjoint"}, 0),
    ("hs_adjoint_f64", 4, L.LOSS_HS, 0, 0, L.F64, {"CPF_ENGINE": "adjoint"}, 0),
    ("state", 4, L.LOSS_STATE, 0, 0, L.F32, {}, 0),
    ("relphase", 4, L.LOSS_RELPHASE, 0, 0, L.F32, {}, 0),
    ("isometry_as_hs", 4, L.LOSS_ISOMETRY, 0b0001, 0, L.F32, {}, 1),
    ("isometry_6q", 6, L.LOSS_ISOMETRY, 0b000011, 0, L.F32, {}, 0),
    ("isometry_8q", 8, L.LOSS_ISOMETRY, 0b00011111, 0, L.F64, {}, 0),
    ("multi_hs", 4, L.LOSS_HS, 0, 7, L.F32, {}, 1),
    ("multi_state", 4, L.LOSS_STATE, 0, 7, L.F64, {}, 0),
]


def _query_kind(kind, mask):
    return L.isometry_kind(mask) if kind == L.LOSS_ISOMETRY else kind


def _need(prog, kind, mask, n_targets, dtype):
    b = C.c_int64()
    if n_targets:
        L.check(L.load().cpf_workspace_bytes_multi(prog._h, kind, dtype, B, n_targets, C.byref(b)))
    else:
        L.check(L.load().cpf_workspace_bytes(prog._h, _query_kind(kind, mask), dtype, B, C.byref(b)))
    return b.value


def _adam_run(prog, kind, mask, n_targets, dtype, pen=None, workspace=None, workspace_bytes=0):
    """cpf_adam_run (or cpf_adam_run_multi) on B samples with fake device buffers."""
    buf = L.CpfAdamBuffers(*([8] * 3), None, *([8] * 5), None, None, 0, workspace, workspace_bytes)
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    ps = C.byref(pen) if pen is not None else None
    lib = L.load()
    if n_targets:
        idx = np.arange(B, dtype=np.int32) % n_targets
        tt = L.CpfTargetTable(kind, n_targets, 16, idx.ctypes.data)
        return lib.cpf_adam_run_multi(prog._h, C.byref(tt), ps, C.byref(ad), dtype, B, 0, 10, C.byref(buf), None)
    spec = L.CpfLossSpec(kind, 16, mask)
    return lib.cpf_adam_run(prog._h, C.byref(spec), ps, C.byref(ad), dtype, B, 0, 10, C.byref(buf), None)


@pytest.fixture(params=ROUTES, ids=[r[0] for r in ROUTES])
def route(request, monkeypatch, lib):
    name, n, kind, mask, n_targets, dtype, env, heis = request.param
    for var in ("CPF_ENGINE", "CPF_NO_LAYERED", "CPF_HEIS_ANY"):
        monkeypatch.delenv(var, raising=False)
    for var, val in env.items():
        monkeypatch.setenv(var, val)
    prog = _chain(n)
    info = L.CpfLaunchInfo()
    L.check(lib.cpf_launch_plan(prog._h, _query_kind(kind, mask), dtype, B, 0, 0, C.byref(info)))
    assert info.engine == heis, name           # the route the case is meant to cover
    return prog, kind, mask, n_targets, dtype


def test_short_workspace_is_refused(route):
    prog, kind, mask, n_targets, dtype = route
    need = _need(prog, kind, mask, n_targets, dtype)
    assert need > 0 and need % 256 == 0
    assert _adam_run(prog, kind, mask, n_targets, dtype, workspace=WS, workspace_bytes=need - 1) == -1
    assert "workspace too small" in _err()
    assert _adam_run(prog, kind, mask, n_targets, dtype, workspace=WS, workspace_bytes=0) == -1
    assert "workspace too small" in _err()


def test_misaligned_workspace_is_refused(route):
    prog, kind, mask, n_targets, dtype = route
    need = _need(prog, kind, mask, n_targets, dtype)
    assert _adam_run(prog, kind, mask, n_targets, dtype, workspace=WS + 8, workspace_bytes=need + 256) == -1
    assert "aligned" in _err()


def test_bad_penalty_is_refused(route):
    prog, kind, mask, n_targets, dtype = route
    pen = L.CpfPenaltySpec()
    pen.kind = 7
    assert _adam_run(prog, kind, mask, n_targets, dtype, pen=pen) == -1
    assert "unknown penalty kind" in _err()
    # every parameter, rotations included: only parameters of CP gates may be penalised
    cp_mask = np.ones(prog.n_params, dtype=np.uint8)
    pen = L.CpfPenaltySpec()
    pen.kind, pen.r, pen.cp_mask = L.PEN_L1, 0.1, cp_mask.ctypes.data
    assert _adam_run(prog, kind, mask, n_targets, dtype, pen=pen) == -2
    assert "does not feed a CP gate" in _err()
    # the same checks come first with a caller-owned workspace too
    assert _adam_run(prog, kind, mask, n_targets, dtype, pen=pen, workspace=WS, workspace_bytes=1 << 40) == -2


def test_bad_penalty_is_refused_by_loss_grad(lib):
    prog = _chain(4)
    spec = L.CpfLossSpec(L.LOSS_HS, 16, 0)
    pen = L.CpfPenaltySpec()
    pen.kind, pen.n_segments, pen.period = L.PEN_PIECEWISE, 0, 1.0
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), C.byref(pen), L.F32, B, C.c_void_p(8), C.c_void_p(8), None,
                             None, None) == -1
    assert "n_segments" in _err()


def test_queries_refuse_an_unknown_dtype(lib):
    prog = _chain(4)
    b, f, x = C.c_int64(), C.c_double(), C.c_double()
    info = L.CpfLaunchInfo()
    for dt in (2, -1):
        assert lib.cpf_workspace_bytes(prog._h, L.LOSS_HS, dt, B, C.byref(b)) == -1 and "dtype" in _err()
        assert lib.cpf_launch_plan(prog._h, L.LOSS_HS, dt, B, 0, 0, C.byref(info)) == -1 and "dtype" in _err()
        assert lib.cpf_eval_cost(prog._h, L.LOSS_HS, dt, C.byref(f), C.byref(x)) == -1 and "dtype" in _err()
        assert lib.cpf_executed_cost(prog._h, L.LOSS_HS, dt, C.byref(f)) == -1 and "dtype" in _err()
        assert lib.cpf_workspace_bytes_multi(prog._h, L.LOSS_HS, dt, B, 3, C.byref(b)) == -1 and "dtype" in _err()


def test_queries_refuse_what_a_loss_call_refuses(lib):
    # full-unitary kinds above 5 qubits: every query entry point, as cpf_workspace_bytes already did
    prog = _chain(6)
    b, f, x = C.c_int64(), C.c_double(), C.c_double()
    info = L.CpfLaunchInfo()
    for kind in (L.LOSS_HS, L.LOSS_RELPHASE, L.isometry_kind(0)):
        assert lib.cpf_workspace_bytes(prog._h, kind, L.F32, B, C.byref(b)) == -2
        assert lib.cpf_launch_plan(prog._h, kind, L.F32, B, 0, 0, C.byref(info)) == -2
        assert lib.cpf_eval_cost(prog._h, kind, L.F32, C.byref(f), C.byref(x)) == -2
        assert lib.cpf_executed_cost(prog._h, kind, L.F32, C.byref(f)) == -2
        assert "n <= 5" in _err()
    for q in (L.LOSS_STATE, L.isometry_kind(1)):
        assert lib.cpf_launch_plan(prog._h, q, L.F32, B, 0, 0, C.byref(info)) == 0
        assert lib.cpf_executed_cost(prog._h, q, L.F32, C.byref(f)) == 0
    # an unknown kind, and a mask on a kind that takes none
    prog = _chain(4)
    for kind in (4, -1, L.LOSS_HS | (1 << 8), L.isometry_kind(1) | (1 << 16)):
        assert lib.cpf_executed_cost(prog._h, kind, L.F32, C.byref(f)) == -1 and "unknown loss kind" in _err()
        assert lib.cpf_launch_plan(prog._h, kind, L.F32, B, 0, 0, C.byref(info)) == -1


def test_zero_batch_checks_the_arguments(lib):
    # batch 0 is a no-op, but only for a call that would be accepted
    prog = _chain(4)
    spec = L.CpfLossSpec(L.LOSS_HS, 16, 0)
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), None, L.F32, 0, None, None, None, None, None) == 0
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), None, 5, 0, None, None, None, None, None) == -1
    pen = L.CpfPenaltySpec()
    pen.kind = 7
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), C.byref(pen), L.F32, 0, None, None, None, None, None) == -1
