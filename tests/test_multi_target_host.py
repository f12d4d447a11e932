"""CPU-side checks of the multi-target entry points (cpf_*_multi, MultiLoss, synthesize_many): symbols and struct
layout, workspace arithmetic, and that bad input is rejected before any device work.  Every call below either needs
no device or fails validation first (the pointers handed to the library are never dereferenced)."""
import ctypes as C

import numpy as np
import pytest
import torch

from cpflow_b200 import _lib as L
from cpflow_b200 import ansatz as A
from cpflow_b200 import topology as T
from cpflow_b200.engine import Loss, MultiLoss, Program, TorchLoss
from cpflow_b200.main import StaticOptions, synthesize_many
from cpflow_b200.optimization import run_adam_batch

MULTI = ("cpf_loss_grad_multi", "cpf_adam_run_multi", "cpf_workspace_bytes_multi")


def _program(n=4, K=40, layer=None):
    anz = A.Ansatz(n, "cp", T.fill_layers(layer or T.chain_layer(n), K), "xyz")
    return Program(n, anz.ops, anz.num_angles)


def test_multi_symbols_and_table_layout(lib):
    for s in MULTI:
        assert s in L.EXPORTS and hasattr(lib, s)
    assert C.sizeof(L.CpfTargetTable) == 4 + 4 + 8 + 8
    assert [f[0] for f in L.CpfTargetTable._fields_] == ["kind", "n_targets", "targets", "target_index"]
    assert L.CpfTargetTable.targets.offset == 8 and L.CpfTargetTable.target_index.offset == 16


def _ws(prog, kind, dtype, batch, n_targets):
    n = C.c_int64()
    rc = L.load().cpf_workspace_bytes_multi(prog._h, kind, dtype, batch, n_targets, C.byref(n))
    return rc, n.value


def _align(b):
    return (b + 255) // 256 * 256


@pytest.mark.parametrize("dtype,rs", [(L.F32, 4), (L.F64, 8)])
def test_workspace_bytes_multi_arithmetic(lib, dtype, rs):
    prog = _program(4, 40)
    N, B = 16, 1000
    # HS on a block-structured template: the Heisenberg-picture kernel's table, 2 N (N + 1) words a target, and the
    # same optimiser state as a single-target run, whose staged target drops out
    rc, one = _ws(prog, L.LOSS_HS, dtype, B, 1)
    assert rc == 0
    single = prog.workspace_bytes(B, L.LOSS_HS, torch.float32 if dtype == L.F32 else torch.float64)
    heis_target = _align(2 * N * (N + 1) * rs)
    assert one == single - heis_target + _align(4 * B) + heis_target
    for T_ in (2, 7, 256):
        rc, many = _ws(prog, L.LOSS_HS, dtype, B, T_)
        assert rc == 0 and many == one - heis_target + _align(T_ * 2 * N * (N + 1) * rs)
    assert _ws(prog, L.LOSS_HS, dtype, 2 * B, 7)[1] > _ws(prog, L.LOSS_HS, dtype, B, 7)[1]
    assert _ws(prog, L.LOSS_HS, dtype, B, 8)[1] > _ws(prog, L.LOSS_HS, dtype, B, 7)[1]
    # state preparation on the interpreter kernel: single-column layout, (N + 1) complex words a target
    rc, st = _ws(prog, L.LOSS_STATE, dtype, B, 5)
    assert rc == 0 and st == _align(prog.info["n_phase"]) + _align(4 * B) + _align(5 * (N + 1) * 2 * rs)


def test_workspace_bytes_multi_rejects_bad_arguments(lib):
    prog = _program(3, 6)
    assert _ws(prog, L.LOSS_HS, L.F32, 10, 0)[0] == -1
    assert _ws(prog, 7, L.F32, 10, 1)[0] == -1
    assert _ws(prog, L.LOSS_HS, 5, 10, 1)[0] == -1
    assert _ws(prog, L.LOSS_HS, L.F32, -1, 1)[0] == -1


def _table(kind, n_targets, index):
    idx = np.ascontiguousarray(index, dtype=np.int32)
    # a non-NULL device address that is never read: every call below fails validation before any CUDA call
    return L.CpfTargetTable(kind, n_targets, 0x1000, idx.ctypes.data), idx


def _loss_grad_multi(prog, table, batch):
    # loss_out / angles NULL: a table that passed validation would still be rejected without touching the device
    return L.load().cpf_loss_grad_multi(prog._h, C.byref(table) if table is not None else None, None, L.F32, batch,
                                        None, None, None, None, None)


def _adam_run_multi(prog, table, batch):
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    buf = L.CpfAdamBuffers()          # all NULL
    return L.load().cpf_adam_run_multi(prog._h, C.byref(table), None, C.byref(ad), L.F32, batch, 0, 10,
                                       C.byref(buf), None)


def _err():
    return L.load().cpf_last_error().decode()


@pytest.mark.parametrize("call", [_loss_grad_multi, _adam_run_multi])
def test_multi_calls_reject_bad_tables_before_device_work(lib, call):
    prog = _program(3, 6)
    tt, idx = _table(L.LOSS_HS, 3, [0, 1, 2, 3, 1])
    assert call(prog, tt, 5) == -1 and "target_index[3] = 3" in _err()
    tt, idx = _table(L.LOSS_HS, 3, [0, -1, 2])
    assert call(prog, tt, 3) == -1 and "target_index[1] = -1" in _err()
    tt, idx = _table(L.LOSS_HS, 0, [0, 0])
    assert call(prog, tt, 2) == -1 and "n_targets" in _err()
    tt, idx = _table(9, 2, [0, 1])
    assert call(prog, tt, 2) == -1 and "unknown loss kind" in _err()
    tt = L.CpfTargetTable(L.LOSS_HS, 2, 0x1000, None)
    assert call(prog, tt, 2) == -1 and "target_index is NULL" in _err()
    # a valid table reaches the next check, which needs no device either
    tt, idx = _table(L.LOSS_RELPHASE, 2, [0, 1, 1, 0])
    assert call(prog, tt, 4) == -1 and "target" not in _err()


def test_multi_full_unitary_losses_keep_the_five_qubit_limit(lib):
    prog = Program(6, [(L.RX, q, -1, q, 0.0) for q in range(6)], 6)
    for kind in (L.LOSS_HS, L.LOSS_RELPHASE):
        tt, idx = _table(kind, 1, [0, 0])
        assert _loss_grad_multi(prog, tt, 2) == -2 and "n <= 5" in _err()
    tt, idx = _table(L.LOSS_STATE, 1, [0, 0])
    assert _loss_grad_multi(prog, tt, 2) == -1 and "n <= 5" not in _err()
    assert _loss_grad_multi(prog, None, 2) == -1 and "NULL" in _err()


def test_multiloss_shapes_and_program_mismatch(lib):
    prog = _program(3, 6)
    with pytest.raises(ValueError):
        MultiLoss("hs", np.zeros((8, 8)))              # one matrix, not a stack
    with pytest.raises(ValueError):
        MultiLoss("state", np.zeros((2, 8, 8)))
    with pytest.raises(ValueError):
        MultiLoss("hs", np.zeros((0, 8, 8)))
    with pytest.raises(ValueError):
        MultiLoss("hs", np.zeros((2, 8, 4)))
    with pytest.raises(ValueError):
        MultiLoss("swap", np.zeros((2, 8, 8)))
    ml = MultiLoss("hs", np.stack([np.eye(4)] * 3))
    assert ml.n_targets == 3 and ml.loss(1).kind == "hs" and ml.loss(1).target.shape == (4, 4)
    angles = torch.zeros(5, prog.n_params)
    with pytest.raises(ValueError, match="dimension 4"):
        prog.loss_grad_multi(angles, ml, [0] * 5)
    ok = MultiLoss("hs", np.stack([np.eye(8)] * 3))
    with pytest.raises(ValueError, match="entries"):
        prog.loss_grad_multi(angles, ok, [0, 1])
    with pytest.raises(TypeError):
        prog.loss_grad_multi(angles, Loss("hs", np.eye(8)), [0] * 5)


def test_run_adam_batch_rejects_user_loss_with_target_index():
    prog = _program(3, 6)
    with pytest.raises(TypeError):
        run_adam_batch(prog, TorchLoss(lambda u: u.abs().sum()), None, torch.zeros(4, prog.n_params), 0.1, 10,
                       target_index=[0, 0, 1, 1])


def test_synthesize_many_argument_handling(lib):
    opts = StaticOptions(num_cp_gates=4, accepted_num_cz_gates=8, num_samples=4)
    layer = T.chain_layer(3)
    tg = np.stack([np.eye(8)] * 2)
    with pytest.raises(ValueError, match="2 targets"):
        synthesize_many(layer, tg, opts, labels=["a", "b", "c"])
    with pytest.raises(ValueError):
        synthesize_many(layer, np.stack([np.eye(4)] * 2), opts)          # 2-qubit targets, 3-qubit layer
    with pytest.raises(ValueError):
        synthesize_many(layer, np.eye(8), opts)                           # not a stack
    with pytest.raises(ValueError):
        synthesize_many(layer, np.ones((2, 4)), opts, loss="state")        # 2-qubit states, 3-qubit layer
    with pytest.raises(TypeError):
        synthesize_many(layer, tg, opts, loss=lambda u: 0.0)
    with pytest.raises(TypeError):
        synthesize_many(layer, tg, opts, loss=TorchLoss(lambda u: u.abs().sum()))
