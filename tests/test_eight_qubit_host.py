"""8-qubit programs, host side: the qubit limit, the refusals that happen before any device work (full-unitary losses,
isometry masks and column counts) and the workspace, cost and launch-plan arithmetic of the state and isometry kinds.
Every library call below either needs no device or fails validation first (its pointers are never dereferenced)."""
import ctypes as C
import math

import numpy as np
import pytest

from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.engine import Loss, clean_ancilla_isometry
from cpflow_b200.topology import chain_layer, fill_layers

N8 = 256


def _chain(K=6):
    return Ansatz(8, "cp", fill_layers(chain_layer(8), K)).program


def _err():
    return L.load().cpf_last_error().decode()


def _mask(anc):
    return sum(1 << q for q in anc)


def _align(b):
    return (b + 255) // 256 * 256


def _fake_calls(prog, kind, mask):
    """Return codes of cpf_loss_grad, cpf_adam_run and cpf_workspace_bytes with fake device pointers."""
    lib = L.load()
    spec = L.CpfLossSpec(kind, 1, mask)
    rc_lg = lib.cpf_loss_grad(prog._h, C.byref(spec), None, L.F32, 4, C.c_void_p(16), C.c_void_p(8), None, None, None)
    err_lg = _err()
    buf = L.CpfAdamBuffers(*([8] * 11), 0, 0, 0)
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    rc_ad = lib.cpf_adam_run(prog._h, C.byref(spec), None, C.byref(ad), L.F64, 4, 0, 5, C.byref(buf), None)
    b = C.c_int64()
    code = L.isometry_kind(mask) if kind == L.LOSS_ISOMETRY else kind
    rc_ws = lib.cpf_workspace_bytes(prog._h, code, L.F32, 4, C.byref(b))
    return rc_lg, err_lg, rc_ad, rc_ws


def test_program_create_limit(lib):
    assert L.MAX_QUBITS == 8
    for n, code in ((8, 0), (9, -2)):
        h = C.c_void_p()
        ops = (L.CpfOp * 1)(L.CpfOp(L.RX, n - 1, -1, 0, 0.0))
        assert lib.cpf_program_create(n, 1, ops, 1, C.byref(h)) == code
        if code == 0:
            info = L.CpfProgramInfo()
            assert lib.cpf_program_get_info(h, C.byref(info)) == 0 and info.n_qubits == 8
            lib.cpf_program_destroy(h)
        else:
            assert not h.value and "outside supported range [2,8]" in _err()


@pytest.mark.parametrize("kind", [L.LOSS_HS, L.LOSS_RELPHASE])
def test_full_unitary_losses_refused_before_device_work(lib, kind):
    prog = _chain()
    rc_lg, err, rc_ad, rc_ws = _fake_calls(prog, kind, 0)
    assert (rc_lg, rc_ad, rc_ws) == (-2, -2, -2)
    assert "n <= 5" in err and "n <= 5" in _err()
    idx = np.zeros(3, dtype=np.int32)
    tt = L.CpfTargetTable(kind, 1, 0x1000, idx.ctypes.data)
    assert lib.cpf_loss_grad_multi(prog._h, C.byref(tt), None, L.F32, 3, C.c_void_p(16), C.c_void_p(8), None, None,
                                   None) == -2
    assert "n <= 5" in _err()
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    buf = L.CpfAdamBuffers()
    assert lib.cpf_adam_run_multi(prog._h, C.byref(tt), None, C.byref(ad), L.F32, 3, 0, 10, C.byref(buf), None) == -2
    assert "n <= 5" in _err()
    b = C.c_int64()
    assert lib.cpf_workspace_bytes_multi(prog._h, kind, L.F32, 3, 1, C.byref(b)) == -2
    assert "n <= 5" in _err()


def test_state_loss_passes_the_checks(lib):
    prog = _chain()
    # the state loss gets past every check; with NULL outputs the call stops at the next argument check
    spec = L.CpfLossSpec(L.LOSS_STATE, 1, 0)
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), None, L.F32, 4, None, None, None, None, None) == -1
    assert "n <= 5" not in _err()
    idx = np.zeros(2, dtype=np.int32)
    tt = L.CpfTargetTable(L.LOSS_STATE, 1, 0x1000, idx.ctypes.data)
    assert lib.cpf_loss_grad_multi(prog._h, C.byref(tt), None, L.F32, 2, None, None, None, None, None) == -1
    assert "n <= 5" not in _err()


@pytest.mark.parametrize("mask,code,words", [
    (1 << 8, -1, "names a qubit >= n"),
    (0, -2, "full-unitary losses need n <= 5"),
    (_mask([0, 7]), -2, "at most k = 32"),           # k = 64
    (_mask([3]), -2, "at most k = 32"),              # k = 128
])
def test_isometry_rejections_before_device_work(lib, mask, code, words):
    prog = _chain()
    rc_lg, err, rc_ad, rc_ws = _fake_calls(prog, L.LOSS_ISOMETRY, mask)
    assert rc_lg == code and rc_ad == code and words in err
    # a mask bit >= 8 does not fit the 8 bits CPF_ISOMETRY_KIND carries: an unknown kind there
    assert rc_ws == (-1 if mask >> 8 else code)
    info = L.CpfLaunchInfo()
    assert lib.cpf_launch_plan(prog._h, L.isometry_kind(mask), L.F32, 100, 0, 0, C.byref(info)) == rc_ws


@pytest.mark.parametrize("anc", [[0, 1, 2, 3, 4, 5, 6, 7], [1, 2, 3, 4, 5, 6, 7], [0, 2, 4, 6], [5, 6, 7],
                                 [0, 3, 7], [1, 2, 3, 4, 5]])
def test_isometry_launch_plan(lib, anc):
    prog = _chain(60)
    k = 2 ** (8 - len(anc))
    for dt in (L.F32, L.F64):
        info = L.CpfLaunchInfo()
        assert lib.cpf_launch_plan(prog._h, L.isometry_kind(_mask(anc)), dt, 1000, 0, 0, C.byref(info)) == 0
        assert info.engine == 0
        assert info.threads_per_sample == 32 * k                 # one warp per input column
        assert info.samples_per_cta == max(1, 128 // (32 * k))
        assert info.block_threads == info.samples_per_cta * info.threads_per_sample
        assert info.max_block_threads == 1024 and info.block_threads <= 1024
        assert info.grid == math.ceil(1000 / info.samples_per_cta)
        assert 0 < info.smem_bytes <= 227 * 1024
        assert info.time_slices == 1 and info.launches_per_run == 1
    if k == 32:
        assert info.block_threads == 1024


def test_state_launch_plan(lib):
    prog = _chain(60)
    for dt in (L.F32, L.F64):
        info = L.CpfLaunchInfo()
        assert lib.cpf_launch_plan(prog._h, L.LOSS_STATE, dt, 1000, 0, 0, C.byref(info)) == 0
        assert info.engine == 0


@pytest.mark.parametrize("anc", [[1, 2, 3, 4, 5, 6, 7], [0, 1, 2, 3, 4, 5, 6, 7], [2, 3, 5], [0, 4, 5, 6]])
def test_eval_and_executed_cost(lib, anc):
    prog = _chain(7)
    k = 2 ** (8 - len(anc))
    code = L.isometry_kind(_mask(anc))
    f_st, b_st = prog.eval_cost(L.LOSS_STATE)
    assert f_st == N8 * (16 * prog.info["n_rotations"] + 4 * prog.info["n_phase"] + 8)
    assert b_st == 6 * prog.n_params * 4 + 8
    f_iso, b_iso = prog.eval_cost(code)
    assert f_iso == pytest.approx(k * f_st) and b_iso == b_st
    G, K = prog.info["n_fused"], prog.info["n_phase"]
    fixed = 232 * G + 80 * K
    e_st = prog.executed_cost(L.LOSS_STATE)
    assert e_st == pytest.approx(N8 * (22 * G + 5.5 * K + 8) + fixed)
    assert prog.executed_cost(code) - fixed == pytest.approx(k * (e_st - fixed))


def test_workspace_bytes(lib):
    prog = _chain(6)
    n_cp = prog.info["n_phase"]
    for dt, rs in ((L.F32, 4), (L.F64, 8)):
        st = C.c_int64()
        L.check(lib.cpf_workspace_bytes(prog._h, L.LOSS_STATE, dt, 50, C.byref(st)))
        st_target = ((N8 + 1) * 2 * rs + 15) // 16 * 16               # one padded column
        assert st.value == _align(n_cp) + _align(st_target)
        for anc in ([1, 2, 3, 4, 5, 6, 7], [0, 2, 4, 6], [5, 6, 7]):
            k = 2 ** (8 - len(anc))
            iso = C.c_int64()
            L.check(lib.cpf_workspace_bytes(prog._h, L.isometry_kind(_mask(anc)), dt, 50, C.byref(iso)))
            assert iso.value == _align(n_cp) + _align(2 * k * N8 * rs)   # W packed column by column
        multi = C.c_int64()
        L.check(lib.cpf_workspace_bytes_multi(prog._h, L.LOSS_STATE, dt, 50, 3, C.byref(multi)))
        assert multi.value == _align(n_cp) + _align(4 * 50) + _align(3 * (N8 + 1) * 2 * rs)


def test_host_isometry_helpers():
    G = np.linalg.qr(np.random.default_rng(2).normal(size=(8, 8)) + 0j)[0]
    W = clean_ancilla_isometry(G, [1, 3, 5, 7, 6], 8)
    loss = Loss("isometry", W, ancillas=[1, 3, 5, 6, 7])
    assert W.shape == (N8, 8) and loss.columns == tuple(s for s in range(N8) if s & 0b01010111 == 0)
    with pytest.raises(ValueError, match="256 x 16"):
        Loss("isometry", np.zeros((N8, 8)), ancillas=[0, 1, 2, 3])
