"""Isometry loss, host side: ABI symbols, the rejections that happen before any device work, the cost and geometry
queries, and the shape checks of Loss('isometry')."""
import ctypes as C
import math

import numpy as np
import pytest

from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.engine import Loss, Program, clean_ancilla_isometry
from cpflow_b200.topology import chain_layer, fill_layers


def _chain(n, K):
    return Ansatz(n, "cp", fill_layers(chain_layer(n), K)).program


def _spec(kind, mask, ptr=1):
    return L.CpfLossSpec(kind, ptr, mask)


def _loss_grad_rc(prog, spec):
    # a fake device pointer: every rejection below must come before the library touches it
    lo = C.c_void_p(8)
    return L.load().cpf_loss_grad(prog._h, C.byref(spec), None, L.F32, 4, C.c_void_p(16), lo, None, None, None)


def test_symbols_and_struct():
    lib = L.load()
    assert L.LOSS_ISOMETRY == 3
    assert [f[0] for f in L.CpfLossSpec._fields_] == ["kind", "target", "ancilla_mask"]
    assert L.CpfLossSpec.ancilla_mask.offset == 16
    assert L.isometry_kind(0b101) == 3 | (5 << 8)
    assert lib.cpf_version() == 200


@pytest.mark.parametrize("n,mask,code,words", [
    (4, 1 << 4, -1, "names a qubit >= n"),
    (6, 1 << 6, -1, "names a qubit >= n"),
    (6, 0, -2, "full-unitary losses need n <= 5"),
    (7, 0, -2, "full-unitary losses need n <= 5"),
    (7, 1, -2, "at most k = 32"),
])
def test_rejections_before_device_work(n, mask, code, words):
    prog = _chain(n, 2)
    assert _loss_grad_rc(prog, _spec(L.LOSS_ISOMETRY, mask)) == code
    assert words in L.load().cpf_last_error().decode()
    buf = L.CpfAdamBuffers(*([8] * 11), 0, 0, 0)
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    assert L.load().cpf_adam_run(prog._h, C.byref(_spec(L.LOSS_ISOMETRY, mask)), None, C.byref(ad), L.F32, 4, 0, 5,
                                 C.byref(buf), None) == code
    b = C.c_int64()
    assert L.load().cpf_workspace_bytes(prog._h, L.isometry_kind(mask), L.F32, 4, C.byref(b)) == code


def test_multi_target_table_refused():
    prog = _chain(3, 2)
    idx = (C.c_int32 * 2)(0, 0)
    tt = L.CpfTargetTable(L.LOSS_ISOMETRY, 1, 8, C.cast(idx, C.c_void_p))
    lo = C.c_void_p(8)
    assert L.load().cpf_loss_grad_multi(prog._h, C.byref(tt), None, L.F32, 2, C.c_void_p(16), lo, None, None,
                                        None) == -2
    assert "isometry" in L.load().cpf_last_error().decode()
    b = C.c_int64()
    assert L.load().cpf_workspace_bytes_multi(prog._h, L.LOSS_ISOMETRY, L.F32, 2, 1, C.byref(b)) == -2


@pytest.mark.parametrize("n,anc", [(3, [1]), (5, [0, 4]), (6, [0]), (7, [0, 3]), (7, [0, 1, 2, 3, 4, 5, 6])])
def test_eval_cost(n, anc):
    prog = _chain(n, 3)
    k = 2 ** (n - len(anc))
    mask = sum(1 << q for q in anc)
    f_iso, b_iso = prog.eval_cost(L.isometry_kind(mask))
    f_st, b_st = prog.eval_cost(L.LOSS_STATE)
    assert f_iso == pytest.approx(k * f_st) and b_iso == b_st


@pytest.mark.parametrize("n,anc", [(6, [0]), (6, [2, 5]), (6, [0, 1, 2, 3, 4, 5]), (7, [0, 6]), (7, [1, 2, 3])])
def test_launch_plan_large(n, anc):
    prog = _chain(n, 60)
    k = 2 ** (n - len(anc))
    mask = sum(1 << q for q in anc)
    for dt in (L.F32, L.F64):
        info = L.CpfLaunchInfo()
        assert L.load().cpf_launch_plan(prog._h, L.isometry_kind(mask), dt, 1000, 0, 0, C.byref(info)) == 0
        assert info.engine == 0
        assert info.threads_per_sample == k * 2 ** (n - 2)
        assert info.block_threads == info.samples_per_cta * info.threads_per_sample
        assert info.block_threads <= info.max_block_threads
        assert info.grid == math.ceil(1000 / info.samples_per_cta)
        assert 0 < info.smem_bytes <= 227 * 1024


def test_launch_plan_small_is_hs():
    prog = _chain(4, 8)
    for mask in (0, 0b0011):
        assert prog.launch_plan(100, L.isometry_kind(mask)) == prog.launch_plan(100, L.LOSS_HS)


def test_workspace_bytes():
    for n, anc in ((4, [1]), (5, [])):
        prog = _chain(n, 6)
        mask = sum(1 << q for q in anc)
        for dt, rs in ((L.F32, 4), (L.F64, 8)):
            hs, iso = C.c_int64(), C.c_int64()
            L.check(L.load().cpf_workspace_bytes(prog._h, L.LOSS_HS, dt, 50, C.byref(hs)))
            L.check(L.load().cpf_workspace_bytes(prog._h, L.isometry_kind(mask), dt, 50, C.byref(iso)))
            v = 2 * 4 ** n * rs                                    # the N x N HS target built from W
            assert iso.value == hs.value + (v + 255) // 256 * 256
    for n, anc in ((6, [0]), (7, [2, 4])):
        prog = _chain(n, 6)
        k = 2 ** (n - len(anc))
        mask = sum(1 << q for q in anc)
        st, iso = C.c_int64(), C.c_int64()
        L.check(L.load().cpf_workspace_bytes(prog._h, L.LOSS_STATE, L.F64, 50, C.byref(st)))
        L.check(L.load().cpf_workspace_bytes(prog._h, L.isometry_kind(mask), L.F64, 50, C.byref(iso)))
        st_target = ((2 ** n + 1) * 2 * 8 + 15) // 16 * 16
        assert iso.value - st.value == (2 * k * 2 ** n * 8 + 255) // 256 * 256 - (st_target + 255) // 256 * 256


def test_loss_shape_checks():
    W = np.zeros((8, 4))
    assert Loss("isometry", W, ancillas=[1]).columns == (0, 1, 4, 5)
    assert Loss("isometry", W, ancillas=[0]).columns == (0, 1, 2, 3)
    with pytest.raises(ValueError, match="needs `ancillas`"):
        Loss("isometry", W)
    with pytest.raises(ValueError, match="8 x 2"):
        Loss("isometry", W, ancillas=[0, 1])
    with pytest.raises(ValueError, match="distinct qubits"):
        Loss("isometry", W, ancillas=[3])
    with pytest.raises(ValueError, match="distinct qubits"):
        Loss("isometry", np.zeros((8, 2)), ancillas=[1, 1])
    with pytest.raises(ValueError, match="N = 2"):
        Loss("isometry", np.zeros((6, 3)), ancillas=[])
    with pytest.raises(ValueError, match="not of 'hs'"):
        Loss("hs", np.eye(8), ancillas=[0])


def test_host_formula_and_helper():
    rng = np.random.default_rng(1)
    G = np.linalg.qr(rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4)))[0]
    W = clean_ancilla_isometry(G, [1], 3)
    loss = Loss("isometry", W, ancillas=[1])
    # U = G on qubits (0, 2) (big-endian), identity on the ancilla: exact
    U = np.zeros((8, 8), complex)
    for a in range(2):
        for i in range(4):
            for j in range(4):
                r = ((i >> 1) << 2) | (a << 1) | (i & 1)
                c = ((j >> 1) << 2) | (a << 1) | (j & 1)
                U[r, c] = G[i, j]
    assert loss(U) == pytest.approx(0.0, abs=1e-12)
    assert loss(np.exp(0.7j) * U) == pytest.approx(0.0, abs=1e-12)
    # A = 0 is the HS loss, k = 1 the state loss
    V = np.linalg.qr(rng.normal(size=(8, 8)) + 1j * rng.normal(size=(8, 8)))[0]
    assert Loss("isometry", V, ancillas=[])(U) == pytest.approx(Loss("hs", V)(U), abs=1e-12)
    assert Loss("isometry", V[:, :1], ancillas=[0, 1, 2])(U) == pytest.approx(Loss("state", V[:, 0])(U), abs=1e-12)
