"""Subspace losses, host side: ABI symbols and query kinds, the refusals made before any device work, the route and
launch geometry each call plans, workspace sizes and costs, and the host formula and checks of Loss('subspace') and
Loss('subspace_relphase').  Library calls that must be refused get fake device pointers, which are never
dereferenced: a call that reached the device would fail with CPF_ERR_CUDA instead of the refusal asserted."""
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.engine import Loss, MultiLoss
from cpflow_b200.topology import chain_layer, fill_layers

# register bits of the single-column kernels on n = 2..8 (inst_f32.cu / inst_f64.cu: engine_rb(n, true))
SINGLE_RB = {2: 2, 3: 2, 4: 1, 5: 1, 6: 2, 7: 2, 8: 3}
KINDS = (L.LOSS_SUBSPACE, L.LOSS_SUBSPACE_RELPHASE)


def _chain(n, K):
    return Ansatz(n, "cp", fill_layers(chain_layer(n), K)).program


def _query(kind, k):
    return L.subspace_kind(k) if kind == L.LOSS_SUBSPACE else L.subspace_relphase_kind(k)


def _err():
    return L.load().cpf_last_error().decode()


def _haar(N, k, seed):
    rng = np.random.default_rng(seed)
    return np.linalg.qr(rng.normal(size=(N, N)) + 1j * rng.normal(size=(N, N)))[0][:, :k]


def _pad(k):
    return 1 << (k - 1).bit_length()


def test_symbols_and_query_kinds():
    assert (L.LOSS_SUBSPACE, L.LOSS_SUBSPACE_RELPHASE) == (6, 7)
    assert L.subspace_kind(3) == 6 | (3 << 8) and L.subspace_relphase_kind(32) == 7 | (32 << 8)
    assert L.load().cpf_version() == 200
    A, B = _haar(8, 3, 1), _haar(8, 3, 2)
    assert Loss("subspace", B, inputs=A).code == L.subspace_kind(3)
    assert Loss("subspace_relphase", B, inputs=A).code == L.subspace_relphase_kind(3)
    prog = _chain(4, 2)
    b = C.c_int64()
    for kind in KINDS:
        assert L.load().cpf_workspace_bytes(prog._h, _query(kind, 2), L.F32, 4, C.byref(b)) == 0
        # bits 16 and up stay an unknown kind, as for the isometry kinds
        assert L.load().cpf_workspace_bytes(prog._h, _query(kind, 2) | (1 << 16), L.F32, 4, C.byref(b)) == -1
        assert "unknown loss kind" in _err()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k,code,words", [
    (2, 0, -1, "1 <= k <= N = 4"),
    (2, 5, -1, "1 <= k <= N = 4"),
    (3, 9, -1, "1 <= k <= N = 8"),
    (5, 33, -1, "1 <= k <= N = 32"),
    (6, 33, -2, "at most k = 32"),
    (8, 64, -2, "at most k = 32"),
    (8, 257, -1, "1 <= k <= N = 256"),
])
def test_refusals_before_device_work(kind, n, k, code, words):
    prog = _chain(n, 2)
    lib = L.load()
    spec = L.CpfLossSpec(kind, 1, k)
    assert lib.cpf_loss_grad(prog._h, C.byref(spec), None, L.F32, 4, C.c_void_p(16), C.c_void_p(8), None, None,
                             None) == code
    assert words in _err()
    buf = L.CpfAdamBuffers(*([8] * 11), 0, 0, 0)
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    assert lib.cpf_adam_run(prog._h, C.byref(spec), None, C.byref(ad), L.F64, 4, 0, 5, C.byref(buf), None) == code
    assert words in _err()
    if k < 256:                      # the query kinds carry k in 8 bits
        b = C.c_int64()
        assert lib.cpf_workspace_bytes(prog._h, _query(kind, k), L.F32, 4, C.byref(b)) == code
        assert words in _err()
        info = L.CpfLaunchInfo()
        assert lib.cpf_launch_plan(prog._h, _query(kind, k), L.F32, 4, 0, 0, C.byref(info)) == code


@pytest.mark.parametrize("kind", KINDS)
def test_multi_target_table_refused(kind):
    lib = L.load()
    for n in (3, 6):
        prog = _chain(n, 2)
        idx = (C.c_int32 * 2)(0, 0)
        tt = L.CpfTargetTable(kind, 1, 8, C.cast(idx, C.c_void_p))
        assert lib.cpf_loss_grad_multi(prog._h, C.byref(tt), None, L.F32, 2, C.c_void_p(16), C.c_void_p(8), None,
                                       None, None) == -2
        assert "one target per call" in _err()
        buf = L.CpfAdamBuffers(*([8] * 11), 0, 0, 0)
        ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
        assert lib.cpf_adam_run_multi(prog._h, C.byref(tt), None, C.byref(ad), L.F32, 2, 0, 5, C.byref(buf),
                                      None) == -2
        assert "one target per call" in _err()
        # the workspace query reads the kind in the query form: a valid k reaches the table refusal, a bare kind is
        # k = 0 and is refused as in cpf_workspace_bytes
        b = C.c_int64()
        assert lib.cpf_workspace_bytes_multi(prog._h, _query(kind, 2), L.F32, 2, 1, C.byref(b)) == -2
        assert "one target per call" in _err()
        assert lib.cpf_workspace_bytes_multi(prog._h, kind, L.F32, 2, 1, C.byref(b)) == -1
        assert "1 <= k <= N" in _err()
        assert lib.cpf_workspace_bytes_multi(prog._h, _query(kind, 2) | (1 << 16), L.F32, 2, 1, C.byref(b)) == -1
        assert "unknown loss kind" in _err()
    with pytest.raises(ValueError, match="one target per call"):
        MultiLoss("subspace", np.zeros((2, 4, 4)))


def test_kind6_small_runs_hs_on_the_heisenberg_kernel(monkeypatch):
    """Kind 6 on n <= 5 is the HS call on V = (N/k) B A^dag: its launch plan, workspace and executed cost are those of
    the HS loss (engine 1 on a layered 4-qubit template; engine 0 under CPF_ENGINE=adjoint)."""
    prog = _chain(4, 6)
    for dtype in (torch.float32, torch.float64):
        for k in (1, 3, 5, 16):
            assert prog.launch_plan(1000, L.subspace_kind(k), dtype)["engine"] == 1
            assert prog.launch_plan(1000, L.subspace_kind(k), dtype) == prog.launch_plan(1000, L.LOSS_HS, dtype)
            # the workspace is the HS call's plus V (N x N complex)
            assert prog.workspace_bytes(50, L.subspace_kind(k), dtype) == prog.workspace_bytes(50, L.isometry_kind(1),
                                                                                               dtype)
            assert prog.executed_cost(L.subspace_kind(k), dtype) == prog.executed_cost(L.LOSS_HS, dtype)
    monkeypatch.setenv("CPF_ENGINE", "adjoint")
    assert prog.launch_plan(1000, L.subspace_kind(3))["engine"] == 0
    # the state-adjoint kernels run it with C = N
    assert prog.executed_cost(L.subspace_kind(3)) == prog.executed_cost(L.LOSS_HS)


# (n, k): on the isometry kernel every k, padded to k' = the next power of two
GEOMETRY = [(2, 1), (2, 3), (3, 5), (4, 3), (5, 7), (5, 32), (6, 3), (6, 5), (6, 8), (7, 2), (7, 17), (8, 1), (8, 3),
            (8, 5), (8, 32)]


@pytest.mark.parametrize("n,k", GEOMETRY)
def test_launch_plan_geometry_is_the_isometry_kinds_with_k_padded(n, k):
    prog = _chain(n, 2 * n)
    kp = _pad(k)
    spt = kp * 2 ** (n - SINGLE_RB[n])
    for dtype in (torch.float32, torch.float64):
        rel = prog.launch_plan(1000, L.subspace_relphase_kind(k), dtype)
        # the relative-phase isometry kind with k' columns (ancillas: the first n - log2 k' qubits)
        mask = (1 << (n - (kp.bit_length() - 1))) - 1
        assert rel == prog.launch_plan(1000, L.isometry_relphase_kind(mask), dtype)
        assert rel["engine"] == 0 and rel["threads_per_sample"] == spt
        assert rel["samples_per_cta"] == max(1, 128 // spt)
        assert rel["block_threads"] % 32 == 0 and rel["block_threads"] <= rel["max_block_threads"]
        assert rel["grid"] == -(-1000 // rel["samples_per_cta"])
        if n >= 6:
            assert prog.launch_plan(1000, L.subspace_kind(k), dtype) == rel
            assert rel == prog.launch_plan(1000, L.isometry_kind(mask), dtype)


@pytest.mark.parametrize("n,k", [(2, 3), (3, 1), (4, 5), (5, 32), (6, 3), (7, 8), (8, 5), (8, 32)])
def test_workspace_and_costs(n, k):
    """On the isometry kernel: penalty mask plus B and A packed to k' columns each; credited C = k, executed C = k'."""
    prog = _chain(n, 6)
    kp = _pad(k)
    info = L.CpfProgramInfo()
    L.check(L.load().cpf_program_get_info(prog._h, C.byref(info)))
    n_cp = max(1, info.n_phase)
    kinds = (L.subspace_relphase_kind(k),) + ((L.subspace_kind(k),) if n >= 6 else ())
    mask = (1 << (n - (kp.bit_length() - 1))) - 1
    for dtype, rs in ((torch.float32, 4), (torch.float64, 8)):
        f_st, b_st = prog.eval_cost(L.LOSS_STATE, dtype)
        for q in kinds:
            assert prog.workspace_bytes(50, q, dtype) == (n_cp + 255) // 256 * 256 + \
                (2 * 2 * kp * 2 ** n * rs + 255) // 256 * 256
            f, b = prog.eval_cost(q, dtype)
            assert f == pytest.approx(k * f_st) and b == b_st
            assert prog.executed_cost(q, dtype) == prog.executed_cost(L.isometry_relphase_kind(mask), dtype)
        if n <= 5:
            f, _ = prog.eval_cost(L.subspace_kind(k), dtype)
            assert f == pytest.approx(k * f_st)


def _brute(kind, A, B, U):
    N, k = A.shape
    t = [sum(np.conj(B[r, c]) * sum(U[r, s] * A[s, c] for s in range(N)) for r in range(N)) for c in range(k)]
    if kind == "subspace":
        return 1 - abs(sum(t)) ** 2 / k ** 2
    return 1 - sum(abs(x) ** 2 for x in t) / k


@pytest.mark.parametrize("n,k", [(2, 1), (2, 3), (3, 2), (3, 5), (4, 4), (5, 7)])
def test_host_formula_against_brute_force(n, k):
    N = 2 ** n
    U = _haar(N, N, n)
    A, B = _haar(N, k, 10 + n), _haar(N, k, 20 + n)
    for kind in Loss.SUBSPACE_KINDS:
        loss = Loss(kind, B, inputs=A)
        assert loss(U) == pytest.approx(_brute(kind, A, B, U), abs=1e-12)
    # zero at a unitary that maps a_c to (a phase times) b_c: U = B' A'^dag on completed bases
    Af = np.linalg.qr(np.concatenate([A, _haar(N, N, 3)], axis=1))[0]
    Bf = np.linalg.qr(np.concatenate([B, _haar(N, N, 4)], axis=1))[0]
    Af[:, :k], Bf[:, :k] = A, B                                 # qr may flip phases of the first k columns
    V = Bf @ Af.conj().T
    assert Loss("subspace", B, inputs=A)(V) == pytest.approx(0.0, abs=1e-12)
    D = np.exp(1j * np.random.default_rng(n).uniform(0, 2 * np.pi, k))
    assert Loss("subspace_relphase", B * D[None, :], inputs=A)(V) == pytest.approx(0.0, abs=1e-12)
    if k > 1:
        assert Loss("subspace", B * D[None, :], inputs=A)(V) > 1e-6
    # kind 6 is invariant under (A, B) -> (A Q, B Q), kind 7 under B -> B D
    Q = _haar(k, k, 7)
    assert Loss("subspace", B @ Q, inputs=A @ Q)(U) == pytest.approx(Loss("subspace", B, inputs=A)(U), abs=1e-12)
    assert Loss("subspace_relphase", B * D[None, :], inputs=A)(U) == pytest.approx(
        Loss("subspace_relphase", B, inputs=A)(U), abs=1e-12)


def test_reductions_to_isometry_and_state():
    n, N = 4, 16
    U = _haar(N, N, 9)
    anc = [1, 3]
    W = _haar(N, 4, 5)
    iso = Loss("isometry", W, ancillas=anc)
    A = np.eye(N)[:, list(iso.columns)]
    assert Loss("subspace", W, inputs=A)(U) == pytest.approx(iso(U), abs=1e-12)
    assert Loss("subspace_relphase", W, inputs=A)(U) == pytest.approx(
        Loss("isometry_relphase", W, ancillas=anc)(U), abs=1e-12)
    psi = _haar(N, 1, 6)
    for kind in Loss.SUBSPACE_KINDS:
        assert Loss(kind, psi, inputs=np.eye(N)[:, :1])(U) == pytest.approx(Loss("state", psi[:, 0])(U), abs=1e-12)


def test_shape_norm_and_inputs_checks():
    A, B = _haar(8, 3, 1), _haar(8, 3, 2)
    for kind in Loss.SUBSPACE_KINDS:
        with pytest.raises(ValueError, match="needs `inputs`"):
            Loss(kind, B)
        with pytest.raises(ValueError, match="same shape"):
            Loss(kind, B, inputs=A[:, :2])
        with pytest.raises(ValueError, match="N = 2\\^n rows"):
            Loss(kind, np.ones((6, 1)) / 6 ** 0.5, inputs=np.ones((6, 1)) / 6 ** 0.5)
        with pytest.raises(ValueError, match="1 <= k <= min\\(N, 32\\) = 4"):
            Loss(kind, _haar(4, 4, 1)[:, [0, 1, 2, 3, 0]], inputs=_haar(4, 4, 2)[:, [0, 1, 2, 3, 0]])
        with pytest.raises(ValueError, match="1 <= k <= min\\(N, 32\\) = 32"):
            Loss(kind, _haar(64, 33, 1), inputs=_haar(64, 33, 2))
        with pytest.raises(ValueError, match="column 1 of inputs has norm 2"):
            Loss(kind, B, inputs=A * np.array([1, 2, 1]))
        with pytest.raises(ValueError, match="column 0 of target has norm"):
            Loss(kind, B * 0.5, inputs=A)
        with pytest.raises(ValueError, match="ancillas are an argument"):
            Loss(kind, B, inputs=A, ancillas=[0])
    for kind, tgt in (("hs", np.eye(8)), ("state", np.eye(8)[:, 0]), ("isometry", np.eye(8)[:, :4])):
        with pytest.raises(ValueError, match=f"inputs are an argument of the 'subspace' losses, not of '{kind}'"):
            Loss(kind, tgt, inputs=A)
    # torch tensors are accepted too
    loss = Loss("subspace", torch.as_tensor(B), inputs=torch.as_tensor(A))
    assert np.array_equal(loss.inputs, A) and loss.ancilla_mask == 3


def test_repr_pickle_and_spec_layout():
    A, B = _haar(8, 3, 1), _haar(8, 3, 2)
    loss = Loss("subspace_relphase", B, inputs=A)
    assert repr(loss) == "Loss('subspace_relphase', target(8, 3), inputs(8, 3))"
    back = pickle.loads(pickle.dumps(loss))
    assert back.kind == loss.kind and np.array_equal(back.target, B) and np.array_equal(back.inputs, A)
    assert back.code == loss.code and back(np.eye(8)) == loss(np.eye(8))
    # a state pickled without `inputs` (an older Loss) still loads
    old = Loss("hs", np.eye(4))
    st = old.__getstate__()
    del st["inputs"]
    o2 = Loss.__new__(Loss)
    o2.__setstate__(st)
    assert o2.inputs is None and o2(np.eye(4)) == pytest.approx(0.0)
    # the device spec: B then A, each N x k row-major, and k in ancilla_mask (a CPU tensor stands in for the device)
    spec = loss.spec(torch.float64, "cpu")
    buf = loss._dev[(torch.float64, "cpu")]
    assert spec.kind == L.LOSS_SUBSPACE_RELPHASE and spec.ancilla_mask == 3 and spec.target == buf.data_ptr()
    assert torch.equal(buf, torch.as_tensor(np.concatenate([B.ravel(), A.ravel()])))
