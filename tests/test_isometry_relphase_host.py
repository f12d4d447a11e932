"""Relative-phase isometry loss, host side: ABI symbols, the rejections that happen before any device work, the launch
geometry and cost queries, and the host formula and shape checks of Loss('isometry_relphase')."""
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.engine import Loss, clean_ancilla_isometry
from cpflow_b200.topology import chain_layer, fill_layers

# register bits of the single-column kernels on n = 2..8 (inst_f32.cu / inst_f64.cu: engine_rb(n, true))
SINGLE_RB = {2: 2, 3: 2, 4: 1, 5: 1, 6: 2, 7: 2, 8: 3}


def _chain(n, K):
    return Ansatz(n, "cp", fill_layers(chain_layer(n), K)).program


def _spec(mask, ptr=1):
    return L.CpfLossSpec(L.LOSS_ISOMETRY_RELPHASE, ptr, mask)


def _rand_unitary(N, seed):
    rng = np.random.default_rng(seed)
    return np.linalg.qr(rng.normal(size=(N, N)) + 1j * rng.normal(size=(N, N)))[0]


def test_symbols_and_macro():
    assert L.LOSS_ISOMETRY_RELPHASE == 5
    assert L.isometry_relphase_kind(0) == 5
    assert L.isometry_relphase_kind(0b101) == 5 | (5 << 8)
    assert L.isometry_relphase_kind(0xff) == 5 | (0xff << 8)
    assert L.load().cpf_version() == 200
    W = np.zeros((8, 4))
    assert Loss("isometry_relphase", W, ancillas=[1]).code == L.isometry_relphase_kind(0b10)
    assert Loss("isometry", W, ancillas=[1]).code == L.isometry_kind(0b10)


@pytest.mark.parametrize("n,mask,code,words", [
    (4, 1 << 4, -1, "names a qubit >= n"),
    (6, 1 << 6, -1, "names a qubit >= n"),
    (6, 0, -2, "= 64)"),
    (7, 1, -2, "= 64)"),
    (8, 0b11, -2, "= 64)"),
])
def test_rejections_before_device_work(n, mask, code, words):
    prog = _chain(n, 2)
    lib = L.load()
    # fake device pointers: every rejection must come before the library touches them
    assert lib.cpf_loss_grad(prog._h, C.byref(_spec(mask)), None, L.F32, 4, C.c_void_p(16), C.c_void_p(8), None,
                             None, None) == code
    assert words in lib.cpf_last_error().decode()
    buf = L.CpfAdamBuffers(*([8] * 11), 0, 0, 0)
    ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
    assert lib.cpf_adam_run(prog._h, C.byref(_spec(mask)), None, C.byref(ad), L.F32, 4, 0, 5, C.byref(buf),
                            None) == code
    assert words in lib.cpf_last_error().decode()
    b = C.c_int64()
    assert lib.cpf_workspace_bytes(prog._h, L.isometry_relphase_kind(mask), L.F32, 4, C.byref(b)) == code
    assert words in lib.cpf_last_error().decode()


def test_multi_target_table_refused():
    lib = L.load()
    for n in (3, 6):
        prog = _chain(n, 2)
        idx = (C.c_int32 * 2)(0, 0)
        tt = L.CpfTargetTable(L.LOSS_ISOMETRY_RELPHASE, 1, 8, C.cast(idx, C.c_void_p))
        assert lib.cpf_loss_grad_multi(prog._h, C.byref(tt), None, L.F32, 2, C.c_void_p(16), C.c_void_p(8), None,
                                       None, None) == -2
        assert "relative-phase isometry" in lib.cpf_last_error().decode()
        buf = L.CpfAdamBuffers(*([8] * 11), 0, 0, 0)
        ad = L.CpfAdamSpec(0.1, 0.9, 0.999, 1e-8)
        assert lib.cpf_adam_run_multi(prog._h, C.byref(tt), None, C.byref(ad), L.F32, 2, 0, 5, C.byref(buf),
                                      None) == -2
        b = C.c_int64()
        assert lib.cpf_workspace_bytes_multi(prog._h, L.LOSS_ISOMETRY_RELPHASE, L.F32, 2, 1, C.byref(b)) == -2


# (n, ancillas): A = 0 where k <= 32, and k = 1, 2, 8, 32 where n allows
GEOMETRY = [(2, []), (2, [0, 1]), (3, []), (3, [1]), (4, []), (4, [0, 3]), (5, []), (5, [0, 1, 2, 3, 4]),
            (6, [0]), (6, [0, 1, 2, 3]), (6, [1, 2, 3, 4, 5]), (7, [0, 3]), (7, [0, 1, 2, 3]), (7, [1, 2, 3, 4, 5, 6]),
            (8, [0, 4, 7]), (8, [2, 3, 4, 5, 6]), (8, [0, 1, 2, 3, 4, 5, 6, 7])]


@pytest.mark.parametrize("n,anc", GEOMETRY)
def test_launch_plan_geometry(n, anc):
    # (a sample's shared-memory store grows with K, and on 2-3 qubits up to 128 samples share a CTA: K = 2n fits)
    prog = _chain(n, 2 * n)
    k = 2 ** (n - len(anc))
    mask = sum(1 << q for q in anc)
    spt = k * 2 ** (n - SINGLE_RB[n])
    for dt in (L.F32, L.F64):
        info = L.CpfLaunchInfo()
        assert L.load().cpf_launch_plan(prog._h, L.isometry_relphase_kind(mask), dt, 1000, 0, 0, C.byref(info)) == 0
        assert info.engine == 0
        assert info.threads_per_sample == spt
        assert info.samples_per_cta == max(1, 128 // spt)
        assert info.block_threads == info.samples_per_cta * info.threads_per_sample
        assert info.block_threads % 32 == 0
        assert info.block_threads <= info.max_block_threads
        assert info.grid == -(-1000 // info.samples_per_cta)
        assert 0 < info.smem_bytes <= 227 * 1024


@pytest.mark.parametrize("n,anc", [(6, [0]), (6, [2, 5]), (7, [0, 6]), (7, [1, 2, 3, 4, 5, 6]), (8, [0, 1, 2])])
def test_large_queries_equal_isometry(n, anc):
    prog = _chain(n, 12)
    mask = sum(1 << q for q in anc)
    rel, iso = L.isometry_relphase_kind(mask), L.isometry_kind(mask)
    for dtype in (torch.float32, torch.float64):
        assert prog.workspace_bytes(50, rel, dtype) == prog.workspace_bytes(50, iso, dtype)
        assert prog.eval_cost(rel, dtype) == prog.eval_cost(iso, dtype)
        assert prog.executed_cost(rel, dtype) == prog.executed_cost(iso, dtype)
        assert prog.launch_plan(1000, rel, dtype) == prog.launch_plan(1000, iso, dtype)


@pytest.mark.parametrize("n,anc", [(2, []), (3, [1]), (4, []), (5, [0, 4])])
def test_small_workspace_and_cost(n, anc):
    """n <= 5 runs the isometry kernel too: penalty mask plus W packed column by column, C = k in the costs."""
    prog = _chain(n, 6)
    k = 2 ** (n - len(anc))
    mask = sum(1 << q for q in anc)
    for dt, rs in ((L.F32, 4), (L.F64, 8)):
        b = C.c_int64()
        L.check(L.load().cpf_workspace_bytes(prog._h, L.isometry_relphase_kind(mask), dt, 50, C.byref(b)))
        info = L.CpfProgramInfo()
        L.check(L.load().cpf_program_get_info(prog._h, C.byref(info)))
        n_cp = max(1, info.n_phase)
        assert b.value == (n_cp + 255) // 256 * 256 + (2 * k * 2 ** n * rs + 255) // 256 * 256
        f_rel, b_rel = C.c_double(), C.c_double()
        f_st, b_st = C.c_double(), C.c_double()
        L.check(L.load().cpf_eval_cost(prog._h, L.isometry_relphase_kind(mask), dt, C.byref(f_rel), C.byref(b_rel)))
        L.check(L.load().cpf_eval_cost(prog._h, L.LOSS_STATE, dt, C.byref(f_st), C.byref(b_st)))
        assert f_rel.value == pytest.approx(k * f_st.value) and b_rel.value == b_st.value


def _brute(W, anc, U):
    """1 - (1/k) sum_c |<W e_c| U |s_c>|^2 with the s_c enumerated bit by bit."""
    N, k = W.shape
    n = N.bit_length() - 1
    cols = [s for s in range(N) if all(not (s >> (n - 1 - q)) & 1 for q in anc)]
    total = 0.0
    for c, s in enumerate(cols):
        t = sum(np.conj(W[r, c]) * U[r, s] for r in range(N))
        total += abs(t) ** 2
    return 1 - total / k


@pytest.mark.parametrize("n,anc", [(2, []), (3, [1]), (4, [0, 2]), (5, [4]), (6, [0, 1, 2])])
def test_host_formula_against_brute_force(n, anc):
    k = 2 ** (n - len(anc))
    U = _rand_unitary(2 ** n, n)
    W = _rand_unitary(2 ** n, 10 + n)[:, :k]
    loss = Loss("isometry_relphase", W, ancillas=anc)
    assert loss(U) == pytest.approx(_brute(W, anc, U), abs=1e-12)
    # invariant under W -> W D for a diagonal phase matrix D
    D = np.exp(1j * np.random.default_rng(n).uniform(0, 2 * np.pi, k))
    assert Loss("isometry_relphase", W * D[None, :], ancillas=anc)(U) == pytest.approx(loss(U), abs=1e-12)
    # zero at a unitary that maps |s_c> to a phase times W e_c
    V = np.zeros((2 ** n, 2 ** n), complex)
    V[:, list(loss.columns)] = W * D[None, :]
    free = [s for s in range(2 ** n) if s not in loss.columns]
    if free:
        q = np.linalg.qr(np.concatenate([W, _rand_unitary(2 ** n, 3)], axis=1))[0]
        V[:, free] = q[:, k:]
    assert loss(V) == pytest.approx(0.0, abs=1e-12)


def test_equals_relphase_for_permutation_targets():
    rng = np.random.default_rng(5)
    for n in (2, 3, 4, 5):
        N = 2 ** n
        perm = rng.permutation(N)
        V = np.zeros((N, N), complex)
        V[perm, np.arange(N)] = np.exp(1j * rng.uniform(0, 2 * np.pi, N))
        U = _rand_unitary(N, 20 + n)
        assert Loss("isometry_relphase", V, ancillas=[])(U) == pytest.approx(Loss("relphase", V)(U), abs=1e-12)


def test_k1_is_state_and_toffoli_phases():
    rng = np.random.default_rng(2)
    U = _rand_unitary(8, 4)
    psi = _rand_unitary(8, 6)[:, 0]
    assert Loss("isometry_relphase", psi[:, None], ancillas=[0, 1, 2])(U) == pytest.approx(
        Loss("state", psi)(U), abs=1e-12)
    # a Toffoli with a phase on each input column, behind clean ancillas, is an optimum
    tof = np.eye(8)[:, [0, 1, 2, 3, 4, 5, 7, 6]]
    W = clean_ancilla_isometry(tof, [3, 4], 5)
    G = tof * np.exp(1j * rng.uniform(0, 2 * np.pi, 8))[None, :]
    Ug = np.kron(G, np.eye(4))                                   # qubits 3, 4 idle
    assert Loss("isometry_relphase", W, ancillas=[3, 4])(Ug) == pytest.approx(0.0, abs=1e-12)
    assert Loss("isometry", W, ancillas=[3, 4])(Ug) > 1e-3


def test_shape_checks_repr_and_pickle():
    W = np.zeros((8, 4), complex)
    W[0, 0] = 1
    loss = Loss("isometry_relphase", W, ancillas=[1])
    assert loss.columns == (0, 1, 4, 5)
    assert repr(loss) == "Loss('isometry_relphase', target(8, 4), ancillas=[1])"
    back = pickle.loads(pickle.dumps(loss))
    assert back.kind == "isometry_relphase" and back.ancillas == (1,) and np.array_equal(back.target, W)
    assert back.code == loss.code
    with pytest.raises(ValueError, match="needs `ancillas`"):
        Loss("isometry_relphase", W)
    with pytest.raises(ValueError, match="8 x 2"):
        Loss("isometry_relphase", W, ancillas=[0, 1])
    with pytest.raises(ValueError, match="distinct qubits"):
        Loss("isometry_relphase", W, ancillas=[3])
    with pytest.raises(ValueError, match="N = 2"):
        Loss("isometry_relphase", np.zeros((6, 3)), ancillas=[])
    for kind, tgt in (("hs", np.eye(8)), ("state", np.eye(8)[:, 0]), ("relphase", np.eye(8))):
        with pytest.raises(ValueError, match=f"ancillas are an argument of the 'isometry' loss, not of '{kind}'"):
            Loss(kind, tgt, ancillas=[0])
