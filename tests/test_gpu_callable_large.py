"""Callable losses on 6-8 qubits on the device: `cpf_adjoint_from_cotangent` (the cotangent mode of the isometry kernel)
against float64 autograd through the oracle's unitary, its consistency with the fused state and isometry gradients,
bitwise determinism, the shared-memory fallback to fewer columns per launch item, the host-driven Adam loop against
the oracle and against the fused kernels (chunked and unchunked), and a known optimum found end to end by `static()`
with a callable HS loss, followed by `refine()`."""
import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

import isometry_ref as R
from cpflow_b200 import _lib as L
from cpflow_b200.engine import Loss, Program, TorchLoss
from cpflow_b200.main import StaticOptions, Synthesize
from cpflow_b200.optimization import run_adam_batch
from cpflow_b200.topology import chain_layer, connected_layer
from oracle import cpflow_oracle as O
from parity_lib import TOL, pen, rel, setup

pytestmark = pytest.mark.gpu
DEV = "cuda"
CDT = {torch.float32: torch.complex64, torch.float64: torch.complex128}


def _cx_program():
    """The 8-qubit gate list of test_gpu_eight_qubit.py: CX gates on register and lane bits, CZ, single rotations and
    one CP gate."""
    ops, p = [], 0
    for q in range(8):
        for kind in (L.RZ, L.RY):
            ops.append((kind, q, -1, p, 0.0)); p += 1
    for q in range(7):
        ops.append((L.CX, q, q + 1, -1, 0.0))
        ops.append((L.RX, q + 1, -1, p, 0.0)); p += 1
        ops.append((L.CZ, 0, q + 1, -1, 0.0))
    ops.append((L.CX, 7, 0, -1, 0.0))
    ops.append((L.CP, 6, 1, p, 0.0)); p += 1
    return Program(8, ops, p)


def _template(n, layer, K):
    anz, _, ops = setup(n, layer, K, "xyz")
    return anz.program, ops


PROGRAMS = {
    "chain6": lambda: _template(6, chain_layer(6), 9),
    "connected6": lambda: _template(6, connected_layer(6), 17),
    "chain7": lambda: _template(7, chain_layer(7), 8),
    "chain8": lambda: _template(8, chain_layer(8), 9),
    "cx8": lambda: (lambda p: (p, p.ops))(_cx_program()),
}


def _angles(B, P, dt, seed):
    return torch.tensor(np.random.default_rng(seed).uniform(0, 2 * np.pi, (B, P)), dtype=dt, device=DEV)


def _cot(B, N, dt, seed):
    rng = np.random.default_rng(seed)
    c = (rng.normal(size=(B, N, N)) + 1j * rng.normal(size=(B, N, N))) / np.sqrt(2 * N)
    return torch.tensor(c, dtype=CDT[dt], device=DEV)


def _autograd_vjp(n, ops, a, cot):
    """grad = 2 Re <cot, dU/dtheta> in float64 through the oracle's unitary."""
    at = torch.tensor(a.cpu().numpy().astype(np.float64), requires_grad=True)
    U = O.program_unitary_batched(n, ops, at)
    (2 * (torch.tensor(cot.cpu().numpy().astype(np.complex128)).conj() * U).real.sum()).backward()
    return at.grad.numpy()


# ---------------------------------------------------------------- VJP parity -----------------------------------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("name", list(PROGRAMS))
def test_vjp_parity(name, dt):
    prog, ops = PROGRAMS[name]()
    n, N = prog.n_qubits, prog.dim
    B = 5 if n == 8 else 7
    a = _angles(B, prog.n_params, dt, 11)
    cot = _cot(B, N, dt, 12)
    g = prog.adjoint_from_cotangent(a, cot).cpu().numpy().astype(np.float64)
    assert rel(g, _autograd_vjp(n, ops, a, cot)) < TOL[dt] * 3


# ---------------------------------------------------------------- consistency with the fused kernels ----------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("name", ["chain6", "chain7", "chain8", "cx8"])
def test_state_seed_gives_the_state_gradient(name, dt):
    prog, _ = PROGRAMS[name]()
    N = prog.dim
    a = _angles(9, prog.n_params, dt, 3)
    psi = unitary_group.rvs(N, random_state=5)[:, 0]
    _, _, gr = prog.loss_grad(a, Loss("state", psi), None)
    U = prog.unitary(a)
    pt = torch.tensor(psi, dtype=CDT[dt], device=DEV)
    t = (pt.conj()[None] * U[:, :, 0]).sum(-1)
    seed = torch.zeros_like(U)
    seed[:, :, 0] = -t[:, None] * pt[None]                 # dL/dconj(U) of L = 1 - |<psi|U e_0>|^2
    g = prog.adjoint_from_cotangent(a, seed.contiguous())
    assert rel(g.cpu().numpy(), gr.cpu().numpy()) < TOL[dt] * 5


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("name,anc", [("chain6", [0, 2]), ("connected6", [5]), ("chain7", [1, 3, 4])])
def test_isometry_seed_gives_the_isometry_gradient(name, anc, dt):
    prog, _ = PROGRAMS[name]()
    n, N = prog.n_qubits, prog.dim
    k = 2 ** (n - len(anc))
    W = unitary_group.rvs(N, random_state=9)[:, :k]
    a = _angles(9, prog.n_params, dt, 4)
    _, _, gr = prog.loss_grad(a, Loss("isometry", W, ancillas=anc), None)
    U = prog.unitary(a)
    cols = R.columns(n, anc)
    Wt = torch.tensor(W, dtype=CDT[dt], device=DEV)
    t = (Wt.conj()[None] * U[:, :, cols]).sum((-1, -2))
    seed = torch.zeros_like(U)
    seed[:, :, cols] = -(t / k ** 2)[:, None, None] * Wt[None]
    g = prog.adjoint_from_cotangent(a, seed.contiguous())
    assert rel(g.cpu().numpy(), gr.cpu().numpy()) < TOL[dt] * 5


# ---------------------------------------------------------------- determinism ----------------------------------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("name", ["chain6", "chain7", "chain8"])
def test_bitwise_determinism(name, dt):
    prog, _ = PROGRAMS[name]()
    B = 37
    a = _angles(B, prog.n_params, dt, 21)
    cot = _cot(B, prog.dim, dt, 22)
    g = prog.adjoint_from_cotangent(a, cot)
    assert torch.equal(g, prog.adjoint_from_cotangent(a, cot))
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(0)).to(DEV)
    assert torch.equal(prog.adjoint_from_cotangent(a[perm].contiguous(), cot[perm].contiguous()), g[perm])
    split = torch.cat([prog.adjoint_from_cotangent(a[:5].contiguous(), cot[:5].contiguous()),
                       prog.adjoint_from_cotangent(a[5:].contiguous(), cot[5:].contiguous())])
    assert torch.equal(split, g)


# ---------------------------------------------------------------- shared-memory fallback -----------------------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_large_program_uses_fewer_columns_per_item(dt):
    """chain_layer(6) with 120 CP gates: in complex128 the store of a 32-column item does not fit 227 KB (the
    isometry kernel's plan for k = 32 says so) and the call runs 16 columns per item; complex64 runs 32."""
    n, K = 6, 120
    prog, ops = _template(n, chain_layer(n), K)
    smem32 = prog.launch_plan(1, L.isometry_kind(1), dt)["smem_bytes"]           # k = 32
    smem16 = prog.launch_plan(1, L.isometry_kind(3), dt)["smem_bytes"]           # k = 16
    if dt == torch.float64:
        assert smem32 > 227 * 1024 >= smem16
    else:
        assert smem32 <= 227 * 1024
    a = _angles(3, prog.n_params, dt, 31)
    cot = _cot(3, prog.dim, dt, 32)
    g = prog.adjoint_from_cotangent(a, cot)
    assert rel(g.cpu().numpy().astype(np.float64), _autograd_vjp(n, ops, a, cot)) < TOL[dt] * 3
    assert torch.equal(prog.adjoint_from_cotangent(a[1:].contiguous(), cot[1:].contiguous()), g[1:])


# ---------------------------------------------------------------- host-driven loop -----------------------------------
def _hs_callable(V):
    V = torch.as_tensor(V)
    N = V.shape[0]

    def hs(u):
        return 1 - torch.abs((u * V.to(u.device, u.dtype).conj()).sum()) ** 2 / N ** 2
    return hs


def test_host_loop_against_the_oracle():
    n, layer, K = 6, chain_layer(6), 9
    anz, oanz, ops = setup(n, layer, K, "xyz")
    V = unitary_group.rvs(64, random_state=2)
    a0 = _angles(6, anz.num_angles, torch.float64, 41)
    T = 15
    call = run_adam_batch(anz.program, TorchLoss(_hs_callable(V)), pen(0.002), a0, 0.1, T)
    res = O.mynimize_repeated(n, ops, "hs", torch.tensor(V), a0.cpu(), 0.1, T, oanz.cp_mask, 0.002,
                              O.make_regularization_function())
    obr = np.array([r["regloss"][1].item() for r in res])
    assert np.abs(call.regloss[:, 1].cpu().numpy() - obr).max() < 1e-9


def _state_callable(psi):
    psi = torch.as_tensor(psi)
    return lambda u: 1 - torch.abs((psi.to(u.device, u.dtype).conj() * u[:, 0]).sum()) ** 2


def _iso_callable(W, cols):
    W = torch.as_tensor(W)
    k = W.shape[1]
    return lambda u: 1 - torch.abs((W.to(u.device, u.dtype).conj() * u[:, cols]).sum()) ** 2 / k ** 2


@pytest.mark.parametrize("case", ["state7", "state8", "iso6"])
def test_host_loop_equals_the_fused_path(case):
    n = {"state7": 7, "state8": 8, "iso6": 6}[case]
    prog, _ = _template(n, chain_layer(n), 7)
    N = prog.dim
    if case == "iso6":
        anc = [0, 2, 3, 5]                                                      # k = 4
        W = unitary_group.rvs(N, random_state=6)[:, :4]
        fused_loss, fn = Loss("isometry", W, ancillas=anc), _iso_callable(W, R.columns(n, anc))
    else:
        psi = unitary_group.rvs(N, random_state=6)[:, 0]
        fused_loss, fn = Loss("state", psi), _state_callable(psi)
    a0 = _angles(7, prog.n_params, torch.float64, 51)
    T, tol = 40, 1e-9
    fused = run_adam_batch(prog, fused_loss, pen(0.002), a0, 0.1, T)
    call = run_adam_batch(prog, TorchLoss(fn), pen(0.002), a0, 0.1, T)
    assert float((fused.regloss - call.regloss).abs().max()) < tol
    assert float((fused.reg - call.reg).abs().max()) < tol
    assert float((fused.params - call.params).abs().max()) < tol * 50
    chunked = run_adam_batch(prog, TorchLoss(fn), pen(0.002), a0, 0.1, T, chunk=3)
    assert float((chunked.regloss - call.regloss).abs().max()) < 1e-12
    assert float((chunked.params - call.params).abs().max()) < 1e-10


# ---------------------------------------------------------------- known optimum end to end ---------------------------
def _cx_staircase(n=6):
    """cx(0,1) then cx(1,2) ... cx(n-2,n-1), big-endian (qubit 0 is the most significant bit)."""
    N = 2 ** n
    U = np.zeros((N, N), complex)
    for x in range(N):
        bits = [(x >> (n - 1 - q)) & 1 for q in range(n)]
        for q in range(n - 1):
            bits[q + 1] ^= bits[q]
        U[sum(b << (n - 1 - q) for q, b in enumerate(bits)), x] = 1
    return U


def _static(K, samples):
    opts = StaticOptions(num_cp_gates=K, accepted_num_cz_gates=2 * K, num_samples=samples, num_gd_iterations=600,
                         random_seed=0)
    syn = Synthesize(chain_layer(6), unitary_loss_func=_hs_callable(_cx_staircase()))
    assert isinstance(syn.unitary_loss_func, TorchLoss)
    return syn.static(opts, save_results=False)


def test_cx_staircase_known_optimum():
    """Every cut of the chain separates qubits the staircase entangles, so it needs 5 CZ on chain_layer(6)."""
    samples = 1000
    res = _static(5, samples)
    at = sorted(d.cz_count for d in res.decompositions)
    print(f"cx staircase, 6 qubits, K = 5, {samples} samples: {at.count(5)} verified at 5 CZ "
          f"({100 * at.count(5) / samples:.1f} %)")
    assert at and at[0] == 5
    d = min(res.decompositions, key=lambda d: d.cz_count)
    assert d.loss < 1e-5
    assert isinstance(d.refine(), str)
    assert d.unitary_loss_func(d.circuit.unitary()) < 1e-5
    assert not _static(4, samples).decompositions
