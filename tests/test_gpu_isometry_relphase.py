"""Relative-phase isometry loss on the device: parity with a float64 autograd reference, the fused Adam loop,
cross-checks with the relphase and isometry kernels, bitwise determinism and end-to-end synthesis with known optima.

The float64 reference, L = 1 - (1/k) sum_c |<W e_c| U |s_c>|^2, is tests/isometry_ref.py's (relphase=True)."""
import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

import isometry_ref as R
from cpflow_b200 import ansatz as A
from cpflow_b200 import _lib as L
from cpflow_b200.engine import Loss, Penalty, Program, clean_ancilla_isometry
from cpflow_b200.gates import u_toff3
from cpflow_b200.main import StaticOptions, Synthesize
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
from cpflow_b200.topology import chain_layer, connected_layer, fill_layers
from oracle import cpflow_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {torch.float64: 1e-12, torch.float32: 1e-5}


# ---------------- helpers ----------------
def _penalty(r=0.002):
    pf = make_regularization_function(RegularizationOptions)
    return Penalty("piecewise", r, pf.segments, pf.period)


def _W(n, anc, seed=0):
    return unitary_group.rvs(2 ** n, random_state=seed)[:, :2 ** (n - len(anc))]


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _anc(n, k):
    """the first n - log2(k) qubits as ancillas"""
    return list(range(n - (k.bit_length() - 1)))


def _check(prog, cp_mask, loss, a, dt):
    # penalise every second CP parameter only: a cp_mask that is not the default
    sub = np.asarray(cp_mask, dtype=np.uint8).copy()
    sub[np.flatnonzero(sub)[1::2]] = 0
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.002, pf.segments, pf.period, cp_mask=sub)
    lo, rg, gr = prog.loss_grad(a.to(dt).contiguous(), loss, pen)
    ol, orr, og = R.loss_and_grad_batched(prog.n_qubits, prog.ops, a.cpu().double(), loss.target, loss.ancillas,
                                          torch.as_tensor(sub), 0.002, O.make_regularization_function(), relphase=True)
    assert float(orr.abs().max()) > 0                               # the penalty takes part
    for x, y in ((lo, ol), (rg, orr), (gr, og)):
        assert _rel(x.cpu().double().numpy(), y.numpy()) < TOL[dt]


def _cx_program(n):
    ops, p = [], 0
    for q in range(n):
        for kind in (L.RZ, L.RY):
            ops.append((kind, q, -1, p, 0.0)); p += 1
    for q in range(n - 1):
        ops.append((L.CX, q, q + 1, -1, 0.0))
        ops.append((L.RX, q + 1, -1, p, 0.0)); p += 1
        ops.append((L.CP, 0, q + 1, p, 0.0)); p += 1
    mask = np.zeros(p, dtype=np.uint8)
    for i, op in enumerate(ops):
        if op[0] == L.CP:
            mask[op[3]] = 1
    return Program(n, ops, p), mask


# k = 1, 2, 8 and 32 where n allows; A = 0 on n <= 5
PARITY = [(n, _anc(n, k)) for n in range(2, 9) for k in (1, 2, 8, 32) if k <= 2 ** n and not (n <= 5 and k == 2 ** n)]
PARITY += [(n, []) for n in range(2, 6)]


# ---------------- parity ----------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", PARITY)
def test_parity_chain(n, anc, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    a = torch.rand(5, anz.num_angles, dtype=torch.float64, device=DEV) * 8 - 2
    _check(anz.program, anz.cp_mask, Loss("isometry_relphase", _W(n, anc, n), ancillas=anc), a, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", [(3, []), (4, [1]), (5, []), (5, [0, 2]), (6, [0]), (6, [1, 2, 3])])
def test_parity_connected(n, anc, dt):
    anz = A.Ansatz(n, "cp", fill_layers(connected_layer(n), 2 * n), "xyz")
    a = torch.rand(5, anz.num_angles, dtype=torch.float64, device=DEV) * 6
    _check(anz.program, anz.cp_mask, Loss("isometry_relphase", _W(n, anc, 20 + n), ancillas=anc), a, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", [(4, []), (4, [2]), (8, [0, 3, 5]), (8, [0, 1, 2, 3, 4, 5, 6])])
def test_parity_cx_gate_list(n, anc, dt):
    prog, mask = _cx_program(n)
    a = torch.rand(5, prog.n_params, dtype=torch.float64, device=DEV) * 6
    _check(prog, mask, Loss("isometry_relphase", _W(n, anc, 3), ancillas=anc), a, dt)


# ---------------- Adam ----------------
@pytest.mark.parametrize("n,anc", [(3, []), (6, [0, 5]), (8, [1, 2, 3, 4, 5])])
def test_adam_against_reference(n, anc):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    loss = Loss("isometry_relphase", _W(n, anc, 7), ancillas=anc)
    B, T = 4, 15
    a0 = torch.rand(B, anz.num_angles, dtype=torch.float64) * 6
    st = anz.program.adam_state(a0.to(DEV).clone())
    anz.program.adam_run(st, loss, _penalty(), 0.1, T)
    params, regloss = R.mynimize_repeated(n, anz.program.ops, loss.target, anc, a0, 0.1, T, torch.as_tensor(anz.cp_mask),
                                          0.002, O.make_regularization_function(), relphase=True)
    assert _rel(st.best_regloss.cpu().numpy(), regloss[:, 1].numpy()) < 1e-9
    assert _rel(st.init_regloss.cpu().numpy(), regloss[:, 0].numpy()) < 1e-9
    assert _rel(st.best_params.cpu().numpy(), params[:, 1].numpy()) < 1e-9


# ---------------- cross-checks with the existing kernels ----------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [3, 4, 5])
def test_permutation_target_is_relphase(n, dt):
    """A = 0 and one unit-modulus entry per column: the relphase kind (full-unitary state-adjoint kernel) computes the
    same loss and gradient."""
    rng = np.random.default_rng(n)
    N = 2 ** n
    V = np.zeros((N, N), complex)
    V[rng.permutation(N), np.arange(N)] = np.exp(1j * rng.uniform(0, 2 * np.pi, N))
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    a = (torch.rand(16, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    r0 = anz.program.loss_grad(a, Loss("isometry_relphase", V, ancillas=[]), _penalty())
    r1 = anz.program.loss_grad(a, Loss("relphase", V), _penalty())
    for x, y in zip(r0, r1):
        assert _rel(x.cpu().double().numpy(), y.cpu().double().numpy()) < TOL[dt]


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [6, 7, 8])
def test_single_column_is_isometry(n, dt):
    """k = 1: the same seed as the isometry kind (t_c = t, k = k^2 = 1), so penalty and gradient are bit-identical;
    the loss is 1 - |t|^2 against the isometry kind's 1 - sqrt(|t|^2)^2."""
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 10), "xyz")
    psi = _W(n, [], 9)[:, :1]
    anc = list(range(n))
    a = (torch.rand(8, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    lr_, rr, gr = anz.program.loss_grad(a, Loss("isometry_relphase", psi, ancillas=anc), _penalty())
    li, ri, gi = anz.program.loss_grad(a, Loss("isometry", psi, ancillas=anc), _penalty())
    assert torch.equal(rr, ri) and torch.equal(gr, gi)
    assert _rel(lr_.cpu().double().numpy(), li.cpu().double().numpy()) < TOL[dt]


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", [(3, [1]), (5, []), (6, [0, 3]), (8, [0, 1, 2, 3])])
def test_column_phases_do_not_matter(n, anc, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    W = _W(n, anc, 11)
    D = np.exp(1j * np.random.default_rng(n).uniform(0, 2 * np.pi, W.shape[1]))
    a = (torch.rand(8, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    r0 = anz.program.loss_grad(a, Loss("isometry_relphase", W, ancillas=anc), _penalty())
    r1 = anz.program.loss_grad(a, Loss("isometry_relphase", W * D[None, :], ancillas=anc), _penalty())
    for x, y in zip(r0, r1):
        assert _rel(x.cpu().double().numpy(), y.cpu().double().numpy()) < TOL[dt]


# ---------------- determinism ----------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", [(2, []), (4, [1]), (5, []), (6, [0]), (7, [0, 3]), (8, [0, 1, 2])])
def test_bitwise_identities(n, anc, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 12), "xyz")
    loss = Loss("isometry_relphase", _W(n, anc, 2), ancillas=anc)
    B = 11
    a = (torch.rand(B, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    one = anz.program.adam_state(a.clone())
    anz.program.adam_run(one, loss, _penalty(), 0.05, 40)
    split = anz.program.adam_state(a.clone())
    for steps in (1, 12, 27):
        anz.program.adam_run(split, loss, _penalty(), 0.05, steps)
    ws = anz.program.adam_state(a.clone())
    ws.workspace = torch.empty(anz.program.workspace_bytes(B, loss.code, dt), dtype=torch.uint8, device=DEV)
    anz.program.adam_run(ws, loss, _penalty(), 0.05, 40)
    for name in ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss"):
        assert torch.equal(getattr(one, name), getattr(split, name)), name
        assert torch.equal(getattr(one, name), getattr(ws, name)), name
    perm = torch.randperm(B, device=DEV)
    lo, rg, gr = anz.program.loss_grad(a, loss, _penalty())
    lp, rp, gp = anz.program.loss_grad(a[perm].contiguous(), loss, _penalty())
    assert torch.equal(lp, lo[perm]) and torch.equal(rp, rg[perm]) and torch.equal(gp, gr[perm])
    l1, r1, g1 = anz.program.loss_grad(a[5:6].contiguous(), loss, _penalty())
    assert torch.equal(l1, lo[5:6]) and torch.equal(r1, rg[5:6]) and torch.equal(g1, gr[5:6])
    l2, r2, g2 = anz.program.loss_grad(a[3:9].contiguous(), loss, _penalty())
    assert torch.equal(l2, lo[3:9]) and torch.equal(g2, gr[3:9])


def test_batched_unitary_loss_matches_host_formula():
    from cpflow_b200.main import batched_unitary_loss
    anz = A.Ansatz(4, "cp", fill_layers(chain_layer(4), 6), "xyz")
    loss = Loss("isometry_relphase", _W(4, [2], 4), ancillas=[2])
    a = torch.rand(6, anz.num_angles, dtype=torch.float64, device=DEV) * 6
    U = anz.program.unitary(a)
    dev = batched_unitary_loss(loss, U)
    assert _rel(dev, np.array([loss(u) for u in U.cpu().numpy()])) < 1e-12
    lo, _, _ = anz.program.loss_grad(a, loss, None)
    assert _rel(lo.cpu().numpy(), dev) < 1e-12


# ---------------- end to end: the relative-phase Toffoli-3 ----------------
def _static_counts(layer, loss, K, samples, steps=1000):
    opts = StaticOptions(num_cp_gates=K, accepted_num_cz_gates=2 * K, num_samples=samples,
                         num_gd_iterations=steps, random_seed=0)
    res = Synthesize(layer, unitary_loss_func=loss).static(opts, save_results=False)
    counts = sorted(d.cz_count for d in res.decompositions)
    hist = {c: counts.count(c) for c in sorted(set(counts))}
    print(f"{loss!r} K={K} samples={samples}: verified decompositions per CZ count {hist}")
    return counts


TRIANGLE = [[0, 1], [0, 2], [1, 2]]


def test_relphase_toffoli3_connected():
    # 6 CP gates in the order 01, 02, 12, 01, 02, 12 contain the Margolus pattern 12, 02, 12.  On a B200, 39 of the
    # 500 samples verified at 3 CZ (7.8 %).
    counts = _static_counts(connected_layer(3), Loss("isometry_relphase", u_toff3, ancillas=[]), 6, 500)
    assert counts and counts[0] <= 3


@pytest.mark.parametrize("n", [6, 8])
def test_relphase_toffoli3_clean_ancillas(n):
    anc = list(range(3, n))
    layer = TRIANGLE + [[q, q + 1] for q in range(2, n - 1)]
    loss = Loss("isometry_relphase", clean_ancilla_isometry(u_toff3, anc, n), ancillas=anc)
    # the triangle, the chain, then the triangle again: 12 (first pass), 02, 12 (second pass) is the Margolus pattern.
    # On a B200, 59 of 1000 samples verified at 3 CZ on 6 qubits (5.9 %) and 34 of 1000 on 8 qubits (3.4 %).
    counts = _static_counts(layer, loss, 3 + (n - 3) + 3, 1000)
    assert counts and counts[0] <= 3


def test_exact_toffoli_not_in_three_gates():
    """Contrast: with 3 CP gates only the data triangle carries entanglers; up to a phase per column the Toffoli fits,
    with one global phase it does not (an exact Toffoli needs at least five two-qubit gates)."""
    n, anc = 6, [3, 4, 5]
    layer = TRIANGLE + [[2, 3], [3, 4], [4, 5]]
    W = clean_ancilla_isometry(u_toff3, anc, n)
    assert not _static_counts(layer, Loss("isometry", W, ancillas=anc), 3, 1000)
