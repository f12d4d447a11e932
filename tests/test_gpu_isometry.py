"""Isometry loss on the device: parity with the float64 reference (tests/isometry_ref.py), the fused Adam loop, the
bitwise identities of both paths (n <= 5: the HS kernels on the scaled, padded target; n = 6, 7: the isometry kernel)
and end-to-end synthesis with known optima."""
import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

import isometry_ref as R
from cpflow_b200 import ansatz as A
from cpflow_b200 import _lib as L
from cpflow_b200.engine import Loss, Penalty, Program, clean_ancilla_isometry
from cpflow_b200.main import StaticOptions, Synthesize
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
from cpflow_b200.topology import chain_layer, fill_layers
from oracle import cpflow_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {torch.float64: 1e-12, torch.float32: 1e-5}


def _penalty(r=0.002):
    pf = make_regularization_function(RegularizationOptions)
    return Penalty("piecewise", r, pf.segments, pf.period)


def _W(n, anc, seed=0):
    k = 2 ** (n - len(anc))
    return unitary_group.rvs(2 ** n, random_state=seed)[:, :k]


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _check(prog, cp_mask, loss, a, dt):
    lo, rg, gr = prog.loss_grad(a.to(dt).contiguous(), loss, _penalty())
    ol, orr, og = R.loss_and_grad_batched(prog.n_qubits, prog.ops, a.cpu().double(), loss.target, loss.ancillas,
                                          torch.as_tensor(cp_mask), 0.002, O.make_regularization_function())
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
        ops.append((L.CZ, 0, q + 1, -1, 0.0))
    return Program(n, ops, p), np.zeros(p, dtype=np.uint8)


PARITY = [(3, [1]), (3, [0, 2]), (4, [0, 3]), (4, [3]), (5, [0]), (5, [1, 4]), (6, [0]), (6, [0, 3]), (6, [5]),
          (7, [0, 6]), (7, [1, 2, 4]), (7, [0, 1, 2, 3, 4, 5, 6])]


@pytest.mark.parametrize("engine", ["default", "adjoint"])
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", PARITY)
def test_parity_layered(monkeypatch, n, anc, dt, engine):
    if engine == "adjoint":
        if n > 5:
            pytest.skip("one engine on 6-7 qubits")
        monkeypatch.setenv("CPF_ENGINE", "adjoint")
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    a = torch.rand(9, anz.num_angles, dtype=torch.float64, device=DEV) * 8 - 2
    _check(anz.program, anz.cp_mask, Loss("isometry", _W(n, anc), ancillas=anc), a, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", [(4, [2]), (6, [1, 4]), (7, [0, 3])])
def test_parity_cx_gate_list(n, anc, dt):
    prog, mask = _cx_program(n)
    a = torch.rand(5, prog.n_params, dtype=torch.float64, device=DEV) * 6
    _check(prog, mask, Loss("isometry", _W(n, anc, 3), ancillas=anc), a, dt)


@pytest.mark.parametrize("n,anc", [(4, [0, 2]), (6, [0, 5])])
def test_adam_against_reference(n, anc):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    loss = Loss("isometry", _W(n, anc, 7), ancillas=anc)
    B, T = 6, 15
    a0 = torch.rand(B, anz.num_angles, dtype=torch.float64) * 6
    freeze = torch.zeros(B, anz.num_angles, dtype=torch.bool)
    freeze[::2, ::5] = True
    for fr in (None, freeze):
        st = anz.program.adam_state(a0.to(DEV).clone(), freeze=None if fr is None else fr.to(DEV, torch.uint8))
        anz.program.adam_run(st, loss, _penalty(), 0.1, T)
        params, regloss = R.mynimize_repeated(n, anz.program.ops, loss.target, anc, a0, 0.1, T,
                                              torch.as_tensor(anz.cp_mask), 0.002, O.make_regularization_function(),
                                              freeze_mask=fr)
        assert _rel(st.best_regloss.cpu().numpy(), regloss[:, 1].numpy()) < 1e-9
        assert _rel(st.init_regloss.cpu().numpy(), regloss[:, 0].numpy()) < 1e-9
        assert _rel(st.best_params.cpu().numpy(), params[:, 1].numpy()) < 1e-9


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [3, 4, 5])
def test_small_is_hs_bitwise(n, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    a = (torch.rand(20, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    V = unitary_group.rvs(2 ** n, random_state=4)
    r0 = anz.program.loss_grad(a, Loss("isometry", V, ancillas=[]), _penalty())
    r1 = anz.program.loss_grad(a, Loss("hs", V), _penalty())
    assert all(torch.equal(x, y) for x, y in zip(r0, r1))
    anc = [0, n - 1]
    loss = Loss("isometry", _W(n, anc, 5), ancillas=anc)
    Vp = np.zeros((2 ** n, 2 ** n), complex)
    Vp[:, list(loss.columns)] = 4 * loss.target                # 2^a with a = 2 ancillas
    r0 = anz.program.loss_grad(a, loss, _penalty())
    r1 = anz.program.loss_grad(a, Loss("hs", Vp), _penalty())
    assert all(torch.equal(x, y) for x, y in zip(r0, r1))
    s0, s1 = anz.program.adam_state(a.clone()), anz.program.adam_state(a.clone())
    anz.program.adam_run(s0, loss, _penalty(), 0.1, 30)
    anz.program.adam_run(s1, Loss("hs", Vp), _penalty(), 0.1, 30)
    assert torch.equal(s0.best_params, s1.best_params) and torch.equal(s0.best_regloss, s1.best_regloss)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,anc", [(6, [0]), (7, [0, 3]), (7, [2, 3, 4, 5])])
def test_large_bitwise_identities(n, anc, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 12), "xyz")
    loss = Loss("isometry", _W(n, anc, 2), ancillas=anc)
    B = 11
    a = (torch.rand(B, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    one = anz.program.adam_state(a.clone())
    anz.program.adam_run(one, loss, _penalty(), 0.05, 40)
    split = anz.program.adam_state(a.clone())
    for steps in (1, 12, 27):
        anz.program.adam_run(split, loss, _penalty(), 0.05, steps)
    for name in ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss"):
        assert torch.equal(getattr(one, name), getattr(split, name)), name
    perm = torch.randperm(B, device=DEV)
    lo, rg, gr = anz.program.loss_grad(a, loss, _penalty())
    lp, rp, gp = anz.program.loss_grad(a[perm].contiguous(), loss, _penalty())
    assert torch.equal(lp, lo[perm]) and torch.equal(rp, rg[perm]) and torch.equal(gp, gr[perm])
    l1, r1, g1 = anz.program.loss_grad(a[5:6].contiguous(), loss, _penalty())
    assert torch.equal(l1, lo[5:6]) and torch.equal(g1, gr[5:6])


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", [6, 7])
def test_single_column_is_state(n, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 10), "xyz")
    psi = _W(n, [], 9)[:, 0]
    a = (torch.rand(8, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    ri = anz.program.loss_grad(a, Loss("isometry", psi[:, None], ancillas=list(range(n))), _penalty())
    rs = anz.program.loss_grad(a, Loss("state", psi), _penalty())
    for x, y in zip(ri, rs):
        assert _rel(x.cpu().double().numpy(), y.cpu().double().numpy()) < TOL[dt]


def _encoder(n):
    """|x>|0...0> -> |x...x> (repetition code), data qubit 0."""
    W = np.zeros((2 ** n, 2), complex)
    W[0, 0] = W[-1, 1] = 1
    return W


def _fanout(n, pairs):
    data = [p[0] for p in pairs]
    anc = [p[1] for p in pairs]
    k = 2 ** len(data)
    W = np.zeros((2 ** n, k), complex)
    for c in range(k):
        row = 0
        for i, (d, a) in enumerate(pairs):
            bit = (c >> (len(pairs) - 1 - i)) & 1
            row |= bit << (n - 1 - d) | bit << (n - 1 - a)
        W[row, c] = 1
    return W, anc


def _static_counts(layer, loss, K, samples=2000, steps=600):
    opts = StaticOptions(num_cp_gates=K, accepted_num_cz_gates=2 * K, num_samples=samples,
                         num_gd_iterations=steps, random_seed=0)
    res = Synthesize(layer, unitary_loss_func=loss).static(opts, save_results=False)
    return sorted(d.cz_count for d in res.decompositions)


@pytest.mark.parametrize("n", [4, 7])
def test_encoder_known_optimum(n):
    loss = Loss("isometry", _encoder(n), ancillas=list(range(1, n)))
    at = _static_counts(chain_layer(n), loss, n - 1)
    assert at and at[0] == n - 1
    below = _static_counts(chain_layer(n), loss, n - 2)
    assert not below


def test_fanout_known_optimum():
    pairs = [[0, 3], [1, 4], [2, 5]]
    W, anc = _fanout(6, pairs)
    loss = Loss("isometry", W, ancillas=anc)
    at = _static_counts(pairs, loss, 3)
    assert at and at[0] == 3
    assert not _static_counts(pairs, loss, 2)


def test_clean_ancilla_helper_on_device():
    G = unitary_group.rvs(4, random_state=3)
    W = clean_ancilla_isometry(G, [1], 3)
    loss = Loss("isometry", W, ancillas=[1])
    anz = A.Ansatz(3, "cp", fill_layers(chain_layer(3), 4), "xyz")
    a = torch.rand(4, anz.num_angles, dtype=torch.float64, device=DEV)
    lo, _, _ = anz.program.loss_grad(a, loss, None)
    U = anz.program.unitary(a).cpu().numpy()
    assert _rel(lo.cpu().numpy(), np.array([loss(u) for u in U])) < 1e-12
