"""Subspace losses on the device: parity with a float64 autograd reference on both routes, reductions to the isometry
and state kinds, invariances, the fused Adam loop (15 steps, and 300 steps checked at every step), bitwise determinism
and end-to-end synthesis with entangled inputs and planted targets.

The float64 reference is tests/subspace_ref.py's."""
import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

import subspace_ref as S
from cpflow_b200 import ansatz as AZ
from cpflow_b200 import _lib as L
from cpflow_b200.engine import Loss, Penalty, Program
from cpflow_b200.main import StaticOptions, Synthesize, batched_unitary_loss
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
from cpflow_b200.topology import chain_layer, connected_layer, fill_layers
from oracle import cpflow_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {torch.float64: 1e-12, torch.float32: 1e-5}
KINDS = ("subspace", "subspace_relphase")


# ---------------- helpers ----------------
def _penalty(r=0.002):
    pf = make_regularization_function(RegularizationOptions)
    return Penalty("piecewise", r, pf.segments, pf.period)


def _haar(N, k, seed):
    return unitary_group.rvs(N, random_state=seed)[:, :k]


def _AB(n, k, seed):
    return _haar(2 ** n, k, seed), _haar(2 ** n, k, seed + 1000)


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _same(r0, r1, dt):
    for x, y in zip(r0, r1):
        assert _rel(x.cpu().double().numpy(), y.cpu().double().numpy()) < TOL[dt]


def _check(prog, cp_mask, loss, a, dt):
    # penalise every second CP parameter only: a cp_mask that is not the default
    sub = np.asarray(cp_mask, dtype=np.uint8).copy()
    sub[np.flatnonzero(sub)[1::2]] = 0
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", 0.002, pf.segments, pf.period, cp_mask=sub)
    lo, rg, gr = prog.loss_grad(a.to(dt).contiguous(), loss, pen)
    ol, orr, og = S.loss_and_grad_batched(prog.n_qubits, prog.ops, a.cpu().double(), loss.inputs, loss.target,
                                          loss.kind, torch.as_tensor(sub), 0.002, O.make_regularization_function())
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


def _anz(n, K, layer=None):
    return AZ.Ansatz(n, "cp", fill_layers(layer or chain_layer(n), K), "xyz")


PARITY = [(n, k) for n in range(2, 9) for k in (1, 2, 3, 8, 32) if k <= 2 ** n]


# ---------------- parity ----------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k", PARITY)
def test_parity_chain(n, k, kind, dt):
    anz = _anz(n, 2 * n)
    a = torch.rand(5, anz.num_angles, dtype=torch.float64, device=DEV) * 8 - 2
    A, B = _AB(n, k, n + 7 * k)
    _check(anz.program, anz.cp_mask, Loss(kind, B, inputs=A), a, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k", [(3, 3), (4, 2), (5, 8), (6, 3), (7, 8)])
def test_parity_connected(n, k, kind, dt):
    anz = _anz(n, 2 * n, connected_layer(n))
    a = torch.rand(5, anz.num_angles, dtype=torch.float64, device=DEV) * 6
    A, B = _AB(n, k, 20 + n)
    _check(anz.program, anz.cp_mask, Loss(kind, B, inputs=A), a, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k", [(4, 3), (4, 16), (8, 5), (8, 32)])
def test_parity_cx_gate_list(n, k, kind, dt):
    prog, mask = _cx_program(n)
    a = torch.rand(5, prog.n_params, dtype=torch.float64, device=DEV) * 6
    A, B = _AB(n, k, 3)
    _check(prog, mask, Loss(kind, B, inputs=A), a, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,k", [(2, 3), (3, 1), (4, 5), (5, 2), (5, 32)])
def test_parity_kind6_small_on_both_engines(n, k, dt, monkeypatch):
    """Kind 6 on n <= 5 is an HS call: on the Heisenberg-picture kernel (layered template) and, under
    CPF_ENGINE=adjoint, on the state-adjoint kernels."""
    anz = _anz(n, 2 * n)
    a = torch.rand(5, anz.num_angles, dtype=torch.float64, device=DEV) * 6
    A, B = _AB(n, k, 40 + n)
    loss = Loss("subspace", B, inputs=A)
    if not (n == 5 and dt == torch.float64):
        assert anz.program.launch_plan(5, loss.code, dt)["engine"] == 1
    _check(anz.program, anz.cp_mask, loss, a, dt)
    monkeypatch.setenv("CPF_ENGINE", "adjoint")
    assert anz.program.launch_plan(5, loss.code, dt)["engine"] == 0
    _check(anz.program, anz.cp_mask, loss, a, dt)


# ---------------- reductions and invariances ----------------
def _anc(n, k):
    """the first n - log2(k) qubits as ancillas"""
    return list(range(n - (k.bit_length() - 1)))


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,k", [(2, 2), (3, 4), (4, 2), (4, 8), (5, 1), (5, 16), (6, 4), (7, 2), (8, 32)])
def test_basis_inputs_are_the_isometry_kinds(n, k, dt):
    anz = _anz(n, 2 * n)
    anc = _anc(n, k)
    W = _haar(2 ** n, k, 60 + n)
    iso = Loss("isometry", W, ancillas=anc)
    A = np.eye(2 ** n)[:, list(iso.columns)]
    a = (torch.rand(8, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    r_iso = anz.program.loss_grad(a, iso, _penalty())
    r_sub = anz.program.loss_grad(a, Loss("subspace", W, inputs=A), _penalty())
    if n <= 5:
        # the same HS call on a bit-identical V
        for x, y in zip(r_sub, r_iso):
            assert torch.equal(x, y)
    else:
        _same(r_sub, r_iso, dt)
    _same(anz.program.loss_grad(a, Loss("subspace_relphase", W, inputs=A), _penalty()),
          anz.program.loss_grad(a, Loss("isometry_relphase", W, ancillas=anc), _penalty()), dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n", range(2, 9))
def test_single_basis_input_is_the_state_kind(n, dt):
    anz = _anz(n, 2 * n)
    psi = _haar(2 ** n, 1, 70 + n)
    a = (torch.rand(8, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    ref = anz.program.loss_grad(a, Loss("state", psi[:, 0]), _penalty())
    for kind in KINDS:
        _same(anz.program.loss_grad(a, Loss(kind, psi, inputs=np.eye(2 ** n)[:, :1]), _penalty()), ref, dt)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("n,k", [(3, 3), (4, 8), (5, 5), (6, 3), (7, 4), (8, 8)])
def test_invariances(n, k, dt):
    """kind 6 under (A, B) -> (A Q, B Q) for a k x k unitary Q; kind 7 under B -> B D for a diagonal phase matrix D"""
    anz = _anz(n, 2 * n)
    A, B = _AB(n, k, 80 + n)
    Q = _haar(k, k, 5) if k > 1 else np.ones((1, 1))
    D = np.exp(1j * np.random.default_rng(n).uniform(0, 2 * np.pi, k))
    a = (torch.rand(8, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    _same(anz.program.loss_grad(a, Loss("subspace", B @ Q, inputs=A @ Q), _penalty()),
          anz.program.loss_grad(a, Loss("subspace", B, inputs=A), _penalty()), dt)
    _same(anz.program.loss_grad(a, Loss("subspace_relphase", B * D[None, :], inputs=A), _penalty()),
          anz.program.loss_grad(a, Loss("subspace_relphase", B, inputs=A), _penalty()), dt)


def test_batched_unitary_loss_matches_host_formula():
    for n, k in ((4, 3), (6, 5)):
        anz = _anz(n, 6)
        A, B = _AB(n, k, 4)
        a = torch.rand(6, anz.num_angles, dtype=torch.float64, device=DEV) * 6
        U = anz.program.unitary(a)
        for kind in KINDS:
            loss = Loss(kind, B, inputs=A)
            dev = batched_unitary_loss(loss, U)
            assert _rel(dev, np.array([loss(u) for u in U.cpu().numpy()])) < 1e-12
            lo, _, _ = anz.program.loss_grad(a, loss, None)
            assert _rel(lo.cpu().numpy(), dev) < 1e-12


# ---------------- Adam ----------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k", [(3, 3), (6, 5), (8, 4)])
def test_adam_against_reference(n, k, kind):
    anz = _anz(n, 2 * n)
    A, B = _AB(n, k, 7)
    loss = Loss(kind, B, inputs=A)
    nb, T = 4, 15
    a0 = torch.rand(nb, anz.num_angles, dtype=torch.float64) * 6
    st = anz.program.adam_state(a0.to(DEV).clone())
    anz.program.adam_run(st, loss, _penalty(), 0.1, T)
    params, regloss = S.mynimize_repeated(n, anz.program.ops, A, B, kind, a0, 0.1, T, torch.as_tensor(anz.cp_mask),
                                          0.002, O.make_regularization_function())
    assert _rel(st.best_regloss.cpu().numpy(), regloss[:, 1].numpy()) < 1e-9
    assert _rel(st.init_regloss.cpu().numpy(), regloss[:, 0].numpy()) < 1e-9
    assert _rel(st.best_params.cpu().numpy(), params[:, 1].numpy()) < 1e-9


@pytest.mark.parametrize("kind,n,k,engine", [("subspace", 4, 3, 1), ("subspace", 6, 3, 0),
                                             ("subspace_relphase", 3, 5, 0), ("subspace_relphase", 6, 4, 0)])
def test_long_adam_run_every_step(kind, n, k, engine):
    """300 fused Adam steps in float64 with history buffers; at every step the recorded loss plus penalty equals the
    reference's at the recorded angles, and the next recorded angles are the reference Adam update from them."""
    anz = _anz(n, 2 * n)
    A, B = _AB(n, k, 90 + n)
    loss = Loss(kind, B, inputs=A)
    nb, T, lr = 6, 300, 0.05
    assert anz.program.launch_plan(nb, loss.code, torch.float64)["engine"] == engine
    a0 = torch.rand(nb, anz.num_angles, dtype=torch.float64) * 6
    st = anz.program.adam_state(a0.to(DEV).clone(), hist_len=T)
    anz.program.adam_run(st, loss, _penalty(), lr, T)
    hp, hr = st.hist_params.cpu(), st.hist_regloss.cpu()
    regloss, pred = S.adam_replay(n, anz.program.ops, A, B, kind, hp, lr, torch.as_tensor(anz.cp_mask), 0.002,
                                  O.make_regularization_function())
    err_l = (hr - regloss).abs().max().item()
    err_p = (hp[:, 1:] - pred).abs().max().item()
    print(f"{kind} n={n} k={k}: worst |regloss - ref| {err_l:.2e}, worst |theta - ref| {err_p:.2e} over {T} steps")
    assert err_l < 1e-12 and err_p < 1e-10
    assert float(hr[:, -1].max()) < float(hr[:, 0].min()) or float(hr[:, -1].mean()) < float(hr[:, 0].mean())


# ---------------- determinism ----------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,k", [(2, 3), (4, 2), (5, 3), (6, 3), (7, 4), (8, 3), (8, 8)])
def test_bitwise_identities(n, k, kind, dt):
    anz = _anz(n, 12)
    A, B = _AB(n, k, 2)
    loss = Loss(kind, B, inputs=A)
    nb = 11
    a = (torch.rand(nb, anz.num_angles, dtype=torch.float64, device=DEV) * 6).to(dt)
    one = anz.program.adam_state(a.clone())
    anz.program.adam_run(one, loss, _penalty(), 0.05, 40)
    split = anz.program.adam_state(a.clone())
    for steps in (1, 12, 27):
        anz.program.adam_run(split, loss, _penalty(), 0.05, steps)
    ws = anz.program.adam_state(a.clone())
    ws.workspace = torch.empty(anz.program.workspace_bytes(nb, loss.code, dt), dtype=torch.uint8, device=DEV)
    anz.program.adam_run(ws, loss, _penalty(), 0.05, 40)
    for name in ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss"):
        assert torch.equal(getattr(one, name), getattr(split, name)), name
        assert torch.equal(getattr(one, name), getattr(ws, name)), name
    perm = torch.randperm(nb, device=DEV)
    lo, rg, gr = anz.program.loss_grad(a, loss, _penalty())
    lp, rp, gp = anz.program.loss_grad(a[perm].contiguous(), loss, _penalty())
    assert torch.equal(lp, lo[perm]) and torch.equal(rp, rg[perm]) and torch.equal(gp, gr[perm])
    l1, r1, g1 = anz.program.loss_grad(a[5:6].contiguous(), loss, _penalty())
    assert torch.equal(l1, lo[5:6]) and torch.equal(r1, rg[5:6]) and torch.equal(g1, gr[5:6])
    l2, r2, g2 = anz.program.loss_grad(a[3:9].contiguous(), loss, _penalty())
    assert torch.equal(l2, lo[3:9]) and torch.equal(g2, gr[3:9])


# ---------------- end to end ----------------
def _static_counts(layer, loss, K, samples, steps=1000):
    opts = StaticOptions(num_cp_gates=K, accepted_num_cz_gates=2 * K, num_samples=samples,
                         num_gd_iterations=steps, random_seed=0)
    res = Synthesize(layer, unitary_loss_func=loss).static(opts, save_results=False)
    counts = sorted(d.cz_count for d in res.decompositions)
    hist = {c: counts.count(c) for c in sorted(set(counts))}
    print(f"{loss!r} K={K} samples={samples}: verified decompositions per CZ count {hist}")
    return counts


def _repetition_hadamard(n):
    """(A, B): |0^n>, |1^n> and GHZ+, GHZ- (the logical Hadamard of the n-qubit repetition code)"""
    N = 2 ** n
    A = np.zeros((N, 2))
    A[0, 0] = A[N - 1, 1] = 1
    B = np.zeros((N, 2))
    B[0, :] = 2 ** -0.5
    B[N - 1, 0], B[N - 1, 1] = 2 ** -0.5, -2 ** -0.5
    return A, B


@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("n,samples", [(3, 500), (6, 1000)])
def test_repetition_code_logical_hadamard(n, samples, inverse):
    """Decode (n - 1 CX), H, encode (n - 1 CX) is a construction with 2(n - 1) CZ.  On a chain its CX run along the
    chain and back, so in the chain template's gate order it needs (n - 1)^2 + 1 CP gates.  The inverse map is the same
    kind-6 objective: B = A H for the 2 x 2 Hadamard H, and (A, A H) -> (A H, A) is the (A, B) -> (A Q, B Q) invariance
    with Q = H.  It adds no new problem; it checks that invariance end to end through static().  On a B200 (seed 0) the
    best verified counts were 3 CZ on 3 qubits (241 of 500 samples) and 10 CZ on 6 qubits (2 of 1000 samples), for the
    map and for its inverse alike."""
    A, B = _repetition_hadamard(n)
    loss = Loss("subspace", A, inputs=B) if inverse else Loss("subspace", B, inputs=A)
    counts = _static_counts(chain_layer(n), loss, (n - 1) ** 2 + 1, samples)
    assert counts and counts[0] <= 2 * (n - 1)


@pytest.mark.parametrize("n", [6, 8])
def test_planted_target(n):
    """Random angles theta* on the template, a Haar-random A with k = 4 and B = U(theta*) A: the same template verifies
    at least one decomposition.  On a B200, 189 of 200 samples verified on 6 qubits and 114 of 200 on 8.

    Verification projects every CP angle within threshold_cp = 0.2 of 0 or pi onto it and freezes it, so a planted
    CP angle that close makes the planted circuit unreachable by verification.  Such angles are drawn again here.  With
    plain uniform angles, the 8-qubit theta* had two CP angles within 0.2 of pi (0.063 and 0.197 away) and none of
    200 samples verified, in complex64 and complex128 alike, although 101 of them reached the entry filter.  The
    fused Adam run was not the cause: from theta* + noise it converged to loss 0 plus the penalty, and its float64
    best losses over 300 steps equalled those of the oracle's float64 Adam (8 samples, tests/subspace_ref.py) to
    the printed digits."""
    K = n
    anz = _anz(n, K)
    rng = np.random.default_rng(n)
    th = rng.uniform(0, 2 * np.pi, anz.num_angles)
    cp = np.flatnonzero(anz.cp_mask)
    while True:
        near = cp[np.min(np.abs(th[cp, None] - np.array([0, np.pi, 2 * np.pi])), axis=1) < 0.3]
        if not near.size:
            break
        th[near] = rng.uniform(0, 2 * np.pi, near.size)
    theta = torch.tensor(th[None], device=DEV)
    U = anz.program.unitary(theta)[0].cpu().numpy()
    A = _haar(2 ** n, 4, 100 + n)
    loss = Loss("subspace", U @ A, inputs=A)
    assert loss(U) == pytest.approx(0.0, abs=1e-12)
    opts = StaticOptions(num_cp_gates=K, accepted_num_cz_gates=2 * K, num_samples=200, num_gd_iterations=1000,
                         random_seed=0)
    res = Synthesize(chain_layer(n), unitary_loss_func=loss).static(opts, save_results=False)
    print(f"planted n={n}: {len(res.decompositions)} of 200 samples verified")
    assert res.decompositions
