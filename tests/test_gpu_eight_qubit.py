"""8-qubit circuits on the device: `cpf_unitary` (column mode), the state loss and the isometry loss against the float64
oracle, the Adam loop, the bitwise identities of the interpreter and isometry kernels, multi-target state preparation
and end-to-end synthesis with known optima (the GHZ state and the repetition-code encoder, 7 CZ each)."""
import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

import cpflow_b200 as cp
import isometry_ref as R
from cpflow_b200 import _lib as L
from cpflow_b200.engine import Loss, MultiLoss, Program
from cpflow_b200.main import StaticOptions, Synthesize
from cpflow_b200.topology import chain_layer, connected_layer
from oracle import cpflow_oracle as O
from parity_lib import TOL, pen, rel, setup

pytestmark = pytest.mark.gpu
DEV = "cuda"
N = 256
LAYERS = [("chain", chain_layer(8), 9), ("connected", connected_layer(8), 28)]


def _cx_program():
    """A gate list that is not a layered template: CX gates (control and target on register and lane bits), CZ and
    single rotations."""
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


def _rel1(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _angles(B, P, dt, seed):
    return torch.tensor(np.random.default_rng(seed).uniform(0, 2 * np.pi, (B, P)), dtype=dt, device=DEV)


def _psi(seed=7):
    return unitary_group.rvs(N, random_state=seed)[:, 0].copy()


def _W(anc, seed=0):
    return unitary_group.rvs(N, random_state=seed)[:, :2 ** (8 - len(anc))]


# ---------------------------------------------------------------- unitary, state loss, Adam --------------------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("name,layer,K", LAYERS)
def test_unitary_and_state_loss_parity(name, layer, K, dt):
    anz, oanz, ops = setup(8, layer, K, "xyz")
    B = 11
    a = _angles(B, anz.num_angles, dt, K)
    a_o = torch.tensor(a.cpu().numpy().astype(np.float64))
    u = anz.program.unitary(a[:3]).cpu().numpy()
    uo = O.program_unitary_batched(8, ops, a_o[:3]).numpy()
    assert np.abs(u - uo).max() < TOL[dt]
    psi = _psi()
    lo, rg, gr = anz.program.loss_grad(a, Loss("state", psi), pen())
    ol, orr, og = O.loss_and_grad_batched(8, ops, a_o, "state", torch.tensor(psi), oanz.cp_mask, 0.01,
                                          O.make_regularization_function())
    assert rel(lo.cpu().numpy(), ol.numpy()) < TOL[dt] and rel(rg.cpu().numpy(), orr.numpy()) < TOL[dt]
    g, og = gr.cpu().numpy().astype(np.float64), og.numpy()
    assert (np.linalg.norm(g - og, axis=1) / np.linalg.norm(og, axis=1)).max() < TOL[dt]
    if dt == torch.float64:
        T = 15
        res = O.mynimize_repeated(8, ops, "state", torch.tensor(psi), a_o[:4], 0.1, T, oanz.cp_mask, 0.002,
                                  O.make_regularization_function())
        st = anz.program.adam_state(a[:4].clone())
        anz.program.adam_run(st, Loss("state", psi), pen(0.002), 0.1, T)
        assert np.abs(st.best_regloss.cpu().numpy() - np.array([r["regloss"][1].item() for r in res])).max() < 1e-9
    with pytest.raises(L.CpflowError, match="n <= 5"):
        anz.program.loss_grad(a, Loss("hs", np.eye(N)), pen())


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_cx_gate_list_parity(dt):
    prog = _cx_program()
    a = _angles(7, prog.n_params, dt, 5)
    a_o = torch.tensor(a.cpu().numpy().astype(np.float64))
    u = prog.unitary(a).cpu().numpy()
    assert np.abs(u - O.program_unitary_batched(8, prog.ops, a_o).numpy()).max() < TOL[dt]
    mask = torch.zeros(prog.n_params, dtype=torch.uint8)
    mask[-1] = 1                                                       # the CP gate's parameter
    psi = _psi(3)
    lo, rg, gr = prog.loss_grad(a, Loss("state", psi), pen())
    ol, orr, og = O.loss_and_grad_batched(8, prog.ops, a_o, "state", torch.tensor(psi), mask, 0.01,
                                          O.make_regularization_function())
    for x, y in ((lo, ol), (rg, orr), (gr, og)):
        assert _rel1(x.cpu().numpy(), y.numpy()) < TOL[dt]


# ---------------------------------------------------------------- isometry loss --------------------------------------
ISO = [[0, 1, 2, 3, 4, 5, 6, 7], [1, 2, 3, 4, 5, 6, 7], [0, 2, 4, 6, 7], [0, 3, 7]]      # k = 1, 2, 8, 32


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("anc", ISO)
def test_isometry_parity(anc, dt):
    anz, oanz, _ = setup(8, chain_layer(8), 16, "xyz")
    cases = [(anz.program, torch.as_tensor(anz.cp_mask))]
    if len(anc) in (3, 7):
        prog = _cx_program()
        mask = torch.zeros(prog.n_params, dtype=torch.uint8)
        mask[-1] = 1
        cases.append((prog, mask))
    loss = Loss("isometry", _W(anc, len(anc)), ancillas=anc)
    for prog, mask in cases:
        a = _angles(9, prog.n_params, torch.float64, 11) * 1.3 - 2
        lo, rg, gr = prog.loss_grad(a.to(dt).contiguous(), loss, pen(0.002))
        ol, orr, og = R.loss_and_grad_batched(8, prog.ops, a.cpu(), loss.target, anc, mask, 0.002,
                                              O.make_regularization_function())
        for x, y in ((lo, ol), (rg, orr), (gr, og)):
            assert _rel1(x.cpu().numpy(), y.numpy()) < TOL[dt]
        info = prog.launch_plan(9, loss.code, dt)
        assert info["threads_per_sample"] == 32 * 2 ** (8 - len(anc))


def test_isometry_adam_against_reference():
    anc = [0, 4, 5, 6, 7]
    anz, oanz, _ = setup(8, chain_layer(8), 10, "xyz")
    loss = Loss("isometry", _W(anc, 7), ancillas=anc)
    B, T = 4, 15
    a0 = torch.rand(B, anz.num_angles, dtype=torch.float64, generator=torch.Generator().manual_seed(1)) * 6
    st = anz.program.adam_state(a0.to(DEV).clone())
    anz.program.adam_run(st, loss, pen(0.002), 0.1, T)
    params, regloss = R.mynimize_repeated(8, anz.program.ops, loss.target, anc, a0, 0.1, T,
                                          torch.as_tensor(anz.cp_mask), 0.002, O.make_regularization_function())
    assert _rel1(st.best_regloss.cpu().numpy(), regloss[:, 1].numpy()) < 1e-9
    assert _rel1(st.init_regloss.cpu().numpy(), regloss[:, 0].numpy()) < 1e-9
    assert _rel1(st.best_params.cpu().numpy(), params[:, 1].numpy()) < 1e-9


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_single_column_isometry_is_state(dt):
    anz, _, _ = setup(8, chain_layer(8), 10, "xyz")
    psi = _psi(9)
    a = _angles(8, anz.num_angles, dt, 4)
    ri = anz.program.loss_grad(a, Loss("isometry", psi[:, None], ancillas=list(range(8))), pen())
    rs = anz.program.loss_grad(a, Loss("state", psi), pen())
    for x, y in zip(ri, rs):
        assert _rel1(x.cpu().double().numpy(), y.cpu().double().numpy()) < TOL[dt]


# ---------------------------------------------------------------- bitwise identities ---------------------------------
LOSSES = [("state", None), ("isometry", [0, 3, 7]), ("isometry", [1, 2, 3, 4, 5, 6, 7])]


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind,anc", LOSSES)
def test_bitwise_identities(kind, anc, dt):
    anz, _, _ = setup(8, chain_layer(8), 12, "xyz")
    prog = anz.program
    loss = Loss("state", _psi(2)) if kind == "state" else Loss("isometry", _W(anc, 2), ancillas=anc)
    B = 11
    a = _angles(B, anz.num_angles, dt, 8)
    names = ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss", "init_reg")
    one = prog.adam_state(a.clone())
    prog.adam_run(one, loss, pen(0.002), 0.05, 40)
    split = prog.adam_state(a.clone())
    for steps in (1, 12, 27):                                   # step split: step0 = 0, 1, 13
        prog.adam_run(split, loss, pen(0.002), 0.05, steps)
    ws = prog.adam_state(a.clone())
    ws.workspace = torch.empty(prog.workspace_bytes(B, loss.code, dt), dtype=torch.uint8, device=DEV)
    prog.adam_run(ws, loss, pen(0.002), 0.05, 40)
    halves = [prog.adam_state(a[:5].clone()), prog.adam_state(a[5:].clone())]   # batch split
    for h in halves:
        prog.adam_run(h, loss, pen(0.002), 0.05, 40)
    for name in names:
        ref = getattr(one, name)
        assert torch.equal(ref, getattr(split, name)), name
        assert torch.equal(ref, getattr(ws, name)), name
        assert torch.equal(ref, torch.cat([getattr(h, name) for h in halves])), name
    perm = torch.randperm(B, device=DEV)
    lo, rg, gr = prog.loss_grad(a, loss, pen())
    lp, rp, gp = prog.loss_grad(a[perm].contiguous(), loss, pen())
    assert torch.equal(lp, lo[perm]) and torch.equal(rp, rg[perm]) and torch.equal(gp, gr[perm])
    pa = prog.adam_state(a[perm].contiguous())
    prog.adam_run(pa, loss, pen(0.002), 0.05, 40)
    for name in names:
        assert torch.equal(getattr(pa, name), getattr(one, name)[perm]), name


# ---------------------------------------------------------------- multi-target state preparation ---------------------
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_multi_target_state_matches_single_target(monkeypatch, dt):
    anz, _, _ = setup(8, chain_layer(8), 16, "xyz")
    B, T = 29, 4
    rng = np.random.default_rng(8)
    tg = rng.normal(size=(T, N)) + 1j * rng.normal(size=(T, N))
    tg /= np.linalg.norm(tg, axis=1, keepdims=True)
    idx = rng.integers(0, T, B)
    a = _angles(B, anz.num_angles, dt, 3)
    lo, rg, gr = anz.program.loss_grad_multi(a, MultiLoss("state", tg), idx, pen())
    monkeypatch.setenv("CPF_NO_LAYERED", "1")
    for t in range(T):
        sel = np.flatnonzero(idx == t)
        if len(sel) == 0:
            continue
        l1, r1, g1 = anz.program.loss_grad(a[torch.as_tensor(sel, device=DEV)].contiguous(), Loss("state", tg[t]), pen())
        assert _rel1(lo.cpu().numpy()[sel], l1.cpu().numpy()) <= TOL[dt]
        assert _rel1(rg.cpu().numpy()[sel], r1.cpu().numpy()) <= TOL[dt]
        assert _rel1(gr.cpu().numpy()[sel], g1.cpu().numpy()) <= TOL[dt] * 10


def _ghz():
    v = np.zeros(N, dtype=complex)
    v[[0, N - 1]] = 1 / np.sqrt(2)
    return v


def _key(d):
    return (d.cz_count, d.loss, np.asarray(d._cp_data[2]).tobytes(), d.unitary.tobytes())


def test_synthesize_many_state_end_to_end():
    plus, zero = np.array([1, 1]) / np.sqrt(2), np.array([1, 0])
    product = plus
    for q in range(7):
        product = np.kron(product, zero if q % 2 else plus)
    rng = np.random.default_rng(29)
    haar = rng.normal(size=N) + 1j * rng.normal(size=N)
    tg = np.stack([_ghz(), product, haar / np.linalg.norm(haar)])
    labels = ["ghz", "product", "haar"]
    # (the GHZ state is found at K = 7 by 0.5 % of the samples: 20 of 4000 with the seed below)
    opts = cp.StaticOptions(num_cp_gates=7, accepted_num_cz_gates=14, num_samples=4000, num_gd_iterations=600)
    res = cp.synthesize_many(chain_layer(8), tg, opts, loss="state", labels=labels)
    assert len(res) == 3
    for t, r in enumerate(res):
        assert r.label == labels[t] and r.loss_function.kind == "state" and np.allclose(r.loss_function.target, tg[t])
        for d in r.decompositions:
            assert d.label == labels[t] and np.allclose(d.unitary_loss_func.target, tg[t])
            assert d.loss <= opts.target_loss and Loss("state", tg[t])(d.unitary) <= 1e-5
            assert d.cz_count <= opts.accepted_num_cz_gates
    print("synthesize_many 8q state, 4000 samples, K = 7: decompositions per target",
          {labels[t]: len(res[t].decompositions) for t in range(3)})
    assert len(res[0].decompositions) >= 1 and len(res[1].decompositions) >= 1
    alone = cp.synthesize_many(chain_layer(8), tg[:1], opts, loss="state", labels=labels[:1])[0]
    assert [_key(d) for d in alone.decompositions] == [_key(d) for d in res[0].decompositions]


# ---------------------------------------------------------------- known optima ---------------------------------------
def _static_counts(loss, K, samples, steps=600):
    opts = StaticOptions(num_cp_gates=K, accepted_num_cz_gates=2 * K, num_samples=samples,
                         num_gd_iterations=steps, random_seed=0)
    res = Synthesize(chain_layer(8), unitary_loss_func=loss).static(opts, save_results=False)
    return sorted(d.cz_count for d in res.decompositions)


def _encoder():
    """|x>|0...0> -> |x...x> on 8 qubits (repetition code), data qubit 0."""
    W = np.zeros((N, 2), complex)
    W[0, 0] = W[-1, 1] = 1
    return W


# Every circuit that entangles all 8 qubits has at least 7 two-qubit gates, so 7 CZ is optimal for both and 6 CP
# gates cannot reach either target.
@pytest.mark.parametrize("name", ["ghz", "encoder"])
def test_known_optimum_seven_cz(name):
    loss = Loss("state", _ghz()) if name == "ghz" else Loss("isometry", _encoder(), ancillas=list(range(1, 8)))
    samples = 4000
    at = _static_counts(loss, 7, samples)
    print(f"{name}: K = 7, {samples} samples: {at.count(7)} verified at 7 CZ ({100 * at.count(7) / samples:.2f} %), "
          f"{len(at)} verified in all")
    assert at and at[0] == 7
    assert not _static_counts(loss, 6, 1000)
