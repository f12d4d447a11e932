"""Multi-target runs on the device (cpf_loss_grad_multi, cpf_adam_run_multi, synthesize_many): every sample must get
what a single-target call on its own target gives on the same kernel family (the runtime-pair Heisenberg kernel,
CPF_HEIS_ANY=1, for HS on block-structured templates; the interpreter kernel, CPF_NO_LAYERED=1, otherwise), and the
results must not depend on how the work is split or laid out."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

import cpflow_b200 as cp
from cpflow_b200 import ansatz as A
from cpflow_b200.engine import Loss, MultiLoss, Penalty
from cpflow_b200.gates import u_toff3, u_toff4
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
from cpflow_b200.topology import chain_layer, connected_layer, fill_layers
from oracle import cpflow_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {torch.float64: 1e-12, torch.float32: 1e-5}
CCZ = np.diag([1, 1, 1, 1, 1, 1, 1, -1]).astype(complex)


def _penalty(r=0.002):
    pf = make_regularization_function(RegularizationOptions)
    return Penalty("piecewise", r, pf.segments, pf.period)


def _targets(kind, n, T, seed=0):
    N = 2 ** n
    rng = np.random.default_rng(seed)
    if kind == "state":
        v = rng.normal(size=(T, N)) + 1j * rng.normal(size=(T, N))
        return v / np.linalg.norm(v, axis=1, keepdims=True)
    return np.stack([unitary_group.rvs(N, random_state=seed * 100 + t) for t in range(T)])


def _single_env(kind):
    return ("CPF_HEIS_ANY", "1") if kind == "hs" else ("CPF_NO_LAYERED", "1")


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


CASES = [(k, n) for k in ("hs", "state", "relphase") for n in (2, 3, 4, 5)] + [("state", 6), ("state", 7)]


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind,n", CASES)
def test_loss_grad_multi_matches_single_target(monkeypatch, kind, n, dt):
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 2 * n), "xyz")
    B, T = 37, 5
    tg = _targets(kind, n, T, seed=n)
    idx = np.random.default_rng(11).integers(0, T, B)
    a = torch.tensor(np.random.default_rng(3).uniform(0, 6.28, (B, anz.num_angles)), dtype=dt, device=DEV)
    pen = _penalty()
    lo, rg, gr = anz.program.loss_grad_multi(a, MultiLoss(kind, tg), idx, pen)
    lo, rg, gr = lo.cpu().numpy(), rg.cpu().numpy(), gr.cpu().numpy()
    monkeypatch.setenv(*_single_env(kind))
    for t in range(T):
        sel = np.flatnonzero(idx == t)
        if len(sel) == 0:
            continue
        l1, r1, g1 = anz.program.loss_grad(a[torch.as_tensor(sel, device=DEV)].contiguous(), Loss(kind, tg[t]), pen)
        assert _rel(lo[sel], l1.cpu().numpy()) <= TOL[dt], (t, kind, n)
        assert _rel(rg[sel], r1.cpu().numpy()) <= TOL[dt]
        assert _rel(gr[sel], g1.cpu().numpy()) <= TOL[dt] * 10
    if dt == torch.float64 and kind != "state" and n <= 4:
        # the oracle's unitary and loss formula for the first samples
        ops = O.ansatz_program(O.cp_ansatz(chain_layer(n), 2 * n))
        U = O.program_unitary_batched(n, ops, torch.tensor(a[:6].cpu().numpy())).numpy()
        for b in range(6):
            assert abs(lo[b] - Loss(kind, tg[idx[b]])(U[b])) < 1e-12


def _adam(anz, init, loss, pen, lr, T, freeze=None, target_index=None, split=None, workspace=False):
    st = anz.program.adam_state(init.clone(), freeze=freeze)
    if workspace:
        n = anz.program.workspace_bytes_multi(st.batch, loss.n_targets, Loss.KINDS[loss.kind], init.dtype)
        st.workspace = torch.empty(n, dtype=torch.uint8, device=DEV)
    for steps in (split or [T]):
        if target_index is None:
            anz.program.adam_run(st, loss, pen, lr, steps)
        else:
            anz.program.adam_run_multi(st, loss, target_index, pen, lr, steps)
    torch.cuda.synchronize()
    return {k: getattr(st, k).cpu().numpy() for k in ("angles", "best_params", "best_regloss", "best_reg",
                                                       "init_regloss", "init_reg", "m", "v")}


@pytest.mark.parametrize("freeze", [False, True])
def test_adam_multi_parity_c3_shape(monkeypatch, freeze):
    """4q chain, K = 40, 3 targets x 32 samples, complex128, 150 steps: each target's samples against a single-target
    run of the same samples on its own target."""
    anz = A.Ansatz(4, "cp", fill_layers(chain_layer(4), 40), "xyz")
    tg = np.stack([u_toff4, unitary_group.rvs(16, random_state=1), unitary_group.rvs(16, random_state=2)])
    S = 32
    init = anz.program.initial_angles(0, 3 * S, dtype=torch.float64)
    idx = np.repeat(np.arange(3), S)
    fr = None
    if freeze:
        fr = torch.zeros(3 * S, anz.num_angles, dtype=torch.uint8, device=DEV)
        fr[:, torch.as_tensor(np.flatnonzero(anz.cp_mask)[::3], device=DEV)] = 1
    pen = _penalty(0.00055)
    many = _adam(anz, init, MultiLoss("hs", tg), pen, 0.1, 150, freeze=fr, target_index=idx)
    monkeypatch.setenv("CPF_HEIS_ANY", "1")
    for t in range(3):
        sl = slice(t * S, (t + 1) * S)
        one = _adam(anz, init[sl].contiguous(), Loss("hs", tg[t]), pen, 0.1, 150,
                    freeze=None if fr is None else fr[sl].contiguous())
        for k in ("init_regloss", "best_regloss", "best_reg", "best_params"):
            assert _rel(many[k][sl], one[k]) < 1e-9, (t, k)
        if freeze:
            assert np.array_equal(many["angles"][sl][:, fr[0].cpu().numpy() > 0],
                                  init[sl].cpu().numpy()[:, fr[0].cpu().numpy() > 0])


@pytest.mark.parametrize("T,tol", [(1, 5e-7), (3, 1e-4)])
def test_adam_multi_parity_c3_shape_f32(monkeypatch, T, tol):
    anz = A.Ansatz(4, "cp", fill_layers(chain_layer(4), 40), "xyz")
    tg = np.stack([u_toff4, unitary_group.rvs(16, random_state=1), unitary_group.rvs(16, random_state=2)])
    S = 32
    init = anz.program.initial_angles(0, 3 * S)
    idx = np.repeat(np.arange(3), S)
    pen = _penalty(0.00055)
    many = _adam(anz, init, MultiLoss("hs", tg), pen, 0.1, T, target_index=idx)
    monkeypatch.setenv("CPF_HEIS_ANY", "1")
    for t in range(3):
        sl = slice(t * S, (t + 1) * S)
        one = _adam(anz, init[sl].contiguous(), Loss("hs", tg[t]), pen, 0.1, T)
        assert _rel(many["init_regloss"][sl], one["init_regloss"]) < 5e-7
        assert _rel(many["best_regloss"][sl], one["best_regloss"]) < tol


def _same(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("kind,dt", [("hs", torch.float32), ("hs", torch.float64), ("state", torch.float32),
                                     ("relphase", torch.float64)])
def test_adam_multi_is_bit_identical_under_reordering_and_splitting(kind, dt):
    n, T = 4, 6
    anz = A.Ansatz(n, "cp", fill_layers(chain_layer(n), 20), "xyz")
    tg = _targets(kind, n, T, seed=5)
    B = 300
    init = anz.program.initial_angles(0, B, dtype=dt)
    idx = np.random.default_rng(1).integers(0, T, B)
    ml, pen = MultiLoss(kind, tg), _penalty()
    ref = _adam(anz, init, ml, pen, 0.05, 40, target_index=idx)
    # permuted samples, index permuted alike
    perm = np.random.default_rng(2).permutation(B)
    got = _adam(anz, init[torch.as_tensor(perm, device=DEV)].contiguous(), ml, pen, 0.05, 40, target_index=idx[perm])
    _same({k: v[np.argsort(perm)] for k, v in got.items()}, ref)
    # the targets split over several calls (each with its own sub-table)
    for group in (np.arange(0, 3), np.arange(3, T)):
        sel = np.flatnonzero(np.isin(idx, group))
        remap = {g: i for i, g in enumerate(group)}
        got = _adam(anz, init[torch.as_tensor(sel, device=DEV)].contiguous(), MultiLoss(kind, tg[group]), pen, 0.05, 40,
                    target_index=np.array([remap[t] for t in idx[sel]]))
        _same(got, {k: v[sel] for k, v in ref.items()})
    # steps split over calls, and a caller-owned workspace
    _same(_adam(anz, init, ml, pen, 0.05, 40, target_index=idx, split=[13, 27]), ref)
    _same(_adam(anz, init, ml, pen, 0.05, 40, target_index=idx, workspace=True), ref)


def test_adam_multi_time_slicing_is_bit_identical(monkeypatch):
    """A batch above one full wave of the Heisenberg kernel, cut into a ring of launches (CPF_HEIS_SLICES)."""
    anz = A.Ansatz(4, "cp", fill_layers(chain_layer(4), 40), "xyz")
    B = 12000
    tg = _targets("hs", 4, 16, seed=9)
    init = anz.program.initial_angles(0, B)
    idx = np.random.default_rng(4).integers(0, 16, B)
    ml, pen = MultiLoss("hs", tg), _penalty(0.00055)
    monkeypatch.setenv("CPF_HEIS_SLICES", "1")
    ref = _adam(anz, init, ml, pen, 0.1, 40, target_index=idx)
    monkeypatch.setenv("CPF_HEIS_SLICES", "2")
    _same(_adam(anz, init, ml, pen, 0.1, 40, target_index=idx), ref)


def _key(d):
    return (d.cz_count, d.loss, np.asarray(d._cp_data[2]).tobytes(), d.unitary.tobytes())


def test_synthesize_many_end_to_end():
    haar = unitary_group.rvs(8, random_state=17)
    tg = np.stack([CCZ, u_toff3, haar])
    labels = ["ccz", "toffoli", "haar"]
    opts = cp.StaticOptions(num_cp_gates=12, accepted_num_cz_gates=14, num_samples=60)
    res = cp.synthesize_many(chain_layer(3), tg, opts, labels=labels)
    assert len(res) == 3
    found = 0
    for t in range(3):
        r = res[t]
        assert r.label == labels[t] and isinstance(r.loss_function, Loss) and r.loss_function.kind == "hs"
        assert np.allclose(r.loss_function.target, tg[t])
        for d in r.decompositions:
            found += 1
            assert d.label == labels[t] and np.allclose(d.unitary_loss_func.target, tg[t])
            assert d.loss <= 1e-5 and Loss("hs", tg[t])(d.unitary) <= 1e-5
            assert d.cz_count <= opts.accepted_num_cz_gates and d._static_options is opts
    assert len(res[0].decompositions) >= 1 and len(res[1].decompositions) >= 1 and found >= 2
    # one target alone gives the same bits as in the group
    alone = cp.synthesize_many(chain_layer(3), tg[1:2], opts, labels=labels[1:2])[0]
    assert [_key(d) for d in alone.decompositions] == [_key(d) for d in res[1].decompositions]


def _state_targets():
    ghz = np.zeros(8, dtype=complex)
    ghz[[0, 7]] = 1 / np.sqrt(2)
    plus, zero = np.array([1, 1]) / np.sqrt(2), np.array([1, 0])
    product = np.kron(np.kron(plus, zero), np.array([np.cos(0.3), np.exp(0.7j) * np.sin(0.3)]))
    rng = np.random.default_rng(23)
    haar = rng.normal(size=8) + 1j * rng.normal(size=8)
    return np.stack([ghz, product, haar / np.linalg.norm(haar)]), ["ghz", "product", "haar"], 2


@pytest.mark.parametrize("kind", ["state", "relphase"])
def test_synthesize_many_end_to_end_state_and_relphase(kind):
    """synthesize_many with the losses that run on InterpSweepMT: every decomposition re-scores below target_loss with
    the single-target loss, labels and targets are carried through, a target alone gives the group's bits."""
    if kind == "state":
        tg, labels, easy = _state_targets()
    else:
        tg, labels, easy = np.stack([u_toff3, CCZ]), ["toffoli", "ccz"], 2
    opts = cp.StaticOptions(num_cp_gates=12, accepted_num_cz_gates=14, num_samples=60)
    res = cp.synthesize_many(chain_layer(3), tg, opts, loss=kind, labels=labels)
    assert len(res) == len(tg)
    for t, r in enumerate(res):
        assert r.label == labels[t] and isinstance(r.loss_function, Loss) and r.loss_function.kind == kind
        assert np.allclose(r.loss_function.target, tg[t])
        for d in r.decompositions:
            assert d.label == labels[t] and np.allclose(d.unitary_loss_func.target, tg[t])
            # the float32 run's own loss passed the filter; the float64 re-score of its angles as in the HS test
            assert d.loss <= opts.target_loss and Loss(kind, tg[t])(d.unitary) <= 1e-5
            assert d.cz_count <= opts.accepted_num_cz_gates and d._static_options is opts
    assert all(len(res[t].decompositions) >= 1 for t in range(easy))
    alone = cp.synthesize_many(chain_layer(3), tg[1:2], opts, loss=kind, labels=labels[1:2])[0]
    assert [_key(d) for d in alone.decompositions] == [_key(d) for d in res[1].decompositions]


def test_synthesize_many_matches_static_statistics():
    """Toffoli-3, all-to-all, 10^4 samples: the share of samples verified at 6 CZ agrees with static() within
    binomial error (same initial batch, trajectories differ only by the kernel family's rounding)."""
    S = 10000
    opts = cp.StaticOptions(num_cp_gates=7, r=0.00131, accepted_num_cz_gates=6, num_samples=S)
    many = cp.synthesize_many(connected_layer(3), np.stack([u_toff3, CCZ]), opts)[0]
    one = cp.Synthesize(connected_layer(3), target_unitary=u_toff3).static(opts, save_results=False)
    p1 = sum(d.cz_count == 6 for d in one.decompositions) / S
    p2 = sum(d.cz_count == 6 for d in many.decompositions) / S
    sigma = np.sqrt(2 * max(p1, 1e-3) * (1 - p1) / S)
    assert 0.1 < p1 < 0.5 and abs(p1 - p2) < 5 * sigma, (p1, p2)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_synthesize_many_is_identical_on_one_and_two_ranks(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    script = os.path.join(ROOT, "tools", "many_ranks.py")
    out = {}
    for world in (1, 2):
        path = str(tmp_path / f"w{world}.json")
        cmd = [sys.executable, script, path] if world == 1 else \
            [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
             "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), script, path]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        out[world] = json.load(open(path))
    assert out[2]["world"] == 2 and out[1]["results"] == out[2]["results"]
    assert sum(len(r) for r in out[1]["results"]) > 0
