"""GPU parity tests: the CUDA engine (through the C ABI, ctypes) against the CPU oracle on the same
seeded inputs, against the committed golden fixtures, and at BASELINE sizes through
size-independent properties.  Tolerances (BASELINE.json north_star): 1e-5 relative in complex64,
1e-12 in complex128; integer / index / PRNG work is bit-exact."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
from scipy.stats import unitary_group

from oracle import cpflow_oracle as O
from conftest import hst
from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.engine import Loss, Penalty, Program
from cpflow_b200.gates import u_toff3, u_toff4
from cpflow_b200.topology import chain_layer, connected_layer, fill_layers

pytestmark = pytest.mark.gpu
DEV = "cuda"
from parity_lib import CONFIGS, KITE4, PF, SQUARE4, STAR4, TOL, measure_adam_loop, measure_loss_grad, pen, rel, setup  # noqa: E402


@pytest.mark.parametrize("n,layer,K,rg", CONFIGS)
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_unitary_loss_grad_parity(n, layer, K, rg, dt):
    """Loss, penalty and gradient of all three losses on a ragged batch of generic angles against the oracle, at
    the contract's tolerance: 1e-5 (complex64) / 1e-12 (complex128).  tools/parity_report.py prints the measured
    maxima of the same function (profiles/parity_r2.txt)."""
    m = measure_loss_grad(n, layer, K, rg, dt)
    tol = TOL[dt]
    assert m["unitary"] < (1e-13 if dt == torch.float64 else 5e-6)
    for kind in ("hs", "relphase", "state"):
        e = m[kind]
        assert e["loss"] < tol and e["reg"] < tol and e["grad"] < tol, (kind, e)
        assert e["loss_only_same_bits"], kind


@pytest.mark.parametrize("layer_name,layer", [("chain", chain_layer(4)), ("star", STAR4)])
@pytest.mark.parametrize("freeze", [False, True])
def test_adam_loop_parity_c3_shape(layer_name, layer, freeze):
    """The kernel the bench times (4 qubits, K = 40, chain and star; HeisSweep) against the oracle's loop over
    T = 150 Adam iterations of 32 samples in complex128: initial / best regloss, best reg, best parameters at 1e-9,
    and the verification variant (projected CP angles frozen, no penalty; cp_utils.py:205-247).  The oracle's
    outputs are the committed fixture tests/golden/adam_c3.npz (make_adam_c3.py; the CPU suite re-derives it)."""
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "adam_c3.npz"))
    expect = {k: z[f"{layer_name}_{int(freeze)}_{k}"] for k in ("init_regloss", "best_regloss", "best_reg", "best_params")}
    m = measure_adam_loop(4, layer, 40, u_toff4, B=32, T=150, freeze=freeze, expect=expect)
    assert m["engine"] == 1, "C3 must run on the Heisenberg kernel"
    assert m["init_regloss"] < 1e-12 and m["best_regloss"] < 1e-9 and m["best_reg"] < 1e-9, m
    assert m["best_params"] < 1e-7, m
    if freeze:
        assert m["frozen_moved"] == 0.0


@pytest.mark.parametrize("T,tol", [(1, 5e-7), (3, 1e-4)])
def test_adam_loop_parity_c3_shape_f32(T, tol):
    """Same kernel in complex64 (the PLAIN instantiation the bench times) against the float32 oracle loop.  Adam's
    first steps move every parameter by ~lr whatever the size of its gradient (update = lr g / (|g| + eps) at step 1),
    so float32 trajectories separate quickly (measured on this case, profiles/grad_accuracy_r2.txt: best-regloss error
    9e-8 after 1 step, 3e-5 after 3, 1e-3 after 6); the complex64 loop is therefore pinned over 1 and 3 iterations
    and the long horizon in complex128 above."""
    m = measure_adam_loop(4, chain_layer(4), 40, u_toff4, B=32, T=T, dt=torch.float32)
    assert m["engine"] == 1
    assert m["init_regloss"] < 5e-7 and m["best_regloss"] < tol and m["best_reg"] < tol, m


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_cotangent_vjp(dt):
    n, layer, K, rg = 4, [[0, 1], [1, 2], [3, 2]], 9, "xyz"
    anz, oanz, ops = setup(n, layer, K, rg)
    B, N = 11, 16
    a = torch.tensor(np.random.default_rng(7).uniform(0, 6.28, (B, anz.num_angles)), dtype=dt, device=DEV)
    cdt = {torch.float32: torch.complex64, torch.float64: torch.complex128}[dt]
    cot = torch.tensor(np.stack([unitary_group.rvs(N, random_state=s) for s in range(B)]), dtype=cdt, device=DEV)
    g = anz.program.adjoint_from_cotangent(a, cot.contiguous()).cpu().numpy()
    at = torch.tensor(a.cpu().numpy().astype(np.float64), requires_grad=True)
    U = O.program_unitary_batched(n, ops, at)
    (2 * (torch.tensor(cot.cpu().numpy().astype(np.complex128)).conj() * U).real.sum()).backward()
    assert rel(g, at.grad.numpy()) < TOL[dt] * 3
    # consistency: HS-loss gradient through the generic entry == built-in loss_grad
    V = unitary_group.rvs(N, random_state=3)
    _, _, gr = anz.program.loss_grad(a, Loss("hs", V), None)
    Ud = anz.program.unitary(a)
    Vt = torch.tensor(V, dtype=cdt, device=DEV)
    t = (Ud * Vt.conj()).sum((-1, -2))
    seed = (-(t / N ** 2)[:, None, None] * Vt[None]).contiguous()   # dL/dconj(U)
    g2 = anz.program.adjoint_from_cotangent(a, seed)
    assert rel(g2.cpu().numpy(), gr.cpu().numpy()) < TOL[dt] * 5


def _oracle_run(n, ops, target, a0, lr, T, cp_mask, r, **kw):
    return O.mynimize_repeated(n, ops, "hs", torch.tensor(target), a0, lr, T, cp_mask, r,
                               O.make_regularization_function(), **kw)


@pytest.mark.parametrize("dt,T,tol", [(torch.float64, 60, 1e-9), (torch.float32, 3, 1e-4)])
def test_adam_loop_parity(dt, T, tol):
    """Whole fused loop vs the oracle loop (optimization.py:28-94, 362): initial regloss, best
    regloss / reg / params.  f32 runs are compared over a short horizon (the trajectories are
    chaotic, see test_adam_loop_parity_c3_shape_f32; per-step parity is what is pinned); split runs must be
    bit-identical to one run over a longer one."""
    n, layer, K = 3, chain_layer(3), 6
    anz, oanz, ops = setup(n, layer, K, "xyz")
    B = 9
    a0 = torch.tensor(np.random.default_rng(0).uniform(0, 2 * np.pi, (B, anz.num_angles)), dtype=dt)
    res = _oracle_run(n, ops, u_toff3, a0, 0.1, T, oanz.cp_mask, 0.002)
    obr = np.array([r["regloss"][1].item() for r in res]); oir = np.array([r["regloss"][0].item() for r in res])
    obp = np.stack([r["params"][1].numpy() for r in res]); oreg = np.array([r["reg"][1].item() for r in res])
    st = anz.program.adam_state(a0.to(DEV).clone())
    anz.program.adam_run(st, Loss("hs", u_toff3), pen(0.002), 0.1, T)
    torch.cuda.synchronize()
    assert np.abs(st.init_regloss.cpu().numpy() - oir).max() < min(tol, 1e-6)
    assert np.abs(st.best_regloss.cpu().numpy() - obr).max() < tol
    assert np.abs(st.best_reg.cpu().numpy() - oreg).max() < tol
    assert np.abs(st.best_params.cpu().numpy() - obp).max() < tol * 50
    Tl = max(T, 24)
    outs = []
    for chunks in ([Tl], [1, Tl // 3, Tl - 1 - Tl // 3]):
        st = anz.program.adam_state(a0.to(DEV).clone())
        for c in chunks:
            anz.program.adam_run(st, Loss("hs", u_toff3), pen(0.002), 0.1, c)
        outs.append((st.best_params.clone(), st.best_regloss.clone(), st.angles.clone(), st.m.clone(), st.v.clone()))
    for x, y in zip(outs[0], outs[1]):
        assert torch.equal(x, y)


def test_adam_history_and_freeze_f64():
    n, layer, K = 3, connected_layer(3), 5
    anz, oanz, ops = setup(n, layer, K, "xyz")
    B, T = 5, 40
    a0 = torch.tensor(np.random.default_rng(1).uniform(0, 2 * np.pi, (B, anz.num_angles)))
    resh = _oracle_run(n, ops, u_toff3, a0, 0.1, T, oanz.cp_mask, 0.002, keep_history=True)
    st = anz.program.adam_state(a0.to(DEV).clone(), hist_len=T)
    anz.program.adam_run(st, Loss("hs", u_toff3), pen(0.002), 0.1, T)
    assert np.abs(st.hist_params.cpu().numpy() - np.stack([r["params"].numpy() for r in resh])).max() < 1e-9
    assert np.abs(st.hist_regloss.cpu().numpy() - np.stack([r["regloss"].numpy() for r in resh])).max() < 1e-10
    # per-sample frozen parameters (verification stage, cp_utils.py:100-108, 205-247): no penalty
    fm = torch.zeros(B, anz.num_angles, dtype=torch.bool)
    rng = np.random.default_rng(2)
    for b in range(B):
        fm[b, rng.choice(anz.num_angles, 6, replace=False)] = True
    res = O.mynimize_repeated(n, ops, "hs", torch.tensor(u_toff3), a0, 0.01, T, freeze_mask=fm)
    st = anz.program.adam_state(a0.to(DEV).clone(), freeze=fm.to(torch.uint8).to(DEV).contiguous())
    anz.program.adam_run(st, Loss("hs", u_toff3), None, 0.01, T)
    assert np.abs(st.best_regloss.cpu().numpy() - np.array([r["regloss"][1].item() for r in res])).max() < 1e-10
    assert torch.equal(st.angles.cpu()[fm], a0[fm])   # frozen entries never move


@pytest.mark.parametrize("kind,env", [("state", {}), ("hs", {"CPF_ENGINE": "adjoint"}), ("hs", {}),
                                      ("hs", {"CPF_NO_LAYERED": "1"})])
def test_history_with_freeze_mask(kind, env):
    """keep_history=True together with a freeze mask: every history row carries the frozen parameters' (unchanged)
    values, on the state-adjoint kernels (state loss, CPF_ENGINE=adjoint), the interpreter and the Heisenberg kernel
    alike; `mynimize_repeated`'s 'reg' / 'loss' histories are then evaluated on complete rows."""
    n, layer, K = 3, connected_layer(3), 5
    anz, oanz, ops = setup(n, layer, K, "xyz")
    B, T = 4, 25
    a0 = torch.tensor(np.random.default_rng(11).uniform(0, 2 * np.pi, (B, anz.num_angles)))
    fm = torch.zeros(B, anz.num_angles, dtype=torch.bool)
    rng = np.random.default_rng(12)
    for b in range(B):
        fm[b, rng.choice(anz.num_angles, 9, replace=False)] = True
    V = unitary_group.rvs(8, random_state=5)
    tgt = V[:, 0].copy() if kind == "state" else V
    res = O.mynimize_repeated(n, ops, kind, torch.tensor(tgt), a0, 0.05, T, oanz.cp_mask, 0.002,
                              O.make_regularization_function(), keep_history=True, freeze_mask=fm)

    def run():
        st = anz.program.adam_state(a0.to(DEV).clone(), freeze=fm.to(torch.uint8).to(DEV).contiguous(), hist_len=T)
        anz.program.adam_run(st, Loss(kind, tgt), pen(0.002), 0.05, T)
        return st
    st = _with_env(env, run)
    hp = st.hist_params.cpu()
    # (Adam divides by sqrt(v): rounding of tiny gradient components is amplified along the trajectory; the
    # single-column state loss has the smallest gradients)
    assert np.abs(hp.numpy() - np.stack([r["params"].numpy() for r in res])).max() < 1e-7
    assert np.abs(st.hist_regloss.cpu().numpy() - np.stack([r["regloss"].numpy() for r in res])).max() < 1e-9
    for b in range(B):      # frozen columns are constant over the whole history
        assert torch.equal(hp[b][:, fm[b]], a0[b][fm[b]][None].expand(T, -1))


def test_constrained_program_equals_freeze_mask():
    """Ansatz.constrained (constant-angle program over the free vector) and the freeze mask are the
    same computation."""
    n, layer, K = 3, chain_layer(3), 6
    anz, oanz, ops = setup(n, layer, K, "xyz")
    a0 = np.random.default_rng(5).uniform(0, 2 * np.pi, anz.num_angles)
    idx = [i for i in range(anz.num_angles) if anz.cp_mask[i]][::2]
    a0[idx] = [0.0, math.pi, 0.0][:len(idx)]
    prog, free_idx = anz.constrained(a0[idx], idx)
    full = torch.tensor(a0[None], device=DEV)
    free = full[:, free_idx].contiguous()
    l1, _, g1 = anz.program.loss_grad(full, Loss("hs", u_toff3), None)
    l2, _, g2 = prog.loss_grad(free, Loss("hs", u_toff3), None)
    assert abs(float(l1 - l2)) < 1e-14
    assert np.abs(g1.cpu().numpy()[0, free_idx] - g2.cpu().numpy()[0]).max() < 1e-13


def test_count_cz_and_projection_bit_exact():
    n, layer, K = 4, chain_layer(4), 25
    anz, oanz, ops = setup(n, layer, K, "xyz")
    rng = np.random.default_rng(11)
    B = 300
    a = rng.uniform(-7, 14, (B, anz.num_angles)).astype(np.float32)
    # put many CP angles near the thresholds
    cp_idx = np.flatnonzero(anz.cp_mask)
    for b in range(B):
        k = rng.choice(cp_idx, 10, replace=False)
        a[b, k] = (rng.choice([0, math.pi, 2 * math.pi, -2 * math.pi, 3 * math.pi], 10)
                   + rng.choice([-0.21, -0.2, -0.19, 0, 0.19, 0.2, 0.21], 10)).astype(np.float32)
    cz, proj, frozen = anz.program.count_cz(torch.tensor(a, device=DEV), 0.2, project=True)
    ocz = np.array([O.count_cz(x * anz.cp_mask, 0.2) for x in a])
    assert np.array_equal(cz.cpu().numpy(), ocz)
    for b in range(0, B, 7):
        po, fo = O.project_cp_angles(a[b], anz.cp_mask, 0.2)
        assert np.array_equal(proj[b].cpu().numpy(), po)
        assert np.array_equal(frozen[b].cpu().numpy().astype(bool), fo)


def test_initial_angles_bit_exact_and_shard_independent():
    """Device threefry sampler == jax 0.3.x semantics restated in the oracle (main.py:541-548)."""
    anz = Ansatz(3, "cp", fill_layers(chain_layer(3), 12))
    P = anz.num_angles
    for seed, total in [(0, 10), (1272950319, 33)]:
        ref = O.generate_initial_angles(seed, P, anz.cp_mask, batch_size=total)
        got = anz.program.initial_angles(seed, total).cpu().numpy()
        assert np.array_equal(got, ref)
        part = anz.program.initial_angles(seed, total, first=4, count=5).cpu().numpy()
        assert np.array_equal(part, ref[4:9])
    ref0 = O.generate_initial_angles(5, P, anz.cp_mask, cp_dist="0", batch_size=6)
    got0 = anz.program.initial_angles(5, 6, cp_dist="0").cpu().numpy()
    assert np.array_equal(got0, ref0)
    # an odd parameter count exercises the padded counter split
    anz2 = Ansatz(3, "cp", fill_layers(chain_layer(3), 3), "xz")
    assert anz2.num_angles % 2 == 0 or True
    ref = O.generate_initial_angles(3, anz2.num_angles, anz2.cp_mask, batch_size=5)
    assert np.array_equal(anz2.program.initial_angles(3, 5).cpu().numpy(), ref)


def test_golden_ansatz_kats_on_gpu(ansatz_kats):
    """Stored converged angle vectors -> stored unitaries, through the CUDA engine."""
    meta, arrs = ansatz_kats
    progs = {}
    worst64 = worst32 = 0.0
    for m in meta:
        sig = (m["n"], str(m["layer"]), m["num_cp_gates"], m["rotation_gates"])
        if sig not in progs:
            progs[sig] = Ansatz(m["n"], "cp", fill_layers(m["layer"], m["num_cp_gates"]), m["rotation_gates"])
        anz = progs[sig]
        ang = arrs["angles_" + m["key"]]
        u64 = anz.unitary(ang, dtype=torch.float64)
        u32 = anz.unitary(ang, dtype=torch.float32)
        worst64 = max(worst64, hst(u64, arrs["u_" + m["key"]]))
        worst32 = max(worst32, hst(u32.astype(np.complex128), arrs["u_" + m["key"]]))
        if m["target"] is not None and m["loss"] is not None:
            lo, _, _ = anz.program.loss_grad(torch.tensor(ang[None], dtype=torch.float64, device=DEV),
                                             Loss("hs", arrs[m["target"]]), None, want_grad=False)
            assert abs(float(lo) - m["loss"]) < 2e-6
    assert worst64 < 1e-12 and worst32 < 5e-6, (worst64, worst32)


def test_golden_gatelists_on_gpu(gatelist_kats):
    """Stored rz/rx/cz circuits as constant-angle programs (the refine-path evaluator, R2)."""
    meta, arrs = gatelist_kats
    name2kind = {"rx": L.RX, "ry": L.RY, "rz": L.RZ, "cz": L.CZ, "cx": L.CX}
    done = 0
    for m in meta[::3]:
        if m["n"] > 5:
            continue
        key = m["key"]
        ops = [(name2kind[k], int(q0), int(q1), -1, float(p))
               for k, q0, q1, p in zip(m["kinds"], arrs["q0_" + key], arrs["q1_" + key], arrs["p_" + key])]
        prog = Program(m["n"], ops, 0)
        u = prog.unitary(torch.zeros(1, 0, dtype=torch.float64, device=DEV))[0].cpu().numpy()
        uo = O.program_unitary_np(m["n"], ops, np.zeros(0))
        assert np.abs(u - uo).max() < 1e-12
        done += 1
    assert done > 40


def test_parametrised_gatelist_and_cx():
    """rz/rx/ry/cz/cx programs with one angle per rotation (circuit_assembly.py:48-81)."""
    rng = np.random.default_rng(4)
    n = 4
    ops, p = [], 0
    for _ in range(40):
        k = rng.integers(0, 6)
        if k <= 2:
            ops.append((int(k), int(rng.integers(n)), -1, p, 0.0)); p += 1
        else:
            q0, q1 = rng.choice(n, 2, replace=False)
            if k == 3:
                ops.append((L.CP, int(q0), int(q1), p, 0.0)); p += 1
            else:
                ops.append((int(k), int(q0), int(q1), -1, 0.0))
    prog = Program(n, ops, p)
    a = torch.tensor(rng.uniform(0, 6.28, (6, p)), device=DEV)
    uo = O.program_unitary_batched(n, ops, a.cpu()).numpy()
    assert np.abs(prog.unitary(a).cpu().numpy() - uo).max() < 1e-13
    V = unitary_group.rvs(16, random_state=9)
    lo, _, gr = prog.loss_grad(a, Loss("hs", V), None)
    ol, _, og = O.loss_and_grad_batched(n, ops, a.cpu(), "hs", torch.tensor(V))
    assert rel(lo.cpu().numpy(), ol.numpy()) < 1e-12 and rel(gr.cpu().numpy(), og.numpy()) < 1e-12


def test_l1_penalty_and_custom_mask():
    n, layer, K = 3, chain_layer(3), 4
    anz, oanz, ops = setup(n, layer, K, "xyz")
    a = torch.tensor(np.random.default_rng(8).uniform(-3, 3, (5, anz.num_angles)), device=DEV)
    mask = anz.cp_mask.copy(); mask[np.flatnonzero(mask)[0]] = 0
    lo, rg_, gr = anz.program.loss_grad(a, Loss("hs", u_toff3), Penalty("l1", 0.3, cp_mask=mask))
    ol, orr, og = O.loss_and_grad_batched(n, ops, a.cpu(), "hs", torch.tensor(u_toff3), mask, 0.3, O.cp_penalty_L1)
    assert rel(rg_.cpu().numpy(), orr.numpy()) < 1e-13 and rel(gr.cpu().numpy(), og.numpy()) < 1e-12
    bad = np.zeros(anz.num_angles, dtype=np.uint8); bad[0] = 1   # a non-CP parameter cannot be penalised
    with pytest.raises(L.CpflowError):
        anz.program.loss_grad(a, Loss("hs", u_toff3), Penalty("l1", 0.3, cp_mask=bad))


def test_edge_cases_and_errors(lib):
    anz = Ansatz(3, "cp", fill_layers(chain_layer(3), 4))
    prog = anz.program
    # empty batch is a no-op
    e = torch.zeros(0, anz.num_angles, device=DEV)
    assert prog.unitary(e).shape == (0, 8, 8)
    lo, _, gr = prog.loss_grad(e, Loss("hs", u_toff3), None)
    assert lo.shape == (0,) and gr.shape == (0, anz.num_angles)
    # single sample, huge angles (range reduction) in f32
    a = torch.tensor([[1e4 * (i % 7 - 3) for i in range(anz.num_angles)]], dtype=torch.float32, device=DEV)
    u = prog.unitary(a)[0].cpu().numpy().astype(np.complex128)
    uo = O.program_unitary_batched(3, O.ansatz_program(O.cp_ansatz(chain_layer(3), 4)),
                                   torch.tensor(a.cpu().numpy().astype(np.float64)))[0].numpy()
    assert np.abs(u - uo).max() < 1e-5
    # NULL / bad arguments come back as error codes, never crashes
    assert lib.cpf_unitary(prog._h, 7, 1, C.c_void_p(a.data_ptr()), C.c_void_p(a.data_ptr()), None) == -1
    assert lib.cpf_unitary(None, 0, 1, None, None, None) == -1
    ls = L.CpfLossSpec(9, a.data_ptr())
    assert lib.cpf_loss_grad(prog._h, C.byref(ls), None, 0, 1, C.c_void_p(a.data_ptr()),
                             C.c_void_p(a.data_ptr()), None, None, None) == -1
    assert b"loss" in lib.cpf_last_error()


@pytest.mark.parametrize("layer_name", ["chain", "star"])
def test_full_size_properties_c3(layer_name):
    """BASELINE config 3 (4q Toffoli, K=40) at the per-GPU batch of the 8-GPU run (12 500): the
    oracle is too slow here, so check size-independent properties."""
    layer = chain_layer(4) if layer_name == "chain" else [[0, 1], [0, 2], [0, 3]]
    anz = Ansatz(4, "cp", fill_layers(layer, 40))
    prog = anz.program
    B = 12500
    a = prog.initial_angles(0, 100000, first=25000, count=B)
    assert float(a.min()) >= 0 and float(a.max()) < 2 * math.pi + 1e-6
    # unitarity of every sample's U
    U = prog.unitary(a)
    eye = torch.eye(16, device=DEV, dtype=U.dtype)
    assert float((U @ U.conj().transpose(1, 2) - eye).abs().max()) < 2e-5
    # loss in [0,1]; gradient agrees with the f64 engine on a slice; batch order does not matter
    lo, rg_, gr = prog.loss_grad(a, Loss("hs", u_toff4), pen(0.001476))
    assert float(lo.min()) >= -1e-6 and float(lo.max()) <= 1 + 1e-6
    lo64, rg64, gr64 = prog.loss_grad(a[:512].double(), Loss("hs", u_toff4), pen(0.001476))
    assert rel(lo[:512].cpu().numpy(), lo64.cpu().numpy()) < 1e-5
    gn = (gr[:512].double() - gr64).norm(dim=1) / gr64.norm(dim=1)
    assert float(gn.max()) < 1e-5
    perm = torch.randperm(B, device=DEV)
    lo_p, _, gr_p = prog.loss_grad(a[perm].contiguous(), Loss("hs", u_toff4), pen(0.001476))
    assert torch.equal(lo_p, lo[perm]) and torch.equal(gr_p, gr[perm])
    # Adam run: best never above the initial regloss, deterministic, chunk-invariant
    st = prog.adam_state(a.clone())
    prog.adam_run(st, Loss("hs", u_toff4), pen(0.001476), 0.1, 30)
    st2 = prog.adam_state(a.clone())
    prog.adam_run(st2, Loss("hs", u_toff4), pen(0.001476), 0.1, 10)
    prog.adam_run(st2, Loss("hs", u_toff4), pen(0.001476), 0.1, 20)
    assert torch.equal(st.best_regloss, st2.best_regloss) and torch.equal(st.angles, st2.angles)
    assert bool((st.best_regloss <= st.init_regloss).all())
    assert torch.equal(st.init_regloss, lo + rg_) or float((st.init_regloss - (lo + rg_)).abs().max()) < 1e-6
    # the best point really has the stored regloss
    lo_b, rg_b, _ = prog.loss_grad(st.best_params, Loss("hs", u_toff4), pen(0.001476), want_grad=False)
    assert float((lo_b + rg_b - st.best_regloss).abs().max()) < 5e-6     # two instantiations of the parameter phase
    assert float((rg_b - st.best_reg).abs().max()) < 1e-6


def _assert_same_run(x, y, dt, ctx=None):
    """(loss, grad, best_regloss, angles[, best_params]) of two engines on the same inputs.  Loss-level
    quantities agree to rounding.  Adam trajectories amplify gradient rounding by lr / (|g| + eps) wherever a
    gradient component is tiny (first steps: update = lr g / (|g| + eps)), so angles are compared at
    1e-10 in f64 and only loosely in f32 (one Adam step is pinned exactly by test_first_adam_step_closed_form)."""
    tol = 1e-12 if dt == torch.float64 else 1e-5
    for a, b in zip(x[:2], y[:2]):
        assert float((a - b).abs().max()) <= tol * max(1.0, float(b.abs().max())), ctx
    assert float((x[2] - y[2]).abs().max()) <= (1e-10 if dt == torch.float64 else 2e-4), ctx
    for a, b in zip(x[3:], y[3:]):
        assert float((a - b).abs().max()) <= (1e-10 if dt == torch.float64 else 2e-2), ctx


def test_first_adam_step_closed_form():
    """optax Adam, first step from zero moments: theta_1 = theta_0 - lr g / (|g| + eps) (bias corrections
    cancel).  Checked against the engine's own gradient so that the float32 arithmetic of the fused update
    (reciprocal bias correction, approximate sqrt / division) is pinned independently of gradient rounding."""
    anz = Ansatz(4, "cp", fill_layers(chain_layer(4), 40))
    V = unitary_group.rvs(16, random_state=2)
    for dt, tol in ((torch.float32, 4e-7), (torch.float64, 1e-15)):
        a = torch.tensor(np.random.default_rng(5).uniform(0, 6.28, (64, anz.num_angles)), dtype=dt, device=DEV)
        _, _, g = anz.program.loss_grad(a, Loss("hs", V), pen())
        st = anz.program.adam_state(a.clone())
        anz.program.adam_run(st, Loss("hs", V), pen(), 0.1, 1)
        # the step against the closed form of the kernel's OWN first moment (m_1 = 0.1 g): components with a tiny
        # gradient move by lr g / (|g| + eps), which amplifies last-bit differences between the gradient of
        # cpf_loss_grad and the one the fused loop computes (two instantiations of the parameter phase)
        gk, a64 = st.m.double() * 10, a.double()
        expect = a64 - 0.1 * gk / (gk.abs() + 1e-8)
        assert float((st.angles.double() - expect).abs().max()) <= tol * 10, dt
        g64 = g.double()
        scale = float(g64.abs().max())
        assert float((st.m.double() - 0.1 * g64).abs().max()) <= max(tol, 2e-6 * scale)
        assert float((st.v.double() - 0.001 * g64 ** 2).abs().max()) <= max(tol, 2e-6 * scale ** 2)


def test_layered_and_interpreter_kernels_agree():
    """Layered templates run on the specialised straight-line kernel (LayerSweep); the same program
    forced onto the interpreter kernel (CPF_NO_LAYERED=1) must give the same numbers."""
    import os
    for n, layer, K, rg in [(4, chain_layer(4), 40, "xyz"), (4, [[0, 1], [0, 2], [0, 3]], 11, "xz"),
                            (3, connected_layer(3), 7, "xyz"), (5, connected_layer(5), 13, "xyz"),
                            (4, connected_layer(4), 9, "zx")]:
        anz = Ansatz(n, "cp", fill_layers(layer, K), rg)
        V = unitary_group.rvs(2 ** n, random_state=2)
        for dt in (torch.float32, torch.float64):
            a = torch.tensor(np.random.default_rng(K).uniform(0, 6.28, (21, anz.num_angles)), dtype=dt, device=DEV)
            outs = []
            for flag in ("0", "1"):
                os.environ["CPF_NO_LAYERED"] = flag
                lo, rg_, gr = anz.program.loss_grad(a, Loss("hs", V), pen())
                st = anz.program.adam_state(a.clone())
                anz.program.adam_run(st, Loss("hs", V), pen(), 0.1, 7)
                outs.append((lo.clone(), gr.clone(), st.best_regloss.clone(), st.angles.clone()))
            os.environ["CPF_NO_LAYERED"] = "0"
            _assert_same_run(outs[0], outs[1], dt)


def _with_env(env, fn):
    import os
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return fn()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_three_engines_agree():
    """HS loss on layered templates runs on the Heisenberg-picture kernel (heis_impl.cuh); the
    state-adjoint LayerSweep kernel (CPF_ENGINE=adjoint) and the interpreter (CPF_NO_LAYERED=1) must give
    the same loss, gradient and Adam trajectory, also for CZ templates and constrained programs."""
    cases = [(4, chain_layer(4), 40, "xyz", "cp"), (4, [[0, 1], [0, 2], [0, 3]], 11, "xz", "cp"),
             (3, connected_layer(3), 7, "xyz", "cp"), (5, chain_layer(5), 9, "xyz", "cp"),
             (4, connected_layer(4), 14, "zyx", "cp"), (3, chain_layer(3), 6, "xyz", "cz"), (2, [[0, 1]], 4, "xyz", "cp")]
    for n, layer, K, rg, ent in cases:
        anz = Ansatz(n, ent, fill_layers(layer, K), rg)
        V = unitary_group.rvs(2 ** n, random_state=4)
        for dt in (torch.float32, torch.float64):
            a = torch.tensor(np.random.default_rng(K).uniform(0, 6.28, (37, anz.num_angles)), dtype=dt, device=DEV)
            progs = [anz.program]
            if ent == "cp":   # constrained program: some CP angles projected to 0 / pi and frozen
                idx = [i for i in range(anz.num_angles) if anz.cp_mask[i]][::2]
                progs.append(anz.constrained([math.pi if j % 2 else 0.0 for j in range(len(idx))], idx)[0])

            def run(prog):
                aa = a[:, :prog.n_params].contiguous()
                p_ = pen() if prog is anz.program and ent == "cp" else None
                lo, rg_, gr = prog.loss_grad(aa, Loss("hs", V), p_)
                st = prog.adam_state(aa.clone())
                prog.adam_run(st, Loss("hs", V), p_, 0.1, 9)
                return lo.clone(), gr.clone(), st.best_regloss.clone(), st.angles.clone(), st.best_params.clone()

            for prog in progs:
                ref = _with_env({"CPF_NO_LAYERED": "1"}, lambda: run(prog))
                adj = _with_env({"CPF_ENGINE": "adjoint"}, lambda: run(prog))
                heis = run(prog)
                _assert_same_run(adj, ref, dt, (n, K, rg, ent, dt, "adjoint"))
                _assert_same_run(heis, ref, dt, (n, K, rg, ent, dt, "heis"))


def test_heis_launch_geometry_edge_cases():
    """Batch sizes around the CTA / wave boundaries and every CTAs-per-SM setting give per-sample results that
    do not depend on the launch geometry (idle sample slots, spare coefficient store, ragged last CTA)."""
    anz = Ansatz(4, "cp", fill_layers(chain_layer(4), 12))
    V = unitary_group.rvs(16, random_state=1)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    a_all = anz.program.initial_angles(3, 4 * n_sm + 50).double()
    lo_ref, _, gr_ref = anz.program.loss_grad(a_all, Loss("hs", V), pen())
    st_ref = anz.program.adam_state(a_all.clone())
    anz.program.adam_run(st_ref, Loss("hs", V), pen(), 0.1, 5)
    for B in (1, 2, 3, 5, n_sm - 1, n_sm, n_sm + 1, 2 * n_sm + 1, 4 * n_sm + 50):
        for env in ({}, {"CPF_HEIS_CTAS": "1"}, {"CPF_HEIS_CTAS": "4", "CPF_HEIS_WARPS": "1"}):
            def run():
                a = a_all[:B].contiguous()
                lo, _, gr = anz.program.loss_grad(a, Loss("hs", V), pen())
                st = anz.program.adam_state(a.clone())
                anz.program.adam_run(st, Loss("hs", V), pen(), 0.1, 5)
                return lo, gr, st
            lo, gr, st = _with_env(env, run)
            assert torch.equal(lo, lo_ref[:B]) and torch.equal(gr, gr_ref[:B]), (B, env)
            assert torch.equal(st.angles, st_ref.angles[:B]) and torch.equal(st.best_params, st_ref.best_params[:B])
            assert torch.equal(st.best_regloss, st_ref.best_regloss[:B])
    # complex64, a batch that fills the SMs: the automatic geometry takes two co-resident CTAs of 8 warps per SM
    # (heis_geometry); one CTA of 16 warps and four small ones must give the same bits
    a32 = anz.program.initial_angles(5, 64 * n_sm)

    def run32():
        st = anz.program.adam_state(a32.clone())
        anz.program.adam_run(st, Loss("hs", V), pen(), 0.1, 7)
        return st
    ref = run32()
    for env in ({"CPF_HEIS_CTAS": "1"}, {"CPF_HEIS_CTAS": "2", "CPF_HEIS_WARPS": "8"}, {"CPF_HEIS_CTAS": "4", "CPF_HEIS_WARPS": "3"},
                {"CPF_HEIS_SYNC": "0"}, {"CPF_HEIS_SYNC": "1"}):
        st = _with_env(env, run32)
        assert torch.equal(st.angles, ref.angles) and torch.equal(st.best_regloss, ref.best_regloss), env
        assert torch.equal(st.best_params, ref.best_params) and torch.equal(st.m, ref.m) and torch.equal(st.v, ref.v), env


@pytest.mark.parametrize("n,layer,K", [(6, chain_layer(6), 9), (6, connected_layer(6), 17), (7, chain_layer(7), 8)])
@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_six_seven_qubit_state_preparation(n, layer, K, dt):
    """BASELINE config 5: 6-qubit (and 7-qubit) state preparation, loss 1 - |<psi|U|0>|^2
    (tutorial/CPFlow_tutorial.ipynb:1318): unitary (column mode), loss / gradient parity and the Adam loop.
    Full-unitary losses are refused with a clear error for n > 5."""
    anz, oanz, ops = setup(n, layer, K, "xyz")
    N, B = 2 ** n, 11
    a = torch.tensor(np.random.default_rng(n + K).uniform(0, 2 * np.pi, (B, anz.num_angles)), dtype=dt, device=DEV)
    a_o = torch.tensor(a.cpu().numpy().astype(np.float64))
    u = anz.program.unitary(a[:3]).cpu().numpy()
    uo = O.program_unitary_batched(n, ops, a_o[:3]).numpy()
    assert np.abs(u - uo).max() < (1e-13 if dt == torch.float64 else 5e-6)
    psi = unitary_group.rvs(N, random_state=7)[:, 0].copy()
    lo, rg_, gr = anz.program.loss_grad(a, Loss("state", psi), pen())
    ol, orr, og = O.loss_and_grad_batched(n, ops, a_o, "state", torch.tensor(psi), oanz.cp_mask, 0.01,
                                          O.make_regularization_function())
    tol = TOL[dt]
    assert rel(lo.cpu().numpy(), ol.numpy()) < tol and rel(rg_.cpu().numpy(), orr.numpy()) < tol
    g, og = gr.cpu().numpy().astype(np.float64), og.numpy()
    assert (np.linalg.norm(g - og, axis=1) / np.linalg.norm(og, axis=1)).max() < tol
    if dt == torch.float64:
        T = 15
        res = O.mynimize_repeated(n, ops, "state", torch.tensor(psi), a_o[:4], 0.1, T, oanz.cp_mask, 0.002,
                                  O.make_regularization_function())
        st = anz.program.adam_state(a[:4].clone())
        anz.program.adam_run(st, Loss("state", psi), pen(0.002), 0.1, T)
        assert np.abs(st.best_regloss.cpu().numpy() - np.array([r["regloss"][1].item() for r in res])).max() < 1e-9
    with pytest.raises(L.CpflowError, match="n <= 5"):
        anz.program.loss_grad(a, Loss("hs", np.eye(N)), pen())


def _heis_run(prog, a, V, p_):
    lo, rg_, gr = prog.loss_grad(a, Loss("hs", V), p_)
    st = prog.adam_state(a.clone())
    prog.adam_run(st, Loss("hs", V), p_, 0.1, 9)
    return lo.clone(), gr.clone(), st.best_regloss.clone(), st.angles.clone(), st.best_params.clone()


def test_any_layer_runs_on_the_heisenberg_kernel():
    """Every block-structured template takes the fast path (VERDICT r1 item 4): the paper's kite and square Toffoli-4
    layers (paper/results/toff4_kite_xyz, toff4_square_xyz), a 5-qubit star, twisted placements and a non-periodic
    block sequence run on HeisSweepAny (qubit pairs dispatched at run time) and agree with the interpreter kernel;
    on the standard layers the run-time-pair kernel (CPF_HEIS_ANY=1) reproduces the compile-time-layer kernel."""
    rng = np.random.default_rng(0)
    irregular = [[int(a), int(b)] for a, b in (rng.permutation(4)[:2] for _ in range(23))]      # no period <= 16
    cases = [(4, KITE4, 25, "xyz"), (4, SQUARE4, 21, "xyz"), (5, [[0, 1], [0, 2], [0, 3], [0, 4]], 13, "xyz"),
             (4, [[3, 1], [2, 0]], 7, "zyx"), (4, irregular, 23, "xz"), (3, [[2, 0], [1, 0]], 5, "xyz")]
    for n, layer, K, rg in cases:
        anz = Ansatz(n, "cp", fill_layers(layer, K), rg)
        V = unitary_group.rvs(2 ** n, random_state=4)
        for dt in (torch.float32, torch.float64):
            if n == 5 and dt == torch.float64:
                continue
            assert anz.program.launch_plan(37, dtype=dt)["engine"] == 1, (layer, dt)
            a = torch.tensor(np.random.default_rng(K).uniform(0, 6.28, (37, anz.num_angles)), dtype=dt, device=DEV)
            ref = _with_env({"CPF_NO_LAYERED": "1"}, lambda: _heis_run(anz.program, a, V, pen()))
            heis = _heis_run(anz.program, a, V, pen())
            _assert_same_run(heis, ref, dt, (n, layer, K, rg, dt))
    for n, layer, K, rg in [(4, chain_layer(4), 40, "xyz"), (3, connected_layer(3), 7, "xyz"), (2, [[0, 1]], 4, "xyz"),
                            (5, chain_layer(5), 9, "xyz")]:
        anz = Ansatz(n, "cp", fill_layers(layer, K), rg)
        V = unitary_group.rvs(2 ** n, random_state=4)
        a = anz.program.initial_angles(1, 37)
        fixed = _heis_run(anz.program, a, V, pen())
        anyk = _with_env({"CPF_HEIS_ANY": "1"}, lambda: _heis_run(anz.program, a, V, pen()))
        # same arithmetic in the same order per block; the sweeps are explicit FMA intrinsics, the scalar parameter
        # phase is compiled once per kernel instantiation (FMA contraction is the compiler's choice there), so the
        # two kernels agree to rounding, not necessarily bit for bit
        assert float((fixed[0] - anyk[0]).abs().max()) <= 2e-7 and float((fixed[1] - anyk[1]).abs().max()) <= 2e-7
        _assert_same_run(fixed, anyk, torch.float32, (n, layer, "any vs fixed"))


def test_time_sliced_runs_are_bit_identical():
    """Batches that are not a whole number of full waves run as a ring of launches over (sample, step-chunk) items
    (heis_impl.cuh: heis_slicing); a sliced run gives the bits of the single launch, with and without a freeze mask."""
    anz = Ansatz(4, "cp", fill_layers(chain_layer(4), 12))
    V = unitary_group.rvs(16, random_state=1)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    plan = anz.program.launch_plan(10 ** 6, n_sm=n_sm)
    slots = plan["samples_per_cta"] * plan["ctas_per_sm"] * n_sm
    assert plan["engine"] == 1 and slots >= n_sm
    B = slots + slots // 3 + 5
    a = anz.program.initial_angles(2, B)
    fm = (torch.rand(B, anz.num_angles, device=DEV) < 0.1).to(torch.uint8)

    def run(freeze):
        st = anz.program.adam_state(a.clone(), freeze=freeze)
        anz.program.adam_run(st, Loss("hs", V), pen() if freeze is None else None, 0.1, 60)
        anz.program.adam_run(st, Loss("hs", V), pen() if freeze is None else None, 0.1, 40)   # resumed, sliced again
        return st
    for freeze in (None, fm):
        ref = _with_env({"CPF_HEIS_SLICES": "1"}, lambda: run(freeze))
        for k in ("0", "2", "3", "20"):
            st = _with_env({"CPF_HEIS_SLICES": k} if k != "0" else {}, lambda: run(freeze))
            for name in ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss", "init_reg"):
                assert torch.equal(getattr(st, name), getattr(ref, name)), (k, name, freeze is not None)


def test_caller_owned_workspace():
    """cpf_workspace_bytes(_multi) + cpf_adam_buffers.workspace (SURVEY.md 8b: 'per-call scratch from a caller-visible
    workspace query'), on every kernel route: a workspace of exactly the size the query gives yields the same bits as
    the library's own pool scratch, one byte less or a misaligned buffer is refused."""
    from cpflow_b200.engine import MultiLoss
    V = unitary_group.rvs(16, random_state=1)
    V64 = unitary_group.rvs(64, random_state=2)
    B = 300
    cases = [  # (name, n, loss, number of targets (0: adam_run), penalty mask on the CP parameters)
        ("hs_heis", 4, Loss("hs", V), 0, False),
        ("hs_heis_cp_mask", 4, Loss("hs", V), 0, True),
        ("state", 4, Loss("state", V[:, 0].copy()), 0, False),
        ("relphase", 4, Loss("relphase", V), 0, False),
        ("isometry_as_hs", 4, Loss("isometry", V[:, :8], ancillas=[0]), 0, False),
        ("isometry_6q", 6, Loss("isometry", V64[:, :16], ancillas=[0, 1]), 0, False),
        ("multi_hs", 4, MultiLoss("hs", np.stack([V, V.conj().T, np.eye(16)])), 3, False),
        ("multi_state", 4, MultiLoss("state", np.stack([V[:, 0], V[:, 1], V[:, 2]])), 3, True),
    ]
    for name, n, loss, n_targets, masked in cases:
        anz = Ansatz(n, "cp", fill_layers(chain_layer(n), 12))
        a = anz.program.initial_angles(4, B)
        p = pen()
        if masked:      # every other CP parameter: the penalty mask takes its own scratch block
            p.cp_mask = np.zeros(anz.num_angles, dtype=np.uint8)
            p.cp_mask[np.flatnonzero(anz.cp_mask)[::2]] = 1
        idx = np.arange(B) % n_targets if n_targets else None

        def run(workspace):
            st = anz.program.adam_state(a.clone())
            st.workspace = workspace
            if n_targets:
                anz.program.adam_run_multi(st, loss, idx, p, 0.1, 20)
            else:
                anz.program.adam_run(st, loss, p, 0.1, 20)
            return st

        need = anz.program.workspace_bytes_multi(B, n_targets, Loss.KINDS[loss.kind]) if n_targets else \
            anz.program.workspace_bytes(B, loss.code)
        if name == "hs_heis":
            assert need >= 16 * B * anz.num_angles           # the packed optimiser state
        ref = run(None)
        st = run(torch.empty(need, dtype=torch.uint8, device=DEV))
        for f in ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss", "init_reg"):
            assert torch.equal(getattr(st, f), getattr(ref, f)), (name, f)
        with pytest.raises(L.CpflowError, match="workspace too small"):
            run(torch.empty(need - 1, dtype=torch.uint8, device=DEV))
        with pytest.raises(L.CpflowError, match="aligned"):
            run(torch.empty(need + 256, dtype=torch.uint8, device=DEV)[8:])


def test_packed_update_matches_the_scalar_update():
    """The packed two-gates-per-thread parameter phase (float runs without freeze mask / history) against the scalar
    loops (the same run with a parameter history, which takes them): the first step is identical up to the rounding
    of the gradient, the loop stays within the usual f32 trajectory tolerances; lane-interleaved state: every
    parameter comes back to its own place (angles, moments, best parameters)."""
    for n, layer, K in ((4, chain_layer(4), 40), (3, chain_layer(3), 7), (4, [[0, 1], [0, 2], [0, 3]], 11)):
        anz = Ansatz(n, "cp", fill_layers(layer, K))
        V = unitary_group.rvs(2 ** n, random_state=n + K)
        a = anz.program.initial_angles(11, 96)
        for T in (1, 12):
            fast = anz.program.adam_state(a.clone())
            anz.program.adam_run(fast, Loss("hs", V), pen(), 0.1, T)
            slow = anz.program.adam_state(a.clone(), hist_len=T)
            anz.program.adam_run(slow, Loss("hs", V), pen(), 0.1, T)
            assert torch.equal(fast.init_regloss, slow.init_regloss) or \
                float((fast.init_regloss - slow.init_regloss).abs().max()) < 2e-6
            tol_a = 2e-5 if T == 1 else 2e-2
            # (T = 1: components with a tiny gradient move by lr g / (|g| + eps); compare moments instead of angles)
            assert float((fast.m - slow.m).abs().max()) < 2e-6 * max(1.0, float(slow.m.abs().max())) or T > 1
            assert float((fast.best_regloss - slow.best_regloss).abs().max()) < 2e-4
            if T > 1:
                assert float((fast.angles - slow.angles).abs().max()) < tol_a
            assert torch.equal(fast.best_params, a) if T == 1 else True


def test_large_angles_leave_the_fast_range_reduction():
    """Half angles beyond the three-constant sin / cos reduction of the packed parameter phase (|theta| > 96 000): the
    warp redoes its coefficients through the scalar loops (heis_kernel: deferred large-argument fix-up), so the
    losses of such a batch equal those of the scalar path (loss_grad mode and a history run)."""
    anz = Ansatz(4, "cp", fill_layers(chain_layer(4), 10))
    V = unitary_group.rvs(16, random_state=3)
    rng = np.random.default_rng(0)
    a = torch.tensor(rng.uniform(-3e5, 3e5, (40, anz.num_angles)), dtype=torch.float32, device=DEV)
    a[::2] = torch.tensor(rng.uniform(0, 6.28, (20, anz.num_angles)), dtype=torch.float32, device=DEV)   # mixed warp
    lo, rg_, _ = anz.program.loss_grad(a, Loss("hs", V), pen(), want_grad=False)
    fast = anz.program.adam_state(a.clone())
    anz.program.adam_run(fast, Loss("hs", V), pen(), 0.1, 1)
    slow = anz.program.adam_state(a.clone(), hist_len=1)
    anz.program.adam_run(slow, Loss("hs", V), pen(), 0.1, 1)
    assert float((fast.init_regloss - (lo + rg_)).abs().max()) < 2e-6
    assert float((fast.init_regloss - slow.init_regloss).abs().max()) < 2e-6
    # the oracle on the same float32 angles (range reduction in double)
    oanz = O.cp_ansatz(chain_layer(4), 10)
    ol = O.loss_and_grad_batched(4, O.ansatz_program(oanz), a.cpu().double(), "hs", torch.tensor(V), oanz.cp_mask, 0.0,
                                 O.make_regularization_function())[0]
    assert float((lo.cpu().double() - ol).abs().max()) < 1e-5


def test_parameters_that_feed_no_gate():
    """A program whose parameter vector is longer than its gates use (the packed optimiser state holds referenced
    parameters only): the unused entries keep their angles, get zero moments and their own value as best parameter."""
    from cpflow_b200.engine import Program
    anz = Ansatz(3, "cp", fill_layers(chain_layer(3), 6))
    ops, P = anz.program.ops, anz.num_angles
    prog = Program(3, ops, P + 3)
    ref = Program(3, ops, P)
    V = unitary_group.rvs(8, random_state=1)
    a = torch.tensor(np.random.default_rng(2).uniform(0, 6.28, (33, P + 3)), dtype=torch.float32, device=DEV)
    for hist in (False, True):
        st = prog.adam_state(a.clone(), hist_len=7 if hist else 0)
        prog.adam_run(st, Loss("hs", V), None, 0.1, 7)
        rf = ref.adam_state(a[:, :P].contiguous().clone(), hist_len=7 if hist else 0)
        ref.adam_run(rf, Loss("hs", V), None, 0.1, 7)
        assert torch.equal(st.angles[:, :P], rf.angles) and torch.equal(st.best_regloss, rf.best_regloss)
        assert torch.equal(st.best_params[:, :P], rf.best_params) and torch.equal(st.m[:, :P], rf.m)
        assert torch.equal(st.angles[:, P:], a[:, P:]) and torch.equal(st.best_params[:, P:], a[:, P:])
        assert float(st.m[:, P:].abs().max()) == 0.0 and float(st.v[:, P:].abs().max()) == 0.0
