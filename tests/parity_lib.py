"""Shared measurement code of the GPU parity tests and of tools/parity_report.py: the CUDA engine
(through the C ABI) against the CPU oracle on identical seeded angle batches.  Error measures are the
ones of SURVEY.md 8(d): loss / reg relative to the batch maximum, gradients norm-wise per sample."""
import os
from collections import namedtuple

import numpy as np
import torch
from scipy.stats import unitary_group

import isometry_ref as IR
from oracle import cpflow_oracle as O
from cpflow_b200 import _lib as L
from cpflow_b200.ansatz import Ansatz
from cpflow_b200.engine import Loss, MultiLoss, Penalty, TorchLoss
from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
from cpflow_b200.topology import chain_layer, connected_layer, fill_layers

PF = make_regularization_function(RegularizationOptions)
# BASELINE.json north_star: 1e-5 relative in complex64, 1e-12 in complex128
TOL = {torch.float64: 1e-12, torch.float32: 1e-5}
STAR4 = [[0, 1], [0, 2], [0, 3]]
KITE4 = [[0, 1], [1, 2], [2, 3], [1, 3]]        # paper/results/toff4_kite_xyz
SQUARE4 = [[0, 1], [1, 2], [2, 3], [3, 0]]      # paper/results/toff4_square_xyz
CONFIGS = [(3, chain_layer(3), 5, "xyz"), (4, STAR4, 10, "xyz"), (2, [[0, 1]], 3, "xz"),
           (5, connected_layer(5), 12, "xyz"), (4, [[3, 1], [2, 0]], 7, "zyx"), (4, chain_layer(4), 40, "xyz"),
           (3, connected_layer(3), 7, "xyz"), (5, chain_layer(5), 9, "xz"), (4, STAR4, 40, "xyz"),
           (4, KITE4, 25, "xyz"), (4, SQUARE4, 21, "xyz"), (5, [[0, 1], [0, 2], [0, 3], [0, 4]], 13, "xyz")]


def pen(r=0.01):
    return Penalty("piecewise", r, PF.segments, PF.period)


def rel(a, b):
    return float(np.abs(a - b).max() / max(1e-30, np.abs(b).max()))


def setup(n, layer, K, rg):
    anz = Ansatz(n, "cp", fill_layers(layer, K), rg)
    oanz = O.cp_ansatz(layer, K, rg)
    return anz, oanz, O.ansatz_program(oanz)


def measure_loss_grad(n, layer, K, rg, dt, B=37, dev="cuda", kinds=("hs", "relphase", "state")):
    """Worst errors of unitary / loss / reg / gradient over a batch of B generic angle vectors.
    Returns {kind: {'loss':, 'reg':, 'grad':}, 'unitary': max abs}.  The oracle sees the dtype-rounded
    inputs, so input rounding is not part of the error."""
    anz, oanz, ops = setup(n, layer, K, rg)
    N = 2 ** n
    a64 = np.random.default_rng(n * 100 + K).uniform(0, 2 * np.pi, (B, anz.num_angles))
    a = torch.tensor(a64, dtype=dt, device=dev)
    a_o = torch.tensor(a.cpu().numpy().astype(np.float64))
    out = {}
    u = anz.program.unitary(a).cpu().numpy()
    uo = O.program_unitary_batched(n, ops, a_o).numpy()
    out["unitary"] = float(np.abs(u - uo).max())
    V = unitary_group.rvs(N, random_state=1)
    for kind in kinds:
        tgt = V[:, 0].copy() if kind == "state" else V
        lo, rg_, gr = anz.program.loss_grad(a, Loss(kind, tgt), pen())
        ol, orr, og = O.loss_and_grad_batched(n, ops, a_o, kind, torch.tensor(tgt), oanz.cp_mask, 0.01,
                                              O.make_regularization_function())
        g, og = gr.cpu().numpy().astype(np.float64), og.numpy()
        gn = np.linalg.norm(g - og, axis=1) / np.linalg.norm(og, axis=1)
        lo2, _, none = anz.program.loss_grad(a, Loss(kind, tgt), pen(), want_grad=False)
        out[kind] = {"loss": rel(lo.cpu().numpy(), ol.numpy()), "reg": rel(rg_.cpu().numpy(), orr.numpy()),
                     "grad": float(gn.max()), "loss_only_same_bits": bool(none is None and torch.equal(lo, lo2))}
    return out


def oracle_run(n, ops, target, a0, lr, T, cp_mask, r, **kw):
    return O.mynimize_repeated(n, ops, "hs", torch.tensor(target), a0, lr, T, cp_mask, r,
                               O.make_regularization_function(), **kw)


def adam_case_inputs(n, layer, K, B, freeze, seed=0, rg="xyz"):
    """Initial angles (float64 copies of the threefry float32 draws) of an Adam-loop parity case; freeze=True is the
    verification variant (cp_utils.py:205-247): a third of the CP angles pulled near 0 / pi, then projected and frozen
    with the oracle's project_cp_angles (cp_utils.py:70-77, 111-141)."""
    oanz = O.cp_ansatz(layer, K, rg)
    a0 = O.generate_initial_angles(seed, oanz.num_angles, oanz.cp_mask, batch_size=B).astype(np.float64)
    if not freeze:
        return a0, None
    rng = np.random.default_rng(seed + 1)
    cp_idx = np.flatnonzero(oanz.cp_mask)
    fm = np.zeros(a0.shape, dtype=bool)
    for b in range(B):
        k = rng.choice(cp_idx, len(cp_idx) // 3, replace=False)
        a0[b, k] = rng.choice([0.0, np.pi], len(k)) + rng.uniform(-0.15, 0.15, len(k))
        po, fo = O.project_cp_angles(a0[b].astype(np.float32), oanz.cp_mask, 0.2)
        a0[b], fm[b] = po.astype(np.float64), fo
    return a0, fm


def oracle_adam_case(n, layer, K, target, B, T, freeze, r=0.001476, lr=0.1, dt=torch.float64):
    """The oracle's loop (optimization.py:28-94, 362) on an Adam-loop parity case -> dict of arrays."""
    oanz = O.cp_ansatz(layer, K, "xyz")
    ops = O.ansatz_program(oanz)
    a0, fm = adam_case_inputs(n, layer, K, B, freeze)
    a0t = torch.tensor(a0).to(dt)
    if freeze:
        res = O.mynimize_repeated(n, ops, "hs", torch.tensor(target), a0t, lr, T, freeze_mask=torch.tensor(fm))
    else:
        res = oracle_run(n, ops, target, a0t, lr, T, oanz.cp_mask, r)
    return {"init_regloss": np.array([x["regloss"][0].item() for x in res]),
            "best_regloss": np.array([x["regloss"][1].item() for x in res]),
            "best_reg": np.array([x["reg"][1].item() for x in res]),
            "best_params": np.stack([x["params"][1].numpy() for x in res])}


def measure_adam_loop(n, layer, K, target, B, T, dt=torch.float64, r=0.001476, lr=0.1, freeze=False, dev="cuda",
                      expect=None):
    """The fused Adam loop (cpf_adam_run) against the oracle loop from the same initial angles: max abs errors of
    init regloss, best regloss, best reg, best params.  `expect`: stored oracle outputs (tests/golden/adam_c3.npz,
    written by tests/golden/make_adam_c3.py); None runs the oracle now."""
    anz, oanz, ops = setup(n, layer, K, "xyz")
    a0, fm = adam_case_inputs(n, layer, K, B, freeze)
    if expect is None:
        expect = oracle_adam_case(n, layer, K, target, B, T, freeze, r, lr, dt)
    a0t = torch.tensor(a0).to(dt).to(dev)
    fmt = torch.tensor(fm).to(torch.uint8).to(dev).contiguous() if freeze else None
    st = anz.program.adam_state(a0t.clone(), freeze=fmt)
    anz.program.adam_run(st, Loss("hs", target), None if freeze else pen(r), lr, T)
    torch.cuda.synchronize()
    out = {k: float(np.abs(getattr(st, k).cpu().numpy() - expect[k]).max())
           for k in ("init_regloss", "best_regloss", "best_reg", "best_params")}
    out["engine"] = anz.program.launch_plan(B, dtype=dt)["engine"]
    if freeze:
        out["frozen_moved"] = float((st.angles[fmt.bool()] - a0t[fmt.bool()]).abs().max()) if fm.any() else 0.0
    return out


# ---- one-step consistency of the fused Adam loop along long runs ----------------------------------------------------
# measure_adam_steps runs the fused loop as a chain of launches that stops at every checkpoint k, snapshots the state,
# runs one step and carries on; the chain must give the same bits as one uninterrupted launch, so each single step
# checked here is a step of the real run.  Each step is compared with the oracle's gradient at the kernel's own theta_k
# (float64, the dtype-rounded angles converted exactly) and with optax's update applied to the kernel's own moments:
# a one-step comparison is well conditioned where whole float32 trajectories are chaotic.
CHECKPOINTS = (0, 1, 2, 3, 10, 100, 1000, 1999)
B1, B2, ADAM_EPS = 0.9, 0.999, 1e-8
# relative error of the update lr * m_hat / (sqrt(v_hat) + eps) given the stored moments: float runs use reciprocal bias
# corrections and approximate sqrt / rcp (<= 2 ulp each, engine.cuh: adam_step_fused), about 8 roundings of 6e-8 in all
UPD_REL = {torch.float32: 1e-6, torch.float64: 1e-14}
_STATE = ("angles", "m", "v", "best_params", "best_regloss", "best_reg", "init_regloss", "init_reg")


def _breakpoints():
    """CP angles on the edges of the penalty's modulus branches and segments, and next to them."""
    two = 2 * np.pi
    edges = sorted({x for lo, hi, _, _ in PF.segments for x in (lo, hi) if np.isfinite(x) and x <= two})
    return [-1e-8, two, -two, 2 * two, -2 * two, 3 * two, -3 * two] + edges + [e - two for e in edges[:4]] + \
           [e + two for e in edges[-4:]]


def adam_steps_inputs(anz, B, dt, big=False, seed=0):
    """Initial angles of a step-consistency case: the threefry batch of static(); CP angles of every third sample
    spread over [-3 pi, 5 pi) (every branch of the penalty's modulus); the breakpoints of _breakpoints() in the CP slots
    of samples 2, 5, 8, ...; big=True: two samples with |theta| > 192000 (half angle beyond the 96000 of the float
    kernels' fast sin / cos reduction), on a rotation and on a CP angle."""
    a = anz.program.initial_angles(seed, B).cpu().numpy().astype(np.float64)
    cp = np.flatnonzero(anz.cp_mask)
    rng = np.random.default_rng(seed + 7)
    for b in range(1, B, 3):
        a[b, cp] = rng.uniform(-3 * np.pi, 5 * np.pi, len(cp))
    for j, x in enumerate(_breakpoints()):
        a[2 + 3 * (j // len(cp)), cp[j % len(cp)]] = x
    if big:
        rot = np.flatnonzero(~np.asarray(anz.cp_mask, dtype=bool))
        a[B - 1, rot[3]] = 2.5e5
        a[B - 3, cp[1]] = -2.6e5
    return torch.tensor(a, dtype=dt)


def _penalty_f32_fix(th, cp_mask, r):
    """(reg, grad) corrections that turn the float64 oracle's penalty into the float32 one at the entries where float32
    arithmetic legitimately gives another penalty.  A float32 kernel reduces a CP angle modulo float32(2 pi) with one
    rounding (a + 2 pi for a in (-2 pi, 0), as jnp.mod does in the reference's own float32).  Two cases differ from the
    float64 reduction by more than rounding:
      - breakpoints: a = -1e-8 gives exactly 2 pi in float32 and 2 pi - 1e-8 in float64, and an angle within an ulp of
        a segment edge can land on either side (another slope);
      - far angles: float32(2 pi) exceeds 2 pi by 1.7e-7, so an angle q periods from [0, 2 pi) is reduced 1.7e-7 q
        away from its float64 reduction (q = 41000 at -2.6e5: 7e-3 rad, a penalty value 5e-3 off on the same slope).
    There the reference's own arithmetic is the oracle's penalty run in float32.  Elsewhere the two agree to the
    rounding of values of order 1 (a few 1e-7), far below VAL_DIFF."""
    pf = O.make_regularization_function()
    out = []
    for dt in (torch.float64, torch.float32):
        a = torch.tensor(th, dtype=dt).requires_grad_(True)
        val = pf(a)
        (s,) = torch.autograd.grad(val.sum(), a)
        out.append((val.detach().double().numpy(), s.double().numpy()))
    (v64, s64), (v32, s32) = out
    dis = ((np.abs(s32 - s64) > 1e-3) | (np.abs(v32 - v64) > VAL_DIFF)) & np.asarray(cp_mask, dtype=bool)[None, :]
    return r * ((v32 - v64) * dis).sum(1), r * (s32 - s64) * dis, int(dis.sum())


# penalty values (of order 1) the float32 and float64 oracles may differ by through rounding alone
VAL_DIFF = 1e-5


# A case of measure_adam_steps: qubits, layer, CP gates, rotation gates, loss kind, ancilla qubits (the isometry kinds),
# number of targets (0: single-target run), samples, freeze, dispatch switches and the expected path.
StepCase = namedtuple("StepCase", "n layer K rg kind anc nt B freeze env path")


def _case(n, layer, K, kind, path, rg="xyz", anc=None, nt=0, B=32, freeze=False, env=None):
    return StepCase(n, layer, K, rg, kind, anc, nt, B, freeze, env or {}, path)


_C4, _C5, _C6, _C7, _C8 = (chain_layer(n) for n in (4, 5, 6, 7, 8))
STEP_CASES = {
    # Heisenberg-picture kernels (compile-time layers, run-time qubit pairs, multi-target; the XZ and generic update
    # loops of heis_su2_loop_any)
    "heis_chain4": _case(4, _C4, 40, "hs", "heis"),
    "heis_chain4_freeze": _case(4, _C4, 40, "hs", "heis", freeze=True),
    "heis_chain4_xz": _case(4, _C4, 20, "hs", "heis", rg="xz"),
    "heis_star4_zyx": _case(4, STAR4, 10, "hs", "heis", rg="zyx"),
    "heis_any_kite4": _case(4, KITE4, 25, "hs", "heis_any", env={"CPF_HEIS_ANY": "1"}),
    "heis_any_mt_chain3": _case(3, chain_layer(3), 8, "hs", "heis_any", nt=3, B=36),
    # the isometry loss on <= 5 qubits: HS on a scaled, padded target (Heisenberg kernel)
    "iso_as_hs_chain4": _case(4, _C4, 12, "isometry", "iso_as_hs", anc=[0]),
    # state-adjoint kernels: LayerSweep (4q full unitary, 5q single column), the interpreter (6-8 qubits, one warp per
    # column on 7-8), multi-target, and the HS seed (5-qubit templates run HS on the Heisenberg kernel in both dtypes;
    # CPF_ENGINE=adjoint sends it to the state-adjoint kernels, where the programs the Heisenberg kernel cannot hold go)
    "adj_hs_chain5": _case(5, _C5, 12, "hs", "state_adjoint", env={"CPF_ENGINE": "adjoint"}),
    "layer_relphase_chain4": _case(4, _C4, 12, "relphase", "state_adjoint"),
    "layer_state_chain5": _case(5, _C5, 12, "state", "state_adjoint"),
    "interp_state_chain6": _case(6, _C6, 9, "state", "state_adjoint"),
    "interp_state_chain7": _case(7, _C7, 8, "state", "state_adjoint", B=16),
    "interp_state_chain8": _case(8, _C8, 9, "state", "state_adjoint", B=12),
    "interp_mt_state_chain4": _case(4, _C4, 12, "state", "state_adjoint", nt=3, B=36),
    "interp_mt_state_chain6": _case(6, _C6, 9, "state", "state_adjoint", nt=3, B=36),
    "interp_mt_state_chain8": _case(8, _C8, 9, "state", "state_adjoint", nt=3, B=12),
    "interp_mt_relphase_chain4": _case(4, _C4, 12, "relphase", "state_adjoint", nt=3, B=36),
    # iso_kernel: the isometry loss on 6-8 qubits (InterpSweepIso), the relative-phase isometry loss on 2-8
    # (InterpSweepIsoPhase, with the single-column register split on 2-5 qubits)
    "iso_chain6_k8": _case(6, _C6, 9, "isometry", "iso", anc=[0, 2, 4]),
    "iso_chain8_k32": _case(8, _C8, 9, "isometry", "iso", anc=[0, 3, 7], B=12),
    "iso_chain8_k32_freeze": _case(8, _C8, 9, "isometry", "iso", anc=[0, 3, 7], B=12, freeze=True),
    "isorel_chain3": _case(3, chain_layer(3), 6, "isometry_relphase", "iso", anc=[]),
    "isorel_chain5_k2": _case(5, _C5, 12, "isometry_relphase", "iso", anc=[0, 1, 3, 4]),
    "isorel_chain7_k8_freeze": _case(7, _C7, 8, "isometry_relphase", "iso", anc=[1, 3, 5, 6], B=16, freeze=True),
    "isorel_chain8_k32": _case(8, _C8, 9, "isometry_relphase", "iso", anc=[1, 4, 6], B=12),
    # the host-driven loop of callable losses, one cpf_adam_step per call; K = 120 in complex128 runs 16 columns per
    # cotangent item (the shared-memory fallback).  Its gradient passes through the materialised U and a second sweep,
    # yet stays within the fused kernels' TOL (profiles/adam_steps_r2.txt), so it is held to the same bounds
    "host_hs_chain6": _case(6, _C6, 9, "hs", "host", B=16),
    "host_hs_chain6_k120": _case(6, _C6, 120, "hs", "host", B=8),
    "host_state_chain8_freeze": _case(8, _C8, 9, "state", "host", B=12, freeze=True),
}


def adam_steps_case(name):
    """The StepCase of measure_adam_steps `name`, one per path the Adam loop dispatches to.  Paths: 'heis' / 'heis_any'
    (Heisenberg-picture kernels with compile-time / run-time qubit pairs), 'iso_as_hs' (Heisenberg kernel on the padded
    isometry target), 'state_adjoint' (engine_kernel: LayerSweep or the interpreter), 'iso' (iso_kernel), 'host'
    (cpf_unitary -> torch loss and cotangent -> cpf_adjoint_from_cotangent -> cpf_adam_step)."""
    return STEP_CASES[name]


def _step_targets(c):
    N, T = 2 ** c.n, max(c.nt, 1)
    if c.kind == "state":
        rng = np.random.default_rng(c.n)
        v = rng.normal(size=(T, N)) + 1j * rng.normal(size=(T, N))
        return v / np.linalg.norm(v, axis=1, keepdims=True)
    U = np.stack([unitary_group.rvs(N, random_state=c.n * 10 + t) for t in range(T)])
    return U[:, :, :2 ** (c.n - len(c.anc))] if c.kind in Loss.ISOMETRY_KINDS else U


def _oracle_loss_grad(c, ops, th, target, cp_mask, r, pf):
    """(loss, reg, grad) of the float64 references at theta [B,P]: the oracle for hs / state / relphase,
    tests/isometry_ref.py for the isometry kinds."""
    th = torch.tensor(th)
    if c.kind in Loss.ISOMETRY_KINDS:
        return IR.loss_and_grad_batched(c.n, ops, th, target, c.anc, cp_mask, r, pf,
                                        relphase=c.kind == "isometry_relphase")
    return O.loss_and_grad_batched(c.n, ops, th, c.kind, torch.tensor(target), cp_mask, r, pf)


def host_loss(kind, target):
    """The 'hs' or 'state' loss as a TorchLoss: the host-driven loop runs it on cpf_unitary's output."""
    V = torch.as_tensor(np.asarray(target))
    if kind == "hs":
        N = V.shape[0]
        return TorchLoss(lambda u: 1 - torch.abs((u * V.to(u.device, u.dtype).conj()).sum()) ** 2 / N ** 2)
    assert kind == "state", kind
    return TorchLoss(lambda u: 1 - torch.abs((V.to(u.device, u.dtype).conj() * u[:, 0]).sum()) ** 2)


def host_steps(prog, st, torch_loss, penalty, lr, steps):
    """`steps` iterations of the host-driven loop (optimization.run_adam_batch with a TorchLoss)."""
    for _ in range(steps):
        U = prog.unitary(st.angles)
        val, cot = torch_loss.value_and_cotangent(U)
        g = prog.adjoint_from_cotangent(st.angles, cot)
        prog.adam_step(st, val.to(st.angles.dtype).contiguous(), g, penalty, lr)


def cotangent_columns(prog, dt):
    """Columns per launch item of cpf_adjoint_from_cotangent on 6-8 qubits: 32, halved until the isometry kernel's
    plan for that many columns fits 227 KB of shared memory (iso_impl.cuh: iso_cot_columns)."""
    for k in (32, 16, 8, 4, 2, 1):
        a = prog.n_qubits - (k.bit_length() - 1)
        if prog.launch_plan(1, L.isometry_kind((1 << a) - 1), dt)["smem_bytes"] <= 227 * 1024:
            return k
    return 0


_NAN_FILLED = ("m", "v", "best_params", "best_regloss", "best_reg", "init_regloss", "init_reg")


def poisoned_state(prog, angles, freeze=None, hist_len=0):
    """prog.adam_state with every output buffer the run must write filled with NaN, so an entry the kernels leave
    unwritten cannot pass as zeroed allocator memory."""
    st = prog.adam_state(angles, freeze=freeze, hist_len=hist_len)
    for k in _NAN_FILLED:
        getattr(st, k).fill_(float("nan"))
    return st


DISPATCH_ENV = ("CPF_HEIS_ANY", "CPF_NO_LAYERED", "CPF_ENGINE")


def with_dispatch_env(env, fn):
    """fn() with exactly the dispatch switches `env`: one inherited from the caller's environment (CPF_NO_LAYERED=1
    would move the LayerSweep cases onto the interpreter) must not change the path a case runs on."""
    saved = {k: os.environ.get(k) for k in DISPATCH_ENV}
    for k in DISPATCH_ENV:
        os.environ.pop(k, None)
    os.environ.update(env)
    try:
        return fn()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def measure_adam_steps(name, dt, checkpoints=CHECKPOINTS, T=2000, r=0.001476, lr=0.1, dev="cuda"):
    """One-step consistency of case `name` (adam_steps_case) in dtype `dt`.  Returns {'engine', 'words_per_sample',
    'threads_per_sample', 'cot_columns', 'chain_identical', 'breakpoint_fixes', 'rows': [per checkpoint k: errors and
    the bounds they are held to]}.
    Bounds, per sample (b1, b2, lr, eps of optax; TOL the gradient contract; e the dtype's machine epsilon;
    gs = max(|g_o|, 1)):
      m:     |m' - (b1 m + (1 - b1) g_o)| <= (1 - b1) TOL gs + 4 e (b1 |m| + (1 - b1) |g_o|)
      v:     |v' - (b2 v + (1 - b2) g_o^2)| <= (1 - b2) TOL gs (2 max|g_o| + TOL gs) + 4 e (b2 |v| + (1 - b2) |g_o^2|)
             (|g^2 - g_o^2| <= |g - g_o| max|g + g_o|; the expected m', v' are O.adam_update's from m, v, count k)
      theta: per entry |theta' - (theta - lr m'/bc1 / (sqrt(v'/bc2) + eps))| <= 4 e max(|theta|, |theta'|)
             + UPD_REL |update|, from the kernel's own m', v' (norms are per sample, over the free entries)
      loss, reg: |x - oracle| <= TOL (the loss scale is 1).
    The gradient scale: every loss here is 1 - (a sum of |overlap|^2 terms) with overlaps of unitary columns and unit
    vectors, so |dL/dtheta| <= 2 for each parameter (HS: |dL/dtheta| <= 2 |t| / N^2 * N / 2; the isometry loss: the
    same with k for N; the relative-phase isometry loss: 2/k sum_c |t_c| |d t_c / d theta| <= 2 / k * k / 2), and
    rounding errors scale with 1 where |g_o| is smaller; hence gs = max(|g_o|, 1) for every kind."""
    return with_dispatch_env(adam_steps_case(name).env,
                             lambda: _measure_adam_steps(adam_steps_case(name), dt, checkpoints, T, r, lr, dev))


def _measure_adam_steps(c, dt, checkpoints, T, r, lr, dev):
    n, kind, nt, B, freeze, path = c.n, c.kind, c.nt, c.B, c.freeze, c.path
    anz, oanz, ops = setup(n, c.layer, c.K, c.rg)
    prog = anz.program
    tg = _step_targets(c)
    idx = np.arange(B) % nt if nt else np.zeros(B, dtype=np.int64)
    loss = MultiLoss(kind, tg) if nt else Loss(kind, tg[0], ancillas=c.anc)
    cot_cols = cotangent_columns(prog, dt) if path == "host" else None
    if path == "host":          # the launch shape of cpf_adjoint_from_cotangent: the isometry kernel, cot_cols columns
        code = L.isometry_kind((1 << (n - (cot_cols.bit_length() - 1))) - 1)
    else:
        code = Loss.KINDS[kind] if nt else loss.code
    plan = prog.launch_plan(B, code, dt)
    # launch_plan reports the same layout for the compile-time kite kernel and HeisSweepAny; the 4q chain, K = 40,
    # tells them apart (HEIS_CHAIN4_WORDS of the tests), so its plan under this case's switches shows which family
    # the Heisenberg dispatcher picks while the case runs
    probe = setup(4, chain_layer(4), 40, "xyz")[0].program.launch_plan(B, Loss.KINDS["hs"], dt)["words_per_sample"]
    fm = None
    if freeze:
        a0, fmask = adam_case_inputs(n, c.layer, c.K, B, True, rg=c.rg)
        init = torch.tensor(a0, dtype=dt)
        fm = torch.tensor(fmask, dtype=torch.uint8, device=dev)
    else:
        init = adam_steps_inputs(anz, B, dt, big=dt == torch.float32 and path == "heis")
    init = init.to(dev)
    pn = None if freeze else pen(r)
    hl = host_loss(kind, tg[0]) if path == "host" else None

    def run(st, steps):
        if path == "host":
            host_steps(prog, st, hl, pn, lr, steps)
        elif nt:
            prog.adam_run_multi(st, loss, idx, pn, lr, steps)
        else:
            prog.adam_run(st, loss, pn, lr, steps)

    def snap(st):
        torch.cuda.synchronize()
        return {k: getattr(st, k).detach().cpu().numpy().copy() for k in _STATE}

    ref = poisoned_state(prog, init.clone(), freeze=fm)
    run(ref, T)
    whole = snap(ref)
    st = poisoned_state(prog, init.clone(), freeze=fm)
    cur, pairs = 0, []
    for k in checkpoints:
        if k > cur:
            run(st, k - cur)
        before = snap(st)
        run(st, 1)
        pairs.append((k, before, snap(st)))
        cur = k + 1
    if T > cur:
        run(st, T - cur)
    chained = snap(st)
    out = {"engine": plan["engine"], "words_per_sample": plan["words_per_sample"],
           "threads_per_sample": plan["threads_per_sample"], "cot_columns": cot_cols, "chain4_probe_words": probe,
           "chain_identical": all(np.array_equal(chained[k], whole[k]) for k in _STATE),
           "breakpoint_fixes": 0, "rows": []}
    free = np.ones(init.shape, dtype=bool) if fm is None else fm.cpu().numpy() == 0
    tol, e = TOL[dt], float(torch.finfo(dt).eps)
    pf = None if freeze else O.make_regularization_function()
    cp_mask = None if freeze else oanz.cp_mask
    for k, s0, s1 in pairs:
        th = s0["angles"].astype(np.float64)
        mk = s0["m"].astype(np.float64) if k else np.zeros_like(th)
        vk = s0["v"].astype(np.float64) if k else np.zeros_like(th)
        lo, rg, g = np.zeros(B), np.zeros(B), np.zeros_like(th)
        for t in range(max(nt, 1)):
            sel = np.flatnonzero(idx == t)
            ol, orr, og = _oracle_loss_grad(c, ops, th[sel], tg[t], cp_mask, r, pf)
            lo[sel], rg[sel], g[sel] = ol.numpy(), orr.numpy(), og.numpy()
        if dt == torch.float32 and not freeze:
            dreg, dg, cnt = _penalty_f32_fix(th, oanz.cp_mask, r)
            rg, g = rg + dreg, g + dg
            out["breakpoint_fixes"] += cnt
        regloss = lo + rg
        gf = np.where(free, g, 0.0)
        gs = np.maximum(np.linalg.norm(gf, axis=1), 1.0)
        m1, v1, th1 = (s1[x].astype(np.float64) for x in ("m", "v", "angles"))
        ost = O.AdamState(torch.tensor(th))        # optax's moment update from the kernel's m_k, v_k, count k
        ost.mu, ost.nu, ost.count = torch.tensor(mk), torch.tensor(vk), k
        O.adam_update(torch.tensor(g), ost, lr, B1, B2, ADAM_EPS)
        m_exp, v_exp = ost.mu.numpy(), ost.nu.numpy()
        em = np.linalg.norm(np.where(free, m1 - m_exp, 0.0), axis=1)
        bm = (1 - B1) * tol * gs + 4 * e * (B1 * np.linalg.norm(mk * free, axis=1) + (1 - B1) * np.linalg.norm(gf, axis=1))
        ev = np.linalg.norm(np.where(free, v1 - v_exp, 0.0), axis=1)
        bv = (1 - B2) * tol * gs * (2 * np.abs(gf).max(1) + tol * gs) + \
            4 * e * (B2 * np.linalg.norm(vk * free, axis=1) + (1 - B2) * np.linalg.norm(gf * gf, axis=1))
        # optax's bias corrections 1 - b^count raise b in the run's dtype (so does O.adam_update): in float32 that is
        # float32(0.999), and 1 - float32(0.999) is 1.3e-5 off 1 - 0.999; evaluated here exactly in float64
        cnt = k + 1
        bc1, bc2 = (1 - float(torch.tensor(b, dtype=dt)) ** cnt for b in (B1, B2))
        upd = lr * (m1 / bc1) / (np.sqrt(v1 / bc2) + ADAM_EPS)
        eth = np.where(free, np.abs(th1 - (th - upd)), 0.0)
        bth = 4 * e * np.maximum(np.abs(th), np.abs(th1)) + UPD_REL[dt] * np.abs(upd) + np.finfo(np.float64).tiny
        row = {"k": k, "m": float(em.max()), "m_ratio": float((em / bm).max()), "v": float(ev.max()),
               "v_ratio": float((ev / bv).max()), "theta": float(eth.max()), "theta_ratio": float((eth / bth).max()),
               "frozen_unchanged": True, "best_ok": True}
        if fm is not None:
            fz = ~free
            # a frozen entry keeps its angle and its moments; the moments of a fresh run start at zero (the state's
            # m, v are NaN before the first launch, so step 0 is held to zero, later steps to k's)
            mz, vz = (np.zeros_like(s1["m"][fz]), np.zeros_like(s1["v"][fz])) if k == 0 else (s0["m"][fz], s0["v"][fz])
            row["frozen_unchanged"] = bool(np.array_equal(s1["angles"][fz], s0["angles"][fz]) and
                                           np.array_equal(s1["m"][fz], mz) and np.array_equal(s1["v"][fz], vz))
        # best tracking: strict improvement of the oracle's regloss at theta_k beyond the tolerance -> theta_k saved,
        # clearly worse -> nothing moves; inside the band either outcome
        if k == 0:
            moved = np.ones(B, dtype=bool)
            errs = [np.abs(s1["init_regloss"] - regloss), np.abs(s1["init_reg"] - rg)]
            row["best_ok"] = bool(np.array_equal(s1["best_regloss"], s1["init_regloss"]) and
                                  np.array_equal(s1["best_reg"], s1["init_reg"]))
        else:
            prev = s0["best_regloss"].astype(np.float64)
            moved = s1["best_regloss"] != s0["best_regloss"]
            row["best_ok"] = bool(np.all(regloss[moved] < prev[moved] + tol) and
                                  np.all(regloss[~moved] >= prev[~moved] - tol) and
                                  np.array_equal(s1["best_params"][~moved], s0["best_params"][~moved]) and
                                  np.array_equal(s1["best_reg"][~moved], s0["best_reg"][~moved]))
            errs = [np.zeros(1)]
        row["best_ok"] = row["best_ok"] and bool(np.array_equal(s1["best_params"][moved], s0["angles"][moved]))
        errs += [np.abs(s1["best_regloss"][moved] - regloss[moved]), np.abs(s1["best_reg"][moved] - rg[moved])]
        row["loss"] = float(max(x.max(initial=0.0) for x in errs))
        row["loss_ratio"] = row["loss"] / tol
        row["improved"] = int(moved.sum())
        out["rows"].append(row)
    return out
