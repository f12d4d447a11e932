"""Procedures to refine approximate circuits (mirror of reference cpflow/exact_decompositions.py).

The reference walks the rotation angles of a {rz, rx, cz} circuit one by one and tries to zero each of
them (or merge it into a later angle on the same wire) while a jitted loss stays below a threshold
(exact_decompositions.py:77-113): O(G^2) sequential loss evaluations of a G-angle circuit.  Here the
circuit is lowered once to a gate program with one parameter per rotation
(`circuit_angle_program`, the job of qiskit_circ_to_jax_unitary, circuit_assembly.py:48-81) and, for
every angle, ALL candidate angle vectors of that step are evaluated in one batched loss-only call of
the CUDA engine (cpf_loss_grad without gradient, complex128); the first candidate in the reference's
order that passes is taken, so the result is the reference's greedy result.

Not provided: the Solovay-Kitaev / Clifford+T stage, `project_circuit` and `move_all_rgates` (qiskit passes
and gate library, exact_decompositions.py:261-269, 374-425, 448-618) and `lasso_angles` (:347-368, an L1 penalty
on every rotation angle; unused by the reference's own drivers); `refine` stops at 'Rational'.
"""
import math
from fractions import Fraction

import numpy as np
import torch

from . import _lib as L
from .circuit import Circuit, Gate, convert_to_ZXZ, cp_to_cz_circuit, gates_count, gates_depth  # noqa: F401
from .engine import Program, TorchLoss
from .matrix_utils import cost_HST

_ROT = {'rx': L.RX, 'ry': L.RY, 'rz': L.RZ}


def bracket_angle(a):
    """trigonometric_utils.py:41-44: the angle in [-pi, pi) that differs from `a` by a multiple of 2 pi."""
    return ((np.asarray(a, dtype=np.float64) + math.pi) % (2 * math.pi)) - math.pi


def check_approximation(circuit, new_circuit, loss=1e-5):
    """exact_decompositions.py:30-33."""
    l = cost_HST(circuit.unitary(), new_circuit.unitary())
    if not l < loss:
        raise ValueError(f'Difference {l} between modified and original circuit is above threshold {loss}.')


def check_loss(circuit, unitary_loss_func, threshold_loss=1e-5):
    """exact_decompositions.py:36-39."""
    loss = unitary_loss_func(circuit.unitary())
    if not loss < threshold_loss:
        raise ValueError(f'Circuit loss {loss} is above threshold {threshold_loss}.')


def circuit_angle_program(qc):
    """{rz, rx, ry, cz} circuit -> (Program with one parameter per rotation in circuit order, angles, wires):
    circuit_assembly.py:48-81."""
    ops, angles, wires = [], [], []
    for g in qc.data:
        if g.name in _ROT:
            ops.append((_ROT[g.name], g.qubits[0], -1, len(angles), 0.0))
            angles.append(float(g.params[0]))
            wires.append(int(g.qubits[0]))
        elif g.name == 'cz':
            ops.append((L.CZ, g.qubits[0], g.qubits[1], -1, 0.0))
        else:
            raise TypeError(f"Gate `{g.name}` not in ['rx', 'ry', 'rz', 'cz'].")
    prog = Program(qc.num_qubits, ops, len(angles))
    return prog, np.array(angles, dtype=np.float64), wires


def _batched_loss(prog, loss, cand, device):
    a = torch.as_tensor(cand, dtype=torch.float64, device=device).contiguous()
    if isinstance(loss, TorchLoss):     # a user loss: evaluated by torch on the candidates' unitaries
        with torch.no_grad():
            return loss.batch(prog.unitary(a)).cpu().numpy()
    lo, _, _ = prog.loss_grad(a, loss, None, want_grad=False)
    return lo.cpu().numpy()


def reduce_all_1q_angles(prog, loss, initial_angles, wires, threshold=1e-5, device='cuda'):
    """exact_decompositions.py:77-113.  For angle k (earlier angles are final): candidate 0 sets it to zero;
    then, for every later angle i on the same wire, the candidates a_i -/+ a_k with a_k = 0.  One batched
    loss call per k; the first passing candidate (reference order) is accepted."""
    angles = np.array(initial_angles, dtype=np.float64)
    G = len(angles)
    for k in range(G):
        later = [i for i in range(k + 1, G) if wires[i] == wires[k]]
        cand = np.repeat(angles[None, :], 1 + 2 * len(later), axis=0)
        cand[:, k] = 0.0
        for j, i in enumerate(later):
            cand[1 + 2 * j, i] = angles[i] - angles[k]
            cand[2 + 2 * j, i] = angles[i] + angles[k]
        losses = _batched_loss(prog, loss, cand, device)
        ok = np.flatnonzero(losses < threshold)
        if len(ok):
            angles = cand[ok[0]]
    return angles


def replace_angles_in_circuit(qc, angles):
    """exact_decompositions.py:116-131."""
    out = Circuit(qc.num_qubits, global_phase=qc.global_phase)
    i = 0
    for g in qc.data:
        if g.name in _ROT:
            out.data.append(Gate(g.name, g.qubits, (float(angles[i]),)))
            i += 1
        else:
            out.data.append(Gate(g.name, g.qubits, g.params))
    return out


def reduce_angles(circuit, unitary_loss_func, reduce_threshold=1e-5, cp_threshold=0.01, device='cuda'):
    """exact_decompositions.py:193-209."""
    qc = cp_to_cz_circuit(circuit.copy(), cp_threshold=cp_threshold)
    check_approximation(circuit, qc, loss=1e-5)
    qc = convert_to_ZXZ(qc)
    prog, angles, wires = circuit_angle_program(qc)
    reduced = reduce_all_1q_angles(prog, unitary_loss_func, angles, wires, threshold=reduce_threshold, device=device)
    qc = replace_angles_in_circuit(qc, bracket_angle(reduced))
    check_loss(qc, unitary_loss_func, threshold_loss=reduce_threshold)
    return qc


def rationalize_rgate(angle, max_denominator, angle_threshold):
    """exact_decompositions.py:247-258."""
    rational = math.pi * Fraction.from_float(angle / math.pi).limit_denominator(max_denominator)
    return float(rational) if abs(rational - angle) < angle_threshold else angle


def rationalize_all_rgates(circuit, max_denominator=32, angle_threshold=1e-3):
    """exact_decompositions.py:212-227."""
    out = Circuit(circuit.num_qubits, global_phase=circuit.global_phase)
    for g in circuit.data:
        if g.name in _ROT:
            out.data.append(Gate(g.name, g.qubits, (rationalize_rgate(g.params[0], max_denominator, angle_threshold),)))
        else:
            out.data.append(Gate(g.name, g.qubits, g.params))
    check_approximation(circuit, out)
    return out


def angle_is_rational(a, power):
    """exact_decompositions.py:239-244: a = pi n / 2^j with j <= power."""
    f = Fraction(a / math.pi).limit_denominator(2 ** power)
    return abs(math.pi * f - a) < 1e-6 and math.log2(f.denominator).is_integer()


def all_rgates_are_rational(circuit, power):
    """exact_decompositions.py:230-236."""
    return all(angle_is_rational(g.params[0], power) for g in circuit.data if g.name in _ROT)


def remove_zero_rgates(circuit):
    """exact_decompositions.py:428-445."""
    out = Circuit(circuit.num_qubits, global_phase=circuit.global_phase)
    for g in circuit.data:
        if g.name in _ROT and abs(g.params[0]) < 1e-5:
            continue
        out.data.append(Gate(g.name, g.qubits, g.params))
    check_approximation(circuit, out)
    return out


def refine(circuit, unitary_loss_func, max_denominator=32, angle_threshold=1e-3, cp_threshold=0.01,
           reduce_threshold=1e-5, recursion_degree=0, recursion_depth=5, verbose=False, device='cuda'):
    """exact_decompositions.py:293-344 without the Solovay-Kitaev stage: returns (circuit, refine_type,
    t_count, t_depth) with refine_type in {'Approximate', 'Rational'}."""
    qc = circuit.copy()
    refine_type, t_count, t_depth = 'Approximate', None, None
    try:
        qc = reduce_angles(qc, unitary_loss_func, reduce_threshold=reduce_threshold, cp_threshold=cp_threshold,
                           device=device)
        qc = remove_zero_rgates(qc)
    except ValueError as e:
        if verbose:
            print(e)
        return qc, refine_type, t_count, t_depth
    try:
        qc = rationalize_all_rgates(qc, max_denominator=max_denominator, angle_threshold=angle_threshold)
        qc = remove_zero_rgates(qc)
        if all_rgates_are_rational(qc, int(math.log2(max_denominator))):
            refine_type = 'Rational'
    except ValueError as e:
        if verbose:
            print(e)
    return qc, refine_type, t_count, t_depth
