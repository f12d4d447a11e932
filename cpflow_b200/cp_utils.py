"""Building, employing and projecting CP templates (mirror of reference cpflow/cp_utils.py).

Sampling, CZ counting and projection run as small CUDA kernels of the C ABI (cpf_initial_angles,
cpf_cz_value, cpf_count_cz); selection over a whole batch is vectorised on the device; the
verification loop is ONE batched `cpf_adam_run` with a per-sample freeze mask instead of the
reference's sequential, re-jitted `mynimize` calls (cp_utils.py:205-247).
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib as L
from .engine import Loss, TorchLoss, _DT, _ptr, _stream
from .optimization import RawResults, run_adam_batch, torch_loss_chunk


def random_cp_angles(anz, num_samples=1, cp_dist='uniform', seed=0, first=0, count=None,
                     dtype=torch.float32, device='cuda'):
    """Batch form of random_cp_angles (cp_utils.py:13-42) under Synthesize._generate_initial_angles
    (main.py:541-548): rows [first, first+count) of the `num_samples` vectors drawn from
    PRNGKey(seed) with jax 0.3.x threefry semantics.  Returns a CUDA tensor [count, P]."""
    if cp_dist not in ('uniform', '0', 'normal'):
        raise ValueError(f"cp_dist {cp_dist!r} not supported")      # cp_utils.py:41-42 prints and returns None
    return anz.program.initial_angles(seed, num_samples, first=first, count=count, cp_dist=cp_dist,
                                      dtype=dtype, device=device)


def cz_value(a, threshold=1e-2, device='cuda'):
    """0 if the CP angle is near 0 (mod 2 pi), 1 if near pi, else 2 (cp_utils.py:45-57); elementwise
    over any array, evaluated by cpf_cz_value.  Returns int32 of the input's shape (numpy in ->
    numpy out, CUDA tensor in -> CUDA tensor out)."""
    is_t = isinstance(a, torch.Tensor)
    t = a if is_t else torch.as_tensor(np.asarray(a, dtype=np.float32))
    if t.dtype not in _DT:
        t = t.to(torch.float32)
    t = t.to(device).contiguous()
    out = torch.empty(t.shape, dtype=torch.int32, device=t.device)
    with torch.cuda.device(t.device):
        L.check(L.load().cpf_cz_value(_DT[t.dtype], t.numel(), _ptr(t), float(threshold), _ptr(out), _stream()))
    return out if is_t else out.cpu().numpy()


def count_cz(angles, threshold=0.2):
    """Number of CZ gates of a template whose CP angles are `angles` (cp_utils.py:59-67)."""
    return int(cz_value(angles, threshold=threshold).sum())


def project_cp_angle(a, threshold=0.2):
    """cp_utils.py:70-77 (host scalar helper; batches use cpf_count_cz's projection output)."""
    a = float(np.float32(a) % np.float32(2 * math.pi))
    if abs(a - math.pi) < threshold:
        return math.pi
    if abs(a) < threshold or abs(a - 2 * math.pi) < threshold:
        return 0
    return a


def insert_params(params, insertion_params, insertion_indices):
    """cp_utils.py:80-97."""
    total = len(params) + len(insertion_params)
    ins = set(int(i) for i in insertion_indices)
    others = [i for i in range(total) if i not in ins]
    res = np.zeros(total, dtype=np.result_type(np.asarray(params).dtype, np.float32))
    res[others] = np.asarray(params)
    res[[int(i) for i in insertion_indices]] = np.asarray(insertion_params)
    return res


def convert_cp_to_cz(anz, angles, threshold=0.2):
    """cp_utils.py:111-141: round CP gates near identity / CZ and freeze them.  Returns
    [circ_func, u_func, free_angles] like the reference; the callables take the free-angle vector.
    `u_func.program` is the constant-folded gate program over the free angles."""
    angles = np.asarray(angles.detach().cpu().numpy() if isinstance(angles, torch.Tensor) else angles)
    t = torch.as_tensor(angles[None].astype(np.float32 if angles.dtype != np.float64 else np.float64)).cuda()
    _, proj, frozen = anz.program.count_cz(t, threshold, project=True)
    frozen = frozen[0].cpu().numpy().astype(bool)
    proj = proj[0].cpu().numpy()
    projected_indices = [int(i) for i in np.flatnonzero(frozen)]
    projected_cp_angles = proj[projected_indices]
    free_idx = [i for i in range(len(angles)) if not frozen[i]]
    free_angles = angles[free_idx]
    circ_func, u_func = _constrained_funcs(anz, projected_cp_angles, projected_indices)
    return [circ_func, u_func, free_angles]


def evaluate_cp_result(res, cp_mask, threshold=0.2):
    """cp_utils.py:144-164: (cz, loss, angles) at the lowest regloss of one learning history."""
    regloss = _np(res['regloss'])
    best_i = int(np.argmin(regloss))
    loss = _np(res['loss'])[best_i]
    angles = _np(res['params'])[best_i]
    cz = count_cz(angles[np.asarray(cp_mask) == 1], threshold=threshold)
    return cz, loss, angles


def _np(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def select_batch(raw, program, threshold_cp=0.2):
    """Vectorised evaluate_cp_result over a device-resident RawResults: returns
    (cz [B] int32, loss [B], angles [B,P]) at each sample's argmin regloss."""
    best_i = torch.argmin(raw.regloss, dim=1)                     # first minimum, like jnp.argmin
    idx = torch.arange(len(raw), device=raw.regloss.device)
    loss = raw.loss[idx, best_i]
    angles = raw.params[idx, best_i].contiguous()
    cz = program.count_cz(angles, threshold_cp)
    return cz, loss, angles


def filter_cp_results(res_list, cp_mask, threshold_cz_count, threshold_loss, threshold_cp=0.2,
                      disable_tqdm=False, program=None):
    """cp_utils.py:167-202: keep histories with cz <= threshold_cz_count and loss <= threshold_loss,
    sorted by cz (stable).  Returns [[cz, res], ...].  A device RawResults (+ its program) is
    filtered on the GPU; any other list of result dicts goes sample by sample like the reference."""
    if isinstance(res_list, RawResults) and isinstance(res_list.regloss, torch.Tensor) and program is not None:
        cz, loss, _ = select_batch(res_list, program, threshold_cp)
        keep = (loss <= threshold_loss)
        if threshold_cz_count != float('inf'):
            keep &= cz <= int(threshold_cz_count)
        sel = torch.nonzero(keep).flatten()
        order = torch.sort(cz[sel], stable=True).indices
        sel = sel[order].cpu().tolist()
        czs = cz.cpu().tolist()
        return [[czs[i], res_list[i]] for i in sel]
    selected = []
    for res in res_list:
        cz, loss, _ = evaluate_cp_result(res, cp_mask, threshold=threshold_cp)
        if cz <= threshold_cz_count and loss <= threshold_loss:
            selected.append([cz, res])
    selected.sort(key=lambda x: x[0])
    return selected


def verify_cp_results(results, anz, unitary_loss_func, options, keep_history=False, dtype=None, device=None):
    """Batched verify_cp_result (cp_utils.py:205-247) for a list of result dicts: project the CP
    angles at each best point, freeze them, and run Adam (no penalty) on the loss from the projected
    point — one fused launch for all candidates.  Returns a list of tuples
    (success, num_cz_gates, circ_func, u_func, best_free_angles) in input order."""
    if keep_history:
        raise NotImplementedError("verify_cp_results keeps no history (the reference's static() never asks)")
    if not len(results):
        return []
    if not isinstance(unitary_loss_func, (Loss, TorchLoss)):
        raise TypeError("unitary_loss_func must be a Loss spec or a TorchLoss")
    prog = anz.program
    picks = []
    for res in results:
        regloss = res['regloss']
        bi = int(torch.argmin(regloss)) if isinstance(regloss, torch.Tensor) else int(np.argmin(regloss))
        p = res['params'][bi]
        picks.append(p if isinstance(p, torch.Tensor) else torch.as_tensor(np.asarray(p)))
    # dtype / device: the caller's (Synthesize passes its own), else those of the stored parameters
    if dtype is None:
        dtype = picks[0].dtype if picks[0].dtype in (torch.float32, torch.float64) else torch.float32
    if device is None:
        device = picks[0].device if picks[0].is_cuda else torch.device('cuda', torch.cuda.current_device())
    angles = torch.stack([p.to(device, dtype) for p in picks]).contiguous()
    cz, proj, frozen = prog.count_cz(angles, options.threshold_cp, project=True)
    raw = run_adam_batch(prog, unitary_loss_func, None, proj, options.learning_rate_at_verification,
                         options.num_gd_iterations_at_verification, freeze=frozen, keep_history=False,
                         chunk=torch_loss_chunk(prog, dtype))
    best_i = torch.argmin(raw.regloss, dim=1)
    idx = torch.arange(len(raw), device=angles.device)
    best_loss = raw.regloss[idx, best_i].cpu().numpy()
    best_full = raw.params[idx, best_i].cpu().numpy()
    frozen_h = frozen.cpu().numpy().astype(bool)
    cz_h = cz.cpu().tolist()
    out = []
    for i in range(len(results)):
        fixed_idx = [int(j) for j in np.flatnonzero(frozen_h[i])]
        fixed_val = best_full[i][fixed_idx]
        free_idx = [j for j in range(anz.num_angles) if not frozen_h[i][j]]
        circ_func, u_func = _constrained_funcs(anz, fixed_val, fixed_idx)
        out.append((bool(best_loss[i] <= options.target_loss), cz_h[i], circ_func, u_func, best_full[i][free_idx]))
    return out


class _Constrained:
    """`constrained_function(f, fixed_params, indices)` of the reference (cp_utils.py:100-108) as a picklable
    top-level callable: f applied to the full angle vector with `fixed_params` inserted at `indices`.  The
    reference stores local closures in `Decomposition._cp_data`; those need dill to be saved."""

    def __init__(self, anz, fixed_params, indices):
        self.anz = anz
        self.fixed_params = np.asarray(fixed_params)
        self.indices = [int(i) for i in indices]

    def full(self, free):
        return insert_params(np.asarray(free), self.fixed_params, self.indices)


class ConstrainedCircuit(_Constrained):
    def __call__(self, free):
        return self.anz.circuit(self.full(free))


class ConstrainedUnitary(_Constrained):
    def __call__(self, free):
        full = self.full(free)
        return self.anz.unitary(full.astype(np.float64 if full.dtype == np.float64 else np.float32))

    @property
    def program(self):
        """The constant-folded gate program over the free angles (Ansatz.constrained)."""
        return self.anz.constrained(self.fixed_params, self.indices)[0]


def _constrained_funcs(anz, fixed_val, fixed_idx):
    return ConstrainedCircuit(anz, fixed_val, fixed_idx), ConstrainedUnitary(anz, fixed_val, fixed_idx)


def verify_cp_result(res, anz, unitary_loss_func, options, keep_history=False, dtype=None, device=None):
    """cp_utils.py:205-247 for one result: (success, num_cz_gates, circ, u, best_angs)."""
    return verify_cp_results([res], anz, unitary_loss_func, options, keep_history=keep_history, dtype=dtype,
                             device=device)[0]
