"""Multi-start optimisation (mirror of reference cpflow/optimization.py:209-419).

The reference hands Python closures to `jit(vmap(...))`; a CUDA kernel cannot run closures, so the
functions here take the same computation as a declarative spec:

    loss_func           -> `ProgramLoss(program, Loss(kind, target))`   (main.py:561)
    regularization_func -> `Penalty` (engine.py) or None                 (main.py:563-564)

Everything else keeps the reference's names, argument meaning and return shapes
(optimization.py:362-382): a list of dicts {'params', 'loss', 'reg', 'regloss'}; without history
'params' is (2, P) = [initial, best-regloss] and the others are (2,).  The whole loop runs inside
one CUDA kernel launch (cpf_adam_run); there is no CPU fallback.
"""
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib as L
from .engine import Loss, MultiLoss, Penalty, Program, TorchLoss

HISTORY_BYTES_LIMIT = 64 << 30


@dataclass
class ProgramLoss:
    """The declarative form of `lambda angles: unitary_loss_func(u_func(angles))`: `loss` is a `Loss` spec (fused
    kernel) or a `TorchLoss` wrapping an arbitrary torch function of the unitary (host-driven loop)."""
    program: Program
    loss: object

    @property
    def num_params(self):
        return self.program.n_params


class RawResults:
    """Result of one batched run, kept as batched tensors; behaves like the reference's list of
    dicts (optimization.py:364-371) and additionally exposes the batch for vectorised selection."""

    def __init__(self, params, regloss, reg):
        # params [B,H,P], regloss [B,H], reg [B,H]   (H = 2 without history, T with history)
        self.params, self.regloss, self.reg = params, regloss, reg
        self.loss = regloss - reg          # optimization.py:368

    def __len__(self):
        return self.params.shape[0]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        return {'params': self.params[i], 'loss': self.loss[i], 'reg': self.reg[i], 'regloss': self.regloss[i]}

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def cpu(self):
        """Device -> host through pinned staging buffers (torch caches pinned allocations), one synchronise."""
        def to_host(t):
            if not t.is_cuda:
                return t
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            h.copy_(t, non_blocking=True)
            return h
        out = [to_host(self.params), to_host(self.regloss), to_host(self.reg)]
        if self.params.is_cuda:
            torch.cuda.current_stream(self.params.device).synchronize()
        return RawResults(*out)

    def numpy(self):
        r = self.cpu()
        out = RawResults.__new__(RawResults)
        out.params, out.regloss, out.reg, out.loss = (r.params.numpy(), r.regloss.numpy(), r.reg.numpy(),
                                                      r.loss.numpy())
        return out


def run_adam_batch(program, loss, penalty, initial_params, learning_rate, num_iterations,
                   freeze=None, keep_history=False, chunk=None, target_index=None):
    """Device-resident core: `initial_params` is a CUDA tensor [B,P] (not modified).  Returns
    RawResults on the device.  Restates jit(vmap(mynimize_particular)) (optimization.py:344-362).
    With `target_index` ([B] ints), `loss` is a MultiLoss and sample b runs against its target target_index[b], all in
    one launch (cpf_adam_run_multi)."""
    if target_index is not None and not isinstance(loss, MultiLoss):
        raise TypeError("target_index needs a MultiLoss(kind, targets): a user loss function runs one target at a "
                        "time on the host-driven loop")
    if not (isinstance(initial_params, torch.Tensor) and initial_params.is_cuda):
        raise L.CpflowError("run_adam_batch needs a CUDA tensor (no CPU fallback)")
    B, P = initial_params.shape
    T = int(num_iterations)
    if keep_history:
        need = B * T * (P + 1) * initial_params.element_size()
        if need > HISTORY_BYTES_LIMIT:
            raise L.CpflowError(f"keep_history=True needs {need / 2**30:.1f} GiB for B={B}, T={T}, P={P}; "
                                "use keep_history=False (the reference default for static())")
    with torch.cuda.device(initial_params.device):
        st = program.adam_state(initial_params.clone(), freeze=freeze, hist_len=T if keep_history else 0)
        if target_index is not None:
            program.adam_run_multi(st, loss, target_index, penalty, learning_rate, T)
        elif isinstance(loss, TorchLoss):
            # user loss outside the engine: the same loop, one iteration at a time (optimization.py:14-25, 61-75)
            for _ in range(T):
                U = program.unitary(st.angles)
                values, cot = loss.value_and_cotangent(U)
                grad = program.adjoint_from_cotangent(st.angles, cot)
                program.adam_step(st, values.to(st.angles.dtype).contiguous(), grad, penalty, learning_rate)
        else:
            program.adam_run(st, loss, penalty, learning_rate, T)
        if keep_history:
            params_h, regloss_h = st.hist_params, st.hist_regloss
            if penalty is not None:
                reg_h = penalty_values(program, params_h.reshape(B * T, P), penalty).reshape(B, T)
            else:
                reg_h = torch.zeros_like(regloss_h)
            return RawResults(params_h, regloss_h, reg_h)
        params = torch.stack([initial_params, st.best_params], 1)
        regloss = torch.stack([st.init_regloss, st.best_regloss], 1)
        reg = torch.stack([st.init_reg, st.best_reg], 1)
        return RawResults(params, regloss, reg)


def penalty_values(program, angles, penalty):
    """vmap(regularization_func)(params) (optimization.py:366): r * sum R(angles * cp_mask) [B]."""
    dummy = Loss('state', np.eye(program.dim)[0])
    _, reg, _ = program.loss_grad(angles.contiguous(), dummy, penalty, want_grad=False)
    return reg


def _as_device_batch(x, dtype, device):
    """Host (numpy / CPU tensor, pinned on the way) or device input -> contiguous CUDA tensor."""
    if isinstance(x, torch.Tensor) and x.is_cuda:
        return x.to(dtype).contiguous()
    t = torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x).to(dtype).contiguous()
    if not t.is_pinned():
        t = t.pin_memory()
    return t.to(device, non_blocking=True)


def mynimize_repeated(loss_func, num_params=None, method='adam', learning_rate=0.1, target_loss=1e-7,
                      u_func=None, initial_params_batch=None, num_repeats=1, regularization_func=None,
                      keep_history=True, compute_losses=True, num_iterations=5000, dtype=torch.float32,
                      device='cuda', freeze_mask=None, return_device=False, zero_regularization=False,
                      **kwargs):
    """Reference optimization.py:269-382 on the CUDA engine.

    loss_func: ProgramLoss; regularization_func: Penalty or None; initial_params_batch: (P,) or
    (B, P) array on the host (numpy / torch) or the device.  Returns one dict for a 1-D input, else
    a list-like of B dicts with host numpy arrays (device tensors if return_device=True)."""
    if not isinstance(loss_func, ProgramLoss):
        raise TypeError("loss_func must be a ProgramLoss(program, Loss(...)): the CUDA engine takes a "
                        "declarative spec instead of a Python closure")
    if method != 'adam':
        raise NotImplementedError(f"method {method!r}: only 'adam' is implemented (the reference marks the "
                                  "others as not well tested, main.py:344)")
    if kwargs:
        raise TypeError(f"unexpected arguments {sorted(kwargs)}")
    if regularization_func is not None and not isinstance(regularization_func, Penalty):
        raise TypeError("regularization_func must be a Penalty spec or None")
    program = loss_func.program
    P = program.n_params
    if num_params is not None and num_params != P:
        raise ValueError(f"num_params={num_params} but the program has {P} parameters")
    if target_loss != 1e-7:
        print('Warning: target loss not yet supported.')   # optimization.py:38-39
    if initial_params_batch is None:
        # optimization.py:304-311: PRNGKey(0) split chain.  Same distribution, drawn on the device.
        init = program.initial_angles(0, num_repeats, dtype=dtype, device=device)
        input_is_vector = num_repeats != 1
    else:
        if num_repeats != 1:
            print('Warning, initial conditions provided and number of repeats will be ignored.')
        shape = tuple(initial_params_batch.shape) if hasattr(initial_params_batch, 'shape') else \
            np.asarray(initial_params_batch).shape
        if len(shape) == 1:
            input_is_vector = False
        elif len(shape) == 2:
            input_is_vector = True
        else:
            raise ValueError('initial parameters must be either 1d or 2d array (multiple initial conditions)')
        init = _as_device_batch(initial_params_batch, dtype, device).reshape(-1, P)
    if freeze_mask is not None:
        freeze_mask = _as_device_batch(freeze_mask, torch.uint8, device).reshape(-1, P)
    raw = run_adam_batch(program, loss_func.loss, regularization_func, init, learning_rate, num_iterations,
                         freeze=freeze_mask, keep_history=keep_history)
    if not return_device:
        raw = raw.numpy()
    if not compute_losses or (regularization_func is None and not zero_regularization):
        # optimization.py:364, 376: without a regularizer 'loss' holds the (reg)loss history
        res = [{'params': raw.params[i], 'loss': raw.regloss[i]} for i in range(len(raw))]
        return res if input_is_vector else res[0]
    return raw if input_is_vector else raw[0]


def mynimize(loss_func, num_params=None, method='adam', learning_rate=0.1, u_func=None, target_loss=1e-7,
             keep_history=True, initial_params=None, num_iterations=5000, **kwargs):
    """Reference optimization.py:209-266 (single start): returns (angles_history, loss_history)."""
    res = mynimize_repeated(loss_func, num_params, method=method, learning_rate=learning_rate,
                            target_loss=target_loss, initial_params_batch=initial_params,
                            keep_history=keep_history, num_iterations=num_iterations, **kwargs)
    return res['params'], res['loss']


def unitary_learn(anz, u_target, num_params=None, method='adam', learning_rate=0.1, target_loss=1e-7,
                  disc_func=None, regularization_options=None, initial_angles=None, num_repeats=1,
                  keep_history=True, **kwargs):
    """Reference optimization.py:385-419: learn `u_target` with the ansatz `anz` (HS loss)."""
    if disc_func is not None:
        raise NotImplementedError("disc_func='swap' (matrix_utils.py:45-49) is outside the accelerated path")
    if regularization_options is not None:
        raise NotImplementedError("construct_penalty_function is deprecated/broken in the reference "
                                  "(penalty.py:101-119)")
    pl = ProgramLoss(anz.program, Loss('hs', u_target))
    res = mynimize_repeated(pl, num_params, method=method, learning_rate=learning_rate, target_loss=target_loss,
                            initial_params_batch=initial_angles, num_repeats=num_repeats,
                            regularization_func=None, zero_regularization=True,  # `lambda x: 0`, :407
                            keep_history=keep_history, **kwargs)
    return res
