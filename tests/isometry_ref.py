"""Float64 autograd references of the isometry losses, built on the oracle's program unitary, penalty and optax Adam.
With t_c = <W e_c| U |s_c> and s_c the basis states whose ancilla qubits (big-endian) are 0:
  'isometry' (one global phase):            L = 1 - |sum_c t_c|^2 / k^2
  'isometry_relphase' (a phase per column): L = 1 - sum_c |t_c|^2 / k"""
import torch

from oracle import cpflow_oracle as O


def columns(n, ancillas):
    bits = sum(1 << (n - 1 - q) for q in ancillas)
    return [s for s in range(2 ** n) if s & bits == 0]


def loss_batched(u, W, cols):
    t = (W.conj()[None] * u[:, :, cols]).sum((-1, -2))
    return 1 - torch.abs(t) ** 2 / W.shape[1] ** 2


def relphase_loss_batched(u, W, cols):
    t = (W.conj()[None] * u[:, :, cols]).sum(-2)                  # [B, k]: t_c = <W e_c| U |s_c>
    return 1 - (torch.abs(t) ** 2).sum(-1) / W.shape[1]


def loss_and_grad_batched(n, ops, angles, W, ancillas, cp_mask=None, r=0.0, penalty_func=None, relphase=False):
    """(loss [B], reg [B], grad [B,P]) with grad = d(loss + reg)/d(angles), as O.loss_and_grad_batched; relphase=True:
    the relative-phase isometry loss."""
    W = torch.as_tensor(W, dtype=torch.complex128)
    a = angles.clone().double().requires_grad_(True)
    u = O.program_unitary_batched(n, ops, a)
    loss = (relphase_loss_batched if relphase else loss_batched)(u, W, columns(n, ancillas))
    reg = O.regularization_value(a, cp_mask, r, penalty_func) if penalty_func is not None else torch.zeros_like(loss)
    (loss + reg).sum().backward()
    return loss.detach(), reg.detach(), a.grad.detach()


def mynimize_repeated(n, ops, W, ancillas, x0, learning_rate, num_iterations, cp_mask=None, r=0.0, penalty_func=None,
                      freeze_mask=None, relphase=False):
    """O.mynimize_repeated for the isometry losses: params [B,2,P] (initial, best) and regloss [B,2]."""
    def lg(p):
        loss, reg, g = loss_and_grad_batched(n, ops, p, W, ancillas, cp_mask, r, penalty_func, relphase)
        return loss + reg, g
    return O.adam_minimize_batched(lg, torch.as_tensor(x0).double(), learning_rate, num_iterations,
                                   freeze_mask=freeze_mask)
