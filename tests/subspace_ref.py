"""Float64 autograd references of the subspace losses, built on the oracle's program unitary, penalty and optax Adam.
With A = [a_0 .. a_{k-1}] the input states, B = [b_0 .. b_{k-1}] their wanted images and t_c = <b_c| U |a_c>:
  'subspace' (one global phase):          L = 1 - |sum_c t_c|^2 / k^2
  'subspace_relphase' (a phase per pair): L = 1 - sum_c |t_c|^2 / k"""
import torch

from oracle import cpflow_oracle as O


def overlaps(u, A, B):
    """t [batch, k]: t_c = <b_c| U |a_c>"""
    return (B.conj()[None] * (u @ A[None])).sum(-2)


def loss_batched(u, A, B, kind):
    t = overlaps(u, A, B)
    k = A.shape[1]
    if kind == "subspace":
        return 1 - torch.abs(t.sum(-1)) ** 2 / k ** 2
    return 1 - (torch.abs(t) ** 2).sum(-1) / k


def loss_and_grad_batched(n, ops, angles, A, B, kind, cp_mask=None, r=0.0, penalty_func=None):
    """(loss [batch], reg [batch], grad [batch,P]) with grad = d(loss + reg)/d(angles), as O.loss_and_grad_batched."""
    A = torch.as_tensor(A, dtype=torch.complex128)
    B = torch.as_tensor(B, dtype=torch.complex128)
    a = angles.clone().double().requires_grad_(True)
    u = O.program_unitary_batched(n, ops, a)
    loss = loss_batched(u, A, B, kind)
    reg = O.regularization_value(a, cp_mask, r, penalty_func) if penalty_func is not None else torch.zeros_like(loss)
    (loss + reg).sum().backward()
    return loss.detach(), reg.detach(), a.grad.detach()


def mynimize_repeated(n, ops, A, B, kind, x0, learning_rate, num_iterations, cp_mask=None, r=0.0, penalty_func=None,
                      freeze_mask=None):
    """O.mynimize_repeated for the subspace losses: params [batch,2,P] (initial, best) and regloss [batch,2]."""
    def lg(p):
        loss, reg, g = loss_and_grad_batched(n, ops, p, A, B, kind, cp_mask, r, penalty_func)
        return loss + reg, g
    return O.adam_minimize_batched(lg, torch.as_tensor(x0).double(), learning_rate, num_iterations,
                                   freeze_mask=freeze_mask)


def adam_replay(n, ops, A, B, kind, hist_params, learning_rate, cp_mask=None, r=0.0, penalty_func=None, chunk=256):
    """Every step of a recorded Adam run, replayed: given the angles theta_0 .. theta_{T-1} a run recorded
    (hist_params [batch,T,P]), returns (regloss [batch,T], predicted [batch,T-1,P]) where regloss[:, i] is the reference
    loss plus penalty at theta_i and predicted[:, i] = theta_i + the optax Adam update from the reference gradients at
    theta_0 .. theta_i.  Each step is checked from the run's own state, so rounding does not compound along the run."""
    Bt, T, P = hist_params.shape
    flat = torch.as_tensor(hist_params, dtype=torch.float64).reshape(Bt * T, P)
    rl, gr = [], []
    for s in range(0, flat.shape[0], chunk):
        lo, rg, g = loss_and_grad_batched(n, ops, flat[s:s + chunk], A, B, kind, cp_mask, r, penalty_func)
        rl.append(lo + rg)
        gr.append(g)
    regloss = torch.cat(rl).reshape(Bt, T)
    grad = torch.cat(gr).reshape(Bt, T, P)
    th = flat.reshape(Bt, T, P)
    st = O.AdamState(th[:, 0])
    pred = torch.empty(Bt, T - 1, P, dtype=torch.float64)
    for i in range(T - 1):
        pred[:, i] = th[:, i] + O.adam_update(grad[:, i], st, learning_rate)
    return regloss, pred
