"""Thin torch-facing wrapper over the C ABI: device buffers are torch CUDA tensors passed as raw
pointers on torch's current stream.  No computation happens here."""
import ctypes as C
import math
import warnings

import numpy as np
import torch

from . import _lib as L

_DT = {torch.float32: L.F32, torch.float64: L.F64}
_CDT = {torch.float32: torch.complex64, torch.float64: torch.complex128}


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _on(t):
    """Context that makes `t`'s device current: the C side launches on the current device (its per-device program
    tables, `cudaGetDevice`) and `_stream()` is torch's current stream OF that device."""
    return torch.cuda.device(t.device)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not (t.is_cuda and t.is_contiguous()):
            raise L.CpflowError("cpflow_b200 needs contiguous CUDA tensors (no CPU fallback)")


class Program:
    """Immutable gate program (cpf_program).  `ops` is a list of (kind, q0, q1, param, const_angle)."""

    def __init__(self, n_qubits, ops, n_params):
        lib = L.load()
        self.n_qubits = int(n_qubits)
        self.n_params = int(n_params)
        self.ops = [tuple(o) for o in ops]
        arr = (L.CpfOp * max(1, len(ops)))()
        for i, (kind, q0, q1, param, const) in enumerate(self.ops):
            arr[i] = L.CpfOp(int(kind), int(q0), int(q1), int(param), float(const))
        h = C.c_void_p()
        L.check(lib.cpf_program_create(self.n_qubits, len(self.ops), arr, self.n_params, C.byref(h)))
        self._h = h
        info = L.CpfProgramInfo()
        L.check(lib.cpf_program_get_info(self._h, C.byref(info)))
        self.info = {f[0]: getattr(info, f[0]) for f in L.CpfProgramInfo._fields_}

    def __reduce__(self):
        # handles are process-local: pickle the description and re-create on load
        return (Program, (self.n_qubits, self.ops, self.n_params))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and L._lib is not None:
            try:
                L._lib.cpf_program_destroy(h)
            except Exception:
                pass
            self._h = None

    @property
    def dim(self):
        return 2 ** self.n_qubits

    def eval_cost(self, loss_kind=L.LOSS_HS, dtype=torch.float32):
        f, b = C.c_double(), C.c_double()
        L.check(L.load().cpf_eval_cost(self._h, int(loss_kind), _DT[dtype], C.byref(f), C.byref(b)))
        return f.value, b.value

    def _note_engine(self, loss, dtype, batch):
        """One warning per program when a Hilbert-Schmidt run does not land on the Heisenberg-picture kernel (a
        non-block-structured gate list, 5 qubits in complex128, more than 32767 parameters or B * P >= 2^32): the
        state-adjoint kernels give the same numbers about five times slower."""
        if loss.kind != "hs" or getattr(self, "_warned_engine", False) or self.n_qubits > 5:
            return
        if self.launch_plan(max(1, int(batch)), L.LOSS_HS, dtype)["engine"] == 0:
            self._warned_engine = True
            warnings.warn(f"cpflow_b200: this {self.n_qubits}-qubit program ({self.info['n_ops']} gates, {dtype}) runs its "
                          "Hilbert-Schmidt loss on the state-adjoint kernels, not on the Heisenberg-picture kernel "
                          "(see Program._note_engine)", RuntimeWarning, stacklevel=3)

    def executed_cost(self, loss_kind=L.LOSS_HS, dtype=torch.float32):
        """Floating-point operations per evaluation the chosen kernel executes (cpf_executed_cost)."""
        f = C.c_double()
        L.check(L.load().cpf_executed_cost(self._h, int(loss_kind), _DT[dtype], C.byref(f)))
        return f.value

    def workspace_bytes(self, batch, loss_kind=L.LOSS_HS, dtype=torch.float32):
        """Device scratch one adam_run on `batch` samples needs (cpf_workspace_bytes); give AdamState.workspace a
        uint8 CUDA tensor of that size to keep the library out of the allocator."""
        n = C.c_int64()
        L.check(L.load().cpf_workspace_bytes(self._h, int(loss_kind), _DT[dtype], int(batch), C.byref(n)))
        return n.value

    def launch_plan(self, batch, loss_kind=L.LOSS_HS, dtype=torch.float32, n_sm=0, regs_per_thread=0):
        """The launch geometry the engine would use for `batch` samples (cpf_launch_plan; needs no device)."""
        info = L.CpfLaunchInfo()
        L.check(L.load().cpf_launch_plan(self._h, int(loss_kind), _DT[dtype], int(batch), int(n_sm),
                                         int(regs_per_thread), C.byref(info)))
        return {name: getattr(info, name) for name, _ in info._fields_ if name != "reserved"}

    # ---- forward / gradients -------------------------------------------------------------
    def unitary(self, angles):
        _need_cuda(angles)
        B = angles.shape[0]
        N = self.dim
        out = torch.empty(B, N, N, dtype=_CDT[angles.dtype], device=angles.device)
        with _on(angles):
            L.check(L.load().cpf_unitary(self._h, _DT[angles.dtype], B, _ptr(angles), _ptr(out), _stream()))
        return out

    def loss_grad(self, angles, loss, penalty=None, want_grad=True):
        _need_cuda(angles)
        B = angles.shape[0]
        dt = angles.dtype
        lo = torch.empty(B, dtype=dt, device=angles.device)
        rg = torch.empty(B, dtype=dt, device=angles.device)
        gr = torch.empty(B, self.n_params, dtype=dt, device=angles.device) if want_grad else None
        ls = loss.spec(dt, angles.device)
        ps = penalty.spec() if penalty is not None else None
        if want_grad:          # loss-only evaluation of arbitrary gate lists (refine) is the state kernels' job
            self._note_engine(loss, dt, B)
        with _on(angles):
            L.check(L.load().cpf_loss_grad(self._h, C.byref(ls), C.byref(ps) if ps is not None else None,
                                           _DT[dt], B, _ptr(angles), _ptr(lo), _ptr(rg), _ptr(gr), _stream()))
        return lo, rg, gr

    def adjoint_from_cotangent(self, angles, cotangent):
        _need_cuda(angles, cotangent)
        B = angles.shape[0]
        gr = torch.empty(B, self.n_params, dtype=angles.dtype, device=angles.device)
        with _on(angles):
            L.check(L.load().cpf_adjoint_from_cotangent(self._h, _DT[angles.dtype], B, _ptr(angles),
                                                        _ptr(cotangent), _ptr(gr), _stream()))
        return gr

    def count_cz(self, angles, threshold=0.2, project=False):
        _need_cuda(angles)
        B = angles.shape[0]
        cz = torch.empty(B, dtype=torch.int32, device=angles.device)
        proj = torch.empty_like(angles) if project else None
        frozen = torch.empty(B, self.n_params, dtype=torch.uint8, device=angles.device) if project else None
        with _on(angles):
            L.check(L.load().cpf_count_cz(self._h, _DT[angles.dtype], B, _ptr(angles), float(threshold),
                                          _ptr(cz), _ptr(proj), _ptr(frozen), _stream()))
        return (cz, proj, frozen) if project else cz

    def initial_angles(self, seed, total_samples, first=0, count=None, cp_dist="uniform",
                       dtype=torch.float32, device="cuda"):
        count = total_samples - first if count is None else count
        out = torch.empty(count, self.n_params, dtype=dtype, device=device)
        code = {"uniform": 0, "0": 1, "normal": 2}.get(cp_dist)
        if code is None:
            raise L.CpflowError(f"cp_dist {cp_dist!r} is not supported on the device sampler")
        with torch.cuda.device(out.device):
            L.check(L.load().cpf_initial_angles(self._h, _DT[dtype], int(seed), int(total_samples), int(first),
                                                int(count), code, _ptr(out), _stream()))
        return out

    # ---- the fused Adam loop ---------------------------------------------------------------
    def adam_state(self, angles, freeze=None, hist_len=0):
        return AdamState(self, angles, freeze, hist_len)

    def adam_run(self, state, loss, penalty, lr, num_steps, b1=0.9, b2=0.999, eps=1e-8):
        dt = state.angles.dtype
        ls = loss.spec(dt, state.angles.device)
        ps = penalty.spec() if penalty is not None else None
        ad = L.CpfAdamSpec(float(lr), float(b1), float(b2), float(eps))
        buf = state.buffers()
        self._note_engine(loss, dt, state.batch)
        with _on(state.angles):
            L.check(L.load().cpf_adam_run(self._h, C.byref(ls), C.byref(ps) if ps is not None else None,
                                          C.byref(ad), _DT[dt], state.batch, state.step, int(num_steps),
                                          C.byref(buf), _stream()))
        state.step += int(num_steps)
        return state


    # ---- many targets in one launch ------------------------------------------------------------
    def workspace_bytes_multi(self, batch, n_targets, loss_kind=L.LOSS_HS, dtype=torch.float32):
        """Device scratch one adam_run_multi over `batch` samples and `n_targets` targets needs
        (cpf_workspace_bytes_multi)."""
        n = C.c_int64()
        L.check(L.load().cpf_workspace_bytes_multi(self._h, int(loss_kind), _DT[dtype], int(batch), int(n_targets),
                                                   C.byref(n)))
        return n.value

    def _target_index(self, loss, target_index, batch):
        """Host int32 copy of `target_index` after the checks that need no device (the library checks the range)."""
        if not isinstance(loss, MultiLoss):
            raise TypeError("the multi-target entry points take a MultiLoss(kind, targets)")
        loss.check_program(self)
        idx = np.ascontiguousarray(
            target_index.detach().cpu().numpy() if isinstance(target_index, torch.Tensor) else target_index,
            dtype=np.int32).reshape(-1)
        if idx.shape[0] != batch:
            raise ValueError(f"target_index has {idx.shape[0]} entries for a batch of {batch}")
        return idx

    def loss_grad_multi(self, angles, loss, target_index, penalty=None, want_grad=True):
        """loss_grad with sample b scored against loss.targets[target_index[b]] (cpf_loss_grad_multi)."""
        B = angles.shape[0]
        idx = self._target_index(loss, target_index, B)
        _need_cuda(angles)
        dt = angles.dtype
        tt = loss.table(dt, angles.device, idx)
        lo = torch.empty(B, dtype=dt, device=angles.device)
        rg = torch.empty(B, dtype=dt, device=angles.device)
        gr = torch.empty(B, self.n_params, dtype=dt, device=angles.device) if want_grad else None
        ps = penalty.spec() if penalty is not None else None
        with _on(angles):
            L.check(L.load().cpf_loss_grad_multi(self._h, C.byref(tt), C.byref(ps) if ps is not None else None,
                                                 _DT[dt], B, _ptr(angles), _ptr(lo), _ptr(rg), _ptr(gr), _stream()))
        return lo, rg, gr

    def adam_run_multi(self, state, loss, target_index, penalty, lr, num_steps, b1=0.9, b2=0.999, eps=1e-8):
        """adam_run with sample b optimised against loss.targets[target_index[b]] (cpf_adam_run_multi); the index
        must be the same for every call that continues the same state."""
        dt = state.angles.dtype
        idx = self._target_index(loss, target_index, state.batch)
        tt = loss.table(dt, state.angles.device, idx)
        ps = penalty.spec() if penalty is not None else None
        ad = L.CpfAdamSpec(float(lr), float(b1), float(b2), float(eps))
        buf = state.buffers()
        with _on(state.angles):
            L.check(L.load().cpf_adam_run_multi(self._h, C.byref(tt), C.byref(ps) if ps is not None else None,
                                                C.byref(ad), _DT[dt], state.batch, state.step, int(num_steps),
                                                C.byref(buf), _stream()))
        state.step += int(num_steps)
        return state

    def adam_step(self, state, loss_values, grad, penalty, lr, b1=0.9, b2=0.999, eps=1e-8):
        """One iteration of the Adam loop for a loss evaluated outside the engine (cpf_adam_step): penalty, best
        tracking and the Adam update on `state`, given loss_values [B] and grad [B,P] = d loss / d theta."""
        _need_cuda(loss_values, grad)
        dt = state.angles.dtype
        ps = penalty.spec() if penalty is not None else None
        ad = L.CpfAdamSpec(float(lr), float(b1), float(b2), float(eps))
        buf = state.buffers()
        with _on(state.angles):
            L.check(L.load().cpf_adam_step(self._h, C.byref(ps) if ps is not None else None, C.byref(ad), _DT[dt],
                                           state.batch, state.step, _ptr(loss_values), _ptr(grad), C.byref(buf),
                                           _stream()))
        state.step += 1
        return state


class AdamState:
    """Device buffers of one multi-start Adam run (cpf_adam_buffers)."""

    def __init__(self, program, angles, freeze=None, hist_len=0):
        _need_cuda(angles, freeze)
        self.program = program
        self.angles = angles  # updated in place
        B, P = angles.shape
        self.batch = B
        dev, dt = angles.device, angles.dtype
        self.m = torch.empty_like(angles)
        self.v = torch.empty_like(angles)
        self.freeze = freeze
        self.best_params = torch.empty_like(angles)
        self.best_regloss = torch.empty(B, dtype=dt, device=dev)
        self.best_reg = torch.empty(B, dtype=dt, device=dev)
        self.init_regloss = torch.empty(B, dtype=dt, device=dev)
        self.init_reg = torch.empty(B, dtype=dt, device=dev)
        self.hist_len = int(hist_len)
        # rows start as the initial angles: parameters that feed no gate are never written by the kernels
        self.hist_params = angles[:, None, :].repeat(1, hist_len, 1).contiguous() if hist_len else None
        self.hist_regloss = torch.zeros(B, hist_len, dtype=dt, device=dev) if hist_len else None
        self.step = 0
        self.workspace = None      # optional caller-owned scratch (uint8 CUDA tensor), see Program.workspace_bytes

    def buffers(self):
        return L.CpfAdamBuffers(
            _ptr(self.angles).value, _ptr(self.m).value, _ptr(self.v).value, _ptr(self.freeze).value,
            _ptr(self.best_params).value, _ptr(self.best_regloss).value, _ptr(self.best_reg).value,
            _ptr(self.init_regloss).value, _ptr(self.init_reg).value, _ptr(self.hist_params).value,
            _ptr(self.hist_regloss).value, self.hist_len, _ptr(self.workspace).value,
            self.workspace.numel() if self.workspace is not None else 0)


class Loss:
    """Declarative loss spec (cpf_loss_spec): 'hs' | 'state' | 'relphase' | 'isometry' and a target array.

    'isometry' takes `ancillas`, the qubits that start in |0>: with k = 2^(n - len(ancillas)) and s_0 < ... < s_{k-1}
    the basis states whose ancilla qubits are 0, the target W is N x k (column c = the wanted image of |s_c>) and the
    loss is 1 - |sum_c <W e_c| U |s_c>|^2 / k^2 (one global phase, like 'hs')."""
    KINDS = {"hs": L.LOSS_HS, "state": L.LOSS_STATE, "relphase": L.LOSS_RELPHASE, "isometry": L.LOSS_ISOMETRY}

    def __init__(self, kind, target, ancillas=None):
        if kind not in self.KINDS:
            raise ValueError(f"unknown loss kind {kind!r}")
        if ancillas is not None and kind != "isometry":
            raise ValueError(f"ancillas are an argument of the 'isometry' loss, not of {kind!r}")
        self.kind = kind
        self.target = np.asarray(target.detach().cpu().numpy() if isinstance(target, torch.Tensor) else target,
                                 dtype=np.complex128)
        self.ancillas = ()
        if kind == "isometry":
            self.ancillas = _check_isometry(self.target, ancillas)
        self._dev = {}

    @property
    def ancilla_mask(self):
        return sum(1 << q for q in self.ancillas)

    @property
    def columns(self):
        """Basis indices s_0 < ... < s_{k-1} of the input columns ('isometry'): ancilla qubits (big-endian) are 0."""
        n = int(self.target.shape[0]).bit_length() - 1
        bits = sum(1 << (n - 1 - q) for q in self.ancillas)
        return tuple(s for s in range(2 ** n) if s & bits == 0)

    @property
    def code(self):
        """The loss-kind argument of the query entry points (workspace_bytes, launch_plan, eval_cost, executed_cost)."""
        return L.isometry_kind(self.ancilla_mask) if self.kind == "isometry" else self.KINDS[self.kind]

    def spec(self, dtype, device):
        key = (dtype, str(device))
        if key not in self._dev:
            self._dev[key] = torch.as_tensor(self.target, dtype=_CDT[dtype]).contiguous().to(device)
        return L.CpfLossSpec(self.KINDS[self.kind], self._dev[key].data_ptr(), self.ancilla_mask)

    def __getstate__(self):
        return {"kind": self.kind, "target": self.target, "ancillas": self.ancillas}

    def __setstate__(self, st):
        self.kind, self.target, self._dev = st["kind"], st["target"], {}
        self.ancillas = tuple(st.get("ancillas", ()))

    def __call__(self, u):
        """Value of the loss at an explicit unitary `u` (host utility with the formulas of
        matrix_utils.py:35-42 and the tutorial's state / relative-phase losses; the optimisation
        itself never goes through here)."""
        u = np.asarray(u.detach().cpu().numpy() if isinstance(u, torch.Tensor) else u)
        n = u.shape[0]
        if self.kind == "hs":
            return float(1 - np.abs((u * self.target.conj()).sum()) ** 2 / n ** 2)
        if self.kind == "state":
            return float(1 - np.abs((self.target.conj() * u[:, 0]).sum()) ** 2)
        if self.kind == "isometry":
            k = self.target.shape[1]
            return float(1 - np.abs((self.target.conj() * u[:, list(self.columns)]).sum()) ** 2 / k ** 2)
        return float(1 - (np.abs(self.target.conj() * u) ** 2).sum() / n)

    def __repr__(self):
        if self.kind == "isometry":
            return f"Loss('isometry', target{tuple(self.target.shape)}, ancillas={list(self.ancillas)})"
        return f"Loss({self.kind!r}, target{tuple(self.target.shape)})"


def _check_isometry(W, ancillas):
    """Shape checks of an 'isometry' target: W is N x k with N = 2^n and k = 2^(n - len(ancillas)); the ancillas are
    distinct qubits in [0, n).  Returns the sorted ancilla tuple."""
    if ancillas is None:
        raise ValueError("the 'isometry' loss needs `ancillas` (the qubits that start in |0>; [] for none)")
    anc = [int(q) for q in ancillas]
    if W.ndim != 2 or W.shape[0] < 2 or W.shape[0] & (W.shape[0] - 1):
        raise ValueError(f"an 'isometry' target is N x k with N = 2^n rows, got shape {W.shape}")
    n = W.shape[0].bit_length() - 1
    if len(set(anc)) != len(anc) or any(q < 0 or q >= n for q in anc):
        raise ValueError(f"ancillas {list(ancillas)} must be distinct qubits in [0, {n})")
    k = 2 ** (n - len(anc))
    if W.shape[1] != k:
        raise ValueError(f"an 'isometry' target with {len(anc)} ancillas on {n} qubits is {2 ** n} x {k}, "
                         f"got shape {W.shape}")
    return tuple(sorted(anc))


def clean_ancilla_isometry(G, ancillas, n):
    """Target W of Loss('isometry', W, ancillas) for a unitary G on the data qubits (the n - len(ancillas) qubits that
    are not ancillas, in increasing order, big-endian) when the ancillas must return to |0>: column c of W is the
    state with the data qubits in G|c> and every ancilla in |0>."""
    G = np.asarray(G, dtype=np.complex128)
    anc = sorted(set(int(q) for q in ancillas))
    if any(q < 0 or q >= n for q in anc):
        raise ValueError(f"ancillas {list(ancillas)} must be qubits in [0, {n})")
    data = [q for q in range(n) if q not in anc]
    k = 2 ** len(data)
    if G.shape != (k, k):
        raise ValueError(f"G acts on {len(data)} data qubits: expected shape {(k, k)}, got {G.shape}")
    rows = [sum(((d >> (len(data) - 1 - i)) & 1) << (n - 1 - q) for i, q in enumerate(data)) for d in range(k)]
    W = np.zeros((2 ** n, k), dtype=np.complex128)
    W[rows, :] = G
    return W


class MultiLoss:
    """Declarative loss over many targets (cpf_target_table): one kind ('hs' | 'state' | 'relphase') and `targets`
    of shape [T, N, N] ('hs', 'relphase') or [T, N] ('state').  Sample b of a multi-target call is scored against
    targets[target_index[b]]."""

    def __init__(self, kind, targets):
        if kind not in Loss.KINDS:
            raise ValueError(f"unknown loss kind {kind!r}")
        t = np.asarray(targets.detach().cpu().numpy() if isinstance(targets, torch.Tensor) else targets,
                       dtype=np.complex128)
        want = 2 if kind == "state" else 3
        if t.ndim != want or t.shape[0] < 1 or (want == 3 and t.shape[1] != t.shape[2]):
            raise ValueError(f"MultiLoss({kind!r}) takes targets of shape " + ("[T, N]" if want == 2 else "[T, N, N]") +
                             f" with T >= 1, got {t.shape}")
        self.kind = kind
        self.targets = t
        self._dev = {}

    @property
    def n_targets(self):
        return self.targets.shape[0]

    def check_program(self, program):
        if self.targets.shape[1] != program.dim:
            raise ValueError(f"targets of dimension {self.targets.shape[1]} for a {program.n_qubits}-qubit program "
                             f"(dimension {program.dim})")

    def table(self, dtype, device, index):
        """cpf_target_table over the device copy of the targets (cached per dtype and device); `index` is the host
        int32 array the table points to and must outlive the call."""
        key = (dtype, str(device))
        if key not in self._dev:
            self._dev[key] = torch.as_tensor(self.targets, dtype=_CDT[dtype]).contiguous().to(device)
        return L.CpfTargetTable(Loss.KINDS[self.kind], self.n_targets, self._dev[key].data_ptr(), index.ctypes.data)

    def loss(self, i):
        """The single-target Loss of target i."""
        return Loss(self.kind, self.targets[i])

    def __getstate__(self):
        return {"kind": self.kind, "targets": self.targets}

    def __setstate__(self, st):
        self.kind, self.targets, self._dev = st["kind"], st["targets"], {}

    def __repr__(self):
        return f"MultiLoss({self.kind!r}, targets{tuple(self.targets.shape)})"


class TorchLoss:
    """An arbitrary user loss `unitary_loss_func(U)` (reference main.py:528-529) written with torch operations:
    a function of ONE unitary (complex tensor [N,N]) returning a real scalar tensor.  It cannot run inside the
    fused kernel, so the optimisation alternates cpf_unitary -> this function and its autograd cotangent ->
    cpf_adjoint_from_cotangent -> cpf_adam_step (optimization.run_adam_batch); the Adam arithmetic, penalty, best
    tracking and freeze masks are the engine's own."""

    def __init__(self, fn):
        if not callable(fn):
            raise TypeError("unitary_loss_func must be a Loss spec or a callable of a torch unitary")
        self.fn = fn
        self._vmap_ok = None

    def batch(self, U):
        """Loss of every unitary of U [B,N,N] -> real tensor [B] (torch.vmap when the function allows it)."""
        if self._vmap_ok is not False:
            try:
                out = torch.vmap(self.fn)(U)
                self._vmap_ok = True
                return out.real if out.is_complex() else out
            except Exception:
                if self._vmap_ok:
                    raise
                self._vmap_ok = False
        out = torch.stack([torch.as_tensor(self.fn(u)) for u in U])
        return out.real if out.is_complex() else out

    def value_and_cotangent(self, U):
        """loss [B] and dL/dconj(U) [B,N,N] (the seed of cpf_adjoint_from_cotangent): torch's gradient of a real
        function with respect to a complex tensor is 2 dL/dconj(U)."""
        U = U.detach().requires_grad_(True)
        with torch.enable_grad():
            loss = self.batch(U)
            (g,) = torch.autograd.grad(loss.sum(), U)
        return loss.detach(), (g / 2).contiguous()

    def __call__(self, u):
        """Value at one explicit unitary (numpy or torch) -> float."""
        t = torch.as_tensor(np.asarray(u)) if not isinstance(u, torch.Tensor) else u
        with torch.no_grad():
            v = self.fn(t)
        v = torch.as_tensor(v)
        return float(v.real if v.is_complex() else v)

    def __repr__(self):
        return f"TorchLoss({getattr(self.fn, '__name__', self.fn)!r})"


class Penalty:
    """Declarative penalty spec (cpf_penalty_spec)."""

    def __init__(self, kind, r, segments=None, period=2 * math.pi, cp_mask=None):
        self.kind = kind
        self.r = float(r)
        self.segments = list(segments or [])
        self.period = float(period)
        self.cp_mask = None if cp_mask is None else np.ascontiguousarray(cp_mask, dtype=np.uint8)
        if len(self.segments) > L.MAX_SEGMENTS:
            raise ValueError("too many penalty segments")

    def spec(self):
        s = L.CpfPenaltySpec()
        s.kind = {"none": L.PEN_NONE, "piecewise": L.PEN_PIECEWISE, "l1": L.PEN_L1}[self.kind]
        s.n_segments = len(self.segments)
        s.r = self.r
        s.period = self.period
        for i, (lo, hi, slope, icpt) in enumerate(self.segments):
            s.lo[i], s.hi[i], s.slope[i], s.intercept[i] = lo, hi, slope, icpt
        s.cp_mask = self.cp_mask.ctypes.data if self.cp_mask is not None else None
        return s
