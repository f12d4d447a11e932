"""User-facing API (mirror of reference cpflow/main.py:242-864): options, Results, Decomposition and
the multi-sample driver `Synthesize`.

Same names, defaults, printed lines and result shapes as the reference; what changes is underneath:
every numeric stage runs in the CUDA engine (sampling, the fused Adam loop, selection, projection,
batched verification), samples shard over the GPUs of one box when a torch.distributed process
group is initialised (cpflow_b200/parallel.py), and losses / penalties are declarative specs
(`Loss`, `PenaltyFunction`) instead of Python closures.
"""
import math
import os
import pickle
from dataclasses import asdict, dataclass

import numpy as np
import torch

from . import parallel as PL
from .ansatz import Ansatz
from .circuit import convert_to_ZXZ, cp_template_cz_count_depth, cp_to_cz_circuit, gates_count, gates_depth
from .cp_utils import (filter_cp_results, random_cp_angles, select_batch, verify_cp_result, verify_cp_results)
from .engine import Loss, MultiLoss, Penalty, TorchLoss
from .optimization import ProgramLoss, RawResults, mynimize_repeated, run_adam_batch
from .penalty import PenaltyFunction, RegularizationOptions, make_regularization_function, tabulate_penalty
from .matrix_utils import theoretical_lower_bound
from .topology import fill_layers, num_qubits_from_layer

try:  # the reference saves with dill; user-supplied callables (a custom unitary_loss_func) need it to be saved
    import dill as _pickler
except ImportError:  # pragma: no cover - spec-based objects (Loss, PenaltyFunction, options, circuits) pickle plainly
    _pickler = pickle

# first bytes of a file written by Results.save(): tells our own files from the reference's dill files
_MAGIC = b'CPFLOW_B200_RESULTS\x01\n'

try:
    from tqdm import tqdm
except ImportError:  # pragma: no cover
    def tqdm(x, **kw):
        return x


def batched_unitary_loss(unitary_loss_func, U):
    """`unitary_loss_func` on a batch U [B,N,N] of device unitaries -> numpy [B].  Declarative `Loss` specs are
    evaluated vectorised on the device with the formulas of `Loss.__call__` (matrix_utils.py:35-42 and the
    tutorial's state / relative-phase losses); any other callable is applied to each unitary in turn."""
    if isinstance(unitary_loss_func, Loss):
        tgt = torch.as_tensor(unitary_loss_func.target).to(U.device, U.dtype)
        n = U.shape[-1]
        if unitary_loss_func.kind == 'hs':
            return (1 - (U * tgt.conj()).sum((-1, -2)).abs() ** 2 / n ** 2).cpu().numpy()
        if unitary_loss_func.kind == 'state':
            return (1 - (tgt.conj() * U[:, :, 0]).sum(-1).abs() ** 2).cpu().numpy()
        if unitary_loss_func.kind == 'isometry':
            k = tgt.shape[1]
            t = (tgt.conj() * U[:, :, list(unitary_loss_func.columns)]).sum((-1, -2))
            return (1 - t.abs() ** 2 / k ** 2).cpu().numpy()
        return (1 - ((tgt.conj() * U).abs() ** 2).sum((-1, -2)) / n).cpu().numpy()
    if isinstance(unitary_loss_func, TorchLoss):
        with torch.no_grad():
            return unitary_loss_func.batch(U).cpu().numpy()
    return np.array([float(unitary_loss_func(u)) for u in U.cpu().numpy()])


class Decomposition:
    """One decomposition: circuit (gate list), its unitary, loss, CZ count / depth (main.py:242-325).

    Attributes mirror the reference: unitary_loss_func, circuit, unitary, label, loss, type,
    cz_count, cz_depth, t_count, t_depth and the provenance fields _cp_data, _static_options,
    _adaptive_options, _decomposer.

    Decompositions made by `Synthesize.static()` come out of ONE batched device evaluation
    (`_from_cp_batch`): unitary, loss and CZ count are there at once; the gate-list `circuit` (CP -> CZ
    rewriting, ZXZ merging: host Python, ~1 ms each) is built on first access.
    """

    def __init__(self, unitary_loss_func, circuit, label='', type='Approximate'):
        self.unitary_loss_func = unitary_loss_func
        self._circuit = circuit
        self.unitary = circuit.unitary()                 # evaluated by the CUDA engine (cpf_unitary)
        self.label = label
        self.loss = self.unitary_loss_func(self.unitary)
        self.type = type
        self.cz_count = gates_count(['cz'], circuit)
        self._cz_depth = gates_depth(['cz'], circuit)
        self.t_count = None
        self.t_depth = None
        self._cp_data = None
        self._static_options = None
        self._adaptive_options = None
        self._decomposer = None

    # ---- lazily materialised fields ----
    @property
    def circuit(self):
        if self.__dict__.get('_circuit') is None:
            u_func, circ_func, angles = self._cp_data
            self._circuit = convert_to_ZXZ(cp_to_cz_circuit(circ_func(angles), cp_threshold=1e-6))
        return self._circuit

    @circuit.setter
    def circuit(self, qc):
        self._circuit = qc

    @property
    def cz_depth(self):
        if self.__dict__.get('_cz_depth') is None:
            self._cz_depth = gates_depth(['cz'], self.circuit)
        return self._cz_depth

    @cz_depth.setter
    def cz_depth(self, v):
        self._cz_depth = v

    @classmethod
    def _from_cp_circuit(cls, unitary_loss_func, u_func, circ_func, angles, label):
        """main.py:281-291: CP template at `angles` -> CZ circuit with merged ZXZ rotations."""
        qc = circ_func(angles)
        qc = cp_to_cz_circuit(qc, cp_threshold=1e-6)
        qc = convert_to_ZXZ(qc)
        d = cls(unitary_loss_func, qc, label=label)
        d._cp_data = [u_func, circ_func, angles]
        return d

    @classmethod
    def _from_cp_batch(cls, unitary_loss_func, anz, full_angles, frozen, label='', device=None):
        """`_from_cp_circuit` for a whole batch of verified results in one device pass.  full_angles [B,P]: the
        template's angle vectors (projected CP angles already inserted); frozen [B,P] bool: which entries are the
        fixed ones (`constrained_function`, cp_utils.py:100-108).  The CZ circuit of main.py:283-286 is the CP
        template with CP(0) dropped, CP(pi) -> CZ and every other CP -> two CZ (exact_decompositions.py:42-74,
        threshold 1e-6), so its unitary is the template's up to a global phase: ONE batched cpf_unitary in
        complex128 gives every `unitary`, the losses are evaluated on that batch, CZ count and depth follow from
        the CP angles, and the gate list is built when `circuit` is first read."""
        from .cp_utils import _constrained_funcs
        full_angles = np.asarray(full_angles)
        frozen = np.asarray(frozen, dtype=bool)
        B = len(full_angles)
        if B == 0:
            return []
        dev = device if device is not None else torch.device('cuda', torch.cuda.current_device())
        a64 = torch.as_tensor(full_angles.astype(np.float64)).to(dev).contiguous()
        U = anz.program.unitary(a64)
        losses = batched_unitary_loss(unitary_loss_func, U)
        U = U.cpu().numpy()
        cp_idx = np.flatnonzero(np.asarray(anz.cp_mask) == 1)
        cz_count, cz_depth = cp_template_cz_count_depth(anz.all_placements, full_angles[:, cp_idx], anz.num_qubits)
        out = []
        for b in range(B):
            fixed_idx = np.flatnonzero(frozen[b])
            free = full_angles[b][~frozen[b]]
            circ_func, u_func = _constrained_funcs(anz, full_angles[b][fixed_idx], fixed_idx)
            d = object.__new__(cls)
            d.unitary_loss_func = unitary_loss_func
            d._circuit = None
            d.unitary = U[b]
            d.label = label
            d.loss = float(losses[b])
            d.type = 'Approximate'
            d.cz_count = int(cz_count[b])
            d._cz_depth = int(cz_depth[b])
            d.t_count = d.t_depth = None
            d._cp_data = [u_func, circ_func, free]
            d._static_options = d._adaptive_options = d._decomposer = None
            out.append(d)
        return out

    def refine(self, max_denominator=32, angle_threshold=0.01, cp_threshold=0.01, reduce_threshold=1e-5,
               recursion_degree=0, recursion_depth=5):
        """main.py:293-319 / exact_decompositions.py:293-344 (angle reduction and rationalisation on the
        forward-only engine; the Solovay-Kitaev / Clifford+T stage needs qiskit and is not provided)."""
        from .exact_decompositions import refine
        qc, refine_type, t_count, t_depth = refine(self.circuit, self.unitary_loss_func,
                                                   max_denominator=max_denominator, angle_threshold=angle_threshold,
                                                   cp_threshold=cp_threshold, reduce_threshold=reduce_threshold)
        self.type = refine_type
        self.circuit = qc
        if refine_type == 'Clifford+T':
            self.t_count, self.t_depth = t_count, t_depth
        return f'Refined to {refine_type}'

    def __repr__(self):
        description = (f"< {self.label}| {self.type} | loss: {self.loss}  | CZ count: {self.cz_count} | "
                       f"CZ depth: {self.cz_depth}  >")
        if self.type == 'Clifford+T':
            description = description[:-1] + f'| T count: {self.t_count} | T depth: {self.t_depth} >'
        return description


@dataclass
class BasicOptions:
    """Options shared by static and adaptive synthesis (main.py:338-367; same names and defaults)."""
    num_samples: int = 100
    method: str = 'adam'
    learning_rate: float = 0.1
    num_gd_iterations: int = 2000
    cp_distribution: str = 'uniform'
    entry_loss: float = 1e-3
    target_loss: float = 1e-6
    threshold_cp: float = 0.2
    learning_rate_at_verification: float = 0.01
    num_gd_iterations_at_verification: int = 5000
    random_seed: int = 0
    rotation_gates: str = 'xyz'


@dataclass
class StaticOptions(BasicOptions):
    """main.py:370-388: fixed template length `num_cp_gates`, regularisation weight `r`, and the CZ
    count below which prospective results are verified."""
    num_cp_gates: int = -1
    r: float = 0.00055
    accepted_num_cz_gates: int = -1

    def __post_init__(self):
        if self.num_cp_gates == -1:
            raise TypeError("Missing required argument 'num_cp_gates'")
        if self.accepted_num_cz_gates == -1:
            raise TypeError("Missing required argument 'accepted_num_cz_gates'")


@dataclass
class AdaptiveOptions(BasicOptions):
    """main.py:391-426."""
    min_num_cp_gates: int = -1
    max_num_cp_gates: int = -1
    r_mean: float = 0.00055
    r_variance: float = 0.5
    max_evals: int = 100
    target_num_cz_gates: int = 0
    stop_if_target_reached: bool = False
    keep_logs: bool = False

    def __post_init__(self):
        if self.min_num_cp_gates == -1:
            raise TypeError("Missing required argument 'min_num_cp_gates'")
        if self.max_num_cp_gates == -1:
            raise TypeError("Missing required argument 'max_num_cp_gates'")

    def get_static(self, num_cp_gates, r):
        basic = {k: v for k, v in asdict(self).items() if k in asdict(BasicOptions())}
        basic['num_cp_gates'] = num_cp_gates
        basic['r'] = r
        basic['accepted_num_cz_gates'] = None
        return StaticOptions(**basic)


@dataclass
class Results:
    """Results of static / adaptive routines (main.py:429-502): save(), load(path),
    best_hyperparameters(), plot_trials()."""
    loss_function: object
    layer: list
    label: str = ''
    trials: object = None
    decompositions: tuple = ()
    save_to: str = ''

    def __post_init__(self):
        if self.save_to == '':
            self.save_to = f'results/{self.label}'

    def save(self):
        """main.py:459-462.  Written to a temporary file and renamed, so an interrupted `adaptive()` run never
        leaves a truncated file behind."""
        os.makedirs(os.path.dirname(self.save_to) or '.', exist_ok=True)
        tmp = f'{self.save_to}.tmp{os.getpid()}'
        try:
            with open(tmp, 'wb') as f:
                f.write(_MAGIC)
                _pickler.dump(self, f)
            os.replace(tmp, self.save_to)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)

    @staticmethod
    def load(path):
        """main.py:464-469.  Files written by this package start with a magic line and are unpickled (with dill
        when installed): like any pickle, only load files you trust.  Anything else is taken for a file written by
        the reference itself (it names cpflow / qiskit / hyperopt / jax classes that are not installed here) and
        goes through `legacy.load_reference_results`, which executes nothing from the file."""
        with open(path, 'rb') as f:
            head = f.read(len(_MAGIC))
            if head == _MAGIC:
                res = _pickler.load(f)
                if not isinstance(res, Results):
                    raise TypeError(f'{path}: holds a {type(res).__name__}, not a Results object')
                return res
        from .legacy import load_reference_results
        return load_reference_results(path)

    def best_hyperparameters(self):
        """Pairs [num_cp_gates, r] ordered by increasing score (main.py:471-477)."""
        results = sorted(self.trials.results, key=lambda res: res['loss'])
        return [[res['num_cp_gates'], res['r']] for res in results]

    def plot_trials(self):
        import matplotlib.pyplot as plt  # optional dependency, as in the reference
        results = self.trials.results
        num = np.array([res['num_cp_gates'] for res in results])
        r = np.array([res['r'] for res in results])
        loss = np.array([res['loss'] for res in results])
        fin = loss < np.inf
        n_best, r_best = self.best_hyperparameters()[0]
        plt.scatter(num[fin], r[fin], c=loss[fin], cmap='jet', edgecolors='black')
        plt.colorbar()
        plt.scatter(num[~fin], r[~fin], marker='x', color='red')
        plt.scatter([n_best], [r_best], marker='*', facecolors='gold', edgecolors='black', s=[250])
        plt.xlabel('Number of CP gates')
        plt.ylabel('r: regularization weight')
        plt.title('Score')


class Trials:
    """Minimal stand-in for hyperopt.Trials: `.results` is the list of objective dicts."""

    def __init__(self):
        self.results = []

    @property
    def trials(self):
        return [{'result': r} for r in self.results]


class Synthesize:
    """Automated synthesis of unitaries into CZ + single-qubit gates (main.py:505-864).

    Args:
        layer: qubit connectivity, e.g. [[0, 1], [1, 2]].
        unitary_loss_func: a `Loss` spec ('hs' | 'state' | 'relphase' with its target; runs inside the fused
            kernel), or any function of the unitary written with torch operations (complex tensor [N,N] -> real
            scalar), as in the reference; the latter runs through a host-driven loop around the engine's kernels.
        target_unitary: if given, the loss is the Hilbert-Schmidt distance to it (matrix_utils.py:35-42).
        label: name used in results / save path.
        cp_regularization_func: `PenaltyFunction` for one CP angle (default: the 'linear' penalty), or any
            2 pi-periodic piecewise-linear callable R(a), which is tabulated.
    """

    def __init__(self, layer, unitary_loss_func=None, target_unitary=None, label=None, cp_regularization_func=None,
                 dtype=torch.float32, device=None):
        self.layer = layer
        self.num_qubits = num_qubits_from_layer(self.layer)
        self.target_unitary = None if target_unitary is None else np.asarray(target_unitary)
        if unitary_loss_func is not None:
            # main.py:528-529: any function of the unitary.  A `Loss` spec runs inside the fused kernel; any other
            # callable (written with torch operations on a complex [N,N] tensor) runs through the host-driven loop
            # cpf_unitary -> loss / autograd cotangent -> cpf_adjoint_from_cotangent -> cpf_adam_step.
            self.unitary_loss_func = unitary_loss_func if isinstance(unitary_loss_func, (Loss, TorchLoss)) \
                else TorchLoss(unitary_loss_func)
        else:
            assert self.target_unitary is not None, 'Neither unitary loss function nor target unitary is provided.'
            assert self.target_unitary.shape == (2 ** self.num_qubits, 2 ** self.num_qubits), \
                'Number of qubits in target unitary and layer do not match.'
            self.unitary_loss_func = Loss('hs', self.target_unitary)
        self.label = label
        if cp_regularization_func:
            # main.py:536-539: any callable R(a).  The kernels consume a segment table: a PenaltyFunction is used
            # as is, any other callable is tabulated (penalty.tabulate_penalty raises with the fit error if it is
            # not a periodic piecewise-linear function of at most 16 pieces).
            self.cp_regularization_func = cp_regularization_func if isinstance(cp_regularization_func, PenaltyFunction) \
                else tabulate_penalty(cp_regularization_func)
        else:
            self.cp_regularization_func = make_regularization_function(RegularizationOptions)
        self.dtype = dtype
        self.device = device

    # ---- helpers ------------------------------------------------------------------------------
    def _device(self):
        if self.device is not None:
            return torch.device(self.device)
        return torch.device('cuda', torch.cuda.current_device())

    def _ansatz(self, options):
        return Ansatz(self.num_qubits, 'cp', fill_layers(self.layer, options.num_cp_gates), options.rotation_gates)

    def _penalty(self, r):
        pf = self.cp_regularization_func
        kind = 'l1' if pf.kind == 'l1' else 'piecewise'
        return Penalty(kind, r, pf.segments, pf.period)

    @staticmethod
    def _generate_initial_angles(seed, anz, cp_dist='uniform', batch_size=1, first=0, count=None,
                                 dtype=torch.float32, device='cuda'):
        """main.py:541-548 with PRNGKey(seed); rows [first, first+count) of the batch, on the device."""
        return random_cp_angles(anz, batch_size, cp_dist=cp_dist, seed=seed, first=first, count=count,
                                dtype=dtype, device=device)

    def _generate_raw(self, options, initial_angles_array=None, keep_history=False, first=0, count=None,
                      return_device=True):
        """main.py:558-587: multi-start Adam on loss + r * sum R(cp angles).  Returns RawResults for
        samples [first, first+count) of the batch (all of it by default)."""
        anz = self._ansatz(options)
        dev = self._device()
        if initial_angles_array is None:
            initial_angles_array = self._generate_initial_angles(
                options.random_seed, anz, cp_dist=options.cp_distribution, batch_size=options.num_samples,
                first=first, count=count, dtype=self.dtype, device=dev)
        raw = mynimize_repeated(
            ProgramLoss(anz.program, self.unitary_loss_func), anz.num_angles, method=options.method,
            learning_rate=options.learning_rate, num_iterations=options.num_gd_iterations,
            initial_params_batch=initial_angles_array, regularization_func=self._penalty(options.r),
            keep_history=keep_history, dtype=self.dtype, device=dev, return_device=return_device)
        return raw

    def _evaluate_raw(self, raw_results, options, disable_tqdm=False):
        """main.py:589-603: keep results with loss <= entry_loss, sorted by CZ count."""
        anz = self._ansatz(options)
        return filter_cp_results(raw_results, anz.cp_mask, float('inf'), options.entry_loss,
                                 threshold_cp=options.threshold_cp, disable_tqdm=disable_tqdm, program=anz.program)

    def _initialize_results(self, save_results, save_to):
        results = Results(self.unitary_loss_func, self.layer, label=self.label)
        if save_results:
            assert self.label or save_to, \
                'To save results on a disk either `label` or `save_to` must be provided. ' \
                'If you insist on not saving the results call the decomposition routine with `save_results=False` flag.'
            if save_to:
                results.save_to = save_to
            try:
                results = Results.load(results.save_to)
            except FileNotFoundError:
                pass
        return results

    def _make_decomposition(self, u_func, circ_func, best_angs, static_options=None, adaptive_options=None,
                            circuit=None):
        if circuit is None:
            circuit = Decomposition._from_cp_circuit(self.unitary_loss_func, u_func, circ_func, best_angs, self.label)
        d = circuit
        d._static_options = static_options
        d._adaptive_options = adaptive_options
        d._decomposer = self
        return d

    # ---- static ---------------------------------------------------------------------------------
    def _prospective(self, options):
        """Stages 1-2 of static() for this rank's shard, then one gather: returns the global, CZ-sorted
        candidate table (global sample index, cz, loss, regloss, angles [P]) on every rank."""
        anz = self._ansatz(options)
        first, count = PL.shard_range(options.num_samples)
        dev = self._device()
        if count > 0:
            raw = self._generate_raw(options, first=first, count=count)
            cz, loss, angles = select_batch(raw, anz.program, options.threshold_cp)
            keep = torch.nonzero(loss <= options.entry_loss).flatten()
            best_i = torch.argmin(raw.regloss, dim=1)
            regloss = raw.regloss[torch.arange(count, device=dev), best_i]
            rec = torch.cat([(keep + first).to(torch.float64)[:, None], cz[keep].to(torch.float64)[:, None],
                             loss[keep].to(torch.float64)[:, None], regloss[keep].to(torch.float64)[:, None],
                             angles[keep].to(torch.float64)], 1)
        else:
            rec = torch.zeros(0, 4 + anz.num_angles, dtype=torch.float64, device=dev)
        rec = PL.gather_rows(rec)
        # sort by cz, ties by global index: the order of the reference's stable sort (cp_utils.py:200)
        order = torch.argsort(rec[:, 1] * (options.num_samples + 1) + rec[:, 0])
        return anz, rec[order]

    def static(self, options, save_results=True, save_to=''):
        """Synthesis with a fixed CP template and regularisation weight (main.py:637-693).

        With an initialised torch.distributed process group the samples are sharded over the ranks
        (one GPU each) and every rank returns the same Results; only rank 0 saves."""
        rank, world = PL.rank_world()
        results = self._initialize_results(save_results, save_to)
        say = print if rank == 0 else (lambda *a, **k: None)
        say('\nStarting decomposition routine with the following options:')
        say('\n', options)
        say('\nComputing raw results...')
        anz, cand = self._prospective(options)
        say('\nSelecting prospective results...')
        cand = cand[cand[:, 1] <= options.accepted_num_cz_gates]
        self.last_prospective_cz_counts = [int(c) for c in cand[:, 1].tolist()]
        successful_results = []
        if len(cand):
            say(f'\nFound {len(cand)}. Verifying...')
            mine = PL.round_robin(len(cand))
            P = anz.num_angles
            dev = self._device()
            if mine:
                angles = cand[mine][:, 4:].to(self.dtype).contiguous()
                cz, proj, frozen = anz.program.count_cz(angles, options.threshold_cp, project=True)
                raw = run_adam_batch(anz.program, self.unitary_loss_func, None, proj,
                                     options.learning_rate_at_verification,
                                     options.num_gd_iterations_at_verification, freeze=frozen)
                bi = torch.argmin(raw.regloss, dim=1)
                ar = torch.arange(len(mine), device=dev)
                out = torch.cat([raw.regloss[ar, bi].to(torch.float64)[:, None], cz.to(torch.float64)[:, None],
                                 raw.params[ar, bi].to(torch.float64), frozen.to(torch.float64)], 1)
            else:
                out = torch.zeros(0, 2 + 2 * P, dtype=torch.float64, device=dev)
            out = PL.gather_round_robin(out, len(cand)).cpu().numpy()
            ok = out[:, 0] <= options.target_loss                    # cp_utils.py:245
            np_dt = np.float32 if self.dtype == torch.float32 else np.float64
            successful_results = Decomposition._from_cp_batch(
                self.unitary_loss_func, anz, out[ok, 2:2 + P].astype(np_dt), out[ok, 2 + P:] > 0.5,
                label=self.label, device=dev)
            for d in successful_results:
                d._static_options = options
                d._decomposer = self
            if successful_results:
                say(f'\n{len(successful_results)} successful. cz counts are:')
                say(sorted([d.cz_count for d in successful_results]))
                results.decompositions = list(results.decompositions) + successful_results
                if save_results and rank == 0:
                    results.save()
            else:
                say('\nAll prospective results failed.')
        else:
            say('\nNo results passed.')
        return results

    # ---- adaptive -------------------------------------------------------------------------------
    def adaptive(self, options, save_results=True, save_to=''):
        """Synthesis with template length and regularisation weight searched over (main.py:695-864).

        The reference drives this loop with hyperopt's TPE; hyperopt is not a dependency here, so the
        proposals come from `cpflow_b200.hyper.TPESampler` (same search space: quniform number of CP
        gates, lognormal r; same score, same seed chain, same resume / verification logic)."""
        from .hyper import TPESampler, next_seed
        rank, world = PL.rank_world()
        say = print if rank == 0 else (lambda *a, **k: None)
        say('\nStarting decomposition routine with the following options:')
        say('\n', options)
        results = self._initialize_results(save_results, save_to)
        if results.trials is not None:
            say('\nFound existing trials, resuming from here.')
            trials = results.trials
            random_seed = trials.results[-1]['random_seed']
            num_existing_trials = len(trials.results)
        else:
            trials = Trials()
            random_seed = options.random_seed
            num_existing_trials = 0
        if results.decompositions:
            scoreboard = sorted(set(d.cz_count for d in results.decompositions))
        else:
            scoreboard = [theoretical_lower_bound(self.num_qubits)]
        if num_existing_trials >= options.max_evals:
            say('Maximum number of evaluations reached.')
        sampler = TPESampler(options.min_num_cp_gates, options.max_num_cp_gates, options.r_mean, options.r_variance)

        for i in range(num_existing_trials, options.max_evals):
            say('\n' + '-' * 42)
            say(f'iteration {i}/{options.max_evals}')
            random_seed = next_seed(random_seed)                       # main.py:798-799
            num_cp_gates, r = sampler.suggest(trials.results, np.random.default_rng(int(random_seed)))
            say(f'\nnum_cp_gates: {num_cp_gates}, r: {r}')
            static_options = options.get_static(num_cp_gates, r)
            static_options.random_seed = random_seed
            static_options.accepted_num_cz_gates = float('inf')
            anz, cand = self._prospective(static_options)
            cz_counts = [int(c) for c in cand[:, 1].tolist()]
            score = float(np.log2((2.0 ** (-np.array(cz_counts, dtype=np.float32))).sum() / options.num_samples)) \
                if cz_counts else -math.inf
            say(f'score: {-score}, cz counts of prospective results: {cz_counts}')
            result = {'loss': -score, 'status': 'ok', 'random_seed': random_seed, 'cz_counts': cz_counts,
                      'num_cp_gates': num_cp_gates, 'r': r, 'layer': self.layer}
            if options.keep_logs:
                # main.py:741-755: the prospective results themselves stay in the trial record, and their pickled
                # form goes into `attachments` together with the options and the loss
                evaluated = [[int(row[1]), {'params': row[4:].to(self.dtype).cpu().numpy()[None],
                                             'loss': row[2:3].cpu().numpy(), 'regloss': row[3:4].cpu().numpy()}]
                             for row in cand]
                result['prospective_decompositions'] = evaluated
                result['attachments'] = {'prospective_decompositions': _pickler.dumps(evaluated),
                                         'static_options': _pickler.dumps(static_options),
                                         'unitary_loss_func': _pickler.dumps(self.unitary_loss_func)}
            trials.results.append(result)
            results.trials = trials
            if save_results and rank == 0:
                results.save()
            current_best_cz = scoreboard[0]
            to_verify = cand[cand[:, 1] < current_best_cz]
            if len(to_verify):
                say(f'\nFound {len(to_verify)} decompositions potentially improving the current best count '
                    f'{current_best_cz}, verifying...')
            else:
                say(f'\nFound no decompositions potentially improving the current best count {current_best_cz}.')
            # the reference verifies one by one and stops at the first success (main.py:833-855);
            # verifying the whole list in one batch and taking the first success is the same result
            if len(to_verify):
                res_list = [{'params': row[4:][None].to(self.dtype), 'regloss': row[3:4], 'loss': row[2:3]}
                            for row in to_verify]
                ver = verify_cp_results(res_list, anz, self.unitary_loss_func, options.get_static(None, None),
                                        dtype=self.dtype, device=self._device())
                for success, num_cz_gates, circ, u, best_angs in ver:
                    if success:
                        say(f'\nFound a new decomposition with {num_cz_gates} gates.')
                        scoreboard.insert(0, num_cz_gates)
                        d = self._make_decomposition(u, circ, best_angs, adaptive_options=options,
                                                     static_options=options.get_static(num_cp_gates, r))
                        results.decompositions = list(results.decompositions) + [d]
                        if save_results and rank == 0:
                            results.save()
                        break
                else:
                    say('\nNone of prospective decompositions passed.')
            if options.stop_if_target_reached and scoreboard[0] <= options.target_num_cz_gates:
                say('\nTarget number of gates reached.')
                break
        return results


def synthesize_many(layer, targets, options, loss='hs', labels=None, cp_regularization_func=None,
                    dtype=torch.float32, device=None, save_results=False):
    """`Synthesize.static(options)` for many targets at once: returns one `Results` per target, in input order.

    Target i gets exactly the work of `Synthesize(layer, unitary_loss_func=Loss(loss, targets[i])).static(options)`
    (for loss='hs' the same as `target_unitary=targets[i]`): the same initial batch (samples 0..S-1 of
    PRNGKey(options.random_seed), drawn once and used for every target), the same entry filter and
    `accepted_num_cz_gates` cut, the same verification with the projected CP angles frozen.  What changes is that all
    T * S samples run in ONE fused Adam launch (cpf_adam_run_multi), and all surviving candidates of all targets are
    verified in one more.  Under torch.distributed the T * S items are sharded over the ranks by global index; every
    rank returns the same list and only rank 0 saves.

    targets: [T, N, N] ('hs', 'relphase') or [T, N] ('state'); labels: None or T labels (needed to save).  A user loss
    function cannot serve several targets in one launch: `loss` is one of 'hs', 'state', 'relphase'."""
    if not isinstance(loss, str):
        raise TypeError("synthesize_many takes a loss kind ('hs', 'state' or 'relphase'); a user loss function runs "
                        "one target at a time (Synthesize(layer, unitary_loss_func=...).static)")
    num_qubits = num_qubits_from_layer(layer)
    ml = MultiLoss(loss, targets)
    if ml.targets.shape[1] != 2 ** num_qubits:
        raise ValueError(f"targets of dimension {ml.targets.shape[1]} for a {num_qubits}-qubit layer")
    T = ml.n_targets
    if labels is None:
        labels = [None] * T
    labels = list(labels)
    if len(labels) != T:
        raise ValueError(f"{len(labels)} labels for {T} targets")
    syns = [Synthesize(layer, unitary_loss_func=ml.loss(i), label=labels[i],
                       cp_regularization_func=cp_regularization_func, dtype=dtype, device=device) for i in range(T)]
    results = [s._initialize_results(save_results, '') for s in syns]
    syn = syns[0]
    rank, world = PL.rank_world()
    say = print if rank == 0 else (lambda *a, **k: None)
    say(f'\nStarting decomposition routine for {T} targets with the following options:')
    say('\n', options)
    anz = syn._ansatz(options)
    P = anz.num_angles
    S = options.num_samples
    dev = syn._device()

    # stage 1: item g = t * S + s (target t, sample s), this rank's contiguous block of the T * S items
    say('\nComputing raw results...')
    first, count = PL.shard_range(T * S)
    if count > 0:
        g = torch.arange(first, first + count, device=dev)
        init = syn._generate_initial_angles(options.random_seed, anz, cp_dist=options.cp_distribution,
                                            batch_size=S, dtype=dtype, device=dev)[g % S].contiguous()
        raw = run_adam_batch(anz.program, ml, syn._penalty(options.r), init, options.learning_rate,
                             options.num_gd_iterations, target_index=(g // S).cpu().numpy())
        cz, lo, angles = select_batch(raw, anz.program, options.threshold_cp)
        keep = torch.nonzero(lo <= options.entry_loss).flatten()
        best_i = torch.argmin(raw.regloss, dim=1)
        regloss = raw.regloss[torch.arange(count, device=dev), best_i]
        gk = g[keep]
        rec = torch.cat([(gk // S).to(torch.float64)[:, None], (gk % S).to(torch.float64)[:, None],
                         cz[keep].to(torch.float64)[:, None], lo[keep].to(torch.float64)[:, None],
                         regloss[keep].to(torch.float64)[:, None], angles[keep].to(torch.float64)], 1)
    else:
        rec = torch.zeros(0, 5 + P, dtype=torch.float64, device=dev)
    rec = PL.gather_rows(rec)
    # grouped by target; within a target sorted by cz, ties by sample index (the order of static())
    order = torch.argsort(rec[:, 1], stable=True)
    order = order[torch.argsort(rec[order, 2], stable=True)]
    order = order[torch.argsort(rec[order, 0], stable=True)]
    cand = rec[order]
    cand = cand[cand[:, 2] <= options.accepted_num_cz_gates]
    cand_t = cand[:, 0].to(torch.int64).cpu().numpy()
    cand_cz = cand[:, 2].to(torch.int64).cpu().numpy()
    for t in range(T):
        syns[t].last_prospective_cz_counts = cand_cz[cand_t == t].tolist()

    # stage 2: every candidate of every target, one multi-target verification run
    if len(cand):
        say(f'\nFound {len(cand)}. Verifying...')
        mine = PL.round_robin(len(cand))
        if mine:
            angles = cand[mine][:, 5:].to(dtype).contiguous()
            cz, proj, frozen = anz.program.count_cz(angles, options.threshold_cp, project=True)
            raw = run_adam_batch(anz.program, ml, None, proj, options.learning_rate_at_verification,
                                 options.num_gd_iterations_at_verification, freeze=frozen,
                                 target_index=cand_t[mine])
            bi = torch.argmin(raw.regloss, dim=1)
            ar = torch.arange(len(mine), device=dev)
            out = torch.cat([raw.regloss[ar, bi].to(torch.float64)[:, None], cz.to(torch.float64)[:, None],
                             raw.params[ar, bi].to(torch.float64), frozen.to(torch.float64)], 1)
        else:
            out = torch.zeros(0, 2 + 2 * P, dtype=torch.float64, device=dev)
        out = PL.gather_round_robin(out, len(cand)).cpu().numpy()
        ok = out[:, 0] <= options.target_loss                    # cp_utils.py:245
        np_dt = np.float32 if dtype == torch.float32 else np.float64
        for t in range(T):
            sel = ok & (cand_t == t)
            ds = Decomposition._from_cp_batch(syns[t].unitary_loss_func, anz, out[sel, 2:2 + P].astype(np_dt),
                                              out[sel, 2 + P:] > 0.5, label=labels[t], device=dev)
            for d in ds:
                d._static_options = options
                d._decomposer = syns[t]
            if ds:
                results[t].decompositions = list(results[t].decompositions) + ds
                if save_results and rank == 0:
                    results[t].save()
        say(f'\n{int(ok.sum())} successful over {T} targets.')
    else:
        say('\nNo results passed.')
    return results
