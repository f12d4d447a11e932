"""cpflow_b200.legacy: reading the reference's stored `Results` files (SURVEY.md §8f N5) without cpflow, qiskit,
hyperopt, jax or dill.  CPU only.  The first test builds a file with the reference's class paths from scratch;
the second reads the reference's own files when CPFLOW_REFERENCE_DIR names a checkout of the reference project
(the files are not part of this repository) and checks them against the committed golden fixtures."""
import json
import os
import pickle
import sys
import types

import numpy as np
import pytest

from cpflow_b200.legacy import load_reference_results
from oracle import cpflow_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("CPFLOW_REFERENCE_DIR", "")


def _fake_class(path):
    """A plain class that pickles under the dotted path `module.Name` (the modules are registered on the fly)."""
    module, name = path.rsplit(".", 1)
    parts = module.split(".")
    for i in range(1, len(parts) + 1):
        m = ".".join(parts[:i])
        if m not in sys.modules:
            sys.modules[m] = types.ModuleType(m)
    cls = type(name, (), {"__module__": module})
    setattr(sys.modules[module], name, cls)
    return cls


def _obj(cls, **state):
    o = cls()
    o.__dict__.update(state)
    return o


@pytest.fixture
def fake_reference_file(tmp_path):
    before = set(sys.modules)
    Results = _fake_class("cpflow.main.Results")
    Decomposition = _fake_class("cpflow.main.Decomposition")
    StaticOptions = _fake_class("cpflow.main.StaticOptions")
    Synthesize = _fake_class("cpflow.main.Synthesize")
    QC = _fake_class("qiskit.circuit.quantumcircuit.QuantumCircuit")
    Qubit = _fake_class("qiskit.circuit.quantumregister.Qubit")
    Trials = _fake_class("hyperopt.base.Trials")
    gates = {n: _fake_class(f"qiskit.circuit.library.standard_gates.{n}.{n.upper()}Gate") for n in ("rx", "rz", "cz")}
    qubits = [Qubit() for _ in range(2)]
    gl = [("rz", [0], [0.3]), ("rx", [1], [1.1]), ("cz", [0, 1], []), ("rx", [0], [-0.7]), ("rz", [1], [2.0])]
    data = [(_obj(gates[n], _name=n, _params=p, _num_qubits=len(q)), [qubits[i] for i in q], []) for n, q, p in gl]
    circ = _obj(QC, _data=data, _qubits=qubits, _global_phase=0.25, name="c")
    ops = [({"rx": 0, "rz": 2, "cz": 4}[n], q[0], q[1] if len(q) > 1 else -1, -1, p[0] if p else 0.0) for n, q, p in gl]
    u = O.program_unitary_np(2, ops, np.zeros(0))
    opts = _obj(StaticOptions, num_samples=7, num_cp_gates=5, r=0.001, accepted_num_cz_gates=3, rotation_gates="xyz",
                some_new_field=object())
    dec = _obj(Decomposition, unitary_loss_func=None, circuit=circ, unitary=u.astype(np.complex64), label="fake",
               loss=np.float32(1e-7), type="Approximate", cz_count=1, cz_depth=1, t_count=None, t_depth=None,
               _cp_data=None, _static_options=opts, _adaptive_options=None,
               _decomposer=_obj(Synthesize, target_unitary=u, layer=[[0, 1]]))
    trials = _obj(Trials, _trials=[{"result": {"loss": 3.0, "status": "ok", "random_seed": 5, "cz_counts": [1, 2],
                                               "num_cp_gates": 4, "r": 0.002, "layer": [[0, 1]]}},
                                   {"result": {"loss": 2.0, "status": "ok", "random_seed": 6, "cz_counts": [1],
                                               "num_cp_gates": 5, "r": 0.001, "layer": [[0, 1]]}}])
    res = _obj(Results, loss_function=None, layer=[[0, 1]], label="fake", trials=trials, decompositions=[dec],
               save_to="results/fake")
    path = tmp_path / "fake_results"
    with open(path, "wb") as f:
        pickle.dump(res, f, protocol=4)
    for m in set(sys.modules) - before:          # the reader must work without these modules
        del sys.modules[m]
    return str(path), u, gl


def test_reads_a_file_with_the_reference_class_paths(fake_reference_file):
    path, u, gl = fake_reference_file
    assert "cpflow" not in sys.modules and "qiskit" not in sys.modules and "hyperopt" not in sys.modules
    res = load_reference_results(path)
    assert res.layer == [[0, 1]] and res.label == "fake" and res.save_to == "results/fake"
    assert [(g.name, list(g.qubits), list(g.params)) for g in res.decompositions[0].circuit.data] == \
        [(n, q, p) for n, q, p in gl]
    d = res.decompositions[0]
    assert d.cz_count == 1 and d.cz_depth == 1 and d.type == "Approximate" and abs(d.loss - 1e-7) < 1e-12
    assert d.circuit.global_phase == 0.25
    assert np.abs(d.unitary - u).max() < 1e-6
    assert d._static_options.num_cp_gates == 5 and d._static_options.num_samples == 7      # unknown fields dropped
    # the circuit that was read reproduces the stored unitary, and the HS loss was rebuilt from the stored target
    uc = O.program_unitary_np(2, [tuple(o) for o in d.circuit.to_ops()], np.zeros(0))
    assert np.abs(uc - u).max() < 1e-12
    assert res.loss_function is not None and res.loss_function.kind == "hs"
    assert res.best_hyperparameters() == [[5, 0.001], [4, 0.002]]
    assert res.trials.results[0]["cz_counts"] == [1, 2]
    assert "some_new_field" not in repr(d)


def test_rejects_other_pickles(tmp_path):
    p = tmp_path / "x"
    with open(p, "wb") as f:
        pickle.dump({"a": 1}, f)
    with pytest.raises(ValueError):
        load_reference_results(str(p))


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "tutorial", "results"))),
                    reason="CPFLOW_REFERENCE_DIR does not name a checkout of the reference project")
def test_reference_files_against_golden_fixtures():
    """Every stored file loads; trials match tests/golden/trials.json; the stored circuits reproduce their stored
    unitaries up to a global phase (the property tests/golden/gatelist_kats pins for a subset; a few refined
    circuits were stored next to the unitary of their unrefined version and agree to ~1e-5 only)."""
    trials = json.load(open(os.path.join(ROOT, "tests", "golden", "trials.json")))
    n_circ = n_tight = 0
    for name, rec in trials.items():
        res = load_reference_results(os.path.join(REF, name))
        assert res.layer == rec["layer"]
        got = [(t["num_cp_gates"], t["r"], t["random_seed"]) for t in res.trials.results]
        assert got == [(t["num_cp_gates"], t["r"], t["random_seed"]) for t in rec["trials"]]
        for d in res.decompositions[:6]:
            n = d.circuit.num_qubits
            uc = O.program_unitary_np(n, [tuple(o) for o in d.circuit.to_ops()], np.zeros(0))
            ov = abs(np.trace(uc.conj().T @ d.unitary)) / 2 ** n
            assert abs(ov - 1) < 1e-3, (name, ov)
            n_tight += abs(ov - 1) < 5e-6
            assert d.cz_count == sum(g.name == "cz" for g in d.circuit.data)
            n_circ += 1
    assert n_circ > 30 and n_tight >= 0.9 * n_circ


def test_results_load_falls_back_to_the_reference_format(fake_reference_file, tmp_path):
    """Results.load (main.py:458-461) reads this package's own files and the reference's."""
    from cpflow_b200.main import Results, Trials
    path, u, _ = fake_reference_file
    res = Results.load(path)
    assert isinstance(res, Results) and res.label == "fake" and len(res.decompositions) == 1
    own = Results(None, [[0, 1]], label="own", trials=Trials(), save_to=str(tmp_path / "own_results"))
    own.trials.results.append({"loss": 1.0, "num_cp_gates": 3, "r": 0.1})
    own.save()
    back = Results.load(own.save_to)
    assert isinstance(back, Results) and back.label == "own" and back.best_hyperparameters() == [[3, 0.1]]
    with pytest.raises(FileNotFoundError):
        Results.load(str(tmp_path / "missing"))


def test_reader_runs_nothing_from_a_crafted_file(tmp_path):
    """A pickle that REDUCEs builtins.eval / os.system / functools.partial must not execute anything: every global
    outside the explicit data allow-list becomes an inert placeholder (legacy.py: _ALLOWED)."""
    import io
    import pickle
    from cpflow_b200 import legacy

    marker = tmp_path / "pwned"

    class Evil:
        def __reduce__(self):
            return (eval, (f"open({str(marker)!r}, 'w').write('x')",))

    class Evil2:
        def __reduce__(self):
            import os
            return (os.system, (f"touch {marker}",))

    class Evil3:
        def __reduce__(self):
            import functools
            return (functools.partial, (exec, f"open({str(marker)!r}, 'w')"))

    for obj in (Evil(), Evil2(), Evil3(), [Evil(), {"a": Evil2()}]):
        out = legacy._Reader(io.BytesIO(pickle.dumps(obj, protocol=4))).load()
        assert not marker.exists()
        assert "inert" in repr(out) or isinstance(out, list)
    for name in ("eval", "exec", "__import__", "getattr", "compile", "open"):
        assert ("builtins", name) not in legacy._ALLOWED
    assert not any(m in ("functools", "copyreg", "os", "posix", "subprocess") for m, _ in legacy._ALLOWED)
