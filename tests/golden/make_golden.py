"""Extract known-answer fixtures from the reference's stored result files.

Run once, given a checkout of the reference project (argument, or CPFLOW_REFERENCE_DIR):

    python tests/golden/make_golden.py /path/to/cpflow

It reads cpflow's dill `Results` pickles (paper/results, paper/results/benchmarks,
tutorial/results — SURVEY.md §4.3 / Appendix A) with the stub unpickler and writes small,
dependency-free fixtures next to this file:

* ``ansatz_kats.npz`` + ``ansatz_kats.json`` — (full angle vector -> stored unitary) pairs that
  pin the ansatz restatement (reference `build_unitary`, main.py:106-146).
* ``gatelist_kats.npz`` + ``gatelist_kats.json`` — stored rz/rx/cz circuits with their stored
  unitary and target (pins gate conventions: gates.py:10-58, circuit_assembly.py:31-45).
* ``trials.json`` — hyperopt trial records (num_cp_gates, r, random_seed, cz_counts) used as
  statistical pins and as threefry `split` known answers (main.py:741-749, 798-799).

Nothing at test time reads the reference checkout; only these committed fixtures are used.
"""
import glob
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import stub_unpickle as su  # noqa: E402

REF = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("CPFLOW_REFERENCE_DIR", "")
FILES = (sorted(glob.glob(f"{REF}/tutorial/results/*"))
         + sorted(f for f in glob.glob(f"{REF}/paper/results/*") if os.path.isfile(f))
         + sorted(glob.glob(f"{REF}/paper/results/benchmarks/*")))

# cap the number of decompositions taken per file to keep fixtures small
MAX_PER_FILE = 12


def cell_payload(cell):
    return type(cell)._fn[0][0] if isinstance(cell, su.Stub) else cell._fn[0][0]


def closure_of(func_stub):
    """(fixed_params, indices) from the pickled `cf` closure (cp_utils.py:100-108)."""
    args = func_stub._fn[0]
    clo = args[4]
    payloads = [c._fn[0][0] for c in clo]
    # free-var order: (f, fixed_params, indices, jax_numpy)
    fixed = su.jax_array(payloads[1]) if not isinstance(payloads[1], (list, tuple)) else np.array(payloads[1])
    idx = list(payloads[2])
    return np.asarray(fixed, dtype=np.float64), idx


def options_dict(opt):
    if opt is None:
        return None
    st = getattr(opt, "_state", None)
    if isinstance(st, dict):
        return {k: (v if isinstance(v, (int, float, str, type(None))) else str(v)) for k, v in st.items()}
    return None


def scalar(x):
    if isinstance(x, (int, float)):
        return float(x)
    try:
        return float(su.jax_array(x).reshape(()))
    except Exception:
        return None


def circuit_gates(circ):
    cs = circ._state
    qubits = cs["_qubits"]
    qidx = {id(q): i for i, q in enumerate(qubits)}
    kinds, q0s, q1s, params = [], [], [], []
    for gate, qargs, _ in cs["_data"]:
        gs = gate._state
        name = gs["_name"]
        qs = [qidx[id(q)] for q in qargs]
        p = [float(x) for x in gs["_params"]] if gs["_params"] else []
        kinds.append(name)
        q0s.append(qs[0])
        q1s.append(qs[1] if len(qs) > 1 else -1)
        params.append(p[0] if p else 0.0)
    gp = cs.get("_global_phase", 0.0)
    try:
        gp = float(gp)
    except Exception:
        gp = 0.0
    return kinds, q0s, q1s, params, gp, len(qubits)


def main():
    if not (REF and os.path.isdir(os.path.join(REF, "tutorial", "results"))):
        raise SystemExit("usage: make_golden.py /path/to/cpflow  (a checkout of the reference project)")
    ans_meta, ans_arrays = [], {}
    gl_meta, gl_arrays = [], {}
    trials_out = {}
    targets = {}
    for path in FILES:
        name = os.path.relpath(path, REF)
        try:
            r = su.load(path)
        except Exception as e:  # pragma: no cover
            print("skip", name, e)
            continue
        st = r._state
        layer = st["layer"]
        decs = list(st["decompositions"])
        # ---- trials
        tr = st.get("trials")
        if tr is not None and hasattr(tr, "_state"):
            rows = []
            for t in tr._state["_trials"]:
                res = t["result"]
                cz = res.get("cz_counts")
                rows.append({
                    "num_cp_gates": int(res["num_cp_gates"]),
                    "r": float(res["r"]),
                    "random_seed": int(res["random_seed"]),
                    "score": float(res["loss"]),
                    "cz_counts": [int(c) for c in cz] if isinstance(cz, (list, tuple)) else int(cz),
                })
            ns = None
            for d in decs:
                ao = options_dict(d._state.get("_adaptive_options"))
                if ao and "num_samples" in ao:
                    ns = ao["num_samples"]
                    break
            trials_out[name] = {"layer": layer, "num_samples": ns, "trials": rows}
        # ---- decompositions
        step = max(1, len(decs) // MAX_PER_FILE)
        picked = decs[::step][:MAX_PER_FILE]
        for di, d in enumerate(picked):
            ds = d._state
            u_stored = np.asarray(su.jax_array(ds["unitary"]), dtype=np.complex128)
            n = int(round(np.log2(u_stored.shape[0])))
            dec = ds.get("_decomposer")
            tgt = None
            if dec is not None and dec._state.get("target_unitary") is not None:
                try:
                    tgt = np.asarray(su.jax_array(dec._state["target_unitary"]), dtype=np.complex128)
                except Exception:
                    tgt = None
            tkey = None
            if tgt is not None:
                tkey = f"target_{len(targets)}"
                for k, v in targets.items():
                    if v.shape == tgt.shape and np.array_equal(v, tgt):
                        tkey = k
                        break
                targets.setdefault(tkey, tgt)
            so = options_dict(ds.get("_static_options"))
            key = f"{len(gl_meta):04d}"
            # gate list KAT
            kinds, q0s, q1s, params, gp, nq = circuit_gates(ds["circuit"])
            gl_arrays[f"u_{key}"] = u_stored
            gl_arrays[f"q0_{key}"] = np.array(q0s, dtype=np.int8)
            gl_arrays[f"q1_{key}"] = np.array(q1s, dtype=np.int8)
            gl_arrays[f"p_{key}"] = np.array(params, dtype=np.float64)
            gl_meta.append({
                "key": key, "file": name, "n": nq, "kinds": kinds, "global_phase": gp,
                "target": tkey, "loss": scalar(ds["loss"]), "cz_count": ds["cz_count"],
                "cz_depth": ds["cz_depth"], "type": ds["type"], "layer": layer,
            })
            # angle KAT (new-layout files only: need rotation_gates in the options)
            cp = ds.get("_cp_data")
            if cp is None or so is None or "rotation_gates" not in so:
                continue
            try:
                fixed, idx = closure_of(cp[0])
                free = np.asarray(su.jax_array(cp[2]), dtype=np.float64)
            except Exception as e:
                print("no angles for", name, di, e)
                continue
            total = len(free) + len(idx)
            full = np.zeros(total)
            others = [i for i in range(total) if i not in set(idx)]
            full[others] = free
            full[idx] = fixed
            akey = f"{len(ans_meta):04d}"
            ans_arrays[f"angles_{akey}"] = full
            ans_arrays[f"frozen_{akey}"] = np.array(idx, dtype=np.int32)
            ans_arrays[f"u_{akey}"] = u_stored
            ans_meta.append({
                "key": akey, "file": name, "n": n, "layer": layer,
                "num_cp_gates": int(so["num_cp_gates"]), "rotation_gates": so["rotation_gates"],
                "target": tkey, "loss": scalar(ds["loss"]), "cz_count": ds["cz_count"],
                "static_options": so,
            })
        print(f"{name}: {len(decs)} decompositions, picked {len(picked)}")
    for k, v in targets.items():
        ans_arrays[k] = v
        gl_arrays[k] = v
    np.savez_compressed(os.path.join(HERE, "ansatz_kats.npz"), **ans_arrays)
    np.savez_compressed(os.path.join(HERE, "gatelist_kats.npz"), **gl_arrays)
    with open(os.path.join(HERE, "ansatz_kats.json"), "w") as f:
        json.dump(ans_meta, f, indent=0)
    with open(os.path.join(HERE, "gatelist_kats.json"), "w") as f:
        json.dump(gl_meta, f, indent=0)
    with open(os.path.join(HERE, "trials.json"), "w") as f:
        json.dump(trials_out, f, indent=0)
    print(len(ans_meta), "angle KATs;", len(gl_meta), "gate-list KATs;", len(targets), "targets;",
          sum(len(v["trials"]) for v in trials_out.values()), "trials")


if __name__ == "__main__":
    main()
