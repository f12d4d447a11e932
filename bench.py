#!/usr/bin/env python
"""Headline benchmark: loss+grad(+Adam step) evaluations per second of the multi-start synthesis
loop on BASELINE.json's metric configuration (4-qubit Toffoli, 40 CP gates, complex64).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --steps K --warmup W    # CPU arm (oracle port of cpflow)

A *step* is one complete stage-1 run of `Synthesize.static()` for this rank's shard of samples:
B = 10^5 independent random initialisations (the sample count of BASELINE configs[2]) x T = 2000
Adam iterations, every iteration = forward sweep + loss + penalty + adjoint sweep + Adam update +
best tracking, all inside ONE launch of the fused engine kernel.  One "eval" = one such iteration
of one sample.  Samples shard over ranks with no data-path collective ("weak" scaling: per-GPU
batch fixed); timing is CUDA events on the launching stream, max over ranks.

Keys beyond the base contract:
  roofline     FP32 CUDA-core roofline of the engine kernel (SURVEY.md §8d: the path is gate
               arithmetic, not HBM or tensor-core bound).  achieved = algorithmic flops per launch
               (C*N*(16*G1+4*K+8) per eval, the adjoint-sweep count; uncompute not credited) / mean
               launch time measured live with CUDA events.  The Heisenberg-picture kernel
               (csrc/heis_impl.cuh) needs fewer executed flops than that count; peak = FP32 FMA issue peak measured live by tools/fp32_peak
               on the same GPU (MEASURED_PEAKS.json carries no FP32 figure).  The HBM side is
               reported next to it (hbm_*), it is not the bound.
  cpu_baseline the CPU oracle (torch restatement of the reference's JAX loop; JAX is not in the
               image) timed on this host, bounded sample.
  e2e          same metric through the public host API (`mynimize_repeated` with HOST buffers):
               pinned H2D of the initial angles and D2H of the result arrays inside the timing.

--dump-outputs DIR writes what the last timed step computed (the AdamState arrays a caller of `adam_run`
receives) for a fixed, seeded sample of the samples, one DIR/<name>.npy per array, so that two builds run with
the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "loss+grad evals/sec (4q Toffoli, 40 CP gates)"
UNIT = "evals/s"
R_WEIGHT = 0.001476          # the reference's stored K=40 trial point (SURVEY.md §8d C3)
LR = 0.1
# --dump-outputs: the AdamState arrays written, and the byte budget that bounds the sampled rows (48 MiB)
DUMP_FIELDS = ("angles", "best_params", "best_regloss", "best_reg", "init_regloss", "init_reg")
DUMP_BYTES = 48 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    # C3 quotes 10^5 samples ACROSS the GPUs of the box: the default splits that batch over the ranks ("strong":
    # 12 500 per GPU at N = 8); --scaling weak keeps 10^5 samples per GPU instead
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--samples", type=int, default=100000, help="global batch (strong) / per-GPU batch (weak)")
    ap.add_argument("--samples-per-gpu", type=int, default=None, help="deprecated alias: implies --scaling weak")
    ap.add_argument("--iters", type=int, default=2000, help="Adam iterations per step (num_gd_iterations)")
    ap.add_argument("--layer", default="chain", choices=["chain", "star"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-static", action="store_true", help="skip the Synthesize.static() wall-time extras")
    ap.add_argument("--no-extras", action="store_true", help="skip the complex128 / 5-qubit / other-loss roofline extras")
    ap.add_argument("--cpu-samples", type=int, default=1024)
    ap.add_argument("--cpu-iters", type=int, default=30)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's results to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the CUDA engine's results: it needs --impl b200")
    if a.samples_per_gpu is not None:
        a.scaling, a.samples = "weak", a.samples_per_gpu
    return a


def shard(args, rank, world):
    """(first global sample index, count, global batch) of this rank."""
    if args.scaling == "weak":
        return rank * args.samples, args.samples, args.samples * world
    base, rem = divmod(args.samples, world)
    return rank * base + min(rank, rem), base + (1 if rank < rem else 0), args.samples


def workload(layer_name):
    from cpflow_b200.topology import chain_layer
    layer = chain_layer(4) if layer_name == "chain" else [[0, 1], [0, 2], [0, 3]]
    return layer, 40


def config_dict(args, n_gpus, extra=None):
    _, per_rank, total = shard(args, 0, n_gpus)
    c = {"workload": f"C3: 4q Toffoli (C3X), {args.layer} connectivity, 40 CP gates, 'xyz' rotations, P=292, "
                     f"HS loss + linear CP penalty r={R_WEIGHT}, Adam lr={LR}, complex64",
         "global_samples": total, "samples_per_gpu": per_rank, "adam_iterations_per_step": args.iters,
         "parallelism": f"samples sharded over {n_gpus} GPU(s), no collective",
         "l2": "GPU arm: flushed between steps (256 MiB write)"}
    if extra:
        c.update(extra)
    return c


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference loop (torch CPU, complex64, all host threads)
# ------------------------------------------------------------------------------------------------
def cpu_oracle_rate(layer, K, samples, iters, repeats=1):
    """evals/s of the oracle's Adam loop (value_and_grad + optax-Adam restatement) on this host."""
    import torch
    from oracle import cpflow_oracle as O
    anz = O.cp_ansatz(layer, K)
    ops = O.ansatz_program(anz)
    tgt = O.toffoli_target(4, torch.complex64)
    R = O.make_regularization_function()
    a0 = torch.tensor(O.generate_initial_angles(0, anz.num_angles, anz.cp_mask, batch_size=samples))
    best = 0.0
    for _ in range(repeats):
        t0 = time.perf_counter()
        O.mynimize_repeated(4, ops, "hs", tgt, a0, LR, iters, anz.cp_mask, R_WEIGHT, R)
        dt = time.perf_counter() - t0
        best = max(best, samples * (iters + 1) / dt)   # the oracle evaluates theta_0 twice like the reference
    return best, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm runs on rank 0 alone and takes the whole host
    torch.set_num_threads(os.cpu_count() or 1)
    layer, K = workload(args.layer)
    for _ in range(args.warmup):
        cpu_oracle_rate(layer, K, min(args.cpu_samples, 256), 2)
    t0 = time.perf_counter()
    rates = []
    for _ in range(args.steps):
        r, threads = cpu_oracle_rate(layer, K, args.cpu_samples, args.cpu_iters)
        rates.append(r)
    dt = time.perf_counter() - t0
    evals = args.steps * args.cpu_samples * (args.cpu_iters + 1)
    value = evals / dt
    sample = (f"{args.cpu_samples} samples x {args.cpu_iters} Adam iterations per step of the same C3 program "
              f"(bounded sample of the {args.samples}x{args.iters} step)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32 (complex64)",
            "data": "synthetic", "config": config_dict(args, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "note": "CPU oracle = torch restatement of cpflow's jit(vmap(value_and_grad)) + optax "
                                     "Adam loop; JAX/optax are not installable in this image"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "host_cores": os.cpu_count()}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# helpers for the CUDA arm
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.stop_flag = threading.Event()
        self.sm, self.reasons, self.power = [], set(), []
        self.sm_max = None
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                     nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
                     nv.nvmlClocksThrottleReasonSyncBoost: "sync_boost",
                     nv.nvmlClocksThrottleReasonApplicationsClocksSetting: "applications_clocks_setting"}
            while not self.stop_flag.is_set():
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:  # NVML missing: report, do not fail the bench
            self.err = repr(e)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=2)
        d = {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max,
             "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.power:
            d["power_w_median"] = statistics.median(self.power)
        if self.err:
            d["error"] = self.err
        return d


def measure_fp32_peak():
    """FP32 FMA issue peak of this GPU, measured now by tools/fp32_peak (built by build())."""
    exe = os.path.join(ROOT, "tools", "fp32_peak")
    src = exe + ".cu"
    try:
        with tempfile.TemporaryDirectory() as tmp:
            if not os.path.exists(exe):     # the tree may be read-only: compile a private copy instead
                exe = os.path.join(tmp, "fp32_peak")
                subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe, src],
                               check=True, capture_output=True)
            out = subprocess.run([exe, "--quick"], capture_output=True, text=True, timeout=120).stdout
        best = {}
        for ln in out.splitlines():
            if ln.startswith("{"):
                d = json.loads(ln)
                best[d["bench"]] = max(best.get(d["bench"], 0.0), d["rate_per_s"])
        peak = max(best.get("ffma_flops", 0.0), best.get("ffma2_flops", 0.0))      # best also carries dfma_flops
        if peak > 0:
            return peak / 1e12, "measured live by tools/fp32_peak (max of FFMA / FFMA2 chains)", best
    except Exception as e:
        return 74.4, f"nominal 148 SM x 128 lanes x 2 x 1.965 GHz (fp32_peak failed: {e!r})", {}
    return 74.4, "nominal 148 SM x 128 lanes x 2 x 1.965 GHz (fp32_peak gave no result)", {}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            for k in ("hbm_gbs", "hbm_gb_s", "hbm"):
                if k in d:
                    return float(d[k]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def static_wall_times():
    """Second half of BASELINE.json's metric: wall time of the whole Synthesize.static() call (sampling, the
    fused Adam stage, selection, batched verification, result objects) on BASELINE configs[0] (README example,
    'one to five minutes' on the reference's CPU path) and configs[1] (Toffoli-3, all-to-all, 10^4 samples)."""
    import contextlib
    import io
    import numpy as np
    import cpflow_b200 as cp
    from cpflow_b200.gates import u_toff3, u_toff4
    from cpflow_b200.topology import chain_layer, connected_layer
    out = {}
    ccz = np.diag([1, 1, 1, 1, 1, 1, 1, -1]).astype(complex)
    cases = [("C1_ccz_chain_K12_B10", chain_layer(3), ccz,
              dict(num_cp_gates=12, accepted_num_cz_gates=10, num_samples=10)),
             ("C2_toffoli3_connected_K7_B10000", connected_layer(3), u_toff3,
              dict(num_cp_gates=7, r=0.00131, accepted_num_cz_gates=6, num_samples=10000)),
             # the metric's own configuration: 10^5 samples, K = 40, chain; the stored K = 40 trial's best prospective
             # count was 21 CZ (1000 samples), so everything up to 22 CZ is verified
             ("C3_toffoli4_chain_K40_B100000", chain_layer(4), u_toff4,
              dict(num_cp_gates=40, r=R_WEIGHT, accepted_num_cz_gates=22, num_samples=100000))]
    for name, layer, target, kw in cases:
        try:
            syn = cp.Synthesize(layer, target_unitary=target, label=name)
            opts = cp.StaticOptions(**kw)
            with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
                syn.static(opts, save_results=False)          # warm-up (module import, allocator, device program)
                t0 = time.perf_counter()
                res = syn.static(opts, save_results=False)
                dt = time.perf_counter() - t0
            cz = sorted(d.cz_count for d in res.decompositions)
            out[name] = {"wall_s": dt, "decompositions": len(cz), "min_cz": cz[0] if cz else None,
                         "prospective": len(syn.last_prospective_cz_counts)}
        except Exception as e:   # an extra must never take the headline down
            out[name] = {"error": repr(e)}
    return out


def other_rooflines(peak_tf, peak_detail):
    """Executed-flop rooflines and rates of the configurations next to the headline (BASELINE configs[3], [4]):
    complex128 (FP64 FMA peak from tools/fp32_peak's DFMA chain), the 5-qubit templates, the paper's kite layer, a layer
    without a compile-time kernel (run-time pair dispatch, HeisSweepAny), and the state-preparation / relative-phase losses on the state-adjoint kernels.  Short launches
    (event-timed, second of two), not part of the headline."""
    import numpy as np
    import torch
    from cpflow_b200 import _lib as L
    from cpflow_b200.ansatz import Ansatz
    from cpflow_b200.engine import Loss, Penalty
    from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
    from cpflow_b200.topology import chain_layer, connected_layer, fill_layers
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", R_WEIGHT, pf.segments, pf.period)
    f64_peak = (peak_detail or {}).get("dfma_flops", 0.0) / 1e12 or None
    cases = [("C4_4q_connected_K61_complex128", 4, connected_layer(4), 61, torch.float64, "hs", 20000, 100),
             ("C4_4q_chain_K40_complex128", 4, chain_layer(4), 40, torch.float64, "hs", 20000, 100),
             ("C5_5q_chain_K60_complex64", 5, chain_layer(5), 60, torch.float32, "hs", 40000, 100),
             ("C5_5q_connected_K60_complex64", 5, connected_layer(5), 60, torch.float32, "hs", 40000, 100),
             ("toffoli4_kite_K25_complex64", 4, [[0, 1], [1, 2], [2, 3], [1, 3]], 25, torch.float32, "hs", 100000, 200),
             ("toffoli4_ring_K24_complex64_anylayer", 4, [[0, 1], [2, 3], [1, 2], [0, 3]], 24, torch.float32, "hs", 100000, 200),
             ("C5_5q_chain_K60_stateprep_complex64", 5, chain_layer(5), 60, torch.float32, "state", 200000, 100),
             ("C5_6q_chain_K60_stateprep_complex64", 6, chain_layer(6), 60, torch.float32, "state", 100000, 100),
             ("toffoli4_chain_K40_relphase_complex64", 4, chain_layer(4), 40, torch.float32, "relphase", 20000, 100)]
    out = {}
    for name, n, layer, K, dt, kind, B, T in cases:
        try:
            anz = Ansatz(n, "cp", fill_layers(layer, K))
            prog = anz.program
            N = 1 << n
            rng = np.random.default_rng(0)
            tgt = np.eye(N, dtype=complex)
            tgt[[N - 2, N - 1]] = tgt[[N - 1, N - 2]]
            if kind == "state":
                tgt = np.zeros(N, dtype=complex)
                tgt[0] = tgt[-1] = 2 ** -0.5                       # GHZ-n
            loss = Loss(kind, tgt)
            lk = {"hs": L.LOSS_HS, "state": L.LOSS_STATE, "relphase": L.LOSS_RELPHASE}[kind]
            a0 = prog.initial_angles(0, B).to(dt)
            ms = None
            for _ in range(2):
                st = prog.adam_state(a0.clone())
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                prog.adam_run(st, loss, pen, LR, T)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
            rate = B * T / (ms * 1e-3)
            fx = prog.executed_cost(lk, dt)
            fc, _ = prog.eval_cost(lk, dt)
            pk = f64_peak if dt == torch.float64 else peak_tf
            out[name] = {"evals_per_s": rate, "engine": "heis" if prog.launch_plan(B, lk, dt)["engine"] == 1 else "state-adjoint",
                         "samples": B, "iters": T, "executed_flops_per_eval": fx, "credited_flops_per_eval": fc,
                         "achieved_tflops": rate * fx / 1e12, "peak_tflops": pk,
                         "frac": (rate * fx / 1e12 / pk) if pk else None,
                         "peak": "DFMA chain (tools/fp32_peak)" if dt == torch.float64 else "FFMA / FFMA2 chain (tools/fp32_peak)"}
            del st, a0
        except Exception as e:      # an extra must never take the headline down
            out[name] = {"error": repr(e)}
    return out


def dump_outputs(out_dir, st, first, B, B_total, world, rank):
    """DIR/<field>.npy for every DUMP_FIELDS array of `st`, restricted to a seeded sample of global sample indices
    (ascending), so that the rows are the same for any split of the batch over ranks.  Rank 0 gathers and writes."""
    import numpy as np
    import torch
    import torch.distributed as dist
    row_bytes = sum(getattr(st, f).element_size() * math.prod(getattr(st, f).shape[1:]) for f in DUMP_FIELDS)
    idx = np.sort(np.random.default_rng(0).choice(B_total, min(B_total, DUMP_BYTES // row_bytes), replace=False))
    rows = torch.as_tensor(idx[(idx >= first) & (idx < first + B)] - first, device=st.angles.device)
    parts = [{f: getattr(st, f).index_select(0, rows).cpu().numpy() for f in DUMP_FIELDS}]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, parts[0])
        parts = gathered
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for f in DUMP_FIELDS:
            np.save(os.path.join(out_dir, f + ".npy"), np.concatenate([p[f] for p in parts]))


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL announces its version there when the communicator is created
        # ("NCCL version ..." with NCCL_DEBUG=VERSION in the image), so creation runs with fd 1 pointed at stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from cpflow_b200.ansatz import Ansatz
    from cpflow_b200.engine import Loss, Penalty
    from cpflow_b200.gates import u_toff4
    from cpflow_b200.optimization import ProgramLoss, mynimize_repeated
    from cpflow_b200.penalty import RegularizationOptions, make_regularization_function
    from cpflow_b200.topology import fill_layers

    layer, K = workload(args.layer)
    anz = Ansatz(4, "cp", fill_layers(layer, K))
    prog = anz.program
    pf = make_regularization_function(RegularizationOptions)
    pen = Penalty("piecewise", R_WEIGHT, pf.segments, pf.period)
    loss = Loss("hs", u_toff4)
    first, B, B_total = shard(args, rank, world)
    T = args.iters
    flops_eval, bytes_eval = prog.eval_cost()
    flops_exec = prog.executed_cost()
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    plan = prog.launch_plan(B, n_sm=n_sm)

    # FP32 peak of this GPU (before the timed region; rank 0's GPU stands for the box)
    peak_tf, peak_src, peak_detail = (measure_fp32_peak() if rank == 0 else (None, None, None))

    # inputs resident in HBM: this rank's shard of the global batch, keyed by global sample index
    a0 = prog.initial_angles(0, B_total, first=first, count=B, device=dev)
    st = prog.adam_state(a0.clone())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def step():
        st.angles.copy_(a0)
        st.step = 0
        prog.adam_run(st, loss, pen, LR, T)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        flush.zero_()
        step()
    barrier()

    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for k in range(args.steps):
        flush.zero_()
        st.angles.copy_(a0)
        st.step = 0
        ev[k][0].record()
        prog.adam_run(st, loss, pen, LR, T)
        ev[k][1].record()
    e1.record()
    barrier()
    clocks = sampler.summary()
    ms_total = e0.elapsed_time(e1)
    launch_ms = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor([ms_total, max(launch_ms), sum(launch_ms) / len(launch_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, _, launch_mean = t.tolist()
    evals_total = B_total * T * args.steps
    value = evals_total / (ms_total * 1e-3)

    # sanity of the work actually done in the timed region (not timed)
    best = st.best_regloss
    assert bool(torch.isfinite(best).all()) and bool((best <= st.init_regloss).all())
    frac_converged = float((best - st.best_reg < 1e-3).float().mean())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, st, first, B, B_total, world, rank)

    # ---- e2e: the public host API with HOST buffers (pinned H2D of inputs, D2H of results) ----
    a0_host = a0.cpu().pin_memory()
    pl = ProgramLoss(prog, loss)

    def e2e_step():
        res = mynimize_repeated(pl, anz.num_angles, learning_rate=LR, num_iterations=T,
                                initial_params_batch=a0_host, regularization_func=pen, keep_history=False,
                                device=dev)
        return res

    for _ in range(2):          # untimed: first use of the pinned staging buffers and of the allocator's blocks
        res = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = evals_total / te.item()
    h2d = a0_host.numel() * a0_host.element_size()
    d2h = int(res.params.nbytes + res.regloss.nbytes + res.reg.nbytes)
    assert np.allclose(res.regloss[:, 1], best.cpu().numpy())   # same computation through both paths

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_pk, hbm_src = hbm_peak()
    credited_tf = flops_eval * B * T / (launch_mean * 1e-3) / 1e12
    achieved_tf = flops_exec * B * T / (launch_mean * 1e-3) / 1e12
    prof = {}
    rp = os.path.join(ROOT, "profiles", "r2_roofline.json")        # ncu capture of this launch shape (tools/ncu_roofline.py)
    if os.path.exists(rp):
        try:
            prof = json.load(open(rp))
        except Exception:
            prof = {}
    traffic = None
    for e in prof.get("launches", []):
        if e.get("samples") == B and e.get("iters") == T:
            traffic = e.get("dram_bytes_per_run")
    roofline = {"bound": "fp32", "kernel": "cpf::heis_kernel<float,4,2,HeisSweep<chain>>",
                "note": "FP32 CUDA-core bound (north_star: no tensor cores, not HBM).  achieved / frac count the flops the "
                        "Heisenberg-picture kernel EXECUTES (cpf_executed_cost, cross-checked against the ncu opcode "
                        "mix in profiles/); frac_credited uses SURVEY.md 8(d)'s adjoint-sweep count, which this "
                        "algorithm undercuts, and is an algorithmic speed-up figure, not a utilisation.",
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                "executed_flops_per_eval": flops_exec,
                "achieved_credited": credited_tf, "frac_credited": credited_tf / peak_tf, "flops_per_eval": flops_eval,
                "pipe_fma_active_pct": prof.get("pipe_fma_cycles_active_pct"),
                "issue_active_pct": prof.get("issue_active_pct"),
                "ncu_executed_flops_per_eval": prof.get("executed_flops_per_eval_from_opcode_mix"),
                "peak_source": peak_src, "evals_per_launch": B * T, "kernel_launches_per_run": plan["launches_per_run"],
                "launch_ms_mean": launch_mean, "traffic": traffic,
                "hbm_algorithmic_bytes_per_eval": bytes_eval,
                "hbm_traffic_gbs": (traffic / (launch_mean * 1e-3) / 1e9) if traffic else None,
                "hbm_peak_gbs": hbm_pk, "hbm_peak_source": hbm_src,
                "hbm_frac": (traffic / (launch_mean * 1e-3) / 1e9 / hbm_pk) if traffic else None,
                "hbm_frac_if_state_streamed": bytes_eval * B * T / (launch_mean * 1e-3) / 1e9 / hbm_pk,
                "peak_detail": peak_detail}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate, threads = cpu_oracle_rate(layer, K, args.cpu_samples, args.cpu_iters)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{args.cpu_samples} samples x {args.cpu_iters} Adam iterations of the same C3 program "
                         f"(torch CPU oracle, complex64)", "host_cores": os.cpu_count()}

    static_wall = None
    if world == 1 and not args.no_static:
        static_wall = static_wall_times()
    extras = None
    if world == 1 and not args.no_extras:
        extras = other_rooflines(peak_tf, peak_detail)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32 (complex64 amplitudes)", "data": "synthetic",
            "config": config_dict(args, world),
            "sanity": {"fraction_of_samples_below_entry_loss": frac_converged},
            "roofline": roofline, "cpu_baseline": cpu, "other_rooflines": extras,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "cpflow_b200.optimization.mynimize_repeated(host arrays)", "timer": "wall clock"},
            "gpu_launches": (plan["launches_per_run"] + 1) * args.steps, "clocks": clocks,
            "static_wall_s": static_wall}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
