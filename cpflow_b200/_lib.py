"""ctypes binding of libcpflow_b200.so (the C ABI declared in include/cpflow_b200.h).

The product path has no CPU fallback: if the CUDA library is missing or a call fails, an
exception is raised.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# CPF_LIB_PATH: load another build of the same library (A/B measurements of kernel variants, tools/)
LIB_PATH = os.environ.get("CPF_LIB_PATH") or os.path.join(HERE, "lib", "libcpflow_b200.so")

MAX_SEGMENTS = 16
MAX_QUBITS = 8

# enums (mirror include/cpflow_b200.h)
RX, RY, RZ, CP, CZ, CX = 0, 1, 2, 3, 4, 5
F32, F64 = 0, 1
LOSS_HS, LOSS_STATE, LOSS_RELPHASE, LOSS_ISOMETRY = 0, 1, 2, 3
LOSS_ISOMETRY_RELPHASE = 5
LOSS_SUBSPACE, LOSS_SUBSPACE_RELPHASE = 6, 7


def isometry_kind(ancilla_mask):
    """CPF_ISOMETRY_KIND: the loss-kind argument of the query entry points for an isometry loss."""
    return LOSS_ISOMETRY | (int(ancilla_mask) << 8)


def isometry_relphase_kind(ancilla_mask):
    """CPF_ISOMETRY_RELPHASE_KIND: the loss-kind argument of the query entry points for a relative-phase isometry
    loss."""
    return LOSS_ISOMETRY_RELPHASE | (int(ancilla_mask) << 8)


def subspace_kind(k):
    """CPF_SUBSPACE_KIND: the loss-kind argument of the query entry points for a subspace loss on k input states."""
    return LOSS_SUBSPACE | (int(k) << 8)


def subspace_relphase_kind(k):
    """CPF_SUBSPACE_RELPHASE_KIND: the loss-kind argument of the query entry points for a relative-phase subspace loss
    on k input states."""
    return LOSS_SUBSPACE_RELPHASE | (int(k) << 8)
PEN_NONE, PEN_PIECEWISE, PEN_L1 = 0, 1, 2


class CpfOp(C.Structure):
    _fields_ = [("kind", C.c_int32), ("q0", C.c_int32), ("q1", C.c_int32), ("param", C.c_int32),
                ("const_angle", C.c_double)]


class CpfLossSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("target", C.c_void_p), ("ancilla_mask", C.c_int32)]


class CpfPenaltySpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_segments", C.c_int32), ("r", C.c_double), ("period", C.c_double),
                ("lo", C.c_double * MAX_SEGMENTS), ("hi", C.c_double * MAX_SEGMENTS),
                ("slope", C.c_double * MAX_SEGMENTS), ("intercept", C.c_double * MAX_SEGMENTS),
                ("cp_mask", C.c_void_p)]


class CpfAdamSpec(C.Structure):
    _fields_ = [("lr", C.c_double), ("b1", C.c_double), ("b2", C.c_double), ("eps", C.c_double)]


class CpfProgramInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_qubits", "n_params", "n_ops", "n_rotations", "n_phase",
                                          "n_fused", "n_sched", "reserved")]


class CpfAdamBuffers(C.Structure):
    _fields_ = [("angles", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("freeze", C.c_void_p),
                ("best_params", C.c_void_p), ("best_regloss", C.c_void_p), ("best_reg", C.c_void_p),
                ("init_regloss", C.c_void_p), ("init_reg", C.c_void_p), ("hist_params", C.c_void_p),
                ("hist_regloss", C.c_void_p), ("hist_len", C.c_int64), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_int64)]


class CpfTargetTable(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_targets", C.c_int32), ("targets", C.c_void_p), ("target_index", C.c_void_p)]


EXPORTS = {
    "cpf_version": (C.c_int, []),
    "cpf_last_error": (C.c_char_p, []),
    "cpf_program_create": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(CpfOp), C.c_int32, C.POINTER(C.c_void_p)]),
    "cpf_program_destroy": (C.c_int, [C.c_void_p]),
    "cpf_program_get_info": (C.c_int, [C.c_void_p, C.POINTER(CpfProgramInfo)]),
    "cpf_unitary": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cpf_loss_grad": (C.c_int, [C.c_void_p, C.POINTER(CpfLossSpec), C.POINTER(CpfPenaltySpec), C.c_int32,
                                C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cpf_adjoint_from_cotangent": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]),
    "cpf_adam_run": (C.c_int, [C.c_void_p, C.POINTER(CpfLossSpec), C.POINTER(CpfPenaltySpec),
                               C.POINTER(CpfAdamSpec), C.c_int32, C.c_int64, C.c_int64, C.c_int64,
                               C.POINTER(CpfAdamBuffers), C.c_void_p]),
    "cpf_workspace_bytes": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_int64)]),
    "cpf_loss_grad_multi": (C.c_int, [C.c_void_p, C.POINTER(CpfTargetTable), C.POINTER(CpfPenaltySpec), C.c_int32,
                                      C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cpf_adam_run_multi": (C.c_int, [C.c_void_p, C.POINTER(CpfTargetTable), C.POINTER(CpfPenaltySpec),
                                     C.POINTER(CpfAdamSpec), C.c_int32, C.c_int64, C.c_int64, C.c_int64,
                                     C.POINTER(CpfAdamBuffers), C.c_void_p]),
    "cpf_workspace_bytes_multi": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int32,
                                            C.POINTER(C.c_int64)]),
    "cpf_adam_step": (C.c_int, [C.c_void_p, C.POINTER(CpfPenaltySpec), C.POINTER(CpfAdamSpec), C.c_int32, C.c_int64,
                                C.c_int64, C.c_void_p, C.c_void_p, C.POINTER(CpfAdamBuffers), C.c_void_p]),
    "cpf_count_cz": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_double, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "cpf_cz_value": (C.c_int, [C.c_int32, C.c_int64, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "cpf_initial_angles": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint64, C.c_int64, C.c_int64, C.c_int64,
                                     C.c_int32, C.c_void_p, C.c_void_p]),
    "cpf_eval_cost": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "cpf_executed_cost": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "cpf_launch_plan": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
}



class CpfLaunchInfo(C.Structure):
    """cpf_launch_info (include/cpflow_b200.h)."""
    _fields_ = [("engine", C.c_int32), ("ctas_per_sm", C.c_int32), ("block_threads", C.c_int32),
                ("samples_per_cta", C.c_int32), ("threads_per_sample", C.c_int32), ("max_block_threads", C.c_int32),
                ("words_per_sample", C.c_int32), ("time_slices", C.c_int32), ("grid", C.c_int64), ("smem_bytes", C.c_int64), ("launches_per_run", C.c_int64)]


_lib = None


class CpflowError(RuntimeError):
    pass


def load():
    """Load the CUDA library; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CpflowError(
            f"{LIB_PATH} not found: build it with `python -m cpflow_b200.build` "
            "(cpflow_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().cpf_last_error()
        raise CpflowError(f"cpflow_b200 error {rc}: {msg.decode() if msg else ''}")
