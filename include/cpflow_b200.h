/*
 * cpflow_b200 — C ABI of the B200-native multi-start variational-synthesis engine.
 *
 * This is the drop-in boundary for the hot path of idnm/cpflow (SURVEY.md §8b).  The
 * reference has no FFI layer: its boundary is the Python call
 *     mynimize_repeated(loss_func, num_params, method, learning_rate, num_iterations,
 *                       initial_params_batch, regularization_func, u_func, keep_history)
 * (reference cpflow/optimization.py:269-382) fed with Python closures.  A kernel cannot run
 * closures, so this ABI takes the same computation as a DECLARATIVE spec:
 *
 *   gate program   <- Ansatz.unitary / build_unitary        (cpflow/main.py:106-146, 186-191)
 *                     qiskit_circ_to_jax_unitary             (cpflow/circuit_assembly.py:48-81)
 *   loss spec      <- cost_HST / user loss closures          (cpflow/matrix_utils.py:35-42,
 *                                                              cpflow/main.py:528-533)
 *   penalty spec   <- make_regularization_function, r*sum R  (cpflow/penalty.py:44-97,
 *                                                              cpflow/main.py:563-564)
 *   adam spec      <- optax.adam(learning_rate)              (cpflow/optimization.py:232, 342)
 *
 * Conventions
 *   - every entry point returns 0 on success, a negative cpf_status on error, and never
 *     throws; cpf_last_error() returns a thread-local message for the last failure;
 *   - all data buffers are CALLER-OWNED DEVICE memory on the current CUDA device unless a
 *     parameter says "host"; complex data is interleaved (re, im) of the call's dtype;
 *   - calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = default
 *     stream) and perform no hidden synchronisation;
 *   - qubit order is big-endian as in the reference: qubit 0 is the MOST significant bit of the
 *     row index of the unitary (cpflow/circuit_assembly.py:31-45);
 *   - a cpf_program is immutable after creation and may be shared by threads and streams;
 *   - a loss call (cpf_loss_grad, cpf_adam_run and their _multi forms) is refused before any CUDA call: loss kind
 *     and mask, qubit limits, target table and target_index, penalty spec and cp_mask, dtype, Adam buffers and the
 *     caller-owned workspace (alignment and size) are all checked first.  The query entry points
 *     (cpf_workspace_bytes(_multi), cpf_launch_plan, cpf_eval_cost, cpf_executed_cost) refuse the same loss kinds
 *     and dtypes with the same codes.
 */
#ifndef CPFLOW_B200_H
#define CPFLOW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPF_VERSION 200 /* 0.2.0 */
#define CPF_MAX_QUBITS 8
#define CPF_MAX_SEGMENTS 16

typedef enum cpf_status {
  CPF_OK = 0,
  CPF_ERR_INVALID = -1,     /* bad argument */
  CPF_ERR_UNSUPPORTED = -2, /* valid request the engine cannot run (e.g. too many qubits) */
  CPF_ERR_CUDA = -3,        /* CUDA runtime failure (message has the CUDA error string) */
  CPF_ERR_NOMEM = -4
} cpf_status;

/* Gate kinds — names and matrices follow cpflow/gates.py:22-58. */
typedef enum cpf_gate_kind {
  CPF_RX = 0, /* exp(-i a X / 2)            gates.py:26-27 */
  CPF_RY = 1, /* exp(-i a Y / 2)            gates.py:30-31 */
  CPF_RZ = 2, /* exp(-i a Z / 2)            gates.py:34-35 */
  CPF_CP = 3, /* diag(1,1,1,exp(i a))       gates.py:51-58 */
  CPF_CZ = 4, /* diag(1,1,1,-1)             gates.py:45-48 */
  CPF_CX = 5  /* CNOT, control q0 target q1 gates.py:40-43 */
} cpf_gate_kind;

/* One primitive gate in time order.  `param` indexes the angle vector, or is -1 for a gate
 * with the constant angle `const_angle` (used for frozen / projected gates). */
typedef struct cpf_op {
  int32_t kind; /* cpf_gate_kind */
  int32_t q0;
  int32_t q1;    /* second qubit of a 2-qubit gate, else -1 */
  int32_t param; /* index into the angle vector or -1 */
  double const_angle;
} cpf_op;

typedef enum cpf_dtype {
  CPF_F32 = 0, /* angles float32, amplitudes complex64  (the reference's default x32 mode) */
  CPF_F64 = 1  /* angles float64, amplitudes complex128 */
} cpf_dtype;

typedef enum cpf_loss_kind {
  CPF_LOSS_HS = 0,       /* 1 - |sum_ij U_ij conj(V_ij)|^2 / N^2   matrix_utils.py:35-42 */
  CPF_LOSS_STATE = 1,    /* 1 - |<psi| U |0>|^2                    tutorial ipynb:1318    */
  CPF_LOSS_RELPHASE = 2, /* 1 - sum_ij |conj(V_ij) U_ij|^2 / N     tutorial ipynb:1507    */
  CPF_LOSS_ISOMETRY = 3  /* 1 - |sum_c <W e_c| U |s_c>|^2 / k^2     (ancilla qubits start in |0>) */
} cpf_loss_kind;

/* ISOMETRY: the qubits of `ancilla_mask` (bit q = qubit q) start in |0>, so only the images of the k = 2^(n - popcount)
 * basis states s_0 < ... < s_{k-1} whose ancilla bits are 0 matter; column c of the N x k target W is the wanted
 * image of |s_c>.  One global phase, like HS: ancilla_mask = 0 is the HS loss, all qubits (k = 1) the state loss.
 * n <= 5 runs on the HS kernels (target 2^a [W at the columns s_c, 0 elsewhere], N = 2^a k: exact scaling); n = 6-8
 * on the isometry kernel with k <= 32 (k > 32 and ancilla_mask = 0 are CPF_ERR_UNSUPPORTED).  Not for multi-target
 * tables.  A mask bit at a position >= n is CPF_ERR_INVALID. */
typedef struct cpf_loss_spec {
  int32_t kind;       /* cpf_loss_kind */
  const void* target; /* device: N*N complex row-major (HS, RELPHASE), N complex (STATE), N*k row-major (ISOMETRY) */
  int32_t ancilla_mask; /* ISOMETRY only (ignored for the other kinds) */
} cpf_loss_spec;

/* cpf_workspace_bytes, cpf_eval_cost, cpf_executed_cost and cpf_launch_plan take a loss kind only: for the isometry
 * loss pass CPF_ISOMETRY_KIND(ancilla_mask), which carries the mask in bits 8-15. */
#define CPF_ISOMETRY_KIND(ancilla_mask) ((int32_t)CPF_LOSS_ISOMETRY | ((int32_t)(ancilla_mask) << 8))

typedef enum cpf_penalty_kind {
  CPF_PEN_NONE = 0,
  CPF_PEN_PIECEWISE = 1, /* first-true-wins piecewise-linear table of (a mod period) */
  CPF_PEN_L1 = 2         /* |a|                                     penalty.py:74-76 */
} cpf_penalty_kind;

/* r * sum_i R(angles_i) over the parameters of CP gates (cpflow/main.py:563-564).
 * PIECEWISE restates cp_penalty_linear (cpflow/penalty.py:44-71): a <- a mod period; the first
 * segment s with lo[s] < a <= hi[s] gives R = slope[s]*a + intercept[s]; no match gives 0.
 * `cp_mask` is an optional HOST array of n_params bytes selecting which parameters are
 * penalised; it may only select parameters of CP gates (NULL = all CP-gate parameters). */
typedef struct cpf_penalty_spec {
  int32_t kind; /* cpf_penalty_kind */
  int32_t n_segments;
  double r;
  double period;
  double lo[CPF_MAX_SEGMENTS];
  double hi[CPF_MAX_SEGMENTS];
  double slope[CPF_MAX_SEGMENTS];
  double intercept[CPF_MAX_SEGMENTS];
  const uint8_t* cp_mask; /* host, nullable */
} cpf_penalty_spec;

/* optax.adam(lr, b1=0.9, b2=0.999, eps=1e-8, eps_root=0) — optax 0.1.1 scale_by_adam. */
typedef struct cpf_adam_spec {
  double lr, b1, b2, eps;
} cpf_adam_spec;

typedef struct cpf_program cpf_program;

typedef struct cpf_program_info {
  int32_t n_qubits;
  int32_t n_params;
  int32_t n_ops;       /* primitive gates given at creation */
  int32_t n_rotations; /* primitive 1-qubit rotations (G1 of SURVEY.md §8) */
  int32_t n_phase;     /* CP + CZ gates (K) */
  int32_t n_fused;     /* fused single-qubit SU(2) gates in the device schedule */
  int32_t n_sched;     /* total ops in the device schedule */
  int32_t reserved;
} cpf_program_info;

/* Device-side state of one Adam run over a batch of B samples.  Every pointer is device
 * memory of the call's dtype unless noted; [B,P] arrays are row-major, P = n_params. */
typedef struct cpf_adam_buffers {
  void* angles;            /* [B,P] in: theta at step `step0`; out: theta after the last step */
  void* m;                 /* [B,P] first moment  (ignored on input when step0 == 0) */
  void* v;                 /* [B,P] second moment (ignored on input when step0 == 0) */
  const uint8_t* freeze;   /* [B,P] nullable; nonzero = parameter is frozen (never updated):
                              the reduced vector of cp_utils.py:100-108 */
  void* best_params;       /* [B,P] params at the lowest regloss so far (optimization.py:70-73) */
  void* best_regloss;      /* [B]   in/out when step0 > 0 */
  void* best_reg;          /* [B]   penalty value at the best point */
  void* init_regloss;      /* [B]   regloss(theta_0), written when step0 == 0 */
  void* init_reg;          /* [B]   penalty(theta_0), written when step0 == 0 */
  void* hist_params;       /* nullable [B,hist_len,P]: row i+1 = theta_{i+1} (optimization.py:52-59) */
  void* hist_regloss;      /* nullable [B,hist_len]:   row i   = regloss(theta_i) */
  int64_t hist_len;        /* number of history rows (the run's total num_iterations) */
  void* workspace;         /* nullable: 256-byte aligned device scratch of at least cpf_workspace_bytes(...) bytes,
                              owned by the caller.  NULL: the library takes its scratch from the device's
                              stream-ordered memory pool on `stream` (and, once per device, raises that pool's
                              release threshold so the blocks are kept between calls) */
  int64_t workspace_bytes;
} cpf_adam_buffers;

int cpf_version(void);
const char* cpf_last_error(void);

/* Build an immutable gate program.  Replaces the closure `anz.unitary` / `u(angles)`
 * (cpflow/main.py:186-191, cpflow/circuit_assembly.py:55-76).  Each parameter may feed at
 * most one gate (true for every program the reference builds). */
int cpf_program_create(int32_t n_qubits, int32_t n_ops, const cpf_op* ops, int32_t n_params,
                       cpf_program** out);
int cpf_program_destroy(cpf_program* prog);
int cpf_program_get_info(const cpf_program* prog, cpf_program_info* info);

/* U_out[B,N,N] (complex, row-major) = unitary of the program at angles[B,P].
 * Replaces Ansatz.unitary under vmap (cpflow/main.py:186-191). */
int cpf_unitary(const cpf_program* prog, int32_t dtype, int64_t batch, const void* angles,
                void* u_out, void* stream);

/* loss[B], reg[B], grad[B,P] = d(loss+reg)/d(angles).  Replaces
 * vmap(value_and_grad(regloss_func)) (cpflow/optimization.py:331-340).  `grad`, `reg` and
 * `penalty` may be NULL. */
int cpf_loss_grad(const cpf_program* prog, const cpf_loss_spec* loss,
                  const cpf_penalty_spec* penalty, int32_t dtype, int64_t batch,
                  const void* angles, void* loss_out, void* reg_out, void* grad_out, void* stream);

/* Generic vector-Jacobian product for a user loss evaluated outside the engine on the
 * materialised unitary (cpflow/main.py:528-529 `unitary_loss_func`): given
 * cotangent[B,N,N] = dL/dconj(U) it returns grad[B,P] = 2 Re <cotangent, dU/dtheta>, on 2-8 qubits.
 * n <= 5 runs on the full-unitary kernels; n = 6-8 on the cotangent mode of the isometry kernel (one launch item
 * per sample and chunk of up to 32 columns, the chunks' gradients added in a fixed order), which needs scratch of
 * batch x (N / columns per item) x P reals from the device's stream-ordered pool.  A sample's gradient does not
 * depend on its batch position or on the batch size.  A program whose shared-memory store does not fit even at one
 * column per item is refused with CPF_ERR_UNSUPPORTED. */
int cpf_adjoint_from_cotangent(const cpf_program* prog, int32_t dtype, int64_t batch,
                               const void* angles, const void* cotangent, void* grad_out,
                               void* stream);

/* `num_steps` fused iterations of: evaluate regloss and gradient at theta_i, track the best
 * (strict <, pre-update params), Adam-update to theta_{i+1}.  Replaces
 * jit(vmap(mynimize_particular)) with method='adam' (cpflow/optimization.py:14-25, 61-75,
 * 91-94, 362).  `step0` is the number of steps already taken (0 for a fresh run); runs may be
 * split into consecutive calls that give results identical to one call. */
int cpf_adam_run(const cpf_program* prog, const cpf_loss_spec* loss,
                 const cpf_penalty_spec* penalty, const cpf_adam_spec* adam, int32_t dtype,
                 int64_t batch, int64_t step0, int64_t num_steps, const cpf_adam_buffers* buf,
                 void* stream);

/* Device scratch one cpf_adam_run (or cpf_loss_grad) call on `batch` samples needs: the packed optimiser state
 * (16 bytes per parameter position and sample on the Heisenberg-picture kernel; positions are the parameters padded
 * to the lanes' pair slots, see heis_impl.cuh: heis_pk_stride), the staged target and the penalty mask.
 * Callers that manage device memory themselves allocate this once and pass it in cpf_adam_buffers.workspace; a call
 * given a smaller or misaligned workspace is refused with CPF_ERR_INVALID (before any CUDA call, as every refusal of a
 * loss call). */
int cpf_workspace_bytes(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch, int64_t* bytes);

/* One iteration of the same loop for a loss that is evaluated OUTSIDE the engine (an arbitrary user
 * `unitary_loss_func(U)`, cpflow/main.py:528-529): the caller evaluates loss[B] on cpf_unitary's output and gets
 * grad[B,P] = d loss / d theta from cpf_adjoint_from_cotangent; this call adds the penalty and its gradient
 * (cpflow/main.py:563-564), tracks the best point (strict <, pre-update parameters; `step` == 0 initialises
 * init_* / best_*), and applies the optax-Adam update (cpflow/optimization.py:14-25, 61-75) in place, honouring
 * `freeze` and the history buffers exactly like cpf_adam_run.  `step` = number of steps already taken. */
int cpf_adam_step(const cpf_program* prog, const cpf_penalty_spec* penalty, const cpf_adam_spec* adam,
                  int32_t dtype, int64_t batch, int64_t step, const void* loss, const void* grad,
                  const cpf_adam_buffers* buf, void* stream);

/* Multi-target runs: many independent targets of one loss kind, optimised on the same program in ONE launch.
 * Sample b of the batch is scored against target target_index[b]; everything else (penalty, Adam, freeze mask,
 * history, split runs with step0 > 0) works exactly as in cpf_loss_grad / cpf_adam_run, and a sample's results are
 * those of a single-target call on its own target run on the same kernel family (the Heisenberg-picture kernel with
 * run-time qubit pairs for HS on block-structured templates, otherwise the interpreter kernel).  Every entry of
 * target_index is checked before any CUDA call: a bad index is CPF_ERR_INVALID with a message. */
typedef struct cpf_target_table {
  int32_t kind;                 /* cpf_loss_kind, as in cpf_loss_spec */
  int32_t n_targets;
  const void* targets;          /* device: n_targets x (N*N complex, row-major) for HS / RELPHASE, n_targets x N for STATE */
  const int32_t* target_index;  /* HOST [batch]: target of each sample, validated in [0, n_targets) */
} cpf_target_table;

int cpf_loss_grad_multi(const cpf_program* prog, const cpf_target_table* table, const cpf_penalty_spec* penalty,
                        int32_t dtype, int64_t batch, const void* angles, void* loss_out, void* reg_out,
                        void* grad_out, void* stream);
int cpf_adam_run_multi(const cpf_program* prog, const cpf_target_table* table, const cpf_penalty_spec* penalty,
                       const cpf_adam_spec* adam, int32_t dtype, int64_t batch, int64_t step0, int64_t num_steps,
                       const cpf_adam_buffers* buf, void* stream);
/* Device scratch of one cpf_adam_run_multi / cpf_loss_grad_multi call: that of cpf_workspace_bytes without the staged
 * target, plus the target table (n_targets packed targets) and the device copy of target_index (4 bytes a sample). */
int cpf_workspace_bytes_multi(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch,
                              int32_t n_targets, int64_t* bytes);

/* cz[B] (int32) = count_cz(angles * cp_mask, threshold) (cpflow/cp_utils.py:45-67): per CP
 * parameter 0 if (a mod 2pi) is within `threshold` of 0 or 2pi, 1 if within of pi, else 2.
 * If `projected` (nullable [B,P]) and `frozen` (nullable uint8 [B,P]) are given they receive the
 * projection of cpflow/cp_utils.py:70-77, 111-141 (near 0 -> 0, near pi -> pi, and the mask). */
int cpf_count_cz(const cpf_program* prog, int32_t dtype, int64_t batch, const void* angles,
                 double threshold, int32_t* cz_out, void* projected, uint8_t* frozen, void* stream);

/* out[n] (int32) = cz_value(angles[i], threshold) elementwise (cpflow/cp_utils.py:45-57): the number
 * of CZ gates a CP gate with that angle costs (0 near 0/2pi, 1 near pi, else 2). */
int cpf_cz_value(int32_t dtype, int64_t n, const void* angles, double threshold, int32_t* out,
                 void* stream);

/* Initial angles of Synthesize._generate_initial_angles (cpflow/main.py:541-548,
 * cpflow/cp_utils.py:13-42, cpflow/trigonometric_utils.py:35-38) with jax 0.3.x threefry
 * semantics: sample s of a batch of `total_samples` drawn from PRNGKey(seed).  Writes samples
 * [first, first+count) to out[count,P]; results do not depend on how the batch is sharded.
 * cp_dist: 0 = 'uniform', 1 = '0' (CP angles zeroed), 2 = 'normal' (CP angles 1.5 * N(0,1), cp_utils.py:38-40). */
int cpf_initial_angles(const cpf_program* prog, int32_t dtype, uint64_t seed,
                       int64_t total_samples, int64_t first, int64_t count, int32_t cp_dist,
                       void* out, void* stream);

/* Algorithmic work of one loss+grad evaluation, SURVEY.md §8(d):
 * flops = C*N*(16*G1 + 4*K + 8), bytes = 6*P*sizeof(real) + 2*sizeof(real); C = N columns (HS, RELPHASE), 1 (STATE),
 * k (ISOMETRY). */
int cpf_eval_cost(const cpf_program* prog, int32_t loss_kind, int32_t dtype, double* flops,
                  double* bytes);

/* Floating-point operations the engine EXECUTES per loss+grad(+Adam) evaluation of one sample on the kernel it would
 * pick for (program, loss, dtype), FMA = 2: the Heisenberg-picture kernel needs far fewer than the credited
 * adjoint-sweep count of cpf_eval_cost (bench.py reports both: roofline.frac is executed flop/s over the measured
 * FP32 peak).  Derived from the fused schedule; cross-checked against the ncu opcode mix (DESIGN.md section 3). */
int cpf_executed_cost(const cpf_program* prog, int32_t loss_kind, int32_t dtype, double* flops);

/* Diagnostics: the launch geometry cpf_adam_run / cpf_loss_grad would use for `batch` samples (no reference
 * counterpart; it makes the geometry rules testable without a device).  engine: 1 = Heisenberg-picture kernel
 * (HS loss on a layered template), 0 = state-adjoint kernel (the remaining fields are 0).  n_sm / regs_per_thread:
 * 0 = 148 SMs / 128 registers (nothing is queried from a device). */
typedef struct cpf_launch_info {
  int32_t engine;
  int32_t ctas_per_sm;        /* co-resident CTAs per SM the geometry was planned for */
  int32_t block_threads;      /* multiple of 32 */
  int32_t samples_per_cta;
  int32_t threads_per_sample;
  int32_t max_block_threads;
  int32_t words_per_sample;   /* shared-memory words (of the real type) per sample */
  int32_t time_slices;        /* launches-in-a-ring factor k a 2000-step cpf_adam_run over `batch` would use (1: one
                                 launch; k > 1: steps cut into k chunks so every launch but the last runs at full
                                 residency — results are bit-identical either way) */
  int64_t grid;
  int64_t smem_bytes;         /* dynamic shared memory per CTA */
  int64_t launches_per_run;   /* engine-kernel launches of that cpf_adam_run (1 unless time-sliced) */
} cpf_launch_info;
int cpf_launch_plan(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch, int32_t n_sm,
                    int32_t regs_per_thread, cpf_launch_info* out);

#ifdef __cplusplus
}
#endif
#endif /* CPFLOW_B200_H */
