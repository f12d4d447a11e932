// C ABI of cpflow_b200 (include/cpflow_b200.h).  Plain pointers and sizes; no exceptions cross
// the boundary.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <mutex>
#include <string>

#include "cpflow_b200.h"
#include "heis_impl.cuh"
#include "iso_impl.cuh"
#include "launch.cuh"
#include "program.hpp"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
int cuda_fail(const char* what, cudaError_t e) {
  return fail(CPF_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CPF_CUDA(call)                                        \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return cuda_fail(#call, e__);     \
  } while (0)

// Per-call scratch (packed optimiser state, staged target, penalty mask): carved from a caller-provided workspace
// (cpf_adam_buffers.workspace, sized by cpf_workspace_bytes) or, without one, taken from the device's stream-ordered
// pool and returned to it when the call has been enqueued.
struct Scratch {
  char* base = nullptr;
  size_t size = 0, used = 0;
  cudaStream_t st = nullptr;
  void* owned[8] = {nullptr};
  int n_owned = 0;
  static size_t align(size_t b) { return (b + 255) & ~(size_t)255; }
  int get(void** out, size_t bytes) {
    bytes = align(bytes ? bytes : 1);
    if (base) {
      if (used + bytes > size)
        return fail(CPF_ERR_INVALID, "workspace too small: cpf_workspace_bytes gives the size this call needs");
      *out = base + used;
      used += bytes;
      return CPF_OK;
    }
    if (n_owned >= 8) return fail(CPF_ERR_NOMEM, "scratch table full");
    cudaError_t e = cudaMallocAsync(out, bytes, st);
    if (e != cudaSuccess) return cuda_fail("cudaMallocAsync(scratch)", e);
    owned[n_owned++] = *out;
    return CPF_OK;
  }
  ~Scratch() { for (int i = 0; i < n_owned; ++i) cudaFreeAsync(owned[i], st); }
};

// per-device copy of the schedule and gate metadata, created on first use
int device_program(const cpf::Program* prog, cpf::DeviceProgram* out) {
  int dev = 0;
  CPF_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(prog->mu);
  auto it = prog->dev.find(dev);
  if (it != prog->dev.end()) { *out = it->second; return CPF_OK; }
  cpf::DeviceProgram d;
  const size_t ns = prog->sched.size() * sizeof(uint32_t);
  const size_t nu = prog->su2.size() * sizeof(cpf::Su2Meta);
  const size_t nc = prog->cp.size() * sizeof(cpf::CpMeta);
  CPF_CUDA(cudaMalloc(&d.sched, ns ? ns : 4));
  CPF_CUDA(cudaMalloc(&d.su2, nu ? nu : 4));
  CPF_CUDA(cudaMalloc(&d.cp, nc ? nc : 4));
  if (ns) CPF_CUDA(cudaMemcpy(d.sched, prog->sched.data(), ns, cudaMemcpyHostToDevice));
  if (nu) CPF_CUDA(cudaMemcpy(d.su2, prog->su2.data(), nu, cudaMemcpyHostToDevice));
  if (nc) CPF_CUDA(cudaMemcpy(d.cp, prog->cp.data(), nc, cudaMemcpyHostToDevice));
  prog->dev[dev] = d;
  *out = d;
  return CPF_OK;
}

// decoded schedule for a kernel configuration with `rb` register bits, cached per device
int device_decoded(const cpf::Program* prog, int rb, cpf::DeviceDecoded* out) {
  if (rb < 0 || rb >= 8)
    return fail(CPF_ERR_UNSUPPORTED, cpf::FULL_UNITARY_LIMIT);
  int dev = 0;
  CPF_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(prog->mu);
  cpf::DeviceProgram& d = prog->dev[dev];
  if (!d.has_dec[rb]) {
    const cpf::DecodedSchedule ds = cpf::decode_schedule(*prog, rb);
    cpf::DeviceDecoded dd;
    const size_t no = ds.ops.size() * sizeof(uint32_t), nr = ds.red.size() * sizeof(uint16_t);
    CPF_CUDA(cudaMalloc(&dd.ops, no ? no : 8));
    CPF_CUDA(cudaMalloc(&dd.red, nr ? nr : 16));
    if (no) CPF_CUDA(cudaMemcpy(dd.ops, ds.ops.data(), no, cudaMemcpyHostToDevice));
    if (nr) CPF_CUDA(cudaMemcpy(dd.red, ds.red.data(), nr, cudaMemcpyHostToDevice));
    dd.n_red = (int)(ds.red.size() / 8);
    d.dec[rb] = dd;
    d.has_dec[rb] = true;
  }
  *out = d.dec[rb];
  return CPF_OK;
}

template <typename R>
int fill_common(const cpf::Program* prog, cpf::KParams<R>& p, int64_t batch, bool single = false) {
  std::memset(&p, 0, sizeof(p));
  cpf::DeviceProgram d;
  int rc = device_program(prog, &d);
  if (rc) return rc;
  cpf::DeviceDecoded dd;
  rc = device_decoded(prog, cpf::engine_rb<R>(prog->n_qubits, single), &dd);
  if (rc) return rc;
  p.dec = dd.ops; p.red = dd.red; p.n_red = dd.n_red;
  p.n_sched = (int)prog->sched.size();
  p.su2 = d.su2; p.n_su2 = (int)prog->su2.size();
  p.cp = d.cp; p.n_cp = (int)prog->cp.size();
  p.P = prog->n_params; p.B = batch;
  p.pen.kind = CPF_PEN_NONE;
  p.nsteps = 1;
  return CPF_OK;
}

// layered templates run on their specialised kernel when one was compiled for the layer
// (CPF_NO_LAYERED=1 forces the interpreter kernel: used by the tests to cover both)
bool layered_kernels(const cpf::Program* prog) {
  const char* e = getenv("CPF_NO_LAYERED");
  return prog->layered && !(e && e[0] == '1');
}

// the state-adjoint kernels: the one compiled for the layer when `layered` and one exists, else the interpreter
template <typename R>
int launch_any(const cpf::KParams<R>& p, const cpf::Program* prog, bool single, bool layered, cudaStream_t st,
               std::string& err) {
  int rc = CPF_OK;
  if (layered && cpf::launch_layered<R>(p, *prog, single, st, err, rc)) return rc;
  return cpf::launch_engine<R>(p, prog->n_qubits, single, st, err);
}

// The penalty in the kernels' form.  Refuses a bad spec and a cp_mask that selects a parameter of no CP gate; the mask
// itself goes to the device with upload_cp_mask.
template <typename R>
int penalty_params(const cpf::Program* prog, const cpf_penalty_spec* pen, cpf::PenaltyT<R>* out) {
  cpf::PenaltyT<R>& q = *out;
  std::memset(&q, 0, sizeof(q));
  q.kind = CPF_PEN_NONE;
  if (!pen || pen->kind == CPF_PEN_NONE) return CPF_OK;
  if (pen->kind != CPF_PEN_PIECEWISE && pen->kind != CPF_PEN_L1)
    return fail(CPF_ERR_INVALID, "unknown penalty kind");
  if (pen->kind == CPF_PEN_PIECEWISE && (pen->n_segments < 1 || pen->n_segments > CPF_MAX_SEGMENTS))
    return fail(CPF_ERR_INVALID, "penalty n_segments out of range");
  if (pen->kind == CPF_PEN_PIECEWISE && !(pen->period > 0))
    return fail(CPF_ERR_INVALID, "penalty period must be positive");
  // only parameters of CP gates may be penalised
  if (pen->cp_mask)
    for (int i = 0; i < prog->n_params; ++i)
      if (pen->cp_mask[i] && !prog->is_cp_param[i])
        return fail(CPF_ERR_UNSUPPORTED, "cp_mask selects a parameter that does not feed a CP gate");
  q.kind = pen->kind; q.nseg = pen->n_segments;
  q.r = (R)pen->r; q.period = (R)pen->period;
  for (int s = 0; s < CPF_MAX_SEGMENTS; ++s) {
    const bool on = pen->kind == CPF_PEN_PIECEWISE && s < pen->n_segments;
    q.lo[s] = on ? (R)pen->lo[s] : (R)INFINITY; q.hi[s] = on ? (R)pen->hi[s] : (R)INFINITY;
    q.slope[s] = on ? (R)pen->slope[s] : R(0); q.icpt[s] = on ? (R)pen->intercept[s] : R(0);
  }
  // ascending, disjoint segments (in the kernel's precision) can be searched instead of scanned
  q.sorted = pen->kind == CPF_PEN_PIECEWISE;
  for (int s = 0; s < pen->n_segments && s < CPF_MAX_SEGMENTS && q.sorted; ++s) {
    if (!(q.lo[s] <= q.hi[s])) q.sorted = 0;
    if (s + 1 < pen->n_segments && !(q.hi[s] <= q.lo[s + 1])) q.sorted = 0;
  }
  return CPF_OK;
}

// the cp_mask as one flag per CP gate, copied into its scratch block
int upload_cp_mask(const cpf::Program* prog, const uint8_t* cp_mask, void* dev, cudaStream_t st) {
  std::string flags(prog->cp.size(), '\0');
  for (size_t k = 0; k < prog->cp.size(); ++k)
    flags[k] = prog->cp[k].pidx >= 0 && cp_mask[prog->cp[k].pidx] ? 1 : 0;
  // pageable source: the runtime stages the bytes before returning, so `flags` may die
  CPF_CUDA(cudaMemcpyAsync(dev, flags.data(), flags.size(), cudaMemcpyHostToDevice, st));
  return CPF_OK;
}

// Per-call scratch (packed optimiser state, staged targets) comes from the device's default stream-ordered pool.
// Its release threshold defaults to 0: freed blocks go back to the driver at the next synchronisation and the
// next call pays for mapping hundreds of megabytes again.  Keep them in the pool (once per device and process).
static void keep_pool_memory() {
  static std::mutex mu;
  static bool done[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return;
  std::lock_guard<std::mutex> lk(mu);
  if (done[dev]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long thr = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  done[dev] = true;
}

// The target-independent part of the heis set-up: per-gate scratch (`aux_pad` bytes at the start of `blk`) followed by
// the packed optimiser state, gate-pattern flags.
template <typename R>
void stage_heis_state(const cpf::Program* prog, cpf::KParams<R>& p, void* blk, size_t aux_pad) {
  const int cpt = cpf::heis_cpt<R>(prog->n_qubits);
  p.pk = reinterpret_cast<char*>(blk) + aux_pad;
  p.aux = reinterpret_cast<R*>(blk);
  // rotation-axis pattern shared by the surface gates (slots < n) and by the block gates (the rest)
  auto pattern = [&](size_t lo, size_t hi) {
    int pat = -1;
    for (size_t g = lo; g < hi && g < prog->su2.size(); ++g) {
      const cpf::Su2Meta& md = prog->su2[g];
      int q = 0;
      for (int k = 0; k < 3; ++k) q |= (md.axis[k] < 0 ? 15 : md.axis[k]) << (4 * k);
      if (pat == -1) pat = q;
      else if (pat != q) return 0xffff;
    }
    return pat < 0 ? 0xffff : pat;
  };
  for (int q = 0; q < 8; ++q) p.last_slot[q] = q < prog->n_qubits ? prog->last_slot[q] : 0;
  p.axp_surface = pattern(0, (size_t)prog->n_qubits);
  p.axp_block = pattern((size_t)prog->n_qubits, prog->su2.size());
  p.su2_all_params = 1;
  int referenced = 0;
  for (const cpf::Su2Meta& md : prog->su2)
    for (int k = 0; k < 3; ++k) {
      if (md.axis[k] >= 0 && md.pidx[k] < 0) p.su2_all_params = 0;
      if (md.pidx[k] >= 0) ++referenced;
    }
  p.cp_all_params = 1;
  for (const cpf::CpMeta& md : prog->cp) {
    if (md.pidx >= 0) ++referenced;
    if (md.pidx < 0 || md.is_cz) p.cp_all_params = 0;
  }
  p.unreferenced_params = referenced != prog->n_params;      // (a parameter feeds at most one gate: program.cpp)
  p.pk_stride = cpf::heis_pk_stride(prog->n_qubits, (1 << prog->n_qubits) / cpt, (int)prog->su2.size(), (int)prog->cp.size());
}

// ---- isometry losses (CPF_LOSS_ISOMETRY, CPF_LOSS_ISOMETRY_RELPHASE) ----
// Largest number of input columns k of the isometry kernel: a sample is k lane groups of 2^(n-RB) threads in one CTA.
constexpr int ISO_MAX_K = 32;

// k input columns (lane groups of the isometry kernel); the ancilla qubits as amplitude-index bits (qubit q is bit
// n - 1 - q, big-endian); the subspace kinds' caller k (0 for the isometry kinds), of which k is the next power of two
struct IsoSpec { int k, amask, sub_k; };
IsoSpec iso_spec(const cpf::Program* prog, int32_t mask) {
  const int n = prog->n_qubits;
  IsoSpec s{1 << (n - __builtin_popcount((unsigned)mask)), 0, 0};
  for (int q = 0; q < n; ++q)
    if ((mask >> q) & 1) s.amask |= 1 << (n - 1 - q);
  return s;
}

// ---- the plan of a loss call ----
// Which kernel runs a loss call and which scratch blocks it needs, decided on the host.  The staged calls and the query
// entry points all read it, so the size cpf_workspace_bytes reports is the sum of the blocks run_staged carves.
enum Route { ROUTE_ADJOINT, ROUTE_HEIS, ROUTE_ISO };
// scratch blocks, in carve order
enum Block { BLK_MASK, BLK_V, BLK_INDEX, BLK_TARGET, BLK_HEIS, N_BLK };

template <typename R>
struct CallPlan {
  Route route;          // the state-adjoint kernels, the Heisenberg-picture kernel (HS on layered templates) or the
                        // isometry kernel (the isometry loss on n >= 6, the relative-phase isometry loss on every n);
                        // each in a single- or a multi-target form
  bool multi;           // sample b is scored against target target_index[b] of a table
  bool layered;         // ROUTE_ADJOINT: try the kernel compiled for the layer before the interpreter
  bool single;          // single-column kernels (state loss, isometry kernel)
  bool iso_as_hs;       // n <= 5 isometry: the HS call on V = 2^a [W at the columns s_c, 0 elsewhere] (iso_impl.cuh:
                        // pack_iso_hs_kernel), built in BLK_V
  bool sub_as_hs;       // n <= 5 subspace loss (one global phase): the HS call on V = (N/k) B A^dag (iso_impl.cuh:
                        // pack_subspace_hs_kernel), built in BLK_V
  int32_t kind;         // the loss the kernel sees
  IsoSpec iso;          // isometry and subspace kinds (the subspace kinds: k = k', the padded group count)
  int n_stage;          // ROUTE_HEIS: SWP::NSTAGE of the kernel chosen
  int cpt, words;       // not ROUTE_ISO: columns per thread and words of one packed target
  size_t heis_aux;      // ROUTE_HEIS: per-gate scratch at the start of BLK_HEIS (the packed state follows, 256-byte aligned)
  cpf::PenaltyT<R> pen;
  bool pen_mask;        // a cp_mask is uploaded: BLK_MASK is carved
  size_t bytes[N_BLK];  // 0: no such block
  // the caller-owned workspace: every block, each 256-byte aligned (BLK_MASK whether or not a cp_mask is given)
  int64_t workspace() const {
    size_t total = 0;
    for (size_t b : bytes) total += Scratch::align(b);
    return (int64_t)total;
  }
};

// Every refusal of a loss call is made here, before any CUDA call.  table != NULL: a multi-target call (`kind` is the
// table's; its target_index, if given, is checked over `batch`).  pen may be NULL.
template <typename R>
int plan_call(const cpf::Program* prog, int32_t kind, int32_t mask, int64_t batch, const cpf_target_table* table,
              const cpf_penalty_spec* pen, CallPlan<R>* pl) {
  const int n = prog->n_qubits;
  *pl = CallPlan<R>();
  const bool sub = kind == CPF_LOSS_SUBSPACE || kind == CPF_LOSS_SUBSPACE_RELPHASE;
  const bool phases = kind == CPF_LOSS_ISOMETRY_RELPHASE || kind == CPF_LOSS_SUBSPACE_RELPHASE;
  if ((kind < CPF_LOSS_HS || kind > CPF_LOSS_ISOMETRY) && !phases && !sub)
    return fail(CPF_ERR_INVALID, "unknown loss kind");
  if (table && kind == CPF_LOSS_ISOMETRY)
    return fail(CPF_ERR_UNSUPPORTED, "multi-target tables do not take the isometry loss (one target per call)");
  if (table && kind == CPF_LOSS_ISOMETRY_RELPHASE)
    return fail(CPF_ERR_UNSUPPORTED,
                "multi-target tables do not take the relative-phase isometry loss (one target per call)");
  if (table && sub)
    return fail(CPF_ERR_UNSUPPORTED, "multi-target tables do not take the subspace losses (one target per call)");
  if (table && table->n_targets < 1) return fail(CPF_ERR_INVALID, "target table: n_targets must be >= 1");
  // HS, relative phase and an isometry without ancillas run on the full-unitary kernels, which stop at 5 qubits.  The
  // relative-phase isometry loss runs on the isometry kernel on every n, so only its k is limited (k <= 32 always
  // holds on n <= 5).
  if (sub) {
    // ancilla_mask carries k; the isometry kernel runs k' = the next power of two groups
    const int N = 1 << n;
    if (mask < 1 || mask > N)
      return fail(CPF_ERR_INVALID, "subspace losses take 1 <= k <= N = " + std::to_string(N) + " input states (k = " +
                                       std::to_string(mask) + ")");
    if (mask > ISO_MAX_K)
      return fail(CPF_ERR_UNSUPPORTED, "subspace losses take at most k = " + std::to_string(ISO_MAX_K) +
                                       " input states (k = " + std::to_string(mask) + ")");
    int kp = 1;
    while (kp < mask) kp <<= 1;
    pl->iso = IsoSpec{kp, 0, mask};
  } else if (kind == CPF_LOSS_ISOMETRY || phases) {
    if (mask < 0 || (mask >> n) != 0)
      return fail(CPF_ERR_INVALID, "ancilla_mask " + std::to_string(mask) + " names a qubit >= n = " + std::to_string(n));
    if (n > 5 && mask == 0 && !phases) return fail(CPF_ERR_UNSUPPORTED, cpf::FULL_UNITARY_LIMIT);
    pl->iso = iso_spec(prog, mask);
    if (n > 5 && pl->iso.k > ISO_MAX_K)
      return fail(CPF_ERR_UNSUPPORTED, "isometry losses on 6-8 qubits take at most k = " + std::to_string(ISO_MAX_K) +
                                       " input columns (k = 2^(n - popcount(ancilla_mask)) = " +
                                       std::to_string(pl->iso.k) + ")");
  } else if (kind != CPF_LOSS_STATE && n > 5) {
    return fail(CPF_ERR_UNSUPPORTED, cpf::FULL_UNITARY_LIMIT);
  }
  for (int64_t b = 0; table && table->target_index && b < batch; ++b) {
    const int32_t t = table->target_index[b];
    if (t < 0 || t >= table->n_targets)
      return fail(CPF_ERR_INVALID, "target_index[" + std::to_string(b) + "] = " + std::to_string(t) +
                                       " is outside [0, n_targets = " + std::to_string(table->n_targets) + ")");
  }
  if (int rc = penalty_params<R>(prog, pen, &pl->pen)) return rc;

  pl->multi = table != nullptr;
  pl->iso_as_hs = kind == CPF_LOSS_ISOMETRY && n <= 5;
  pl->sub_as_hs = kind == CPF_LOSS_SUBSPACE && n <= 5;
  pl->kind = pl->iso_as_hs || pl->sub_as_hs ? CPF_LOSS_HS : kind;
  const bool iso_route = pl->kind == CPF_LOSS_ISOMETRY || phases || pl->kind == CPF_LOSS_SUBSPACE;
  pl->single = pl->kind == CPF_LOSS_STATE || iso_route;
  pl->layered = layered_kernels(prog);
  // The Heisenberg-picture kernel keeps parameter and slot indices in 16 bits of shared memory (heis_impl.cuh: HSu2,
  // HCp) and B * P below 2^32.  CPF_ENGINE=adjoint forces the state-adjoint kernels (tests cover both engines).
  const char* eng = getenv("CPF_ENGINE");
  bool heis = pl->kind == CPF_LOSS_HS && pl->layered && prog->n_params <= 32767 && prog->su2.size() <= 32767 &&
              !(eng && std::strcmp(eng, "adjoint") == 0) &&
              (unsigned long long)batch * (unsigned long long)prog->n_params < (1ull << 32);
  if (heis) {
    cpf::KParams<R> dummy;
    std::string err;
    int rc = 0;
    heis = cpf::launch_heis<R>(dummy, *prog, nullptr, err, rc, true, &pl->n_stage);
  }
  pl->route = iso_route ? ROUTE_ISO : heis ? ROUTE_HEIS : ROUTE_ADJOINT;

  pl->bytes[BLK_MASK] = prog->cp.empty() ? 1 : prog->cp.size();
  pl->pen_mask = pl->pen.kind != CPF_PEN_NONE && pen->cp_mask && !prog->cp.empty();
  if (pl->iso_as_hs || pl->sub_as_hs) pl->bytes[BLK_V] = ((size_t)2 << (2 * n)) * sizeof(R);
  if (pl->route == ROUTE_ISO) {
    // W packed column by column; the subspace kinds: B and then A, each packed to k' columns
    pl->bytes[BLK_TARGET] = ((size_t)pl->iso.k << (n + 1)) * sizeof(R) * (sub ? 2 : 1);
    return CPF_OK;
  }
  pl->cpt = heis ? cpf::heis_cpt<R>(n) : pl->single ? 1 : cpf::cpt_for<R>(n);
  pl->words = heis ? cpf::heis_target_words<R>(n, pl->cpt) : cpf::target_words<R>(n, pl->cpt, pl->single);
  if (table) {
    // the kernels read index and targets (back to back) from global memory: no shared-memory copy, no padding
    pl->bytes[BLK_INDEX] = (size_t)batch * sizeof(int32_t);
    pl->bytes[BLK_TARGET] = (size_t)table->n_targets * (size_t)pl->words * sizeof(R);
  } else {
    pl->bytes[BLK_TARGET] = ((size_t)pl->words * sizeof(R) + 15) & ~(size_t)15;
  }
  if (heis) {
    const size_t aux = (size_t)batch * (prog->su2.empty() ? 1 : prog->su2.size()) * 4 * sizeof(R);
    pl->heis_aux = (aux + 255) & ~(size_t)255;      // the packed state starts on a 256-byte boundary (blocks of 16 positions)
    // lane-interleaved packed optimiser state (heis_impl.cuh: heis_pk_stride words per sample)
    const int tps = (1 << n) / pl->cpt;
    pl->bytes[BLK_HEIS] = pl->heis_aux + (size_t)batch *
                          (size_t)cpf::heis_pk_stride(n, tps, (int)prog->su2.size(), (int)prog->cp.size()) * sizeof(R);
  }
  return CPF_OK;
}

// the buffers every Adam entry point needs
int check_adam_buffers(const cpf_adam_buffers* buf) {
  if (!buf->angles || !buf->m || !buf->v || !buf->best_params || !buf->best_regloss || !buf->best_reg ||
      !buf->init_regloss || !buf->init_reg)
    return fail(CPF_ERR_INVALID, "a required cpf_adam_buffers pointer is NULL");
  if ((buf->hist_params || buf->hist_regloss) && buf->hist_len <= 0)
    return fail(CPF_ERR_INVALID, "history buffers given with hist_len <= 0");
  return CPF_OK;
}

// the table's own pointers; everything else about it is checked by plan_call
int check_table_pointers(const cpf_target_table* tt, int64_t batch) {
  if (!tt) return fail(CPF_ERR_INVALID, "target table is NULL");
  if (!tt->targets) return fail(CPF_ERR_INVALID, "target table: targets is NULL");
  if (batch > 0 && !tt->target_index) return fail(CPF_ERR_INVALID, "target table: target_index is NULL");
  return CPF_OK;
}

// A planned loss call: check the caller's workspace, carve every scratch block, then upload the program, stage the
// penalty mask and the target and launch.  Nothing touches the device before the blocks are carved.  `target` is the
// loss spec's or the table's; `set_mode` fills the mode fields of KParams; grad_out, if given, is zeroed first, and so
// are the moments of a fresh Adam run off the Heisenberg kernel.
template <typename R, typename SetMode>
int run_staged(const cpf::Program* prog, const CallPlan<R>& pl, const void* target, const cpf_target_table* table,
               const cpf_penalty_spec* pen, int64_t batch, void* workspace, int64_t workspace_bytes, void* grad_out,
               cudaStream_t st, SetMode set_mode) {
  Scratch sc;
  sc.st = st;
  if (workspace) {
    if (((uintptr_t)workspace & 255) != 0) return fail(CPF_ERR_INVALID, "workspace must be 256-byte aligned");
    if (workspace_bytes < pl.workspace())
      return fail(CPF_ERR_INVALID, "workspace too small: cpf_workspace_bytes gives the size this call needs");
    sc.base = (char*)workspace;
    sc.size = (size_t)workspace_bytes;
  } else if (pl.route == ROUTE_HEIS) {
    keep_pool_memory();
  }
  void* blk[N_BLK] = {};
  for (int b = 0; b < N_BLK; ++b)
    if (pl.bytes[b] && (b != BLK_MASK || pl.pen_mask))
      if (int rc = sc.get(&blk[b], pl.bytes[b])) return rc;

  const int n = prog->n_qubits;
  cpf::KParams<R> p;
  int rc = fill_common(prog, p, batch, pl.single);
  if (rc) return rc;
  set_mode(p);
  p.pen = pl.pen;
  if (blk[BLK_MASK]) {
    if ((rc = upload_cp_mask(prog, pen->cp_mask, blk[BLK_MASK], st))) return rc;
    p.cp_pen = (const uint8_t*)blk[BLK_MASK];
  }
  if (pl.iso_as_hs) {
    rc = cpf::launch_pack_iso<R>((const R*)target, (R*)blk[BLK_V], n, pl.iso.k, pl.iso.amask, true, st);
    if (rc) return fail(rc, "pack_iso launch failed");
    target = blk[BLK_V];
  } else if (pl.sub_as_hs) {
    rc = cpf::launch_pack_subspace_hs<R>((const R*)target, (R*)blk[BLK_V], n, pl.iso.sub_k, st);
    if (rc) return fail(rc, "pack_subspace_hs launch failed");
    target = blk[BLK_V];
  }
  R* packed = (R*)blk[BLK_TARGET];
  p.target_packed = packed;
  p.loss_kind = pl.kind;
  if (pl.multi) {
    // pageable source: the runtime stages the bytes before returning
    CPF_CUDA(cudaMemcpyAsync(blk[BLK_INDEX], table->target_index, (size_t)batch * sizeof(int32_t),
                             cudaMemcpyHostToDevice, st));
    rc = pl.route == ROUTE_HEIS
             ? cpf::launch_pack_targets_heis<R>((const R*)target, packed, n, pl.cpt, table->n_targets, st)
             : cpf::launch_pack_targets<R>((const R*)target, packed, n, pl.cpt, pl.single, table->n_targets, st);
    if (rc) return fail(rc, "pack_targets launch failed");
    p.target_index = (const int32_t*)blk[BLK_INDEX];
  } else if (pl.route == ROUTE_ISO && pl.iso.sub_k) {
    // B and A, each packed column by column to k' columns; the k' - k padding columns are zero
    const int k = pl.iso.sub_k, kp = pl.iso.k;
    const size_t col = (size_t)2 << n;                // reals per packed column
    if (k != kp) CPF_CUDA(cudaMemsetAsync(packed, 0, pl.bytes[BLK_TARGET], st));
    rc = cpf::launch_pack_iso<R>((const R*)target, packed, n, k, 0, false, st);
    if (!rc) rc = cpf::launch_pack_iso<R>((const R*)target + col * k, packed + col * kp, n, k, 0, false, st);
    if (rc) return fail(rc, "pack_iso launch failed");
    p.iso_k = kp;
    p.inputs_packed = packed + col * kp;
    p.sub_k = k;
  } else if (pl.route == ROUTE_ISO) {
    rc = cpf::launch_pack_iso<R>((const R*)target, packed, n, pl.iso.k, pl.iso.amask, false, st);
    if (rc) return fail(rc, "pack_iso launch failed");
    p.iso_k = pl.iso.k;
    p.iso_amask = pl.iso.amask;
  } else {
    const size_t bytes = pl.bytes[BLK_TARGET];
    if (bytes != (size_t)pl.words * sizeof(R)) CPF_CUDA(cudaMemsetAsync(packed, 0, bytes, st));
    rc = pl.route == ROUTE_HEIS ? cpf::launch_pack_target_heis<R>((const R*)target, packed, n, pl.cpt, st)
                                : cpf::launch_pack_target<R>((const R*)target, packed, n, pl.cpt, pl.single, st);
    if (rc) return fail(rc, "pack_target launch failed");
    p.target_bytes = (int)bytes;
  }
  if (pl.route == ROUTE_HEIS) stage_heis_state(prog, p, blk[BLK_HEIS], pl.heis_aux);
  if (grad_out) CPF_CUDA(cudaMemsetAsync(grad_out, 0, (size_t)batch * prog->n_params * sizeof(R), st));
  // A fresh Adam run starts every moment at zero.  The kernels' updates never visit frozen parameters or those that
  // feed no gate, so these keep the zeros.  The Heisenberg kernel writes every moment from its packed state; for the
  // other kernels the zeros are set here.  Written in engine_kernel's first pass instead, they changed that kernel's
  // code and cost 8 % of the 8-qubit state-preparation rate (one B200 at 1000 W: 9.8 -> 9.0 M evals/s).
  if (p.mode == cpf::M_ADAM && p.step0 == 0 && pl.route != ROUTE_HEIS) {
    CPF_CUDA(cudaMemsetAsync(p.m, 0, (size_t)batch * prog->n_params * sizeof(R), st));
    CPF_CUDA(cudaMemsetAsync(p.v, 0, (size_t)batch * prog->n_params * sizeof(R), st));
  }

  std::string err;
  if (pl.route == ROUTE_ISO) {
    rc = pl.kind == CPF_LOSS_ISOMETRY_RELPHASE ? cpf::launch_iso_phase<R>(p, n, st, err)
         : pl.kind == CPF_LOSS_SUBSPACE        ? cpf::launch_sub<R>(p, n, st, err)
         : pl.kind == CPF_LOSS_SUBSPACE_RELPHASE ? cpf::launch_sub_phase<R>(p, n, st, err)
                                                 : cpf::launch_iso<R>(p, n, st, err);
  } else if (pl.route == ROUTE_HEIS) {
    if (!(pl.multi ? cpf::launch_heis_multi<R>(p, *prog, st, err, rc) : cpf::launch_heis<R>(p, *prog, st, err, rc, false))) {
      rc = CPF_ERR_UNSUPPORTED;
      err = "no Heisenberg-picture kernel for this program";
    }
  } else {
    rc = pl.multi ? cpf::launch_engine_multi<R>(p, n, pl.single, st, err) : launch_any<R>(p, prog, pl.single, pl.layered, st, err);
  }
  return rc ? fail(rc, err) : CPF_OK;
}

template <typename R>
int run_unitary(const cpf::Program* prog, int64_t batch, const void* angles, void* u_out, cudaStream_t st) {
  cpf::KParams<R> p;
  // 6-8 qubits: a column per virtual sample on the single-column kernels (engine_impl.cuh: colmode)
  const bool colmode = prog->n_qubits > 5;
  int rc = fill_common(prog, p, colmode ? batch << prog->n_qubits : batch, colmode);
  if (rc) return rc;
  p.mode = cpf::M_UNITARY;
  p.colmode = colmode ? 1 : 0;
  p.angles = (R*)angles; p.u_out = (R*)u_out;
  std::string err;
  rc = launch_any<R>(p, prog, colmode, layered_kernels(prog), st, err);
  return rc ? fail(rc, err) : CPF_OK;
}

// table != NULL: multi-target call (kind = table->kind, target = table->targets)
template <typename R>
int run_loss_grad(const cpf::Program* prog, int32_t kind, int32_t mask, const void* target, const cpf_penalty_spec* pen,
                  int64_t batch, const void* angles, void* loss_out, void* reg_out, void* grad_out,
                  cudaStream_t st, const cpf_target_table* table = nullptr) {
  CallPlan<R> pl;
  if (int rc = plan_call<R>(prog, kind, mask, batch, table, pen, &pl)) return rc;
  if (batch == 0) return CPF_OK;
  if (!loss_out) return fail(CPF_ERR_INVALID, "loss_out is NULL");
  if (!angles && prog->n_params > 0) return fail(CPF_ERR_INVALID, "angles is NULL");
  return run_staged<R>(prog, pl, target, table, pen, batch, nullptr, 0, grad_out, st, [&](cpf::KParams<R>& p) {
    p.mode = cpf::M_LOSSGRAD;
    p.angles = (R*)angles; p.loss_out = (R*)loss_out; p.reg_out = (R*)reg_out; p.grad_out = (R*)grad_out;
  });
}

// 6-8 qubits: the cotangent mode of the isometry kernel (iso_impl.cuh: InterpSweepIsoCot), one launch item per
// (sample, chunk of k_c columns), each item's gradient in a scratch row; the rows of a sample are then added in chunk
// order.  k_c depends on the program and the precision only, so a sample's gradient does not depend on the batch.
template <typename R>
int run_cotangent_iso(const cpf::Program* prog, int64_t batch, const void* angles, const void* cot, void* grad_out,
                      cudaStream_t st) {
  const int n = prog->n_qubits;
  cpf::KParams<R> p;
  int rc = fill_common(prog, p, batch, true);
  if (rc) return rc;
  const int kc = cpf::iso_cot_columns(n, cpf::engine_rb<R>(n, true), p.n_su2, p.n_cp, p.n_sched, p.n_red, sizeof(R));
  if (kc == 0)
    return fail(CPF_ERR_UNSUPPORTED, "program too large for cpf_adjoint_from_cotangent on " + std::to_string(n) +
                                     " qubits: the shared-memory store of one column does not fit 227 KB");
  const int n_chunks = (1 << n) / kc;
  p.mode = cpf::M_COTANGENT;
  p.B = batch * n_chunks;
  p.iso_k = kc;
  p.angles = (R*)angles; p.cot = (const R*)cot;
  Scratch sc;
  sc.st = st;
  R* partial = nullptr;
  const size_t pbytes = (size_t)p.B * prog->n_params * sizeof(R);
  rc = sc.get((void**)&partial, pbytes);
  if (rc) return rc;
  // parameters that feed no gate get no row entry from the kernel
  CPF_CUDA(cudaMemsetAsync(partial, 0, pbytes, st));
  p.grad_out = partial;
  std::string err;
  rc = cpf::launch_iso_cot<R>(p, n, st, err);
  if (rc) return fail(rc, err);
  rc = cpf::launch_cot_reduce<R>(partial, (R*)grad_out, batch, prog->n_params, n_chunks, st);
  return rc ? fail(rc, "cot_reduce launch failed") : CPF_OK;
}

template <typename R>
int run_cotangent(const cpf::Program* prog, int64_t batch, const void* angles, const void* cot,
                  void* grad_out, cudaStream_t st) {
  if (prog->n_qubits > 5) return run_cotangent_iso<R>(prog, batch, angles, cot, grad_out, st);
  cpf::KParams<R> p;
  int rc = fill_common(prog, p, batch);
  if (rc) return rc;
  p.mode = cpf::M_COTANGENT;
  p.angles = (R*)angles; p.cot = (const R*)cot; p.grad_out = (R*)grad_out;
  CPF_CUDA(cudaMemsetAsync(grad_out, 0, (size_t)batch * prog->n_params * sizeof(R), st));
  std::string err;
  rc = launch_any<R>(p, prog, false, layered_kernels(prog), st, err);
  return rc ? fail(rc, err) : CPF_OK;
}

template <typename R>
int run_adam(const cpf::Program* prog, int32_t kind, int32_t mask, const void* target, const cpf_penalty_spec* pen,
             const cpf_adam_spec* adam, int64_t batch, int64_t step0, int64_t num_steps,
             const cpf_adam_buffers* buf, cudaStream_t st, const cpf_target_table* table = nullptr) {
  CallPlan<R> pl;
  if (int rc = plan_call<R>(prog, kind, mask, batch, table, pen, &pl)) return rc;
  if (batch == 0 || num_steps == 0) return CPF_OK;
  if (int rc = check_adam_buffers(buf)) return rc;
  if (num_steps > 2000000000LL) return fail(CPF_ERR_INVALID, "num_steps too large");
  return run_staged<R>(prog, pl, target, table, pen, batch, buf->workspace, buf->workspace_bytes, nullptr, st,
                       [&](cpf::KParams<R>& p) {
    p.mode = cpf::M_ADAM;
    p.lr = (R)adam->lr; p.b1 = (R)adam->b1; p.b2 = (R)adam->b2; p.eps = (R)adam->eps;
    p.omb1 = (R)(1.0 - adam->b1); p.omb2 = (R)(1.0 - adam->b2);
    p.step0 = step0; p.nsteps = (int)num_steps;
    p.angles = (R*)buf->angles; p.m = (R*)buf->m; p.v = (R*)buf->v; p.freeze = buf->freeze;
    p.best_params = (R*)buf->best_params; p.best_regloss = (R*)buf->best_regloss;
    p.best_reg = (R*)buf->best_reg; p.init_regloss = (R*)buf->init_regloss; p.init_reg = (R*)buf->init_reg;
    p.hist_params = (R*)buf->hist_params; p.hist_regloss = (R*)buf->hist_regloss; p.hist_len = buf->hist_len;
  });
}

// The plan behind a query entry point's loss-kind argument: an isometry kind carries its ancilla mask in bits 8-15
// (CPF_ISOMETRY_KIND, CPF_ISOMETRY_RELPHASE_KIND), a subspace kind its k (CPF_SUBSPACE_KIND,
// CPF_SUBSPACE_RELPHASE_KIND); any other use of bits 8-31 makes an unknown kind.
template <typename R>
int plan_query(const cpf::Program* prog, int32_t arg, int64_t batch, CallPlan<R>* pl) {
  const int32_t base = arg & ~0xff00;
  const int32_t kind = base == CPF_LOSS_ISOMETRY || base == CPF_LOSS_ISOMETRY_RELPHASE || base == CPF_LOSS_SUBSPACE ||
                               base == CPF_LOSS_SUBSPACE_RELPHASE || (arg >> 8) == 0
                           ? arg & 0xff
                           : -1;
  return plan_call<R>(prog, kind, (arg >> 8) & 0xff, batch, nullptr, nullptr, pl);
}

// ---- count_cz / projection (cp_utils.py:45-77, 111-141) ----
template <typename R>
__global__ void count_cz_kernel(const cpf::CpMeta* cp, int n_cp, int P, long long B, const R* angles,
                                R threshold, int32_t* cz_out, R* projected, uint8_t* frozen) {
  const long long b = (long long)blockIdx.x * blockDim.y + threadIdx.y;
  if (b >= B) return;
  const R two_pi = R(2.0 * M_PI), pi = R(M_PI);
  if (projected)
    for (int i = threadIdx.x; i < P; i += 32) projected[b * P + i] = angles[b * P + i];
  if (frozen)
    for (int i = threadIdx.x; i < P; i += 32) frozen[b * P + i] = 0;
  __syncwarp();
  int cz = 0;
  for (int k = threadIdx.x; k < n_cp; k += 32) {
    const int pidx = cp[k].pidx;
    if (pidx < 0) continue;
    const R a0 = angles[b * P + pidx];
    const R a = cpf::pymod(a0, two_pi);
    int val = 2;
    if (a < threshold || cpf::abs_r(a - two_pi) < threshold) val = 0;
    else if (cpf::abs_r(a - pi) < threshold) val = 1;
    cz += val;
    // project_cp_angle tests pi first, then 0 / 2pi (cp_utils.py:70-77)
    int proj = -1;
    if (cpf::abs_r(a - pi) < threshold) proj = 1;
    else if (cpf::abs_r(a) < threshold || cpf::abs_r(a - two_pi) < threshold) proj = 0;
    if (proj >= 0) {
      if (projected) projected[b * P + pidx] = proj ? pi : R(0);
      if (frozen) frozen[b * P + pidx] = 1;
    }
  }
  for (int m = 16; m >= 1; m >>= 1) cz += __shfl_xor_sync(0xffffffffu, cz, m);
  if (threadIdx.x == 0 && cz_out) cz_out[b] = cz;
}

// ---- elementwise cz_value (cp_utils.py:45-57) ----
template <typename R>
__global__ void cz_value_kernel(const R* angles, long long n, R threshold, int32_t* out) {
  const R two_pi = R(2.0 * M_PI), pi = R(M_PI);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const R a = cpf::pymod(angles[i], two_pi);
    int val = 2;
    if (a < threshold || cpf::abs_r(a - two_pi) < threshold) val = 0;
    else if (cpf::abs_r(a - pi) < threshold) val = 1;
    out[i] = val;
  }
}

// ---- one optimiser step for a loss evaluated outside the engine (cpf_adam_step) ----
// One warp per sample: penalty and its gradient (main.py:563-564), best tracking with strict < on the pre-update
// parameters (optimization.py:61-75), optax Adam (optimization.py:22-23), history rows (optimization.py:52-59).
template <typename R>
__global__ void adam_step_kernel(const cpf::PenaltyT<R> pen, const uint8_t* __restrict__ pen_mask, int P, long long B,
                                 long long step, R lr, R b1, R b2, R eps, R omb1, R omb2, const R* __restrict__ loss,
                                 const R* __restrict__ grad, R* angles, R* m, R* v, const uint8_t* __restrict__ freeze,
                                 R* best_params, R* best_regloss, R* best_reg, R* init_regloss, R* init_reg,
                                 R* hist_params, R* hist_regloss, long long hist_len) {
  const long long b = (long long)blockIdx.x * blockDim.y + threadIdx.y;
  if (b >= B) return;
  const int lane = threadIdx.x;
  const size_t off = (size_t)b * P;
  R reg_part = R(0);
  if (pen.kind != CPF_PEN_NONE && pen_mask)
    for (int i = lane; i < P; i += 32)
      if (pen_mask[i]) {
        R val, slope;
        cpf::penalty_eval(pen, angles[off + i], val, slope);
        reg_part += val;
      }
  for (int d = 16; d >= 1; d >>= 1) reg_part += __shfl_xor_sync(0xffffffffu, reg_part, d);
  const R reg = cpf::mul_rn(pen.kind != CPF_PEN_NONE ? pen.r : R(0), reg_part);
  const R regloss = cpf::add_rn(loss[b], reg);
  const bool improved = step == 0 || regloss < best_regloss[b];
  __syncwarp();
  if (lane == 0) {
    if (step == 0) { init_regloss[b] = regloss; init_reg[b] = reg; }
    if (improved) { best_regloss[b] = regloss; best_reg[b] = reg; }
    if (hist_regloss && step < hist_len) hist_regloss[b * hist_len + step] = regloss;
  }
  const R bc1 = cpf::bias_corr(b1, R(step + 1)), bc2 = cpf::bias_corr(b2, R(step + 1));
  for (int i = lane; i < P; i += 32) {
    R th = angles[off + i];
    if (improved) best_params[off + i] = th;
    if (hist_params && step == 0) hist_params[(size_t)b * hist_len * P + i] = th;
    if (!(freeze && freeze[off + i])) {
      R g = grad[off + i];
      if (pen.kind != CPF_PEN_NONE && pen_mask && pen_mask[i]) {
        R val, slope;
        cpf::penalty_eval(pen, th, val, slope);
        g = cpf::add_rn(g, cpf::mul_rn(pen.r, slope));
      }
      const cpf::AdamOut<R> o = cpf::adam_step(g, th, step == 0 ? R(0) : m[off + i], step == 0 ? R(0) : v[off + i],
                                               b1, omb1, b2, omb2, bc1, bc2, eps, -lr);
      th = o.th;
      m[off + i] = o.mu; v[off + i] = o.nu; angles[off + i] = th;
    } else if (step == 0) {                 // a frozen parameter keeps the zero moments a fresh run starts from
      m[off + i] = R(0); v[off + i] = R(0);
    }
    if (hist_params && step + 1 < hist_len) hist_params[((size_t)b * hist_len + step + 1) * P + i] = th;
  }
}

// ---- jax 0.3.x threefry initial angles (main.py:541-548, cp_utils.py:13-42) ----
__host__ __device__ inline void threefry2x32(uint32_t k0, uint32_t k1, uint32_t& x0, uint32_t& x1) {
  const uint32_t ks[3] = {k0, k1, k0 ^ k1 ^ 0x1BD11BDAu};
  const int rot[2][4] = {{13, 15, 26, 6}, {17, 29, 16, 24}};
  x0 += ks[0]; x1 += ks[1];
  for (int g = 0; g < 5; ++g) {
    for (int r = 0; r < 4; ++r) {
      x0 += x1;
      const int s = rot[g & 1][r];
      x1 = (x1 << s) | (x1 >> (32 - s));
      x1 ^= x0;
    }
    x0 += ks[(g + 1) % 3];
    x1 += ks[(g + 2) % 3] + (uint32_t)(g + 1);
  }
}
// element i of jax's threefry_2x32(key, iota(n)): the count array is split in two halves
__host__ __device__ inline uint32_t threefry_iota(uint32_t k0, uint32_t k1, uint32_t n, uint32_t i) {
  const uint32_t h = (n + 1) / 2;  // odd n is padded with one zero
  uint32_t x0, x1;
  if (i < h) {
    x0 = i; x1 = (h + i < n) ? h + i : 0u;
    threefry2x32(k0, k1, x0, x1);
    return x0;
  }
  x0 = i - h; x1 = i;
  threefry2x32(k0, k1, x0, x1);
  return x1;
}

// jax 0.3.x random.normal in float32 from 32 random bits: u = max(lo, f * (1 - lo) + lo) with lo = nextafter(-1, 0)
// and f the uniform [0, 1) float of the bits, then sqrt(2) * erf_inv(u) with XLA's single-precision erf_inv
// (Giles' polynomial approximation, xla/client/lib/math.cc: ErfInv32).  No reference artefact stores normal draws
// ("parity unpinned"); the oracle restates the same arithmetic.
__host__ __device__ inline float erfinv_xla_f32(float x) {
  float w = -logf((1.0f - x) * (1.0f + x));
  float p;
  if (w < 5.0f) {
    w = w - 2.5f;
    p = 2.81022636e-08f;
    p = 3.43273939e-07f + p * w; p = -3.5233877e-06f + p * w; p = -4.39150654e-06f + p * w;
    p = 0.00021858087f + p * w; p = -0.00125372503f + p * w; p = -0.00417768164f + p * w;
    p = 0.246640727f + p * w; p = 1.50140941f + p * w;
  } else {
    w = sqrtf(w) - 3.0f;
    p = -0.000200214257f;
    p = 0.000100950558f + p * w; p = 0.00134934322f + p * w; p = -0.00367342844f + p * w;
    p = 0.00573950773f + p * w; p = -0.0076224613f + p * w; p = 0.00943887047f + p * w;
    p = 1.00167406f + p * w; p = 2.83297682f + p * w;
  }
  return p * x;
}
__device__ inline float normal_from_bits(uint32_t bits) {
  const float lo = -0.99999994f;                                      // nextafter(-1, 0)
  const float f = __uint_as_float((bits >> 9) | 0x3f800000u) - 1.0f;
  const float u = fmaxf(lo, __fadd_rn(__fmul_rn(f, 2.0f), lo));       // float32(1 - lo) == 2
  return __fmul_rn(1.41421354f, erfinv_xla_f32(u));
}

template <typename R>
__global__ void initial_angles_kernel(const cpf::CpMeta* cp, int n_cp, int P, uint32_t seed_hi,
                                      uint32_t seed_lo, long long total, long long first,
                                      long long count, int cp_dist, R* out) {
  const long long s = (long long)blockIdx.x;
  if (s >= count) return;
  const long long g = first + s;
  __shared__ uint32_t sub[4];
  if (threadIdx.x == 0) {
    // key, *subkeys = split(PRNGKey(seed), total + 1); sample g uses subkeys[g] = row g + 1
    const uint32_t n1 = (uint32_t)(2 * (total + 1));
    const uint32_t r = (uint32_t)(g + 1);
    const uint32_t a0 = threefry_iota(seed_hi, seed_lo, n1, 2 * r);
    const uint32_t a1 = threefry_iota(seed_hi, seed_lo, n1, 2 * r + 1);
    // key, subkey = split(k): subkey is row 1 of a (2,2) split (cp_utils.py:31)
    sub[0] = threefry_iota(a0, a1, 4, 2);
    sub[1] = threefry_iota(a0, a1, 4, 3);
    if (cp_dist == 2) {
      // second split, of the FIRST split's key half (row 0): its row 1 seeds random.normal (cp_utils.py:39)
      const uint32_t k0 = threefry_iota(a0, a1, 4, 0), k1 = threefry_iota(a0, a1, 4, 1);
      sub[2] = threefry_iota(k0, k1, 4, 2);
      sub[3] = threefry_iota(k0, k1, 4, 3);
    }
  }
  __syncthreads();
  const float two_pi = 6.2831855f;  // float32(2*pi)
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    const uint32_t bits = threefry_iota(sub[0], sub[1], (uint32_t)P, (uint32_t)i);
    const float f = __uint_as_float((bits >> 9) | 0x3f800000u) - 1.0f;
    float a = fmaxf(0.0f, __fadd_rn(__fmul_rn(f, two_pi), 0.0f));
    out[s * P + i] = (R)a;
  }
  if (cp_dist == 1) {
    __syncthreads();
    for (int k = threadIdx.x; k < n_cp; k += blockDim.x)
      if (cp[k].pidx >= 0) out[s * P + cp[k].pidx] = R(0);
  } else if (cp_dist == 2) {
    // 'normal' (cp_utils.py:38-40): key, subkey = split(key) once more, CP angles = 1.5 * random.normal(subkey, (P,))
    __syncthreads();
    for (int k = threadIdx.x; k < n_cp; k += blockDim.x)
      if (cp[k].pidx >= 0) {
        const uint32_t bits = threefry_iota(sub[2], sub[3], (uint32_t)P, (uint32_t)cp[k].pidx);
        out[s * P + cp[k].pidx] = (R)__fmul_rn(1.5f, normal_from_bits(bits));
      }
  }
}

}  // namespace

template <typename R>
static int run_adam_step(const cpf::Program* prog, const cpf_penalty_spec* pen, const cpf_adam_spec* adam, int64_t batch,
                         int64_t step, const void* loss, const void* grad, const cpf_adam_buffers* buf, cudaStream_t st) {
  // the penalty mask is per parameter here ([P], not [n_cp])
  cpf::PenaltyT<R> pt;
  int rc = penalty_params<R>(prog, pen, &pt);
  if (rc) return rc;
  uint8_t* mask_dev = nullptr;
  if (pt.kind != CPF_PEN_NONE && prog->n_params > 0) {
    std::string mask((size_t)prog->n_params, '\0');
    for (int i = 0; i < prog->n_params; ++i)
      mask[i] = prog->is_cp_param[i] && (!pen->cp_mask || pen->cp_mask[i]) ? 1 : 0;
    CPF_CUDA(cudaMallocAsync((void**)&mask_dev, mask.size(), st));
    CPF_CUDA(cudaMemcpyAsync(mask_dev, mask.data(), mask.size(), cudaMemcpyHostToDevice, st));
  }
  dim3 block(32, 8);
  const unsigned grid = (unsigned)((batch + 7) / 8);
  adam_step_kernel<R><<<grid, block, 0, st>>>(
      pt, mask_dev, prog->n_params, batch, step, (R)adam->lr, (R)adam->b1, (R)adam->b2, (R)adam->eps,
      (R)(1.0 - adam->b1), (R)(1.0 - adam->b2), (const R*)loss, (const R*)grad, (R*)buf->angles, (R*)buf->m, (R*)buf->v,
      buf->freeze, (R*)buf->best_params, (R*)buf->best_regloss, (R*)buf->best_reg, (R*)buf->init_regloss,
      (R*)buf->init_reg, (R*)buf->hist_params, (R*)buf->hist_regloss, buf->hist_len);
  cudaError_t e = cudaGetLastError();
  if (mask_dev) cudaFreeAsync(mask_dev, st);
  if (e != cudaSuccess) return cuda_fail("adam_step_kernel", e);
  return CPF_OK;
}

template <typename R>
static int workspace_t(const cpf::Program* prog, int32_t loss_kind, int64_t batch, const cpf_target_table* table,
                       int64_t* bytes) {
  CallPlan<R> pl;
  // cpf_workspace_bytes_multi is a query entry point too: a subspace kind carries its k in bits 8-15 there, and a k
  // out of range (a bare kind 6 or 7 is k = 0) is refused as in cpf_workspace_bytes before the table is
  const int32_t base = loss_kind & ~0xff00;
  if (table && (base == CPF_LOSS_SUBSPACE || base == CPF_LOSS_SUBSPACE_RELPHASE)) {
    if (int rc = plan_query<R>(prog, loss_kind, batch, &pl)) return rc;
    loss_kind = base;
  }
  const int rc = table ? plan_call<R>(prog, loss_kind, 0, batch, table, nullptr, &pl)
                       : plan_query<R>(prog, loss_kind, batch, &pl);
  if (!rc) *bytes = pl.workspace();
  return rc;
}

template <typename R>
static int launch_plan_t(const cpf::Program* prog, int32_t loss_kind, int64_t batch, int n_sm, int regs,
                         cpf_launch_info* out, int adam_steps = 2000) {
  CallPlan<R> pl;
  if (int rc = plan_query<R>(prog, loss_kind, batch, &pl)) return rc;
  const int n = prog->n_qubits, N = 1 << n, n_su2 = (int)prog->su2.size(), n_cp = (int)prog->cp.size();
  if (pl.route == ROUTE_ISO) {
    // the isometry kernel's geometry (iso_impl.cuh: iso_geometry); co-residency is not planned (ctas_per_sm = 0)
    const int k = pl.iso.k, rb = cpf::engine_rb<R>(n, true);
    const cpf::DecodedSchedule ds = cpf::decode_schedule(*prog, rb);
    const int n_red = ds.red.empty() ? 1 : (int)(ds.red.size() / 8);
    const cpf::IsoGeometry g = cpf::iso_geometry(n, rb, k, n_su2, n_cp, (int)prog->sched.size(), n_red, sizeof(R));
    out->block_threads = g.block;
    out->samples_per_cta = g.spb;
    out->threads_per_sample = g.spt;
    out->max_block_threads = n <= 6 ? 512 : 1024;          // __launch_bounds__ of iso_kernel
    out->words_per_sample = cpf::iso_sample_words(cpf::coef_stride_words(n_su2, n_cp), k, cpf::iso_sum_stride(n_su2, n_cp));
    out->time_slices = 1;
    out->grid = (batch + g.spb - 1) / g.spb;
    out->smem_bytes = (int64_t)g.smem;
    out->launches_per_run = 1;
    return CPF_OK;
  }
  out->engine = pl.route == ROUTE_HEIS ? 1 : 0;
  if (pl.route != ROUTE_HEIS) return CPF_OK;
  const int tps = N / pl.cpt;
  const int maxt = 2 * N * pl.cpt * (int)(sizeof(R) / 4) <= 64 ? 512 : 256;       // HCfg::MAXT
  const int stride = cpf::heis_coef_stride(n_su2, n_cp, pl.n_stage);
  const size_t fixed = pl.bytes[BLK_TARGET] + cpf::heis_meta_bytes(n_su2, n_cp);
  const cpf::HeisGeometry g = cpf::heis_geometry(batch, fixed, (size_t)stride * sizeof(R), tps, maxt,
                                                 regs > 0 ? regs : 128, n_sm > 0 ? n_sm : 148);
  out->ctas_per_sm = g.ctas; out->block_threads = g.block; out->samples_per_cta = g.spb; out->grid = g.grid;
  out->smem_bytes = (int64_t)g.smem; out->threads_per_sample = tps; out->max_block_threads = maxt;
  out->words_per_sample = stride;
  // time slices an Adam run of `adam_steps` iterations over this batch would be cut into (1 = one launch)
  const cpf::HeisSlicing sl = cpf::heis_slicing(batch, adam_steps > 0 ? adam_steps : 2000, fixed,
                                                (size_t)stride * sizeof(R), tps, maxt, regs > 0 ? regs : 128,
                                                n_sm > 0 ? n_sm : 148, true);
  out->time_slices = sl.k;
  out->launches_per_run = sl.k > 1 ? (batch * sl.k + sl.slots - 1) / sl.slots : 1;
  return CPF_OK;
}

template <typename R>
static int eval_cost_t(const cpf::Program* p, int32_t loss_kind, double* flops, double* bytes) {
  CallPlan<R> pl;
  if (int rc = plan_query<R>(p, loss_kind, 1, &pl)) return rc;
  const double N = (double)(1 << p->n_qubits);
  // isometry kinds: C = k; subspace kinds: C = the caller's k on either route
  const double C = pl.kind == CPF_LOSS_STATE ? 1.0 : pl.iso.sub_k ? (double)pl.iso.sub_k : pl.iso.k ? (double)pl.iso.k : N;
  const double rs = (double)sizeof(R);
  if (flops) *flops = C * N * (16.0 * p->n_rot + 4.0 * p->n_phase + 8.0);
  if (bytes) *bytes = 6.0 * p->n_params * rs + 2.0 * rs;
  return CPF_OK;
}

template <typename R>
static int executed_cost_t(const cpf::Program* p, int32_t loss_kind, double* flops) {
  CallPlan<R> pl;
  if (int rc = plan_query<R>(p, loss_kind, 1, &pl)) return rc;
  const double N = (double)(1 << p->n_qubits), n = p->n_qubits, K = (double)p->cp.size(), G = (double)p->su2.size();
  if (pl.route == ROUTE_HEIS) {
    // heis_kernel (heis_impl.cuh), FMA = 2 flop, per sample and step:
    //   forward   block: 3 diagonal phases on N/4 rows (6 flop per complex amplitude) + 2 Ry in lifting form (3 shears on
    //             re and im): N^2 (4.5 + 12); surface gate: phase on N/2 rows + Ry: 9 N^2; pending phases at the end: 3 N^2
    //   backward  fused gate: Rx exchange + merged Rz on the N^2 real coefficients: 4.5 N^2; ZZ pair rotations
    //             (lifting): 3 N^2 per block; outgoing Rz of the last gate per qubit: 3 N^2
    //   pivot     Walsh-Hadamard transform (re, im) + seed of h: N^2 (2 n + 6)
    //   update    per fused gate: chain rule, 3 x Adam, 3 x sin/cos, SU(2) products, ZYZ data, staging: ~232;
    //             per entangler: Adam, sin/cos, penalty, merged diagonal: ~80
    *flops = N * N * (28.5 * K + 19.5 * n + 2.0 * n + 6.0) + 232.0 * G + 80.0 * K;
  } else {
    // state-adjoint kernels: the credited count plus the uncompute of phi (6 flop per amplitude and rotation on
    // fused gates, 1.5 per phase gate), with fused gates instead of primitive rotations: C N (22 G + 5.5 K + 8);
    // an isometry runs as an HS call on n <= 5 and on the isometry kernel with C = k on n >= 6, the relative-phase
    // isometry on the isometry kernel on every n.  The subspace losses: C = N on the HS route, and on the isometry kernel
    // C = k', the padded group count, not the caller's k: the zero groups run full sweeps too, and this entry point
    // counts executed work (cpf_eval_cost credits C = k)
    const double C = pl.kind == CPF_LOSS_STATE ? 1.0 : pl.route == ROUTE_ISO ? (double)pl.iso.k : N;
    *flops = C * N * (22.0 * G + 5.5 * K + 8.0) + 232.0 * G + 80.0 * K;
  }
  return CPF_OK;
}

extern "C" {

int cpf_version(void) { return CPF_VERSION; }
const char* cpf_last_error(void) { return g_err.c_str(); }

int cpf_program_create(int32_t n_qubits, int32_t n_ops, const cpf_op* ops, int32_t n_params,
                       cpf_program** out) {
  if (!out) return fail(CPF_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (n_ops < 0 || n_params < 0 || (n_ops > 0 && !ops)) return fail(CPF_ERR_INVALID, "bad ops / sizes");
  cpf::Program* p = new (std::nothrow) cpf::Program();
  if (!p) return fail(CPF_ERR_NOMEM, "out of memory");
  try {
    p->n_qubits = n_qubits; p->n_params = n_params;
    p->ops.assign(ops, ops + n_ops);
    std::string err = cpf::compile_program(*p);
    if (!err.empty()) {
      delete p;
      return fail(n_qubits > CPF_MAX_QUBITS ? CPF_ERR_UNSUPPORTED : CPF_ERR_INVALID, err);
    }
  } catch (const std::exception& e) {
    delete p;
    return fail(CPF_ERR_NOMEM, e.what());
  }
  *out = reinterpret_cast<cpf_program*>(p);
  return CPF_OK;
}

int cpf_program_destroy(cpf_program* prog) {
  if (!prog) return CPF_OK;
  cpf::Program* p = reinterpret_cast<cpf::Program*>(prog);
  int cur = 0;
  cudaGetDevice(&cur);
  for (auto& kv : p->dev) {
    cudaSetDevice(kv.first);
    cudaFree(kv.second.sched); cudaFree(kv.second.su2); cudaFree(kv.second.cp);
    for (int r = 0; r < 8; ++r)
      if (kv.second.has_dec[r]) { cudaFree(kv.second.dec[r].ops); cudaFree(kv.second.dec[r].red); }
  }
  cudaSetDevice(cur);
  delete p;
  return CPF_OK;
}

int cpf_program_get_info(const cpf_program* prog, cpf_program_info* info) {
  if (!prog || !info) return fail(CPF_ERR_INVALID, "NULL argument");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  info->n_qubits = p->n_qubits; info->n_params = p->n_params; info->n_ops = (int)p->ops.size();
  info->n_rotations = p->n_rot; info->n_phase = p->n_phase; info->n_fused = (int)p->su2.size();
  info->n_sched = (int)p->sched.size(); info->reserved = 0;
  return CPF_OK;
}

#define CPF_DISPATCH(dtype, CALL)                                   \
  try {                                                             \
    if ((dtype) == CPF_F32) { using R = float; return CALL; }       \
    if ((dtype) == CPF_F64) { using R = double; return CALL; }      \
    return fail(CPF_ERR_INVALID, "unknown dtype");                  \
  } catch (const std::exception& e) {                               \
    return fail(CPF_ERR_NOMEM, e.what());                           \
  }

int cpf_unitary(const cpf_program* prog, int32_t dtype, int64_t batch, const void* angles, void* u_out,
                void* stream) {
  if (!prog || batch < 0) return fail(CPF_ERR_INVALID, "NULL program / bad batch");
  if (batch == 0) return CPF_OK;
  if (!u_out) return fail(CPF_ERR_INVALID, "u_out is NULL");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  if (!angles && p->n_params > 0) return fail(CPF_ERR_INVALID, "angles is NULL");
  CPF_DISPATCH(dtype, (run_unitary<R>(p, batch, angles, u_out, (cudaStream_t)stream)));
}

int cpf_loss_grad(const cpf_program* prog, const cpf_loss_spec* loss, const cpf_penalty_spec* penalty,
                  int32_t dtype, int64_t batch, const void* angles, void* loss_out, void* reg_out,
                  void* grad_out, void* stream) {
  if (!prog || batch < 0) return fail(CPF_ERR_INVALID, "NULL program / bad batch");
  if (!loss || !loss->target) return fail(CPF_ERR_INVALID, "loss spec / target is NULL");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_loss_grad<R>(p, loss->kind, loss->ancilla_mask, loss->target, penalty, batch, angles,
                                        loss_out, reg_out, grad_out, (cudaStream_t)stream)));
}

int cpf_adjoint_from_cotangent(const cpf_program* prog, int32_t dtype, int64_t batch, const void* angles,
                               const void* cotangent, void* grad_out, void* stream) {
  if (!prog || batch < 0) return fail(CPF_ERR_INVALID, "NULL program / bad batch");
  if (batch == 0) return CPF_OK;
  if (!angles || !cotangent || !grad_out) return fail(CPF_ERR_INVALID, "NULL argument");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_cotangent<R>(p, batch, angles, cotangent, grad_out, (cudaStream_t)stream)));
}

int cpf_adam_run(const cpf_program* prog, const cpf_loss_spec* loss, const cpf_penalty_spec* penalty,
                 const cpf_adam_spec* adam, int32_t dtype, int64_t batch, int64_t step0, int64_t num_steps,
                 const cpf_adam_buffers* buf, void* stream) {
  if (!prog || !adam || !buf || batch < 0 || step0 < 0 || num_steps < 0)
    return fail(CPF_ERR_INVALID, "NULL argument / negative size");
  if (!loss || !loss->target) return fail(CPF_ERR_INVALID, "loss spec / target is NULL");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_adam<R>(p, loss->kind, loss->ancilla_mask, loss->target, penalty, adam, batch, step0,
                                   num_steps, buf, (cudaStream_t)stream)));
}

int cpf_workspace_bytes(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch, int64_t* bytes) {
  if (!prog || !bytes || batch < 0) return fail(CPF_ERR_INVALID, "NULL argument / negative batch");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (workspace_t<R>(p, loss_kind, batch, nullptr, bytes)));
}

int cpf_loss_grad_multi(const cpf_program* prog, const cpf_target_table* table, const cpf_penalty_spec* penalty,
                        int32_t dtype, int64_t batch, const void* angles, void* loss_out, void* reg_out,
                        void* grad_out, void* stream) {
  if (!prog || batch < 0) return fail(CPF_ERR_INVALID, "NULL program / bad batch");
  if (int rc = check_table_pointers(table, batch)) return rc;
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_loss_grad<R>(p, table->kind, 0, table->targets, penalty, batch, angles, loss_out, reg_out,
                                        grad_out, (cudaStream_t)stream, table)));
}

int cpf_adam_run_multi(const cpf_program* prog, const cpf_target_table* table, const cpf_penalty_spec* penalty,
                       const cpf_adam_spec* adam, int32_t dtype, int64_t batch, int64_t step0, int64_t num_steps,
                       const cpf_adam_buffers* buf, void* stream) {
  if (!prog || !adam || !buf || batch < 0 || step0 < 0 || num_steps < 0)
    return fail(CPF_ERR_INVALID, "NULL argument / negative size");
  if (int rc = check_table_pointers(table, batch)) return rc;
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_adam<R>(p, table->kind, 0, table->targets, penalty, adam, batch, step0, num_steps, buf,
                                   (cudaStream_t)stream, table)));
}

int cpf_workspace_bytes_multi(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch,
                              int32_t n_targets, int64_t* bytes) {
  if (!prog || !bytes || batch < 0) return fail(CPF_ERR_INVALID, "NULL argument / negative batch");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  const cpf_target_table tt{loss_kind, n_targets, nullptr, nullptr};
  CPF_DISPATCH(dtype, (workspace_t<R>(p, loss_kind, batch, &tt, bytes)));
}

int cpf_adam_step(const cpf_program* prog, const cpf_penalty_spec* penalty, const cpf_adam_spec* adam, int32_t dtype,
                  int64_t batch, int64_t step, const void* loss, const void* grad, const cpf_adam_buffers* buf,
                  void* stream) {
  if (!prog || !adam || !buf || batch < 0 || step < 0) return fail(CPF_ERR_INVALID, "NULL argument / negative size");
  if (batch == 0) return CPF_OK;
  if (!loss || !grad) return fail(CPF_ERR_INVALID, "loss / grad is NULL");
  if (int rc = check_adam_buffers(buf)) return rc;
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_adam_step<R>(p, penalty, adam, batch, step, loss, grad, buf, (cudaStream_t)stream)));
}

int cpf_count_cz(const cpf_program* prog, int32_t dtype, int64_t batch, const void* angles, double threshold,
                 int32_t* cz_out, void* projected, uint8_t* frozen, void* stream) {
  if (!prog || batch < 0) return fail(CPF_ERR_INVALID, "NULL program / bad batch");
  if (batch == 0) return CPF_OK;
  if (!angles) return fail(CPF_ERR_INVALID, "angles is NULL");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  cpf::DeviceProgram d;
  int rc = device_program(p, &d);
  if (rc) return rc;
  dim3 block(32, 8);
  const unsigned grid = (unsigned)((batch + 7) / 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == CPF_F32)
    count_cz_kernel<float><<<grid, block, 0, st>>>(d.cp, (int)p->cp.size(), p->n_params, batch,
                                                   (const float*)angles, (float)threshold, cz_out,
                                                   (float*)projected, frozen);
  else if (dtype == CPF_F64)
    count_cz_kernel<double><<<grid, block, 0, st>>>(d.cp, (int)p->cp.size(), p->n_params, batch,
                                                    (const double*)angles, threshold, cz_out,
                                                    (double*)projected, frozen);
  else
    return fail(CPF_ERR_INVALID, "unknown dtype");
  CPF_CUDA(cudaGetLastError());
  return CPF_OK;
}

int cpf_cz_value(int32_t dtype, int64_t n, const void* angles, double threshold, int32_t* out, void* stream) {
  if (n < 0 || (n > 0 && (!angles || !out))) return fail(CPF_ERR_INVALID, "NULL argument / bad size");
  if (n == 0) return CPF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
  if (dtype == CPF_F32)
    cz_value_kernel<float><<<grid, 256, 0, st>>>((const float*)angles, n, (float)threshold, out);
  else if (dtype == CPF_F64)
    cz_value_kernel<double><<<grid, 256, 0, st>>>((const double*)angles, n, threshold, out);
  else
    return fail(CPF_ERR_INVALID, "unknown dtype");
  CPF_CUDA(cudaGetLastError());
  return CPF_OK;
}

int cpf_initial_angles(const cpf_program* prog, int32_t dtype, uint64_t seed, int64_t total_samples,
                       int64_t first, int64_t count, int32_t cp_dist, void* out, void* stream) {
  if (!prog || !out || total_samples < 0 || first < 0 || count < 0 || first + count > total_samples)
    return fail(CPF_ERR_INVALID, "bad sample range");
  if (cp_dist < 0 || cp_dist > 2) return fail(CPF_ERR_UNSUPPORTED, "cp_dist must be 0 ('uniform'), 1 ('0') or 2 ('normal')");
  if (2 * (total_samples + 1) > 0xffffffffLL) return fail(CPF_ERR_UNSUPPORTED, "too many samples for a 32-bit counter");
  if (count == 0) return CPF_OK;
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  cpf::DeviceProgram d;
  int rc = device_program(p, &d);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t hi = (uint32_t)(seed >> 32), lo = (uint32_t)(seed & 0xffffffffu);
  if (dtype == CPF_F32)
    initial_angles_kernel<float><<<(unsigned)count, 128, 0, st>>>(d.cp, (int)p->cp.size(), p->n_params, hi, lo,
                                                                total_samples, first, count, cp_dist, (float*)out);
  else if (dtype == CPF_F64)
    initial_angles_kernel<double><<<(unsigned)count, 128, 0, st>>>(d.cp, (int)p->cp.size(), p->n_params, hi, lo,
                                                                 total_samples, first, count, cp_dist, (double*)out);
  else
    return fail(CPF_ERR_INVALID, "unknown dtype");
  CPF_CUDA(cudaGetLastError());
  return CPF_OK;
}

int cpf_eval_cost(const cpf_program* prog, int32_t loss_kind, int32_t dtype, double* flops, double* bytes) {
  if (!prog) return fail(CPF_ERR_INVALID, "NULL program");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (eval_cost_t<R>(p, loss_kind, flops, bytes)));
}

int cpf_executed_cost(const cpf_program* prog, int32_t loss_kind, int32_t dtype, double* flops) {
  if (!prog || !flops) return fail(CPF_ERR_INVALID, "NULL argument");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (executed_cost_t<R>(p, loss_kind, flops)));
}

int cpf_launch_plan(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch, int32_t n_sm,
                    int32_t regs_per_thread, cpf_launch_info* out) {
  if (!prog || !out) return fail(CPF_ERR_INVALID, "NULL argument");
  if (batch < 0) return fail(CPF_ERR_INVALID, "negative batch");
  std::memset(out, 0, sizeof(*out));
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (launch_plan_t<R>(p, loss_kind, batch, n_sm, regs_per_thread, out)));
}

}  // extern "C"
