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
template <typename R>
int launch_any(const cpf::KParams<R>& p, const cpf::Program* prog, bool single, cudaStream_t st,
               std::string& err) {
  const char* e = getenv("CPF_NO_LAYERED");
  const bool no_layered = e && e[0] == '1';
  int rc = CPF_OK;
  if (prog->layered && !no_layered && cpf::launch_layered<R>(p, *prog, single, st, err, rc)) return rc;
  return cpf::launch_engine<R>(p, prog->n_qubits, single, st, err);
}

template <typename R>
int fill_penalty(const cpf::Program* prog, const cpf_penalty_spec* pen, cpf::KParams<R>& p, Scratch& sc) {
  cudaStream_t st = sc.st;
  if (!pen || pen->kind == CPF_PEN_NONE) return CPF_OK;
  if (pen->kind != CPF_PEN_PIECEWISE && pen->kind != CPF_PEN_L1)
    return fail(CPF_ERR_INVALID, "unknown penalty kind");
  if (pen->kind == CPF_PEN_PIECEWISE && (pen->n_segments < 1 || pen->n_segments > CPF_MAX_SEGMENTS))
    return fail(CPF_ERR_INVALID, "penalty n_segments out of range");
  if (pen->kind == CPF_PEN_PIECEWISE && !(pen->period > 0))
    return fail(CPF_ERR_INVALID, "penalty period must be positive");
  p.pen.kind = pen->kind; p.pen.nseg = pen->n_segments;
  p.pen.r = (R)pen->r; p.pen.period = (R)pen->period;
  for (int s = 0; s < CPF_MAX_SEGMENTS; ++s) {
    const bool on = pen->kind == CPF_PEN_PIECEWISE && s < pen->n_segments;
    p.pen.lo[s] = on ? (R)pen->lo[s] : (R)INFINITY; p.pen.hi[s] = on ? (R)pen->hi[s] : (R)INFINITY;
    p.pen.slope[s] = on ? (R)pen->slope[s] : R(0); p.pen.icpt[s] = on ? (R)pen->intercept[s] : R(0);
  }
  // ascending, disjoint segments (in the kernel's precision) can be searched instead of scanned
  p.pen.sorted = pen->kind == CPF_PEN_PIECEWISE;
  for (int s = 0; s < pen->n_segments && s < CPF_MAX_SEGMENTS && p.pen.sorted; ++s) {
    if (!(p.pen.lo[s] <= p.pen.hi[s])) p.pen.sorted = 0;
    if (s + 1 < pen->n_segments && !(p.pen.hi[s] <= p.pen.lo[s + 1])) p.pen.sorted = 0;
  }
  if (pen->cp_mask) {
    // only parameters of CP gates may be penalised
    for (int i = 0; i < prog->n_params; ++i)
      if (pen->cp_mask[i] && !prog->is_cp_param[i])
        return fail(CPF_ERR_UNSUPPORTED, "cp_mask selects a parameter that does not feed a CP gate");
    std::string flags(prog->cp.size(), '\0');
    for (size_t k = 0; k < prog->cp.size(); ++k)
      flags[k] = prog->cp[k].pidx >= 0 && pen->cp_mask[prog->cp[k].pidx] ? 1 : 0;
    if (!flags.empty()) {
      uint8_t* dev = nullptr;
      int rc = sc.get((void**)&dev, flags.size());
      if (rc) return rc;
      // pageable source: the runtime stages the bytes before returning, so `flags` may die
      CPF_CUDA(cudaMemcpyAsync(dev, flags.data(), flags.size(), cudaMemcpyHostToDevice, st));
      p.cp_pen = dev;
    }
  }
  return CPF_OK;
}

template <typename R>
int stage_target(const cpf::Program* prog, const cpf_loss_spec* loss, cpf::KParams<R>& p, bool single, Scratch& sc) {
  cudaStream_t st = sc.st;
  const int cpt = single ? 1 : cpf::cpt_for<R>(prog->n_qubits);
  const int words = cpf::target_words<R>(prog->n_qubits, cpt, single);
  const size_t bytes = ((size_t)words * sizeof(R) + 15) & ~(size_t)15;
  R* packed = nullptr;
  int rc = sc.get((void**)&packed, bytes);
  if (rc) return rc;
  if (bytes != (size_t)words * sizeof(R)) CPF_CUDA(cudaMemsetAsync(packed, 0, bytes, st));
  rc = cpf::launch_pack_target<R>((const R*)loss->target, packed, prog->n_qubits, cpt, single, st);
  if (rc) return fail(rc, "pack_target launch failed");
  p.target_packed = packed;
  p.target_bytes = (int)bytes;
  p.loss_kind = loss->kind;
  return CPF_OK;
}

struct cpf_loss_spec_kind_only { int32_t kind; };

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

// ---- Heisenberg-picture kernels (heis_impl.cuh): HS loss on layered templates ----
// CPF_ENGINE=adjoint forces the state-adjoint kernels (tests cover both engines).
template <typename R>
bool use_heis(const cpf::Program* prog, const cpf_loss_spec* loss) {
  if (loss->kind != CPF_LOSS_HS || !prog->layered) return false;
  // the kernel's shared-memory metadata holds parameter and slot indices in 16 bits (heis_impl.cuh: HSu2, HCp)
  if (prog->n_params > 32767 || prog->su2.size() > 32767) return false;
  const char* e = getenv("CPF_ENGINE");
  if (e && std::strcmp(e, "adjoint") == 0) return false;
  const char* nl = getenv("CPF_NO_LAYERED");
  if (nl && nl[0] == '1') return false;
  cpf::KParams<R> dummy;
  std::string err;
  int rc = 0;
  return cpf::launch_heis<R>(dummy, *prog, nullptr, err, rc, true);
}

// bytes of the two heis scratch blocks: staged target; per-gate scratch followed by the packed optimiser state
template <typename R>
void heis_scratch_sizes(const cpf::Program* prog, int64_t batch, size_t* target_bytes, size_t* aux_pad, size_t* pk_bytes) {
  const int cpt = cpf::heis_cpt<R>(prog->n_qubits);
  const int words = cpf::heis_target_words<R>(prog->n_qubits, cpt);
  *target_bytes = ((size_t)words * sizeof(R) + 15) & ~(size_t)15;
  const size_t aux_bytes = (size_t)batch * (prog->su2.empty() ? 1 : prog->su2.size()) * 4 * sizeof(R);
  *aux_pad = (aux_bytes + 255) & ~(size_t)255;      // the packed state starts on a 256-byte boundary (blocks of 16 positions)
  // lane-interleaved packed optimiser state (heis_impl.cuh: heis_pk_stride words per sample)
  const int tps = (1 << prog->n_qubits) / cpt;
  *pk_bytes = (size_t)batch * (size_t)cpf::heis_pk_stride(prog->n_qubits, tps, (int)prog->su2.size(), (int)prog->cp.size()) *
              sizeof(R);
}

template <typename R>
int stage_heis_state(const cpf::Program* prog, cpf::KParams<R>& p, Scratch& sc);

template <typename R>
int stage_heis(const cpf::Program* prog, const cpf_loss_spec* loss, cpf::KParams<R>& p, Scratch& sc) {
  cudaStream_t st = sc.st;
  if (!sc.base) keep_pool_memory();
  const int cpt = cpf::heis_cpt<R>(prog->n_qubits);
  const int words = cpf::heis_target_words<R>(prog->n_qubits, cpt);
  size_t bytes, aux_pad, pk_bytes;
  heis_scratch_sizes<R>(prog, p.B, &bytes, &aux_pad, &pk_bytes);
  R* packed = nullptr;
  int rc = sc.get((void**)&packed, bytes);
  if (rc) return rc;
  if (bytes != (size_t)words * sizeof(R)) CPF_CUDA(cudaMemsetAsync(packed, 0, bytes, st));
  rc = cpf::launch_pack_target_heis<R>((const R*)loss->target, packed, prog->n_qubits, cpt, st);
  if (rc) return fail(rc, "pack_target_heis launch failed");
  p.target_packed = packed;
  p.target_bytes = (int)bytes;
  p.loss_kind = loss->kind;
  return stage_heis_state(prog, p, sc);
}

// the target-independent part of the heis set-up: per-gate scratch and packed optimiser state, gate-pattern flags
template <typename R>
int stage_heis_state(const cpf::Program* prog, cpf::KParams<R>& p, Scratch& sc) {
  const int cpt = cpf::heis_cpt<R>(prog->n_qubits);
  size_t bytes, aux_pad, pk_bytes;
  heis_scratch_sizes<R>(prog, p.B, &bytes, &aux_pad, &pk_bytes);
  R* aux = nullptr;
  // one block: per-gate scratch, then the packed optimiser state (32-byte aligned)
  int rc = sc.get((void**)&aux, aux_pad + pk_bytes);
  if (rc) return rc;
  p.pk = reinterpret_cast<char*>(aux) + aux_pad;
  p.aux = aux;
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
  return CPF_OK;
}

// HS and relative-phase losses run on the full-unitary kernels, which stop at 5 qubits: refused before any CUDA call.
int check_full_unitary(const cpf::Program* prog, int32_t kind) {
  if ((kind == CPF_LOSS_HS || kind == CPF_LOSS_RELPHASE) && prog->n_qubits > 5)
    return fail(CPF_ERR_UNSUPPORTED, cpf::FULL_UNITARY_LIMIT);
  return CPF_OK;
}

// ---- isometry loss (CPF_LOSS_ISOMETRY) ----
// Largest number of input columns k of the 6-8 qubit kernel: a sample is k lane groups of 2^(n-RB) threads in one CTA.
constexpr int ISO_MAX_K = 32;

// Everything about an isometry request that can be refused is refused here, before any CUDA call.
int check_iso(const cpf::Program* prog, int32_t mask) {
  const int n = prog->n_qubits;
  if (mask < 0 || (mask >> n) != 0)
    return fail(CPF_ERR_INVALID, "ancilla_mask " + std::to_string(mask) + " names a qubit >= n = " + std::to_string(n));
  if (n > 5 && mask == 0)
    return fail(CPF_ERR_UNSUPPORTED, cpf::FULL_UNITARY_LIMIT);
  const int k = 1 << (n - __builtin_popcount((unsigned)mask));
  if (n > 5 && k > ISO_MAX_K)
    return fail(CPF_ERR_UNSUPPORTED, "isometry losses on 6-8 qubits take at most k = " + std::to_string(ISO_MAX_K) +
                                     " input columns (k = 2^(n - popcount(ancilla_mask)) = " + std::to_string(k) + ")");
  return CPF_OK;
}

// k input columns; the ancilla qubits as amplitude-index bits (qubit q is bit n - 1 - q, big-endian)
struct IsoSpec { int k, amask; };
IsoSpec iso_spec(const cpf::Program* prog, int32_t mask) {
  const int n = prog->n_qubits;
  IsoSpec s{1 << (n - __builtin_popcount((unsigned)mask)), 0};
  for (int q = 0; q < n; ++q)
    if ((mask >> q) & 1) s.amask |= 1 << (n - 1 - q);
  return s;
}

// The query entry points take a loss kind only: an isometry kind carries its ancilla mask in bits 8-15
// (CPF_ISOMETRY_KIND).  Splits and checks such an argument.
int split_kind(const cpf::Program* prog, int32_t arg, int32_t* kind, int32_t* mask) {
  *kind = arg & 0xff;
  *mask = (arg >> 8) & 0xff;
  if (*kind < CPF_LOSS_HS || *kind > CPF_LOSS_ISOMETRY || (arg >> 16) != 0 || (*kind != CPF_LOSS_ISOMETRY && *mask))
    return fail(CPF_ERR_INVALID, "unknown loss kind");
  return *kind == CPF_LOSS_ISOMETRY ? check_iso(prog, *mask) : CPF_OK;
}

// n <= 5: the isometry loss is the HS loss on V = 2^a [W at the columns s_c, 0 elsewhere] (iso_impl.cuh:
// pack_iso_hs_kernel), built in scratch; `hs` becomes the spec of that HS call.
template <typename R>
int stage_iso_as_hs(const cpf::Program* prog, const cpf_loss_spec* loss, Scratch& sc, cpf_loss_spec* hs) {
  const int n = prog->n_qubits;
  const IsoSpec is = iso_spec(prog, loss->ancilla_mask);
  R* v = nullptr;
  int rc = sc.get((void**)&v, ((size_t)2 << (2 * n)) * sizeof(R));
  if (rc) return rc;
  rc = cpf::launch_pack_iso<R>((const R*)loss->target, v, n, is.k, is.amask, true, sc.st);
  if (rc) return fail(rc, "pack_iso launch failed");
  *hs = cpf_loss_spec{};
  hs->kind = CPF_LOSS_HS;
  hs->target = v;
  return CPF_OK;
}

// n >= 6: W packed column by column for the isometry kernel
template <typename R>
int stage_iso(const cpf::Program* prog, const cpf_loss_spec* loss, cpf::KParams<R>& p, Scratch& sc) {
  const int n = prog->n_qubits;
  const IsoSpec is = iso_spec(prog, loss->ancilla_mask);
  R* packed = nullptr;
  int rc = sc.get((void**)&packed, ((size_t)is.k << (n + 1)) * sizeof(R));
  if (rc) return rc;
  rc = cpf::launch_pack_iso<R>((const R*)loss->target, packed, n, is.k, is.amask, false, sc.st);
  if (rc) return fail(rc, "pack_iso launch failed");
  p.target_packed = packed;
  p.target_bytes = 0;
  p.loss_kind = CPF_LOSS_ISOMETRY;
  p.iso_k = is.k;
  p.iso_amask = is.amask;
  return CPF_OK;
}

int check_loss(const cpf::Program* prog, const cpf_loss_spec* loss) {
  if (!loss || !loss->target) return fail(CPF_ERR_INVALID, "loss spec / target is NULL");
  if (loss->kind < CPF_LOSS_HS || loss->kind > CPF_LOSS_ISOMETRY)
    return fail(CPF_ERR_INVALID, "unknown loss kind");
  return loss->kind == CPF_LOSS_ISOMETRY ? check_iso(prog, loss->ancilla_mask) : check_full_unitary(prog, loss->kind);
}

// Everything a multi-target call needs to know is checked here, before any CUDA call.
int check_table(const cpf::Program* prog, const cpf_target_table* tt, int64_t batch) {
  if (!tt) return fail(CPF_ERR_INVALID, "target table is NULL");
  if (tt->kind == CPF_LOSS_ISOMETRY)
    return fail(CPF_ERR_UNSUPPORTED, "multi-target tables do not take the isometry loss (one target per call)");
  if (tt->kind < CPF_LOSS_HS || tt->kind > CPF_LOSS_RELPHASE) return fail(CPF_ERR_INVALID, "unknown loss kind");
  if (tt->n_targets < 1) return fail(CPF_ERR_INVALID, "target table: n_targets must be >= 1");
  if (!tt->targets) return fail(CPF_ERR_INVALID, "target table: targets is NULL");
  if (batch > 0 && !tt->target_index) return fail(CPF_ERR_INVALID, "target table: target_index is NULL");
  if (int rc = check_full_unitary(prog, tt->kind)) return rc;
  for (int64_t b = 0; b < batch; ++b) {
    const int32_t t = tt->target_index[b];
    if (t < 0 || t >= tt->n_targets)
      return fail(CPF_ERR_INVALID, "target_index[" + std::to_string(b) + "] = " + std::to_string(t) +
                                       " is outside [0, n_targets = " + std::to_string(tt->n_targets) + ")");
  }
  return CPF_OK;
}

// bytes of the multi-target table of the kernel a call runs on (targets back to back in the kernel's packed layout)
template <typename R>
size_t multi_table_bytes(const cpf::Program* prog, int32_t kind, bool heis, int32_t n_targets) {
  const bool single = kind == CPF_LOSS_STATE;
  const int n = prog->n_qubits;
  const int words = heis ? cpf::heis_target_words<R>(n, cpf::heis_cpt<R>(n))
                         : cpf::target_words<R>(n, single ? 1 : cpf::cpt_for<R>(n), single);
  return (size_t)n_targets * (size_t)words * sizeof(R);
}

// Multi-target staging: the index array (host, checked by check_table) goes to the device, all targets are packed in
// one launch; the kernels read both from global memory (p.target_bytes = 0: no shared-memory copy).
template <typename R>
int stage_multi(const cpf::Program* prog, const cpf_target_table* tt, cpf::KParams<R>& p, bool heis, Scratch& sc) {
  cudaStream_t st = sc.st;
  if (heis && !sc.base) keep_pool_memory();
  const bool single = tt->kind == CPF_LOSS_STATE;
  const int n = prog->n_qubits;
  int32_t* idx = nullptr;
  R* table = nullptr;
  int rc = sc.get((void**)&idx, (size_t)p.B * sizeof(int32_t));
  if (!rc) rc = sc.get((void**)&table, multi_table_bytes<R>(prog, tt->kind, heis, tt->n_targets));
  if (rc) return rc;
  // pageable source: the runtime stages the bytes before returning
  CPF_CUDA(cudaMemcpyAsync(idx, tt->target_index, (size_t)p.B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  rc = heis ? cpf::launch_pack_targets_heis<R>((const R*)tt->targets, table, n, cpf::heis_cpt<R>(n), tt->n_targets, st)
            : cpf::launch_pack_targets<R>((const R*)tt->targets, table, n, single ? 1 : cpf::cpt_for<R>(n), single,
                                          tt->n_targets, st);
  if (rc) return fail(rc, "pack_targets launch failed");
  p.target_packed = table;
  p.target_bytes = 0;
  p.target_index = idx;
  p.loss_kind = tt->kind;
  return heis ? stage_heis_state(prog, p, sc) : CPF_OK;
}

// Launch of a staged call: the single-target kernels, or (table != NULL) their multi-target variants.
template <typename R>
int launch_staged(const cpf::KParams<R>& p, const cpf::Program* prog, const cpf_target_table* table, bool heis,
                  bool single, cudaStream_t st, std::string& err) {
  int rc = CPF_OK;
  if (table) {
    if (heis) cpf::launch_heis_multi<R>(p, *prog, st, err, rc);
    else rc = cpf::launch_engine_multi<R>(p, prog->n_qubits, single, st, err);
  } else {
    if (heis) cpf::launch_heis<R>(p, *prog, st, err, rc, false);
    else rc = launch_any<R>(p, prog, single, st, err);
  }
  return rc;
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
  rc = launch_any<R>(p, prog, colmode, st, err);
  return rc ? fail(rc, err) : CPF_OK;
}

// table != NULL: multi-target call (loss->kind = table->kind, loss->target unused)
template <typename R>
int run_loss_grad(const cpf::Program* prog, const cpf_loss_spec* loss, const cpf_penalty_spec* pen,
                  int64_t batch, const void* angles, void* loss_out, void* reg_out, void* grad_out,
                  cudaStream_t st, const cpf_target_table* table = nullptr) {
  cpf::KParams<R> p;
  Scratch sc;
  sc.st = st;
  cpf_loss_spec hs;
  const bool iso = loss->kind == CPF_LOSS_ISOMETRY && prog->n_qubits > 5;    // else n <= 5: an HS call on V
  if (loss->kind == CPF_LOSS_ISOMETRY && !iso) {
    int rc = stage_iso_as_hs<R>(prog, loss, sc, &hs);
    if (rc) return rc;
    loss = &hs;
  }
  const bool single = loss->kind == CPF_LOSS_STATE || iso;
  int rc = fill_common(prog, p, batch, single);
  if (rc) return rc;
  p.mode = cpf::M_LOSSGRAD;
  p.angles = (R*)angles; p.loss_out = (R*)loss_out; p.reg_out = (R*)reg_out; p.grad_out = (R*)grad_out;
  const bool heis = use_heis<R>(prog, loss) && (unsigned long long)batch * (unsigned long long)prog->n_params < (1ull << 32);
  rc = fill_penalty(prog, pen, p, sc);
  if (!rc && table) rc = stage_multi(prog, table, p, heis, sc);
  else if (!rc && iso) rc = stage_iso(prog, loss, p, sc);
  else if (!rc) rc = heis ? stage_heis(prog, loss, p, sc) : stage_target(prog, loss, p, single, sc);
  if (!rc && grad_out) {
    cudaError_t e = cudaMemsetAsync(grad_out, 0, (size_t)batch * prog->n_params * sizeof(R), st);
    if (e != cudaSuccess) rc = cuda_fail("cudaMemsetAsync(grad)", e);
  }
  std::string err;
  if (!rc) {
    rc = iso ? cpf::launch_iso<R>(p, prog->n_qubits, st, err) : launch_staged<R>(p, prog, table, heis, single, st, err);
    if (rc) fail(rc, err);
  }
  return rc;
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
  rc = launch_any<R>(p, prog, false, st, err);
  return rc ? fail(rc, err) : CPF_OK;
}

template <typename R>
int run_adam(const cpf::Program* prog, const cpf_loss_spec* loss, const cpf_penalty_spec* pen,
             const cpf_adam_spec* adam, int64_t batch, int64_t step0, int64_t num_steps,
             const cpf_adam_buffers* buf, cudaStream_t st, const cpf_target_table* table = nullptr) {
  cpf::KParams<R> p;
  const bool iso = loss->kind == CPF_LOSS_ISOMETRY && prog->n_qubits > 5;    // else n <= 5: an HS call on V
  const bool single = loss->kind == CPF_LOSS_STATE || iso;
  int rc = fill_common(prog, p, batch, single);
  if (rc) return rc;
  p.mode = cpf::M_ADAM;
  p.lr = (R)adam->lr; p.b1 = (R)adam->b1; p.b2 = (R)adam->b2; p.eps = (R)adam->eps;
  p.omb1 = (R)(1.0 - adam->b1); p.omb2 = (R)(1.0 - adam->b2);
  p.step0 = step0; p.nsteps = (int)num_steps;
  p.angles = (R*)buf->angles; p.m = (R*)buf->m; p.v = (R*)buf->v; p.freeze = buf->freeze;
  p.best_params = (R*)buf->best_params; p.best_regloss = (R*)buf->best_regloss;
  p.best_reg = (R*)buf->best_reg; p.init_regloss = (R*)buf->init_regloss; p.init_reg = (R*)buf->init_reg;
  p.hist_params = (R*)buf->hist_params; p.hist_regloss = (R*)buf->hist_regloss; p.hist_len = buf->hist_len;
  Scratch sc;
  sc.st = st;
  if (buf->workspace) {
    if (((uintptr_t)buf->workspace & 255) != 0) return fail(CPF_ERR_INVALID, "workspace must be 256-byte aligned");
    sc.base = (char*)buf->workspace;
    sc.size = buf->workspace_bytes > 0 ? (size_t)buf->workspace_bytes : 0;
  }
  cpf_loss_spec hs;
  if (loss->kind == CPF_LOSS_ISOMETRY && !iso) {
    rc = stage_iso_as_hs<R>(prog, loss, sc, &hs);
    if (rc) return rc;
    loss = &hs;
  }
  const bool heis = use_heis<R>(prog, loss) && (unsigned long long)batch * (unsigned long long)prog->n_params < (1ull << 32);
  rc = fill_penalty(prog, pen, p, sc);
  if (!rc && table) rc = stage_multi(prog, table, p, heis, sc);
  else if (!rc && iso) rc = stage_iso(prog, loss, p, sc);
  else if (!rc) rc = heis ? stage_heis(prog, loss, p, sc) : stage_target(prog, loss, p, single, sc);
  std::string err;
  if (!rc) {
    rc = iso ? cpf::launch_iso<R>(p, prog->n_qubits, st, err) : launch_staged<R>(p, prog, table, heis, single, st, err);
    if (rc) fail(rc, err);
  }
  return rc;
}

// bytes of scratch one cpf_adam_run / cpf_loss_grad needs (the blocks Scratch::get hands out, each 256-byte aligned)
template <typename R>
int64_t workspace_bytes_t(const cpf::Program* prog, int32_t loss_kind, int32_t mask, int64_t batch) {
  size_t total = Scratch::align(prog->cp.empty() ? 1 : prog->cp.size());          // penalty mask
  if (loss_kind == CPF_LOSS_ISOMETRY) {
    const int n = prog->n_qubits;
    if (n > 5) return (int64_t)(total + Scratch::align(((size_t)iso_spec(prog, mask).k << (n + 1)) * sizeof(R)));
    total += Scratch::align(((size_t)2 << (2 * n)) * sizeof(R));                   // V of the HS call
    loss_kind = CPF_LOSS_HS;
  }
  cpf_loss_spec ls{};
  ls.kind = loss_kind;
  const bool single = loss_kind == CPF_LOSS_STATE;
  const bool heis = use_heis<R>(prog, &ls) && (unsigned long long)batch * (unsigned long long)prog->n_params < (1ull << 32);
  if (heis) {
    size_t tb, ap, pk;
    heis_scratch_sizes<R>(prog, batch, &tb, &ap, &pk);
    total += Scratch::align(tb) + Scratch::align(ap + pk);
  } else {
    const int cpt = single ? 1 : cpf::cpt_for<R>(prog->n_qubits);
    total += Scratch::align((((size_t)cpf::target_words<R>(prog->n_qubits, cpt, single) * sizeof(R)) + 15) & ~(size_t)15);
  }
  return (int64_t)total;
}

template <typename R>
int64_t workspace_bytes_multi_t(const cpf::Program* prog, int32_t loss_kind, int64_t batch, int32_t n_targets) {
  cpf_loss_spec ls{};
  ls.kind = loss_kind;
  const bool heis = use_heis<R>(prog, &ls) && (unsigned long long)batch * (unsigned long long)prog->n_params < (1ull << 32);
  size_t total = Scratch::align(prog->cp.empty() ? 1 : prog->cp.size());          // penalty mask
  total += Scratch::align((size_t)batch * sizeof(int32_t));                         // target_index
  total += Scratch::align(multi_table_bytes<R>(prog, loss_kind, heis, n_targets));  // target table
  if (heis) {
    size_t tb, ap, pk;
    heis_scratch_sizes<R>(prog, batch, &tb, &ap, &pk);
    total += Scratch::align(ap + pk);
  }
  return (int64_t)total;
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
  cpf::KParams<R> p;
  std::memset(&p, 0, sizeof(p));
  // fill_penalty validates the spec and converts the table; the per-parameter mask is rebuilt here ([P], not [n_cp])
  int rc;
  {
    Scratch sc;
    sc.st = st;
    rc = fill_penalty(prog, pen, p, sc);
  }
  if (rc) return rc;
  uint8_t* mask_dev = nullptr;
  if (p.pen.kind != CPF_PEN_NONE && prog->n_params > 0) {
    std::string mask((size_t)prog->n_params, '\0');
    for (int i = 0; i < prog->n_params; ++i)
      mask[i] = prog->is_cp_param[i] && (!pen->cp_mask || pen->cp_mask[i]) ? 1 : 0;
    CPF_CUDA(cudaMallocAsync((void**)&mask_dev, mask.size(), st));
    CPF_CUDA(cudaMemcpyAsync(mask_dev, mask.data(), mask.size(), cudaMemcpyHostToDevice, st));
  }
  dim3 block(32, 8);
  const unsigned grid = (unsigned)((batch + 7) / 8);
  adam_step_kernel<R><<<grid, block, 0, st>>>(
      p.pen, mask_dev, prog->n_params, batch, step, (R)adam->lr, (R)adam->b1, (R)adam->b2, (R)adam->eps,
      (R)(1.0 - adam->b1), (R)(1.0 - adam->b2), (const R*)loss, (const R*)grad, (R*)buf->angles, (R*)buf->m, (R*)buf->v,
      buf->freeze, (R*)buf->best_params, (R*)buf->best_regloss, (R*)buf->best_reg, (R*)buf->init_regloss,
      (R*)buf->init_reg, (R*)buf->hist_params, (R*)buf->hist_regloss, buf->hist_len);
  cudaError_t e = cudaGetLastError();
  if (mask_dev) cudaFreeAsync(mask_dev, st);
  if (e != cudaSuccess) return cuda_fail("adam_step_kernel", e);
  return CPF_OK;
}

template <typename R>
static int launch_plan_t(const cpf::Program* prog, const cpf_loss_spec_kind_only& lk, int64_t batch, int n_sm, int regs,
                         cpf_launch_info* out, int adam_steps = 2000) {
  cpf_loss_spec ls{};
  ls.kind = lk.kind;
  const bool heis = use_heis<R>(prog, &ls) && (unsigned long long)batch * (unsigned long long)prog->n_params < (1ull << 32);
  out->engine = heis ? 1 : 0;
  if (!heis) return CPF_OK;
  const int n = prog->n_qubits, N = 1 << n, cpt = cpf::heis_cpt<R>(n), tps = N / cpt;
  const int maxt = 2 * N * cpt * (int)(sizeof(R) / 4) <= 64 ? 512 : 256;          // HCfg::MAXT
  const int n_su2 = (int)prog->su2.size(), n_cp = (int)prog->cp.size();
  int n_stage = n;                                                                // SWP::NSTAGE of the kernel chosen
  {
    cpf::KParams<R> dummy;
    std::string e2;
    int rc2 = 0;
    cpf::launch_heis<R>(dummy, *prog, nullptr, e2, rc2, true, &n_stage);
  }
  const int stride = cpf::heis_coef_stride(n_su2, n_cp, n_stage);
  const size_t target = (((size_t)cpf::heis_target_words<R>(n, cpt) * sizeof(R)) + 15) & ~(size_t)15;
  const cpf::HeisGeometry g = cpf::heis_geometry(batch, target + cpf::heis_meta_bytes(n_su2, n_cp),
                                                 (size_t)stride * sizeof(R), tps, maxt, regs > 0 ? regs : 128,
                                                 n_sm > 0 ? n_sm : 148);
  out->ctas_per_sm = g.ctas; out->block_threads = g.block; out->samples_per_cta = g.spb; out->grid = g.grid;
  out->smem_bytes = (int64_t)g.smem; out->threads_per_sample = tps; out->max_block_threads = maxt;
  out->words_per_sample = stride;
  // time slices an Adam run of `adam_steps` iterations over this batch would be cut into (1 = one launch)
  const cpf::HeisSlicing sl = cpf::heis_slicing(batch, adam_steps > 0 ? adam_steps : 2000,
                                                target + cpf::heis_meta_bytes(n_su2, n_cp), (size_t)stride * sizeof(R), tps,
                                                maxt, regs > 0 ? regs : 128, n_sm > 0 ? n_sm : 148, true);
  out->time_slices = sl.k;
  out->launches_per_run = sl.k > 1 ? (batch * sl.k + sl.slots - 1) / sl.slots : 1;
  return CPF_OK;
}

// the isometry kernel's geometry (iso_impl.cuh: iso_geometry); co-residency is not planned (ctas_per_sm = 0)
template <typename R>
static int iso_plan_t(const cpf::Program* prog, int32_t mask, int64_t batch, cpf_launch_info* out) {
  const int n = prog->n_qubits, n_su2 = (int)prog->su2.size(), n_cp = (int)prog->cp.size();
  const int k = iso_spec(prog, mask).k;
  const int rb = cpf::engine_rb<R>(n, true);
  const cpf::DecodedSchedule ds = cpf::decode_schedule(*prog, rb);
  const int n_red = ds.red.empty() ? 1 : (int)(ds.red.size() / 8);
  const cpf::IsoGeometry g = cpf::iso_geometry(n, rb, k, n_su2, n_cp, (int)prog->sched.size(), n_red, sizeof(R));
  out->engine = 0;
  out->block_threads = g.block;
  out->samples_per_cta = g.spb;
  out->threads_per_sample = g.spt;
  out->max_block_threads = n == 6 ? 512 : 1024;          // __launch_bounds__ of iso_kernel
  out->words_per_sample = cpf::iso_sample_words(cpf::coef_stride_words(n_su2, n_cp), k, cpf::iso_sum_stride(n_su2, n_cp));
  out->time_slices = 1;
  out->grid = (batch + g.spb - 1) / g.spb;
  out->smem_bytes = (int64_t)g.smem;
  out->launches_per_run = 1;
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
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  int rc = check_loss(p, loss);
  if (rc) return rc;
  if (batch == 0) return CPF_OK;
  if (!loss_out) return fail(CPF_ERR_INVALID, "loss_out is NULL");
  if (!angles && p->n_params > 0) return fail(CPF_ERR_INVALID, "angles is NULL");
  CPF_DISPATCH(dtype, (run_loss_grad<R>(p, loss, penalty, batch, angles, loss_out, reg_out, grad_out,
                                        (cudaStream_t)stream)));
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
  int rc = check_loss(reinterpret_cast<const cpf::Program*>(prog), loss);
  if (rc) return rc;
  if (batch == 0 || num_steps == 0) return CPF_OK;
  if (!buf->angles || !buf->m || !buf->v || !buf->best_params || !buf->best_regloss || !buf->best_reg ||
      !buf->init_regloss || !buf->init_reg)
    return fail(CPF_ERR_INVALID, "a required cpf_adam_buffers pointer is NULL");
  if ((buf->hist_params || buf->hist_regloss) && buf->hist_len <= 0)
    return fail(CPF_ERR_INVALID, "history buffers given with hist_len <= 0");
  if (num_steps > 2000000000LL) return fail(CPF_ERR_INVALID, "num_steps too large");
  if (batch == 0 || num_steps == 0) return CPF_OK;
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  CPF_DISPATCH(dtype, (run_adam<R>(p, loss, penalty, adam, batch, step0, num_steps, buf,
                                   (cudaStream_t)stream)));
}

int cpf_workspace_bytes(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch, int64_t* bytes) {
  if (!prog || !bytes || batch < 0) return fail(CPF_ERR_INVALID, "NULL argument / negative batch");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  int32_t kind, mask;
  int rc = split_kind(p, loss_kind, &kind, &mask);
  if (!rc) rc = check_full_unitary(p, kind);
  if (rc) return rc;
  *bytes = dtype == CPF_F64 ? workspace_bytes_t<double>(p, kind, mask, batch) : workspace_bytes_t<float>(p, kind, mask, batch);
  return CPF_OK;
}

int cpf_loss_grad_multi(const cpf_program* prog, const cpf_target_table* table, const cpf_penalty_spec* penalty,
                        int32_t dtype, int64_t batch, const void* angles, void* loss_out, void* reg_out,
                        void* grad_out, void* stream) {
  if (!prog || batch < 0) return fail(CPF_ERR_INVALID, "NULL program / bad batch");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  int rc = check_table(p, table, batch);
  if (rc) return rc;
  if (batch == 0) return CPF_OK;
  if (!loss_out) return fail(CPF_ERR_INVALID, "loss_out is NULL");
  if (!angles && p->n_params > 0) return fail(CPF_ERR_INVALID, "angles is NULL");
  const cpf_loss_spec loss{table->kind, table->targets, 0};
  CPF_DISPATCH(dtype, (run_loss_grad<R>(p, &loss, penalty, batch, angles, loss_out, reg_out, grad_out,
                                        (cudaStream_t)stream, table)));
}

int cpf_adam_run_multi(const cpf_program* prog, const cpf_target_table* table, const cpf_penalty_spec* penalty,
                       const cpf_adam_spec* adam, int32_t dtype, int64_t batch, int64_t step0, int64_t num_steps,
                       const cpf_adam_buffers* buf, void* stream) {
  if (!prog || !adam || !buf || batch < 0 || step0 < 0 || num_steps < 0)
    return fail(CPF_ERR_INVALID, "NULL argument / negative size");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  int rc = check_table(p, table, batch);
  if (rc) return rc;
  if (batch == 0 || num_steps == 0) return CPF_OK;
  if (!buf->angles || !buf->m || !buf->v || !buf->best_params || !buf->best_regloss || !buf->best_reg ||
      !buf->init_regloss || !buf->init_reg)
    return fail(CPF_ERR_INVALID, "a required cpf_adam_buffers pointer is NULL");
  if ((buf->hist_params || buf->hist_regloss) && buf->hist_len <= 0)
    return fail(CPF_ERR_INVALID, "history buffers given with hist_len <= 0");
  if (num_steps > 2000000000LL) return fail(CPF_ERR_INVALID, "num_steps too large");
  const cpf_loss_spec loss{table->kind, table->targets, 0};
  CPF_DISPATCH(dtype, (run_adam<R>(p, &loss, penalty, adam, batch, step0, num_steps, buf, (cudaStream_t)stream,
                                   table)));
}

int cpf_workspace_bytes_multi(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch,
                              int32_t n_targets, int64_t* bytes) {
  if (!prog || !bytes || batch < 0) return fail(CPF_ERR_INVALID, "NULL argument / negative batch");
  if (loss_kind == CPF_LOSS_ISOMETRY)
    return fail(CPF_ERR_UNSUPPORTED, "multi-target tables do not take the isometry loss (one target per call)");
  if (loss_kind < CPF_LOSS_HS || loss_kind > CPF_LOSS_RELPHASE) return fail(CPF_ERR_INVALID, "unknown loss kind");
  if (n_targets < 1) return fail(CPF_ERR_INVALID, "n_targets must be >= 1");
  if (dtype != CPF_F32 && dtype != CPF_F64) return fail(CPF_ERR_INVALID, "unknown dtype");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  if (int rc = check_full_unitary(p, loss_kind)) return rc;
  *bytes = dtype == CPF_F64 ? workspace_bytes_multi_t<double>(p, loss_kind, batch, n_targets)
                            : workspace_bytes_multi_t<float>(p, loss_kind, batch, n_targets);
  return CPF_OK;
}

int cpf_adam_step(const cpf_program* prog, const cpf_penalty_spec* penalty, const cpf_adam_spec* adam, int32_t dtype,
                  int64_t batch, int64_t step, const void* loss, const void* grad, const cpf_adam_buffers* buf,
                  void* stream) {
  if (!prog || !adam || !buf || batch < 0 || step < 0) return fail(CPF_ERR_INVALID, "NULL argument / negative size");
  if (batch == 0) return CPF_OK;
  if (!loss || !grad) return fail(CPF_ERR_INVALID, "loss / grad is NULL");
  if (!buf->angles || !buf->m || !buf->v || !buf->best_params || !buf->best_regloss || !buf->best_reg ||
      !buf->init_regloss || !buf->init_reg)
    return fail(CPF_ERR_INVALID, "a required cpf_adam_buffers pointer is NULL");
  if ((buf->hist_params || buf->hist_regloss) && buf->hist_len <= 0)
    return fail(CPF_ERR_INVALID, "history buffers given with hist_len <= 0");
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
  int32_t kind, mask;
  int rc = split_kind(p, loss_kind, &kind, &mask);
  if (rc) return rc;
  const double N = (double)(1 << p->n_qubits);
  const double C = kind == CPF_LOSS_STATE ? 1.0 : kind == CPF_LOSS_ISOMETRY ? (double)iso_spec(p, mask).k : N;
  const double rs = dtype == CPF_F64 ? 8.0 : 4.0;
  if (flops) *flops = C * N * (16.0 * p->n_rot + 4.0 * p->n_phase + 8.0);
  if (bytes) *bytes = 6.0 * p->n_params * rs + 2.0 * rs;
  return CPF_OK;
}

int cpf_executed_cost(const cpf_program* prog, int32_t loss_kind, int32_t dtype, double* flops) {
  if (!prog || !flops) return fail(CPF_ERR_INVALID, "NULL argument");
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  const double N = (double)(1 << p->n_qubits), n = p->n_qubits, K = (double)p->cp.size(), G = (double)p->su2.size();
  int32_t kind, mask;
  int rc = split_kind(p, loss_kind, &kind, &mask);
  if (rc) return rc;
  // isometry: n <= 5 runs as an HS call; n >= 6 on the isometry kernel, the state-adjoint count with C = k
  const bool iso = kind == CPF_LOSS_ISOMETRY && p->n_qubits > 5;
  if (kind == CPF_LOSS_ISOMETRY && !iso) kind = CPF_LOSS_HS;
  cpf_loss_spec ls{};
  ls.kind = kind;
  const bool heis = dtype == CPF_F64 ? use_heis<double>(p, &ls) : use_heis<float>(p, &ls);
  if (heis) {
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
    // fused gates, 1.5 per phase gate), with fused gates instead of primitive rotations: C N (22 G + 5.5 K + 8)
    const double C = kind == CPF_LOSS_STATE ? 1.0 : iso ? (double)iso_spec(p, mask).k : N;
    *flops = C * N * (22.0 * G + 5.5 * K + 8.0) + 232.0 * G + 80.0 * K;
  }
  return CPF_OK;
}

int cpf_launch_plan(const cpf_program* prog, int32_t loss_kind, int32_t dtype, int64_t batch, int32_t n_sm,
                    int32_t regs_per_thread, cpf_launch_info* out) {
  if (!prog || !out) return fail(CPF_ERR_INVALID, "NULL argument");
  if (batch < 0) return fail(CPF_ERR_INVALID, "negative batch");
  std::memset(out, 0, sizeof(*out));
  const cpf::Program* p = reinterpret_cast<const cpf::Program*>(prog);
  int32_t kind, mask;
  int rc = split_kind(p, loss_kind, &kind, &mask);
  if (rc) return rc;
  if (kind == CPF_LOSS_ISOMETRY && p->n_qubits > 5)
    return dtype == CPF_F64 ? iso_plan_t<double>(p, mask, batch, out) : iso_plan_t<float>(p, mask, batch, out);
  const cpf_loss_spec_kind_only lk{kind == CPF_LOSS_ISOMETRY ? CPF_LOSS_HS : kind};   // n <= 5: an HS call
  return dtype == CPF_F64 ? launch_plan_t<double>(p, lk, batch, n_sm, regs_per_thread, out)
                          : launch_plan_t<float>(p, lk, batch, n_sm, regs_per_thread, out);
}

}  // extern "C"
