// Host launcher for engine_kernel instantiations.
#pragma once
#include <string>

#include "engine_impl.cuh"

namespace cpf {

// refusal of HS and relative-phase losses above 5 qubits (the full-unitary kernels stop at n = 5)
constexpr char FULL_UNITARY_LIMIT[] =
    "full-unitary losses need n <= 5 qubits (6-8 qubits: state preparation, isometries and cpf_unitary only)";

inline int coef_stride_words(int n_su2, int n_cp) {
  int w = (coef_words(n_su2, n_cp) + 3) & ~3;
  if (w == 0) w = 4;
  if (((w / 4) & 1) == 0) w += 4;  // odd number of 16-byte groups: samples of a warp hit distinct banks
  return w;
}

template <typename R>
inline int target_words(int n, int cpt, bool single) {
  const int N = 1 << n;
  return (single ? 1 : N / cpt) * (N + 1) * 2 * cpt;
}

template <typename R, int NQ, int RB, int CPT, bool SINGLE, typename SW = InterpSweep<R, NQ, RB, CPT, SINGLE>>
int launch_one(KParams<R> p, cudaStream_t st, std::string& err) {
  using C = Cfg<R, NQ, RB, CPT, SINGLE>;
  if (!SW::USES_SCHED) { p.n_sched = 0; p.n_red = 0; }
  p.coef_stride = coef_stride_words(p.n_su2, p.n_cp);
  // CTA barrier at the sweep starts for the straight-line layered sweeps (the warps of a CTA then share the
  // instruction cache: state preparation n = 5 54.5 -> 66.1 M evals/s, relative-phase loss 24 -> 29.6 M); the
  // interpreter's sweep is a small loop and runs without.  CPF_ENGINE_SYNC overrides (measurements).
  p.sync_sweeps = SW::USES_SCHED ? 0 : 3;
  if (const char* e = getenv("CPF_ENGINE_SYNC")) { int v = atoi(e); if (v >= 0 && v <= 3) p.sync_sweeps = v; }
  const size_t smem = (size_t)p.target_bytes + (size_t)((p.n_sched + 1) & ~1) * 8 + (size_t)p.n_red * 16 +
                      (size_t)C::SPB * p.coef_stride * sizeof(R);
  if (smem > 227 * 1024) {
    err = "program too large for the shared-memory coefficient store (" + std::to_string(smem) + " bytes)";
    return CPF_ERR_UNSUPPORTED;
  }
  auto kern = engine_kernel<R, NQ, RB, CPT, SINGLE, SW>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) { err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); return CPF_ERR_CUDA; }
  const long long grid = (p.B + C::SPB - 1) / C::SPB;
  if (grid <= 0) return CPF_OK;
  if (grid > 2147483647LL) { err = "batch too large for one launch"; return CPF_ERR_UNSUPPORTED; }
  kern<<<(unsigned)grid, C::BLOCK, smem, st>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) { err = std::string("kernel launch: ") + cudaGetErrorString(e); return CPF_ERR_CUDA; }
  return CPF_OK;
}

// columns per thread chosen for each (dtype, n)
template <typename R> constexpr int cpt_for(int n) { return 1; }
template <> constexpr int cpt_for<float>(int n) { return 2; }

template <typename R> int launch_engine(const KParams<R>& p, int n_qubits, bool single,
                                        cudaStream_t st, std::string& err);
// Specialised kernels for layered templates (inst_layer_*.cu).  Returns true and sets `rc` when a
// kernel compiled for this layer exists; false means "use the interpreter kernel".
template <typename R> bool launch_layered(const KParams<R>& p, const Program& prog, bool single,
                                          cudaStream_t st, std::string& err, int& rc);
// register bits of the kernel configuration launch_engine picks (selects the decoded schedule)
template <typename R> int engine_rb(int n_qubits, bool single);
template <typename R> int launch_pack_target(const R* src, R* dst, int n_qubits, int cpt, bool single,
                                             cudaStream_t st);

}  // namespace cpf
