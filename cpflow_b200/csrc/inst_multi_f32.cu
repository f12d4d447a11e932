// Multi-target kernels, float32 / complex64: the runtime-pair Heisenberg sweep (HeisSweepAnyMT) for the HS loss on
// block-structured templates, and the interpreter kernel (InterpSweepMT) for every other loss and template.  Register
// bits and columns per thread are those of the single-target dispatch (inst_f32.cu, inst_heis_f32.cu): the decoded
// schedule (engine_rb) and the heis target packing (heis_cpt) are shared with it.
#include <algorithm>

#include "heis_impl.cuh"
#include "launch.cuh"

namespace cpf {

template <>
bool launch_heis_multi<float>(const KParams<float>& p, const Program& prog, cudaStream_t st, std::string& err, int& rc) {
  switch (prog.n_qubits) {
    case 2: rc = launch_heis_sized<float, 2, 2, HeisSweepAnyMT<float, 2, 2>>(p, st, err); return true;
    case 3: rc = launch_heis_sized<float, 3, 2, HeisSweepAnyMT<float, 3, 2>>(p, st, err); return true;
    case 4: rc = launch_heis_sized<float, 4, 2, HeisSweepAnyMT<float, 4, 2>>(p, st, err); return true;
    case 5: rc = launch_heis_sized<float, 5, 1, HeisSweepAnyMT<float, 5, 1>>(p, st, err); return true;
  }
  return false;
}

template <>
int launch_engine_multi<float>(const KParams<float>& p, int n, bool single, cudaStream_t st, std::string& err) {
  if (single) {
    switch (n) {
      case 2: return launch_one<float, 2, 2, 1, true, InterpSweepMT<float, 2, 2, 1, true>>(p, st, err);
      case 3: return launch_one<float, 3, 2, 1, true, InterpSweepMT<float, 3, 2, 1, true>>(p, st, err);
      case 4: return launch_one<float, 4, 1, 1, true, InterpSweepMT<float, 4, 1, 1, true>>(p, st, err);
      case 5: return launch_one<float, 5, 1, 1, true, InterpSweepMT<float, 5, 1, 1, true>>(p, st, err);
      case 6: return launch_one<float, 6, 2, 1, true, InterpSweepMT<float, 6, 2, 1, true>>(p, st, err);
      case 7: return launch_one<float, 7, 2, 1, true, InterpSweepMT<float, 7, 2, 1, true>>(p, st, err);
      case 8: return launch_one<float, 8, 3, 1, true, InterpSweepMT<float, 8, 3, 1, true>>(p, st, err);
    }
  } else {
    switch (n) {
      case 2: return launch_one<float, 2, 2, 2, false, InterpSweepMT<float, 2, 2, 2, false>>(p, st, err);
      case 3: return launch_one<float, 3, 2, 2, false, InterpSweepMT<float, 3, 2, 2, false>>(p, st, err);
      case 4: return launch_one<float, 4, 2, 2, false, InterpSweepMT<float, 4, 2, 2, false>>(p, st, err);
      case 5: return launch_one<float, 5, 4, 2, false, InterpSweepMT<float, 5, 4, 2, false>>(p, st, err);
    }
  }
  err = single ? "unsupported number of qubits" : FULL_UNITARY_LIMIT;
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_pack_targets_heis<float>(const float* src, float* dst, int n, int cpt, int n_targets, cudaStream_t st) {
  const int N = 1 << n;
  for (int t0 = 0; t0 < n_targets; t0 += 65535)      // (grid.y limit)
    pack_targets_heis_kernel<float><<<dim3(1, (unsigned)std::min(n_targets - t0, 65535)), 256, 0, st>>>(
        src + (size_t)t0 * N * N * 2, dst + (size_t)t0 * heis_target_words<float>(n, cpt), N, cpt);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

template <>
int launch_pack_targets<float>(const float* src, float* dst, int n, int cpt, bool single, int n_targets, cudaStream_t st) {
  const int N = 1 << n;
  for (int t0 = 0; t0 < n_targets; t0 += 65535)
    pack_targets_kernel<float><<<dim3(1, (unsigned)std::min(n_targets - t0, 65535)), 256, 0, st>>>(
        src + (size_t)t0 * (single ? N : N * N) * 2, dst + (size_t)t0 * target_words<float>(n, cpt, single), N, cpt,
        single ? 1 : 0);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
