// float64 / complex128 instantiations of the engine (reference semantics in double).
#include "launch.cuh"

namespace cpf {

template <>
int launch_engine<double>(const KParams<double>& p, int n, bool single, cudaStream_t st, std::string& err) {
  if (single) {
    switch (n) {
      case 2: return launch_one<double, 2, 2, 1, true>(p, st, err);
      case 3: return launch_one<double, 3, 2, 1, true>(p, st, err);
      // (register bits as in inst_f32.cu: more lanes per sample = more resident warps)
      case 4: return launch_one<double, 4, 1, 1, true>(p, st, err);
      case 5: return launch_one<double, 5, 1, 1, true>(p, st, err);
      case 6: return launch_one<double, 6, 2, 1, true>(p, st, err);
      case 7: return launch_one<double, 7, 2, 1, true>(p, st, err);
      case 8: return launch_one<double, 8, 3, 1, true>(p, st, err);
    }
  } else {
    switch (n) {
      case 2: return launch_one<double, 2, 2, 1, false>(p, st, err);
      case 3: return launch_one<double, 3, 2, 1, false>(p, st, err);
      case 4: return launch_one<double, 4, 3, 1, false>(p, st, err);
      case 5: return launch_one<double, 5, 5, 1, false>(p, st, err);
    }
  }
  err = single ? "unsupported number of qubits" : FULL_UNITARY_LIMIT;
  return CPF_ERR_UNSUPPORTED;
}

template <>
int engine_rb<double>(int n, bool single) {
  if (single) {
    switch (n) {
      case 2: return 2; case 3: return 2; case 4: return 1; case 5: return 1; case 6: return 2; case 7: return 2;
      case 8: return 3;
    }
  } else {
    switch (n) { case 2: return 2; case 3: return 2; case 4: return 3; case 5: return 5; }
  }
  return -1;
}

template <>
int launch_pack_target<double>(const double* src, double* dst, int n, int cpt, bool single, cudaStream_t st) {
  pack_target_kernel<double><<<8, 256, 0, st>>>(src, dst, 1 << n, cpt, single ? 1 : 0);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
