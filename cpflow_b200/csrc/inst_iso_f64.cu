// Isometry kernels on 6-8 qubits, float64 / complex128 (iso_impl.cuh).  The decoded schedule is the one of the single-column
// kernels (engine_rb: 2 register bits on 6-7 qubits, 3 on 8).
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_iso<double>(const KParams<double>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 6: return launch_iso_sized<double, 6>(p, st, err);
    case 7: return launch_iso_sized<double, 7>(p, st, err);
    case 8: return launch_iso_sized<double, 8>(p, st, err);
  }
  err = "the isometry kernel runs 6-8 qubits (n <= 5: the HS kernels)";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_pack_iso<double>(const double* src, double* dst, int n, int k, int amask, bool as_hs, cudaStream_t st) {
  if (as_hs) pack_iso_hs_kernel<double><<<8, 256, 0, st>>>(src, dst, n, k, amask);
  else pack_iso_kernel<double><<<8, 256, 0, st>>>(src, dst, 1 << n, k);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
