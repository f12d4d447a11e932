// Cotangent mode of the isometry kernel on 6-8 qubits, double / complex128 (iso_impl.cuh: InterpSweepIsoCot): the
// vector-Jacobian product of cpf_adjoint_from_cotangent, one launch item per (sample, chunk of columns), and the sum
// of the chunks' gradients.
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_iso_cot<double>(const KParams<double>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 6: return launch_iso_sized<double, 6, InterpSweepIsoCot<double, 6>>(p, st, err);
    case 7: return launch_iso_sized<double, 7, InterpSweepIsoCot<double, 7>>(p, st, err);
    case 8: return launch_iso_sized<double, 8, InterpSweepIsoCot<double, 8>>(p, st, err);
  }
  err = "the cotangent kernel of the isometry family runs 6-8 qubits (n <= 5: the full-unitary kernels)";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_cot_reduce<double>(const double* partial, double* grad, long long batch, int P, int n_chunks, cudaStream_t st) {
  const long long blocks = (batch * P + 255) / 256;
  cot_reduce_kernel<double><<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, st>>>(partial, grad, batch, P, n_chunks);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
