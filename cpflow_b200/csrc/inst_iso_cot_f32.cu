// Cotangent mode of the isometry kernel on 6-8 qubits, float / complex64 (iso_impl.cuh: InterpSweepIsoCot): the
// vector-Jacobian product of cpf_adjoint_from_cotangent, one launch item per (sample, chunk of columns), and the sum
// of the chunks' gradients.
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_iso_cot<float>(const KParams<float>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 6: return launch_iso_sized<float, 6, InterpSweepIsoCot<float, 6>>(p, st, err);
    case 7: return launch_iso_sized<float, 7, InterpSweepIsoCot<float, 7>>(p, st, err);
    case 8: return launch_iso_sized<float, 8, InterpSweepIsoCot<float, 8>>(p, st, err);
  }
  err = "the cotangent kernel of the isometry family runs 6-8 qubits (n <= 5: the full-unitary kernels)";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_cot_reduce<float>(const float* partial, float* grad, long long batch, int P, int n_chunks, cudaStream_t st) {
  const long long blocks = (batch * P + 255) / 256;
  cot_reduce_kernel<float><<<(unsigned)(blocks < 4096 ? blocks : 4096), 256, 0, st>>>(partial, grad, batch, P, n_chunks);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
