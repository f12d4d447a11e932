// Subspace kernels, float32 / complex64 (iso_impl.cuh: InterpSweepSub, InterpSweepSubPhase): the isometry kernel with forward sweeps
// that start from the caller's input states.  CPF_LOSS_SUBSPACE runs here on 6-8 qubits (n <= 5: the HS kernels on
// V = (N/k) B A^dag), CPF_LOSS_SUBSPACE_RELPHASE on 2-8.  The decoded schedule is the one of the single-column kernels
// (engine_rb: 2, 2, 1, 1, 2, 2, 3 register bits on 2-8 qubits), which launch_iso_sized checks against the sweep type's.
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_sub<float>(const KParams<float>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 6: return launch_iso_sized<float, 6, InterpSweepSub<float, 6>>(p, st, err);
    case 7: return launch_iso_sized<float, 7, InterpSweepSub<float, 7>>(p, st, err);
    case 8: return launch_iso_sized<float, 8, InterpSweepSub<float, 8>>(p, st, err);
  }
  err = "the subspace kernel runs 6-8 qubits (n <= 5: the HS kernels)";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_sub_phase<float>(const KParams<float>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 2: return launch_iso_sized<float, 2, InterpSweepSubPhase<float, 2>>(p, st, err);
    case 3: return launch_iso_sized<float, 3, InterpSweepSubPhase<float, 3>>(p, st, err);
    case 4: return launch_iso_sized<float, 4, InterpSweepSubPhase<float, 4>>(p, st, err);
    case 5: return launch_iso_sized<float, 5, InterpSweepSubPhase<float, 5>>(p, st, err);
    case 6: return launch_iso_sized<float, 6, InterpSweepSubPhase<float, 6>>(p, st, err);
    case 7: return launch_iso_sized<float, 7, InterpSweepSubPhase<float, 7>>(p, st, err);
    case 8: return launch_iso_sized<float, 8, InterpSweepSubPhase<float, 8>>(p, st, err);
  }
  err = "the relative-phase subspace kernel runs 2-8 qubits";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_pack_subspace_hs<float>(const float* src, float* dst, int n, int k, cudaStream_t st) {
  pack_subspace_hs_kernel<float><<<8, 256, 0, st>>>(src, dst, 1 << n, k);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
