// Subspace kernels, double / complex128 (iso_impl.cuh: InterpSweepSub, InterpSweepSubPhase): the isometry kernel with forward sweeps
// that start from the caller's input states.  CPF_LOSS_SUBSPACE runs here on 6-8 qubits (n <= 5: the HS kernels on
// V = (N/k) B A^dag), CPF_LOSS_SUBSPACE_RELPHASE on 2-8.  The decoded schedule is the one of the single-column kernels
// (engine_rb: 2, 2, 1, 1, 2, 2, 3 register bits on 2-8 qubits), which launch_iso_sized checks against the sweep type's.
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_sub<double>(const KParams<double>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 6: return launch_iso_sized<double, 6, InterpSweepSub<double, 6>>(p, st, err);
    case 7: return launch_iso_sized<double, 7, InterpSweepSub<double, 7>>(p, st, err);
    case 8: return launch_iso_sized<double, 8, InterpSweepSub<double, 8>>(p, st, err);
  }
  err = "the subspace kernel runs 6-8 qubits (n <= 5: the HS kernels)";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_sub_phase<double>(const KParams<double>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 2: return launch_iso_sized<double, 2, InterpSweepSubPhase<double, 2>>(p, st, err);
    case 3: return launch_iso_sized<double, 3, InterpSweepSubPhase<double, 3>>(p, st, err);
    case 4: return launch_iso_sized<double, 4, InterpSweepSubPhase<double, 4>>(p, st, err);
    case 5: return launch_iso_sized<double, 5, InterpSweepSubPhase<double, 5>>(p, st, err);
    case 6: return launch_iso_sized<double, 6, InterpSweepSubPhase<double, 6>>(p, st, err);
    case 7: return launch_iso_sized<double, 7, InterpSweepSubPhase<double, 7>>(p, st, err);
    case 8: return launch_iso_sized<double, 8, InterpSweepSubPhase<double, 8>>(p, st, err);
  }
  err = "the relative-phase subspace kernel runs 2-8 qubits";
  return CPF_ERR_UNSUPPORTED;
}

template <>
int launch_pack_subspace_hs<double>(const double* src, double* dst, int n, int k, cudaStream_t st) {
  pack_subspace_hs_kernel<double><<<8, 256, 0, st>>>(src, dst, 1 << n, k);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
