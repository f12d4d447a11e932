// Relative-phase isometry kernels on 2-8 qubits, float32 / complex64 (iso_impl.cuh: InterpSweepIsoPhase).  The decoded
// schedule is the one of the single-column kernels on every n (engine_rb: 2, 2, 1, 1, 2, 2, 3 register bits on 2-8
// qubits), which launch_iso_sized checks against the sweep type's.
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_iso_phase<float>(const KParams<float>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 2: return launch_iso_sized<float, 2, InterpSweepIsoPhase<float, 2>>(p, st, err);
    case 3: return launch_iso_sized<float, 3, InterpSweepIsoPhase<float, 3>>(p, st, err);
    case 4: return launch_iso_sized<float, 4, InterpSweepIsoPhase<float, 4>>(p, st, err);
    case 5: return launch_iso_sized<float, 5, InterpSweepIsoPhase<float, 5>>(p, st, err);
    case 6: return launch_iso_sized<float, 6, InterpSweepIsoPhase<float, 6>>(p, st, err);
    case 7: return launch_iso_sized<float, 7, InterpSweepIsoPhase<float, 7>>(p, st, err);
    case 8: return launch_iso_sized<float, 8, InterpSweepIsoPhase<float, 8>>(p, st, err);
  }
  err = "the relative-phase isometry kernel runs 2-8 qubits";
  return CPF_ERR_UNSUPPORTED;
}

}  // namespace cpf
