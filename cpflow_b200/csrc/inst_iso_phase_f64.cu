// Relative-phase isometry kernels on 2-8 qubits, double / complex128 (iso_impl.cuh: InterpSweepIsoPhase).  The decoded
// schedule is the one of the single-column kernels on every n (engine_rb: 2, 2, 1, 1, 2, 2, 3 register bits on 2-8
// qubits), which launch_iso_sized checks against the sweep type's.
#include "iso_impl.cuh"

namespace cpf {

template <>
int launch_iso_phase<double>(const KParams<double>& p, int n, cudaStream_t st, std::string& err) {
  switch (n) {
    case 2: return launch_iso_sized<double, 2, InterpSweepIsoPhase<double, 2>>(p, st, err);
    case 3: return launch_iso_sized<double, 3, InterpSweepIsoPhase<double, 3>>(p, st, err);
    case 4: return launch_iso_sized<double, 4, InterpSweepIsoPhase<double, 4>>(p, st, err);
    case 5: return launch_iso_sized<double, 5, InterpSweepIsoPhase<double, 5>>(p, st, err);
    case 6: return launch_iso_sized<double, 6, InterpSweepIsoPhase<double, 6>>(p, st, err);
    case 7: return launch_iso_sized<double, 7, InterpSweepIsoPhase<double, 7>>(p, st, err);
    case 8: return launch_iso_sized<double, 8, InterpSweepIsoPhase<double, 8>>(p, st, err);
  }
  err = "the relative-phase isometry kernel runs 2-8 qubits";
  return CPF_ERR_UNSUPPORTED;
}

}  // namespace cpf
