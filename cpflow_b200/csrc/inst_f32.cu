// float32 / complex64 instantiations of the engine (the reference's default x32 mode).
// launch_one<R, NQ, RB, CPT, SINGLE>: RB register bits, NQ-RB lane bits, CPT packed columns.
#include <cstdlib>

#include "launch.cuh"

namespace cpf {

// Register bits of the single-column kernels (state preparation, column-mode unitary).  A sample's coefficient store
// (8 words per fused gate) lives in shared memory, so few lanes per sample mean few resident warps: with 3 / 4 register
// bits the 5-7 qubit templates ran 4 warps per SM.  Measured on B200 (state preparation, K = 60, evals/s;
// profiles/r2_exp_single_rb.txt): n = 4: 2 bits 61 M, 1 bit 92 M, 0 bits 86 M; n = 5: 3 bits 22 M, 2: 35 M, 1: 47 M,
// 0: 36 M; n = 6: 3 bits 21 M, 2: 35 M, 1: 28 M; n = 7: 4 bits 7.5 M, 3: 15.7 M, 2: 20.5 M.  n = 8: 3 bits, the fewest
// that keep a column in one warp (32 lanes).
static int single_rb_f32(int n) {
  switch (n) {
    case 2: return 2; case 3: return 2; case 4: return 1; case 5: return 1; case 6: return 2; case 7: return 2;
    case 8: return 3;
  }
  return -1;
}

template <>
int launch_engine<float>(const KParams<float>& p, int n, bool single, cudaStream_t st, std::string& err) {
  if (single) {
    switch (n) {
      case 2: return launch_one<float, 2, 2, 1, true>(p, st, err);
      case 3: return launch_one<float, 3, 2, 1, true>(p, st, err);
      case 4: return launch_one<float, 4, 1, 1, true>(p, st, err);
      case 5: return launch_one<float, 5, 1, 1, true>(p, st, err);
      case 6: return launch_one<float, 6, 2, 1, true>(p, st, err);
      case 7: return launch_one<float, 7, 2, 1, true>(p, st, err);
      case 8: return launch_one<float, 8, 3, 1, true>(p, st, err);
    }
  } else {
    switch (n) {
      case 2: return launch_one<float, 2, 2, 2, false>(p, st, err);
      case 3: return launch_one<float, 3, 2, 2, false>(p, st, err);
      case 4: return launch_one<float, 4, 2, 2, false>(p, st, err);
      case 5: return launch_one<float, 5, 4, 2, false>(p, st, err);
    }
  }
  err = single ? "unsupported number of qubits" : FULL_UNITARY_LIMIT;
  return CPF_ERR_UNSUPPORTED;
}

template <>
int engine_rb<float>(int n, bool single) {
  if (single) {
    return single_rb_f32(n);
  } else {
    switch (n) { case 2: return 2; case 3: return 2; case 4: return 2; case 5: return 4; }
  }
  return -1;
}

template <>
int launch_pack_target<float>(const float* src, float* dst, int n, int cpt, bool single, cudaStream_t st) {
  pack_target_kernel<float><<<8, 256, 0, st>>>(src, dst, 1 << n, cpt, single ? 1 : 0);
  return cudaGetLastError() == cudaSuccess ? CPF_OK : CPF_ERR_CUDA;
}

}  // namespace cpf
