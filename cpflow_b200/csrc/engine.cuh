// sm_100a device engine for the cpflow hot path (SURVEY.md §8a rows A1-A11, A15).
//
// One launch runs, for every sample of the batch and `nsteps` times:
//   parameter phase : sin/cos of the angles, fuse up to three rotations into one SU(2)
//                     (gates.py:22-35, main.py:77-80, main.py:122-124), CP phases (gates.py:51-58),
//                     penalty value (penalty.py:44-71)
//   forward sweep   : apply the gate schedule to the identity -> U      (main.py:106-146)
//   loss            : HS / state-prep / relative-phase trace reduction  (matrix_utils.py:35-42)
//   best tracking   : strict <, pre-update parameters                   (optimization.py:70-73)
//   adjoint sweep   : walk the schedule backwards with inverse gates, O(1) memory; per gate
//                     accumulate Im<lambda|sigma_a|phi> (SURVEY.md Appendix B)
//   update phase    : gradients from the Pauli sums, penalty slope, optax Adam
//                     (optimization.py:14-25), then the next parameter phase.
//
// Data layout.  The n amplitude-index bits of a column are split into RB "register bits" (the
// low bits: 2^RB amplitudes of a column live in one thread's registers at compile-time indices)
// and LB = n - RB "lane bits" (the high bits select one of 2^LB lanes).  A gate on a register bit
// is a register-local butterfly (one unrolled code block per register bit); a gate on a lane bit
// exchanges the partner amplitudes with __shfl_xor_sync on a RUNTIME lane mask, so one code block
// serves every lane-bit qubit.  Keeping RB small keeps the unrolled code inside the SM's
// instruction cache: the first version of this kernel held whole columns in registers (RB = n)
// and ncu showed 58% of all stall cycles were instruction-fetch misses (profiles/r1_v0_*).
// With CPT = 2 two columns are packed in float2 registers and the gate arithmetic issues as packed
// FFMA2/FMUL2 (fma.rn.f32x2, sm_100+): the FP32 pipe saturates at half the issue slots, which
// leaves room for the SHFL/LDS/integer traffic.  The TPS = (2^n / CPT) * 2^LB threads of a sample
// sit in one warp; cross-column sums (loss trace, per-gate Pauli sums) are xor-butterflies.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "program.hpp"

namespace cpf {

enum Mode : int { M_ADAM = 0, M_LOSSGRAD = 1, M_UNITARY = 2, M_COTANGENT = 3 };

template <typename R>
struct PenaltyT {
  int kind, nseg;
  int sorted;   // segments ascending and disjoint (hi[s] <= lo[s + 1]; slots >= nseg hold +inf): binary search allowed
  R r, period;
  R lo[CPF_MAX_SEGMENTS], hi[CPF_MAX_SEGMENTS], slope[CPF_MAX_SEGMENTS], icpt[CPF_MAX_SEGMENTS];
};

template <typename R>
struct KParams {
  const uint32_t* dec; int n_sched;   // decoded schedule: 2 words per op (program.hpp)
  const uint16_t* red; int n_red;     // reduce tables: 8 offsets per group
  const Su2Meta* su2; int n_su2;
  const CpMeta* cp; int n_cp;
  const uint8_t* cp_pen;  // device [n_cp] or null: which CP params are penalised
  int P; long long B;
  int mode, loss_kind;
  const R* target_packed; int target_bytes;
  R lr, b1, b2, eps, omb1, omb2;
  long long step0; int nsteps;
  R* angles; R* m; R* v; const uint8_t* freeze;
  R* best_params; R* best_regloss; R* best_reg; R* init_regloss; R* init_reg;
  R* hist_params; R* hist_regloss; long long hist_len;
  R* loss_out; R* reg_out; R* grad_out;
  R* u_out; const R* cot;
  void* pk;         // heis_kernel: [B][pk_stride] lane-interleaved optimiser state {theta, m, v, best} (heis_impl.cuh: Pk4)
  R* aux;           // heis_kernel: [B][n_su2][4] half-angle cos/sin of the 2nd and 3rd fused rotations
  int coef_stride;  // R words per sample in shared memory
  int spb;          // heis_kernel: sample slots used per CTA
  int sync_sweeps;  // heis_kernel: CTA barrier at the start of the forward (bit 0) / backward (bit 1) sweep
  // heis_kernel, time-sliced Adam runs (heis_impl.cuh: launch_heis_sized): the launch covers positions
  // [ring_start, ring_end) of a ring that walks `ring_visits` times over the B samples; position c is sample c % B on
  // its visit c / B, i.e. its steps [step0 + visit * nsteps, + nsteps).  Unsliced: ring_start = 0, ring_end = B.
  long long ring_start, ring_end;
  int colmode;      // engine_kernel<SINGLE>, M_UNITARY: virtual sample b = (sample b / N, column b % N)
  int axp_surface, axp_block;   // heis_kernel: packed rotation axes shared by the surface / block gates
  int su2_all_params;           // heis_kernel: every rotation of every fused gate is a parameter (no constant angles)
  int unreferenced_params;      // heis_kernel: some parameters feed no gate
  int cp_all_params;            // heis_kernel: every entangler is a CP gate with a parameter (no CZ, no constant angle)
  int pk_stride;                // heis_kernel: words of R per sample in the packed optimiser state (heis_pk_stride)
  int last_slot[8];             // heis_kernel: slot of the last fused gate on each qubit
  PenaltyT<R> pen;
  // multi-target kernels (sweep types with MULTI_TARGET, engine_impl.cuh): device [B], sample b is scored against the
  // packed target target_index[b] of the table at target_packed (nothing is staged: target_bytes = 0)
  const int32_t* target_index;
  // isometry kernels (iso_impl.cuh): k input columns per sample, and the ancilla qubits as amplitude-index bits
  int iso_k, iso_amask;
  // subspace kernels (iso_impl.cuh: sweep types with INPUTS): the input states packed like the target ([iso_k][N]
  // complex, columns >= sub_k zero) and the caller's k, which normalises the loss.  Appended last, so the kernels
  // without inputs keep their parameter layout.
  const R* inputs_packed; int sub_k;
};

// ------------------------------------------------------------------------------------------
// packed-vector abstraction: V holds CPT lanes of R
// ------------------------------------------------------------------------------------------
template <typename R, int CPT> struct VT;
template <> struct VT<float, 1> {
  using V = float;
  static __device__ __forceinline__ V bc(float a) { return a; }
  static __device__ __forceinline__ V mul(V a, V b) { return a * b; }
  static __device__ __forceinline__ V fma(V a, V b, V c) { return fmaf(a, b, c); }
  static __device__ __forceinline__ V sub(V a, V b) { return a - b; }
  static __device__ __forceinline__ float hsum(V a) { return a; }
  static __device__ __forceinline__ float get(V a, int) { return a; }
  static __device__ __forceinline__ V onehot(int j, int col0) { return j == col0 ? 1.f : 0.f; }
  static __device__ __forceinline__ V make(float a, float) { return a; }
};
template <> struct VT<double, 1> {
  using V = double;
  static __device__ __forceinline__ V bc(double a) { return a; }
  static __device__ __forceinline__ V mul(V a, V b) { return a * b; }
  static __device__ __forceinline__ V fma(V a, V b, V c) { return ::fma(a, b, c); }
  static __device__ __forceinline__ V sub(V a, V b) { return a - b; }
  static __device__ __forceinline__ double hsum(V a) { return a; }
  static __device__ __forceinline__ double get(V a, int) { return a; }
  static __device__ __forceinline__ V onehot(int j, int col0) { return j == col0 ? 1.0 : 0.0; }
  static __device__ __forceinline__ V make(double a, double) { return a; }
};
template <> struct VT<float, 2> {
  using V = float2;
  static __device__ __forceinline__ V bc(float a) { return make_float2(a, a); }
  static __device__ __forceinline__ V mul(V a, V b) { return __fmul2_rn(a, b); }
  static __device__ __forceinline__ V fma(V a, V b, V c) { return __ffma2_rn(a, b, c); }
  static __device__ __forceinline__ V sub(V a, V b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }
  static __device__ __forceinline__ float hsum(V a) { return a.x + a.y; }
  static __device__ __forceinline__ float get(V a, int k) { return k ? a.y : a.x; }
  static __device__ __forceinline__ V onehot(int j, int col0) {
    return make_float2(j == col0 ? 1.f : 0.f, j == col0 + 1 ? 1.f : 0.f);
  }
  static __device__ __forceinline__ V make(float a, float b) { return make_float2(a, b); }
};

// ------------------------------------------------------------------------------------------
// scalar helpers
// ------------------------------------------------------------------------------------------
static __device__ __noinline__ void sincos_slow_f(float x, float* s, float* c) { sincosf(x, s, c); }

// sin/cos with Cody-Waite reduction and the Cephes single-precision kernels (~1 ulp), no
// local-memory slow path inlined.  XLA-class accuracy is required for 1e-5 parity.
template <typename R> struct SinCos { R s, c; };

static __device__ __noinline__ SinCos<float> sincos_nr(float x) {
  float s, c;
  if (fabsf(x) > 48000.f) { sincos_slow_f(x, &s, &c); return {s, c}; }
  float j = rintf(x * 0.636619747f);
  float r = fmaf(j, -1.57079601e+00f, x);
  r = fmaf(j, -3.13916473e-07f, r);
  r = fmaf(j, -5.39030253e-15f, r);
  int q = __float2int_rn(j);
  float r2 = r * r;
  float sp = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
  sp = fmaf(sp, r2, -1.6666654611e-1f);
  sp = fmaf(sp * r2, r, r);
  float cp = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
  cp = fmaf(cp, r2, 4.166664568298827e-2f);
  cp = fmaf(cp * r2, r2, fmaf(r2, -0.5f, 1.0f));
  float ss = (q & 1) ? cp : sp;
  float cc = (q & 1) ? sp : cp;
  s = (q & 2) ? -ss : ss;
  c = ((q + 1) & 2) ? -cc : cc;
  return {s, c};
}
static __device__ __noinline__ SinCos<double> sincos_nr(double x) {
  double s, c;
  sincos(x, &s, &c);
  return {s, c};
}
// out-of-line on purpose: the parameter phase must stay small so that the whole hot loop fits
// in the SM instruction cache.
__device__ __forceinline__ void sincos_r(float x, float& s, float& c) { auto r = sincos_nr(x); s = r.s; c = r.c; }
__device__ __forceinline__ void sincos_r(double x, double& s, double& c) { auto r = sincos_nr(x); s = r.s; c = r.c; }

// IEEE operations that must NOT be contracted into FMAs (optax/XLA evaluate the Adam update and
// the penalty line as separate multiplies and adds; the oracle does the same).
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float rsqrt_r(float a) { return rsqrtf(a); }
__device__ __forceinline__ double rsqrt_r(double a) { return 1.0 / sqrt(a); }
__device__ __forceinline__ float sqrt_r(float a) { return sqrtf(a); }
__device__ __forceinline__ double sqrt_r(double a) { return sqrt(a); }
// 1 - b^t (optax bias correction); float: exp2(t*log2 b), ~1e-7 relative like an f32 pow
// 1 - b^t (optax bias correction).  Not 1 - exp2(t log2 b): for b2 = 0.999 and the first steps that cancels to a
// relative error of 1e-4 (5e-5 on the step size; the first-step closed-form test saw it as a uniform 2.4e-6 offset
// of every parameter); -expm1(t log b) keeps 1e-7.
static __device__ __noinline__ float bias_corr(float b, float t) { return -expm1f(t * logf(b)); }
static __device__ __noinline__ double bias_corr(double b, double t) { return 1.0 - pow(b, t); }
__device__ __forceinline__ float fmod_r(float a, float b) { return fmodf(a, b); }
__device__ __forceinline__ double fmod_r(double a, double b) { return fmod(a, b); }
__device__ __forceinline__ float abs_r(float a) { return fabsf(a); }
__device__ __forceinline__ double abs_r(double a) { return fabs(a); }

template <typename R>
__device__ __forceinline__ R shfl_xor_r(R x, int m) { return __shfl_xor_sync(0xffffffffu, x, m); }

template <int TPS, typename R>
__device__ __forceinline__ R sample_sum(R x) {
#pragma unroll
  for (int m = TPS / 2; m >= 1; m >>= 1) x += shfl_xor_r(x, m);
  return x;
}

// jnp.mod semantics (result has the sign of the divisor; period > 0)
template <typename R>
static __device__ __noinline__ R pymod(R a, R period) {
  R r = fmod_r(a, period);
  if (r != R(0) && r < R(0)) r = add_rn(r, period);
  return r;
}

// penalty value and slope at angle a (penalty.py:44-76)
template <typename R>
__device__ __forceinline__ void penalty_eval(const PenaltyT<R>& pen, R a, R& val, R& slope) {
  val = R(0); slope = R(0);
  if (pen.kind == CPF_PEN_PIECEWISE) {
    R am = pymod(a, pen.period);
#pragma unroll 1
    for (int s = 0; s < pen.nseg; ++s) {
      if (pen.lo[s] < am && am <= pen.hi[s]) {
        val = add_rn(mul_rn(pen.slope[s], am), pen.icpt[s]);
        slope = pen.slope[s];
        break;
      }
    }
  } else if (pen.kind == CPF_PEN_L1) {
    val = abs_r(a);
    slope = a > R(0) ? R(1) : (a < R(0) ? R(-1) : R(0));
  }
}

// Same values as penalty_eval, shaped for the per-gate loops of heis_kernel: the common ranges of jnp.mod are
// handled inline (a in [0, p): a; [p, 2p): a - p exactly; (-p, 0): a + p rounded once, as the fmod route does),
// and the first-true-wins search over the (disjoint) segments runs branch-free from the last segment down.
template <typename R>
__device__ __forceinline__ void penalty_eval_fast(const PenaltyT<R>& pen, R a, R& val, R& slope) {
  val = R(0); slope = R(0);
  if (pen.kind == CPF_PEN_PIECEWISE) {
    const R per = pen.period;
    R am;
    if (a >= R(0) && a < per) am = a;
    else if (a >= per && a < per + per) am = a - per;
    else if (a < R(0) && a > -per) am = add_rn(a, per);
    else am = pymod(a, per);
    R sl = R(0), ic = R(0);
    bool found = false;
    if (pen.sorted) {
      // ascending disjoint segments (every table penalty.py builds): at most one matches, branch-free lower bound
      // over hi[] (16 slots, the unused ones +inf)
      static_assert(CPF_MAX_SEGMENTS == 16, "lower bound below is written for 16 slots");
      int s = pen.hi[7] < am ? 8 : 0;
      s += pen.hi[s + 3] < am ? 4 : 0;
      s += pen.hi[s + 1] < am ? 2 : 0;
      s += pen.hi[s] < am ? 1 : 0;
      found = pen.lo[s] < am && am <= pen.hi[s];
      sl = pen.slope[s]; ic = pen.icpt[s];
    } else {
#pragma unroll
      for (int s = CPF_MAX_SEGMENTS - 1; s >= 0; --s) {
        const bool in = s < pen.nseg && pen.lo[s] < am && am <= pen.hi[s];
        sl = in ? pen.slope[s] : sl;
        ic = in ? pen.icpt[s] : ic;
        found = found || in;
      }
    }
    if (found) { val = add_rn(mul_rn(sl, am), ic); slope = sl; }
  } else if (pen.kind == CPF_PEN_L1) {
    val = abs_r(a);
    slope = a > R(0) ? R(1) : (a < R(0) ? R(-1) : R(0));
  }
}

// optax 0.1.1 scale_by_adam + scale(-lr), one parameter (optimization.py:22-23); out of line
template <typename R> struct AdamOut { R th, mu, nu; };
template <typename R>
static __device__ __noinline__ AdamOut<R> adam_step(R g, R th, R mu, R nu, R b1, R omb1, R b2, R omb2,
                                                    R bc1, R bc2, R eps, R neg_lr) {
  mu = add_rn(mul_rn(omb1, g), mul_rn(b1, mu));
  nu = add_rn(mul_rn(omb2, mul_rn(g, g)), mul_rn(b2, nu));
  const R mu_hat = mu / bc1, nu_hat = nu / bc2;
  const R upd = mu_hat / add_rn(sqrt_r(nu_hat), eps);
  th = add_rn(th, mul_rn(neg_lr, upd));
  return {th, mu, nu};
}

// The same step inside the fused loops of the kernels.  double: the exact IEEE sequence above.  float: reciprocal bias
// corrections (ibc = 1 / bc, computed once per step), approximate sqrt and reciprocal (<= 2 ulp each) instead of three
// IEEE divisions and a square root per parameter (in the state-adjoint kernels these were 9 % of the time of a
// state-preparation run); the arithmetic of heis_impl.cuh: adam_inl.
__device__ __forceinline__ AdamOut<double> adam_step_fused(double g, double th, double mu, double nu, double b1, double omb1,
                                                           double b2, double omb2, double bc1, double bc2, double, double,
                                                           double eps, double neg_lr) {
  mu = add_rn(mul_rn(omb1, g), mul_rn(b1, mu));
  nu = add_rn(mul_rn(omb2, mul_rn(g, g)), mul_rn(b2, nu));
  const double mu_hat = mu / bc1, nu_hat = nu / bc2;
  th = add_rn(th, mul_rn(neg_lr, mu_hat / add_rn(sqrt(nu_hat), eps)));
  return {th, mu, nu};
}
__device__ __forceinline__ AdamOut<float> adam_step_fused(float g, float th, float mu, float nu, float b1, float omb1,
                                                          float b2, float omb2, float, float, float ibc1, float ibc2,
                                                          float eps, float neg_lr) {
  mu = add_rn(mul_rn(omb1, g), mul_rn(b1, mu));
  nu = add_rn(mul_rn(omb2, mul_rn(g, g)), mul_rn(b2, nu));
  const float mu_hat = mu * ibc1, nu_hat = nu * ibc2;
  float rt, iv;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rt) : "f"(nu_hat));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iv) : "f"(add_rn(rt, eps)));
  th = add_rn(th, mul_rn(neg_lr, mul_rn(mu_hat, iv)));
  return {th, mu, nu};
}

// rotate vector (x,y,z) by angle with cos C, sin S about coordinate axis `a` (right-handed):
// R_a(theta) sigma_b R_a(theta)^dagger = sum_c [Rot_a(theta)]_{cb} sigma_c
template <typename R>
__device__ __forceinline__ void rot_axis(int a, R C, R S, R& x, R& y, R& z) {
  if (a == 0) { R ny = C * y - S * z, nz = S * y + C * z; y = ny; z = nz; }
  else if (a == 1) { R nz = C * z - S * x, nx = S * z + C * x; z = nz; x = nx; }
  else if (a == 2) { R nx = C * x - S * y, ny = S * x + C * y; x = nx; y = ny; }
}

// SU(2) element (alpha, beta) of a rotation about axis a with half-angle cos c / sin s:
// [[alpha, -conj(beta)], [beta, conj(alpha)]]  (gates.py:22-35)
template <typename R>
__device__ __forceinline__ void su2_of(int a, R c, R s, R& ar, R& ai, R& br, R& bi) {
  ar = c; ai = R(0); br = R(0); bi = R(0);
  if (a == 0) bi = -s;        // Rx: beta = -i s
  else if (a == 1) br = s;    // Ry: beta = s
  else if (a == 2) ai = -s;   // Rz: alpha = c - i s
}

// (alpha, beta) <- (a2, b2) * (alpha, beta):  alpha = a2 a - conj(b2) b ; beta = b2 a + conj(a2) b
template <typename R>
__device__ __forceinline__ void su2_mul(R a2r, R a2i, R b2r, R b2i, R& ar, R& ai, R& br, R& bi) {
  const R nar = a2r * ar - a2i * ai - (b2r * br + b2i * bi);
  const R nai = a2r * ai + a2i * ar - (b2r * bi - b2i * br);
  const R nbr = b2r * ar - b2i * ai + (a2r * br + a2i * bi);
  const R nbi = b2r * ai + b2i * ar + (a2r * bi - a2i * br);
  ar = nar; ai = nai; br = nbr; bi = nbi;
}

// ------------------------------------------------------------------------------------------
// gate application on the register/lane-split columns
// ------------------------------------------------------------------------------------------
template <typename V> struct ShflV;
template <> struct ShflV<float> {
  static __device__ __forceinline__ float x(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
};
template <> struct ShflV<double> {
  static __device__ __forceinline__ double x(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
};
template <> struct ShflV<float2> {
  static __device__ __forceinline__ float2 x(float2 v, int m) {
    return make_float2(__shfl_xor_sync(0xffffffffu, v.x, m), __shfl_xor_sync(0xffffffffu, v.y, m));
  }
};

template <typename R, int RB, int CPT>
struct Cols {
  using T = VT<R, CPT>;
  using V = typename T::V;
  static constexpr int NA = 1 << RB;  // amplitudes of a column held by one thread

  // ---- register-bit butterfly: x' = alpha x - conj(beta) y ; y' = beta x + conj(alpha) y ----
  template <int BP>
  static __device__ __forceinline__ void su2_reg(V (&re)[NA], V (&im)[NA], R ar, R ai, R br, R bi) {
    constexpr int M = 1 << BP;
    const V Ar = T::bc(ar), Ai = T::bc(ai), nAi = T::bc(-ai);
    const V Br = T::bc(br), nBr = T::bc(-br), Bi = T::bc(bi), nBi = T::bc(-bi);
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if (j & M) continue;
      const V xr = re[j], xi = im[j], yr = re[j | M], yi = im[j | M];
      re[j] = T::fma(nBi, yi, T::fma(nBr, yr, T::fma(nAi, xi, T::mul(Ar, xr))));
      im[j] = T::fma(Bi, yr, T::fma(nBr, yi, T::fma(Ai, xr, T::mul(Ar, xi))));
      re[j | M] = T::fma(Ai, yi, T::fma(Ar, yr, T::fma(nBi, xi, T::mul(Br, xr))));
      im[j | M] = T::fma(nAi, yr, T::fma(Ar, yi, T::fma(Bi, xr, T::mul(Br, xi))));
    }
  }

  // Pauli sums S_a = Im <lam| sigma_a |phi> for a register bit
  template <int BP>
  static __device__ __forceinline__ void pauli_reg(const V (&pr)[NA], const V (&pi)[NA],
                                                   const V (&lr)[NA], const V (&li)[NA],
                                                   R& sx, R& sy, R& sz) {
    constexpr int M = 1 << BP;
    V xp = T::bc(R(0)), xn = xp, yp = xp, yn = xp, zp = xp, zn = xp;
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if (j & M) continue;
      const int k = j | M;
      zp = T::fma(lr[j], pi[j], zp); zn = T::fma(li[j], pr[j], zn);
      zp = T::fma(li[k], pr[k], zp); zn = T::fma(lr[k], pi[k], zn);
      xp = T::fma(lr[j], pi[k], xp); xn = T::fma(li[j], pr[k], xn);
      xp = T::fma(lr[k], pi[j], xp); xn = T::fma(li[k], pr[j], xn);
      yp = T::fma(lr[k], pr[j], yp); yn = T::fma(lr[j], pr[k], yn);
      yp = T::fma(li[k], pi[j], yp); yn = T::fma(li[j], pi[k], yn);
    }
    sx = T::hsum(T::sub(xp, xn));
    sy = T::hsum(T::sub(yp, yn));
    sz = T::hsum(T::sub(zp, zn));
  }

  // ---- lane-bit butterfly: new = A * mine + B * partner with per-lane (A, B) ----
  //   my bit 0: A = alpha,       B = -conj(beta)
  //   my bit 1: A = conj(alpha), B = beta
  static __device__ __forceinline__ void lane_coef(bool mybit, R ar, R ai, R br, R bi,
                                                   R& Ar, R& Ai, R& Br, R& Bi) {
    Ar = ar; Ai = mybit ? -ai : ai;
    Br = mybit ? br : -br; Bi = bi;
  }
  static __device__ __forceinline__ void mix(V (&re)[NA], V (&im)[NA], const V (&qr)[NA],
                                             const V (&qi)[NA], R Ar, R Ai, R Br, R Bi) {
    const V vAr = T::bc(Ar), vAi = T::bc(Ai), nAi = T::bc(-Ai);
    const V vBr = T::bc(Br), vBi = T::bc(Bi), nBi = T::bc(-Bi);
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const V mr = re[j], mi = im[j];
      re[j] = T::fma(nBi, qi[j], T::fma(vBr, qr[j], T::fma(nAi, mi, T::mul(vAr, mr))));
      im[j] = T::fma(vBi, qr[j], T::fma(vBr, qi[j], T::fma(vAi, mr, T::mul(vAr, mi))));
    }
  }
  static __device__ __forceinline__ void su2_lane(V (&re)[NA], V (&im)[NA], int lm, bool mybit,
                                                  R ar, R ai, R br, R bi) {
    V qr[NA], qi[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) { qr[j] = ShflV<V>::x(re[j], lm); qi[j] = ShflV<V>::x(im[j], lm); }
    R Ar, Ai, Br, Bi;
    lane_coef(mybit, ar, ai, br, bi, Ar, Ai, Br, Bi);
    mix(re, im, qr, qi, Ar, Ai, Br, Bi);
  }
  // adjoint step on a lane bit: Pauli sums (this lane's share) then the inverse butterfly on both
  // phi and lambda, sharing the partner exchange.
  static __device__ __forceinline__ void bwd_lane(V (&pr)[NA], V (&pi)[NA], V (&lr)[NA], V (&li)[NA],
                                                  int lm, bool mybit, bool want_sums, R ar, R ai,
                                                  R br, R bi, R& sx, R& sy, R& sz) {
    V qr[NA], qi[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) { qr[j] = ShflV<V>::x(pr[j], lm); qi[j] = ShflV<V>::x(pi[j], lm); }
    if (want_sums) {
      V xp = T::bc(R(0)), xn = xp, yp = xp, zp = xp, zn = xp;
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        zp = T::fma(lr[j], pi[j], zp); zn = T::fma(li[j], pr[j], zn);   // Im(conj(l) p), own
        xp = T::fma(lr[j], qi[j], xp); xn = T::fma(li[j], qr[j], xn);   // Im(conj(l) partner)
        yp = T::fma(lr[j], qr[j], yp); yp = T::fma(li[j], qi[j], yp);   // Re(conj(l) partner)
      }
      const R z = T::hsum(T::sub(zp, zn)), y = T::hsum(yp);
      sx = T::hsum(T::sub(xp, xn));
      sz = mybit ? -z : z;
      sy = mybit ? y : -y;
    }
    R Ar, Ai, Br, Bi;
    lane_coef(mybit, ar, -ai, -br, -bi, Ar, Ai, Br, Bi);   // inverse gate
    mix(pr, pi, qr, qi, Ar, Ai, Br, Bi);
#pragma unroll
    for (int j = 0; j < NA; ++j) { qr[j] = ShflV<V>::x(lr[j], lm); qi[j] = ShflV<V>::x(li[j], lm); }
    mix(lr, li, qr, qi, Ar, Ai, Br, Bi);
  }

  // ---- diagonal two-qubit phases: multiply amplitudes whose register bits RM are all set ----
  // (the lane-bit part of the |11> condition is folded into (c, s) by the caller: lanes that do not
  // satisfy it pass (1, 0))
  template <int RM>
  static __device__ __forceinline__ void phase(V (&re)[NA], V (&im)[NA], R c, R s) {
    const V C = T::bc(c), S = T::bc(s), nS = T::bc(-s);
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if ((j & RM) != RM) continue;
      const V xr = re[j], xi = im[j];
      re[j] = T::fma(nS, xi, T::mul(C, xr));
      im[j] = T::fma(S, xr, T::mul(C, xi));
    }
  }
  // rows whose bits SET are all set and whose bits CLR are all clear get the phase (c, s)
  template <int SET, int CLR>
  static __device__ __forceinline__ void phase_mask(V (&re)[NA], V (&im)[NA], R c, R s) {
    const V C = T::bc(c), S = T::bc(s), nS = T::bc(-s);
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if ((j & SET) != SET || (j & CLR) != 0) continue;
      const V xr = re[j], xi = im[j];
      re[j] = T::fma(nS, xi, T::mul(C, xr));
      im[j] = T::fma(S, xr, T::mul(C, xi));
    }
  }
  // real rotation Ry = [[c, -s], [s, c]] on a register bit: 4 FMA per amplitude
  template <int BP>
  static __device__ __forceinline__ void ry_reg(V (&re)[NA], V (&im)[NA], R c, R s) {
    constexpr int M = 1 << BP;
    const V C = T::bc(c), S = T::bc(s), nS = T::bc(-s);
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if (j & M) continue;
      const V xr = re[j], xi = im[j], yr = re[j | M], yi = im[j | M];
      re[j] = T::fma(nS, yr, T::mul(C, xr));
      im[j] = T::fma(nS, yi, T::mul(C, xi));
      re[j | M] = T::fma(C, yr, T::mul(S, xr));
      im[j | M] = T::fma(C, yi, T::mul(S, xi));
    }
  }
  // The same rotation by phi in [0, pi/2] (c = cos phi >= 0, s = sin phi >= 0) as three shears (lifting steps):
  // [[c, -s], [s, c]] = [[1, t], [0, 1]] [[1, 0], [s, 1]] [[1, t], [0, 1]] with t = -tan(phi/2) = -s / (1 + c)
  // in [-1, 0]: 3 FMA per amplitude, exactly orthogonal up to rounding, no scaling.
  template <int BP>
  static __device__ __forceinline__ void ry_lift(V (&re)[NA], V (&im)[NA], R t, R s) {
    constexpr int M = 1 << BP;
    const V Tt = T::bc(t), S = T::bc(s);
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if (j & M) continue;
      V xr = T::fma(Tt, re[j | M], re[j]), xi = T::fma(Tt, im[j | M], im[j]);
      const V yr = T::fma(S, xr, re[j | M]), yi = T::fma(S, xi, im[j | M]);
      re[j] = T::fma(Tt, yr, xr); im[j] = T::fma(Tt, yi, xi);
      re[j | M] = yr; im[j | M] = yi;
    }
  }
  // ---- CNOT on amplitude-index bit positions (cpos controls, tpos is flipped); `la` is this
  // thread's lane part of the amplitude index.  Used by 'cx' templates only. ----
  static __device__ __forceinline__ V selv(bool p, V a, V b) { return p ? a : b; }
  template <int BP>
  static __device__ __forceinline__ void cnot_reg(V (&re)[NA], V (&im)[NA], int cpos, int la) {
    constexpr int M = 1 << BP;
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if (j & M) continue;
      const bool c = ((((la << RB) | j) >> cpos) & 1) != 0;
      const V a = re[j], b = re[j | M], ai = im[j], bi = im[j | M];
      re[j] = selv(c, b, a); re[j | M] = selv(c, a, b);
      im[j] = selv(c, bi, ai); im[j | M] = selv(c, ai, bi);
    }
  }
  static __device__ __forceinline__ void cnot_lane(V (&re)[NA], V (&im)[NA], int cpos, int lm, int la) {
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const bool c = ((((la << RB) | j) >> cpos) & 1) != 0;
      const V qr = ShflV<V>::x(re[j], lm), qi = ShflV<V>::x(im[j], lm);
      re[j] = selv(c, qr, re[j]); im[j] = selv(c, qi, im[j]);
    }
  }
  template <int RM>
  static __device__ __forceinline__ R phase_sum(const V (&pr)[NA], const V (&pi)[NA],
                                                const V (&lr)[NA], const V (&li)[NA]) {
    V p = T::bc(R(0)), n = p;
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if ((j & RM) != RM) continue;
      p = T::fma(lr[j], pi[j], p); n = T::fma(li[j], pr[j], n);
    }
    return T::hsum(T::sub(p, n));
  }
};

// ---- compile-time dispatch over register bit positions / register masks ---------------------
#define CPF_BP_SWITCH(RB, bp, ...)                                             \
  switch (bp) {                                                                \
    case 0: if constexpr (RB > 0) { constexpr int BP = 0; __VA_ARGS__; } break; \
    case 1: if constexpr (RB > 1) { constexpr int BP = 1; __VA_ARGS__; } break; \
    case 2: if constexpr (RB > 2) { constexpr int BP = 2; __VA_ARGS__; } break; \
    case 3: if constexpr (RB > 3) { constexpr int BP = 3; __VA_ARGS__; } break; \
    case 4: if constexpr (RB > 4) { constexpr int BP = 4; __VA_ARGS__; } break; \
    default: break;                                                            \
  }
#define CPF_RM_CASE(RB, I, ...)                                                \
  case I: if constexpr (I < (1 << RB)) { constexpr int RM = I; __VA_ARGS__; } break;
// RM has at most two bits set (a two-qubit gate)
#define CPF_RM_SWITCH(RB, rm, ...)                                             \
  switch (rm) {                                                                \
    CPF_RM_CASE(RB, 0, __VA_ARGS__) CPF_RM_CASE(RB, 1, __VA_ARGS__) CPF_RM_CASE(RB, 2, __VA_ARGS__)    \
    CPF_RM_CASE(RB, 3, __VA_ARGS__) CPF_RM_CASE(RB, 4, __VA_ARGS__) CPF_RM_CASE(RB, 5, __VA_ARGS__)    \
    CPF_RM_CASE(RB, 6, __VA_ARGS__) CPF_RM_CASE(RB, 8, __VA_ARGS__) CPF_RM_CASE(RB, 9, __VA_ARGS__)    \
    CPF_RM_CASE(RB, 10, __VA_ARGS__) CPF_RM_CASE(RB, 12, __VA_ARGS__) CPF_RM_CASE(RB, 16, __VA_ARGS__) \
    CPF_RM_CASE(RB, 17, __VA_ARGS__) CPF_RM_CASE(RB, 18, __VA_ARGS__) CPF_RM_CASE(RB, 20, __VA_ARGS__) \
    CPF_RM_CASE(RB, 24, __VA_ARGS__)                                           \
    default: break;                                                            \
  }

// ------------------------------------------------------------------------------------------
// kernel configuration
// ------------------------------------------------------------------------------------------
template <typename R, int NQ, int RB, int CPT, bool SINGLE>
struct Cfg {
  static constexpr int N = 1 << NQ;
  static constexpr int LB = NQ - RB;
  static constexpr int NA = 1 << RB;
  static constexpr int COLS = SINGLE ? 1 : N;
  static constexpr int TPS = (COLS / CPT) << LB;     // threads per sample (<= 32)
#ifndef CPF_SINGLE_BLOCK
#define CPF_SINGLE_BLOCK 128
#endif
  static constexpr int BLOCK = SINGLE ? CPF_SINGLE_BLOCK : 128;
  static constexpr int SPB = BLOCK / TPS;            // samples per block
  static_assert(RB >= 0 && RB <= NQ, "bad register/lane split");
  static_assert(TPS >= 1 && TPS <= 32, "a sample must fit in one warp");
};

// per-sample coefficient storage (R words, program.hpp: coef_words): su2 gate g at [8g, 8g+8) =
//   {alpha_r, alpha_i, beta_r, beta_i, c2, s2, c3, s3}; the adjoint sweep overwrites the first
//   three words with the Pauli sums (Sx, Sy, Sz).  Phase gate k (CP or CZ) at [8*n_su2 + 4k, +4) =
//   {cos a, sin a, -, -}; word 0 is overwritten with the |11> sum.

// Sum 8 per-thread partials over the TPS lanes of a sample with a transposing butterfly: the first
// steps halve the number of live values (each lane sends the half its partner keeps), so 8 sums
// over 32 lanes cost 4+2+1+1+1 = 9 shuffles instead of 40.  Afterwards the lanes whose low
// (non-halving) bits are zero hold complete sums: lane bits (from the top) select the slot group.
// dst[slot] is the word offset in the sample's coefficient store (0xffff: unused).
template <int TPS> struct Red8 {
  static constexpr int LOG = TPS >= 32 ? 5 : TPS >= 16 ? 4 : TPS >= 8 ? 3 : TPS >= 4 ? 2 : TPS >= 2 ? 1 : 0;
  static constexpr int H = LOG < 3 ? LOG : 3;     // halving steps
  static constexpr int CNT = 8 >> H;              // values left per lane
};
// After the call acc[0..CNT) of the lanes with `writer` hold the complete sums of slots
// slot0 .. slot0+CNT-1.
template <int TPS, typename R>
__device__ __forceinline__ void reduce8(R (&acc)[8], int ls, int& slot0, bool& writer) {
  constexpr int H = Red8<TPS>::H, CNT = Red8<TPS>::CNT;
  slot0 = 0;
#pragma unroll
  for (int s = 0; s < H; ++s) {
    const int m = TPS >> (s + 1);
    const int cnt = 8 >> (s + 1);
    const bool up = (ls & m) != 0;
    if (up) slot0 += cnt;
#pragma unroll
    for (int k = 0; k < cnt; ++k) {
      const R send = up ? acc[k] : acc[k + cnt];
      const R keep = up ? acc[k + cnt] : acc[k];
      acc[k] = keep + shfl_xor_r(send, m);
    }
  }
#pragma unroll
  for (int m = (TPS >> H) / 2; m >= 1; m >>= 1) {
#pragma unroll
    for (int k = 0; k < CNT; ++k) acc[k] += shfl_xor_r(acc[k], m);
  }
  writer = (ls & ((TPS >> H) - 1)) == 0;
}
template <int TPS, typename R>
__device__ __forceinline__ void reduce8_store(R (&acc)[8], const uint16_t* dst, R* coef, int ls) {
  int slot0; bool writer;
  reduce8<TPS>(acc, ls, slot0, writer);
  if (writer) {
#pragma unroll
    for (int k = 0; k < Red8<TPS>::CNT; ++k) {
      const uint32_t o = dst[slot0 + k];
      if (o != 0xffffu) coef[o] = acc[k];
    }
  }
}

}  // namespace cpf
