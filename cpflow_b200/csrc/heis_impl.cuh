// Heisenberg-picture engine kernel for the HS loss on layered templates (the Synthesize.static()
// hot path: cost_HST of matrix_utils.py:35-42 over build_unitary of main.py:106-146).
//
// The adjoint sweep of engine_impl.cuh propagates two N x N complex states (phi, lambda) backwards:
// 22 FMA per amplitude and fused gate plus a cross-lane reduction for every gradient entry.  Here
// the backward sweep runs in the Heisenberg picture instead (tools/heisenberg_model.py is the numpy
// statement of the same math, checked against the oracle by tests/test_heisenberg_model.py):
//
//   forward   Y = U V^dag, started from V^dag (staged in shared memory by TMA) instead of the identity:
//             t = Tr(V^dag U) = Tr(Y), loss = 1 - |t|^2/N^2.  All n row bits of a column live in
//             registers (CPT = 2 columns packed in float2 -> FFMA2), so the forward sweep has no
//             shuffles at all: lane = column group.
//   pivot     dL/dtheta_k = Tr(H_k sigma) with H_k = Herm(s Z_k), s = i conj(t)/N^2,
//             Z_k = G_k..G_1 V^dag G_M..G_{k+1}, Z_M = Y.  H is Hermitian, so its Pauli coefficients
//             h[x, z] = Re(i^{|x&z|} s W[x,z]),  W[x,z] = sum_r (-1)^{|z&r|} Y[r, r^x]
//             are N^2 REAL numbers: one xor-shuffle all-to-all gathers the x-diagonals (lane = x >> PB)
//             and a register-local Walsh-Hadamard transform over r produces W.
//   backward  H_{k-1} = G_k^dag H_k G_k acts on h by real linear maps.  Every fused gate is used as
//             Rz(phi_out + pi/2) Rx(theta) Rz(phi_in - pi/2): Rx mixes (h_Y, h_Z) (2 FFMA2 + 1 SHFL per packed pair
//             when the qubit's x bit is a lane bit, the exchanged value is the raw register), Rz mixes
//             (h_X, h_Y) inside a lane (4 FFMA2); the Rz factors of consecutive gates on a qubit, the Rz halves of
//             CP(a) ~ Rz Rz exp(i a/4 ZZ) and the pending phases commute and are undone as ONE rotation per gate;
//             the ZZ part is a pair rotation by a/2 in lifting form (three shears).
//             Every gradient entry is ONE coefficient of h (X: h[b,0], Y: h[b,b], Z: h[0,b]; CP:
//             -(h[0,0]-h[0,b1]-h[0,b2]+h[0,b1|b2])/2): no reductions.
//
// Shared memory per sample: 8 words per fused gate + 3 per entangler + a staging area for the coefficients of
// ONE layer of the backward sweep (produced just in time from the forward data), see HEIS_SU2_WORDS below.
// Per sample and eval for C3 (n = 4, K = 40): ~4.9 k warp instructions (x 1/4 warp) instead of ~22 k.
#pragma once
#include <atomic>
#include <cmath>

#include "engine_impl.cuh"

namespace cpf {

// Shared-memory slot of a fused one-qubit gate, 8 words: ty, sy (lifting form of Ry: ty = -sy / (1 + cy)) | u_out |
// u_in (surface) / A (lower-qubit gate) / A B e^{ia} (higher-qubit gate) | B (lower-qubit gate) / r * penalty
// slope of the block's entangler (higher-qubit gate, word 6).  The backward sweep overwrites words 0, 1, 4 with the
// gradient sums (S_X, S_Y, S_Z); u_out stays (the parameter phase needs it to bring the sums back to the gate's
// output frame).  The coefficients of the backward sweep are NOT kept per gate: they are produced one layer at a
// time in a staging area (HEIS_STAGE_WORDS per gate of a layer), which keeps the per-sample footprint small enough
// for 64 resident samples (16 warps) per SM on C3.
constexpr int HEIS_SU2_WORDS = 8;
// Staged coefficients of a gate of the backward sweep (Z-X-Z form, see backward()), 8 words: two rows
// (cos theta, -+sin theta, cos zeta | 1, sin zeta | 0): row 0 for lanes that hold (I, Z) of the gate's qubit, row 1
// for lanes that hold (X, Y).  A lane picks its row by address: no selects.
constexpr int HEIS_STAGE_WORDS = 8;
constexpr int HEIS_CP_WORDS = 3;     // cos(a/2) >= 0, sin(a/2), -tan(a/4); word 0 <- dL/da after the backward sweep

inline int heis_coef_stride(int n_su2, int n_cp, int n_stage) {
  int w = (HEIS_SU2_WORDS * n_su2 + HEIS_CP_WORDS * n_cp + HEIS_STAGE_WORDS * n_stage + 3) & ~3;
  if (w == 0) w = 4;
  if (((w / 4) & 1) == 0) w += 4;   // odd number of 16-byte groups: samples of a warp hit distinct banks
  return w;
}
template <typename R> inline int heis_target_words(int n, int cpt) {
  const int N = 1 << n;
  return (N / cpt) * (N + 1) * 2 * cpt;
}

// Gate metadata as the kernel reads it, staged in shared memory by the prologue (the global-memory records of
// program.hpp sat on the critical path of every gate update: a dependent L2 round trip before the load of the
// packed state).  Constant angles (pidx < 0) stay in the global records.
struct __align__(8) HSu2 { int16_t pidx[3]; uint16_t axes; };                   // axes: 4 bits per rotation, 15 = unused
struct __align__(8) HCp { int16_t pidx; uint16_t flags; int16_t prev_lo, prev_hi; };   // flags: 1 penalised, 2 CZ, bits [4,7) lower qubit, [8,11) higher qubit
__host__ __device__ inline int heis_meta_bytes(int n_su2, int n_cp) { return (8 * (n_su2 + n_cp) + 15) & ~15; }

template <typename R, int NQ, int CPT>
struct HCfg {
  static constexpr int N = 1 << NQ;
  static constexpr int PB = CPT == 2 ? 1 : 0;   // x bits of a thread held in registers
  static constexpr int XR = 1 << PB;
  static constexpr int TPS = N / CPT;           // threads per sample
  // forward state registers: 2 * N * CPT words (x2 for double) -> register cap 128 (512 threads) or 255 (256)
#ifndef CPF_F64_MAXT
#define CPF_F64_MAXT 512
#endif
  static constexpr int MAXT = 2 * N * CPT * (int)(sizeof(R) / 4) <= 64 ? (sizeof(R) == 8 && NQ >= 4 ? CPF_F64_MAXT : 512) : 256;
  static_assert(TPS >= 1 && TPS <= 32, "a sample must fit in one warp");
};

// A CTA barrier at the start of each sweep keeps the warps of a CTA on the same instruction-cache lines (a barrier
// per layer, the first design, cost 7 %; none at all 20 %).  fwd / bwd: barrier before the forward / backward sweep.
struct LayerBar {
  bool fwd, bwd;
};

// Store to shared memory under a predicate, without a branch (the compiler turns `if (lane == k) s[i] = v`
// into BSSY / BRA / BSYNC sequences inside the sweeps).
__device__ __forceinline__ void sts_if(bool on, float* q, float v) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %0, 0; @p st.shared.f32 [%1], %2; }" ::"r"((int)on),
               "r"((unsigned)__cvta_generic_to_shared(q)), "f"(v) : "memory");
}
__device__ __forceinline__ void sts_if(bool on, double* q, double v) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %0, 0; @p st.shared.f64 [%1], %2; }" ::"r"((int)on),
               "r"((unsigned)__cvta_generic_to_shared(q)), "d"(v) : "memory");
}

// two adjacent words in one predicated store (q 8 / 16 bytes aligned): two predicated scalar stores under the same
// predicate come out of ptxas as a BSSY / BRA / BSYNC region
__device__ __forceinline__ void sts2_if(bool on, float* q, float v0, float v1) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %0, 0; @p st.shared.v2.f32 [%1], {%2, %3}; }" ::"r"((int)on),
               "r"((unsigned)__cvta_generic_to_shared(q)), "f"(v0), "f"(v1) : "memory");
}
__device__ __forceinline__ void sts2_if(bool on, double* q, double v0, double v1) {
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %0, 0; @p st.shared.v2.f64 [%1], {%2, %3}; }" ::"r"((int)on),
               "r"((unsigned)__cvta_generic_to_shared(q)), "d"(v0), "d"(v1) : "memory");
}

template <typename V> struct AddV;
template <> struct AddV<float> { static __device__ __forceinline__ float add(float a, float b) { return a + b; }
                                 static __device__ __forceinline__ float sub(float a, float b) { return a - b; } };
template <> struct AddV<double> { static __device__ __forceinline__ double add(double a, double b) { return a + b; }
                                  static __device__ __forceinline__ double sub(double a, double b) { return a - b; } };
template <> struct AddV<float2> {
  static __device__ __forceinline__ float2 add(float2 a, float2 b) { return __fadd2_rn(a, b); }
  static __device__ __forceinline__ float2 sub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
};

// Layered template (same slot order as LayerSweep, program.cpp: detect_layered): surface SU2 of qubit q
// in slot q; block k = phase gate k on the qubit pair of position k % NBL, SU2 of the pair's lower
// qubit in slot NQ + 2k, of its higher qubit in slot NQ + 2k + 1.
template <typename R, int NQ, int CPT, int NBL, unsigned long long LOQ, unsigned long long HIQ>
struct HeisSweep {
  using CO = Cols<R, NQ, CPT>;
  using T = VT<R, CPT>;
  using V = typename T::V;
  static constexpr int N = 1 << NQ, PB = CPT == 2 ? 1 : 0, XR = 1 << PB, TPS = N / CPT;
  static constexpr int SW = HEIS_SU2_WORDS, CW = HEIS_CP_WORDS, STW = HEIS_STAGE_WORDS;
  static constexpr int NSTAGE = 2 * NBL > NQ ? 2 * NBL : NQ;   // gates staged at a time (one layer / the surface)
  static __host__ __device__ constexpr int lo_q(int j) { return (int)((LOQ >> (4 * j)) & 15); }
  static __host__ __device__ constexpr int hi_q(int j) { return (int)((HIQ >> (4 * j)) & 15); }

  // ------------------------------- forward: row operations on Y -------------------------------
  // Every fused gate is used in ZYZ form G ~ diag(1, u_out) Ry diag(1, u_in) (global phase dropped: the HS
  // loss and the Hermitian part that seeds the backward sweep do not see it).  u_in merges with the block's
  // CP phase and with the u_out still pending on the same qubits into one diagonal (1, B, A, A B e^{ia}),
  // prepared by the parameter phase: a block costs 3 + 4 + 4 = 11 FMA per amplitude instead of 1 + 8 + 8.
  // Slot words during the forward sweep: 0 ty = -sy / (1 + cy); 1 sy; [2,4) u_out; lower-qubit slot [4,8) A, B;
  // higher-qubit slot [4,6) A B e^{ia}; surface slots [4,6) u_in.
  template <int BP>
  static __device__ __forceinline__ void ry_fwd(V (&yr)[N], V (&yi)[N], const R* cf) {
    CO::template ry_lift<BP>(yr, yi, cf[0], cf[1]);
  }
  template <int Q>
  static __device__ __forceinline__ void surface_fwd(V (&yr)[N], V (&yi)[N], const R* coef) {
    if constexpr (Q < NQ) {
      constexpr int BP = NQ - 1 - Q;
      CO::template phase_mask<(1 << BP), 0>(yr, yi, coef[SW * Q + 4], coef[SW * Q + 5]);
      ry_fwd<BP>(yr, yi, coef + SW * Q);
      surface_fwd<Q + 1>(yr, yi, coef);
    }
  }
  template <int Q>
  static __device__ __forceinline__ void tail_fwd(const KParams<R>& p, V (&yr)[N], V (&yi)[N], const R* coef) {
    if constexpr (Q < NQ) {
      const R* cf = coef + SW * p.last_slot[Q];
      CO::template phase_mask<(1 << (NQ - 1 - Q)), 0>(yr, yi, cf[2], cf[3]);
      tail_fwd<Q + 1>(p, yr, yi, coef);
    }
  }
  // one block on amplitude bits PA (lower qubit) / PC (higher qubit); cl: slot of the lower-qubit gate
  template <int PA, int PC>
  static __device__ __forceinline__ void block_fwd(const R* cl, V (&yr)[N], V (&yi)[N]) {
    const R* ch = cl + SW;
    R ar, ai, br, bi;
    Vec4Load<R>::ld(cl + 4, ar, ai, br, bi);
    CO::template phase_mask<(1 << PA), (1 << PC)>(yr, yi, ar, ai);
    CO::template phase_mask<(1 << PC), (1 << PA)>(yr, yi, br, bi);
    CO::template phase_mask<(1 << PA) | (1 << PC), 0>(yr, yi, ch[4], ch[5]);
    ry_fwd<PA>(yr, yi, cl);
    ry_fwd<PC>(yr, yi, ch);
  }
  // CHECKED: the (one) partial layer at the end of the template; full layers run without the per-block tests (an
  // early exit after every block costs a compare, a branch and ~8 register moves that bring the state back to the
  // loop's register assignment)
  template <int J, bool CHECKED>
  static __device__ __forceinline__ void blocks_fwd(int k0, int K, const R* cs, V (&yr)[N], V (&yi)[N]) {
    if constexpr (J < NBL) {
      if (CHECKED && k0 + J >= K) return;
      block_fwd<NQ - 1 - lo_q(J), NQ - 1 - hi_q(J)>(cs + 2 * SW * J, yr, yi);
      blocks_fwd<J + 1, CHECKED>(k0, K, cs, yr, yi);
    }
  }
  static __device__ __forceinline__ void forward(const KParams<R>& p, const LayerBar lb, const HCp*, const R* coef,
                                                 V (&yr)[N], V (&yi)[N]) {
    surface_fwd<0>(yr, yi, coef);
    const int K = p.n_cp;
    const R* cs = coef + SW * NQ;
    if (lb.fwd) __syncthreads();
    int k0 = 0;
#pragma unroll 1
    for (; k0 + NBL <= K; k0 += NBL) {
      blocks_fwd<0, false>(k0, K, cs, yr, yi);
      cs += 2 * SW * NBL;
    }
    if (k0 < K) blocks_fwd<0, true>(k0, K, cs, yr, yi);
    tail_fwd<0>(p, yr, yi, coef);
  }

  // ------------------ pivot: gather the x-diagonals, Walsh-Hadamard transform over r ------------------
  // Before: lane l holds Y[r, l*CPT + k] (k = packed component).  Round d: every lane exchanges its rows
  // r >> PB == d with lane l ^ d, in place.  After: lane m holds, in slot r, Y[r, ((m ^ (r>>PB)) << PB) | k],
  // i.e. the element of diagonal x = (m << PB) | (k ^ (r & PB-bit)) at row r.
  static __device__ __forceinline__ void gather_wht(V (&yr)[N], V (&yi)[N]) {
#pragma unroll
    for (int d = 1; d < TPS; ++d) {
#pragma unroll
      for (int r0 = 0; r0 < CPT; ++r0) {
        const int r = d * CPT + r0;
        yr[r] = ShflV<V>::x(yr[r], d);
        yi[r] = ShflV<V>::x(yi[r], d);
      }
    }
    if constexpr (CPT == 2) {
      // butterfly over row bit 0: slot r0 = 0 holds (x0 = 0, x0 = 1), slot r0 = 1 holds (x0 = 1, x0 = 0)
#pragma unroll
      for (int r = 0; r < N; r += 2) {
        const V ur = yr[r], wr = yr[r + 1], ui = yi[r], wi = yi[r + 1];
        yr[r] = T::make(ur.x + wr.y, ur.y + wr.x); yr[r + 1] = T::make(ur.x - wr.y, ur.y - wr.x);
        yi[r] = T::make(ui.x + wi.y, ui.y + wi.x); yi[r + 1] = T::make(ui.x - wi.y, ui.y - wi.x);
      }
    }
#pragma unroll
    for (int j = PB; j < NQ; ++j) {
#pragma unroll
      for (int r = 0; r < N; ++r) {
        if (r & (1 << j)) continue;
        const V ar = yr[r], br = yr[r | (1 << j)], ai = yi[r], bi = yi[r | (1 << j)];
        yr[r] = AddV<V>::add(ar, br); yr[r | (1 << j)] = AddV<V>::sub(ar, br);
        yi[r] = AddV<V>::add(ai, bi); yi[r | (1 << j)] = AddV<V>::sub(ai, bi);
      }
    }
  }

  // ------------------------------- backward: real maps on h -------------------------------
  // h[xr][z] is held packed over xr: hv[z] = (h[0][z], h[1][z]) for CPT = 2 (scalar for CPT = 1), so every map
  // whose coefficients do not depend on xr issues as FFMA2; only gates on amplitude bit 0 (x bit = xr) are scalar.
  //
  // Z-X-Z form with merged Rz factors (tools/heisenberg_model.py: grad_hs_zxz).  G ~ Rz(phi_out) Ry(theta) Rz(phi_in)
  // = Rz(phi_out + pi/2) Rx(theta) Rz(phi_in - pi/2).  Rx mixes (Y, Z): for a lane-bit qubit both sit in register
  // slot z | BM of the two paired lanes, so the exchange is the raw register (no send computation): 2 FMA + SHFL per
  // packed pair; Rz mixes (X, Y), which one lane holds: 4 FMA.  Everything between the Rx of consecutive gates on
  // a qubit is Z-type and commutes, so a gate's outgoing Rz is undone together with the incoming Rz of the NEXT
  // gate on that qubit: per gate, undo Rx(theta), then Rz(zeta) with e^{i zeta} = (A or B of the forward sweep's
  // merged diagonal) e^{i a/2}.  6 instead of 8 packed instructions per pair, and nothing to select.
  // cf: the gate's staged rows; words 0, 1, 4 of the gate's slot sl receive (S_X, S_Y, S_Z) = entries of h in the
  // frame where the gate's own Rz(phi_out + pi/2) is already undone (the parameter phase rotates them back).
  template <int B>
  static __device__ __forceinline__ void su2_bwd(V (&hv)[N], const R* cf, R* sl, int m) {
    constexpr int BM = 1 << B;
    if constexpr (B < PB) {
      const bool own = m == 0;
      sts2_if(own, sl, T::get(hv[0], 1), T::get(hv[BM], 1)); sts_if(own, sl + 4, T::get(hv[BM], 0));
      // x bit = xr: I = h[0][z], Z = h[0][z|1], X = h[1][z], Y = h[1][z|1]
      R ct, st, cz, sz;
      Vec4Load<R>::ld(cf + 4, ct, st, cz, sz);
      // (scalar on purpose: Rx mixes the two halves of hv[z | BM] = (Z, Y); the packed form ct (Z, Y) + (-st, st) (Y, Z)
      // was measured: the same FMA-pipe time, plus two register moves per pair for the swapped operand)
#pragma unroll
      for (int z = 0; z < N; ++z) {
        if (z & BM) continue;
        const R X = T::get(hv[z], 1), Y = T::get(hv[z | BM], 1), Z = T::get(hv[z | BM], 0);
        const R Y1 = ct * Y + st * Z;
        hv[z] = T::make(T::get(hv[z], 0), cz * X + sz * Y1);
        hv[z | BM] = T::make(ct * Z - st * Y, cz * Y1 - sz * X);
      }
    } else {
      // x bit is lane bit J: lanes with the bit clear hold (I, Z), lanes with it set hold (X, Y)
      constexpr int J = B - PB;
      const bool mb = ((m >> J) & 1) != 0;
      const bool own = m == (1 << J);
      sts2_if(own, sl, T::get(hv[0], 0), T::get(hv[BM], 0));
      sts_if(m == 0, sl + 4, T::get(hv[BM], 0));
      R ct, st, cz, sz;
      Vec4Load<R>::ld(cf + (mb ? 4 : 0), ct, st, cz, sz);
      const V kct = T::bc(ct), kst = T::bc(st), kcz = T::bc(cz), ksz = T::bc(sz), knz = T::bc(-sz);
#pragma unroll
      for (int z = 0; z < N; ++z) {
        if (z & BM) continue;
        const V recv = ShflV<V>::x(hv[z | BM], 1 << J);
        const V e1 = T::fma(kst, recv, T::mul(kct, hv[z | BM]));   // (X, Y) lanes: Y' = ct Y + st Z; (I, Z): Z' = ct Z - st Y
        const V e0 = hv[z];
        hv[z] = T::fma(ksz, e1, T::mul(kcz, e0));                  // X' = cz X + sz Y'      (identity on (I, Z) lanes)
        hv[z | BM] = T::fma(knz, e0, T::mul(kcz, e1));             // Y'' = cz Y' - sz X
      }
    }
  }
  // Rz alone (the outgoing Rz of the last gate on a qubit, undone before the sweep starts): (X, Y) -> (c X + s Y, c Y - s X)
  template <int B>
  static __device__ __forceinline__ void rz_bwd(V (&hv)[N], R c, R s, int m) {
    constexpr int BM = 1 << B;
    if constexpr (B < PB) {
#pragma unroll
      for (int z = 0; z < N; ++z) {
        if (z & BM) continue;
        const R X = T::get(hv[z], 1), Y = T::get(hv[z | BM], 1);
        hv[z] = T::make(T::get(hv[z], 0), c * X + s * Y);
        hv[z | BM] = T::make(T::get(hv[z | BM], 0), c * Y - s * X);
      }
    } else {
      const bool mb = ((m >> (B - PB)) & 1) != 0;
      const V kc = T::bc(mb ? c : R(1)), ks = T::bc(mb ? s : R(0)), kn = T::bc(mb ? -s : R(0));
#pragma unroll
      for (int z = 0; z < N; ++z) {
        if (z & BM) continue;
        const V e0 = hv[z], e1 = hv[z | BM];
        hv[z] = T::fma(ks, e1, T::mul(kc, e0));
        hv[z | BM] = T::fma(kn, e0, T::mul(kc, e1));
      }
    }
  }

  // x bit of amplitude bit B (B >= PB) for this lane
  template <int B>
  static __device__ __forceinline__ bool xlane(int m) { return ((m >> (B - PB)) & 1) != 0; }

  // Entangler of a block on amplitude bits (B1, B2).  CP(a) ~ Rz_1(a/2) Rz_2(a/2) exp(i (a/4) Z1 Z2): the two Rz
  // join the merged Rz rotation of the block's fused gates (stage_layer: zeta), what remains rotates,
  // for coefficients whose x bits on the two qubits differ, the pairs (e00, e11) and (e01, e10) of every
  // (z1, z2) quad by a/2.  cf: cos(a/2), sin(a/2); word 0 receives dL/da = -(h_II - h_ZI - h_IZ + h_ZZ)/2
  // (Z-type coefficients: they do not see the Rz shuffle).
  // Both pair rotations in lifting form (three shears each: 6 instead of 8 FMA-pipe instructions per quad): the
  // parameter phase keeps cos(a/2) >= 0 (CP(a) = CP(a - 2 pi)), so t = -tan(a/4) = -s / (1 + c) lies in [-1, 1].
  template <typename E>
  static __device__ __forceinline__ void zz_quad(E& e00, E& e01, E& e10, E& e11, E tl, E sl, E t2, E s2) {
    using O = VT<R, sizeof(E) == sizeof(R) ? 1 : 2>;
    E a = O::fma(tl, e11, e00), b = O::fma(t2, e10, e01);
    e11 = O::fma(sl, a, e11); e10 = O::fma(s2, b, e10);
    e00 = O::fma(tl, e11, a); e01 = O::fma(t2, e10, b);
  }
  template <int B1, int B2>
  static __device__ __forceinline__ void phase_bwd(V (&hv)[N], R* cf, int m) {
    constexpr int M1 = 1 << B1, M2 = 1 << B2;
    const R s = cf[1], t = cf[2];
    const R g11 = R(-0.5) * ((T::get(hv[0], 0) - T::get(hv[M1], 0)) - (T::get(hv[M2], 0) - T::get(hv[M1 | M2], 0)));
    __syncwarp();
    sts_if(m == 0, cf, g11);
    if constexpr (B1 >= PB && B2 >= PB) {
      // both x bits are lane bits: one case per lane, packed arithmetic over xr
      const bool x1 = xlane<B1>(m), x2 = xlane<B2>(m), on = x1 != x2;
      const V tl = T::bc(on ? t : R(0)), sl = T::bc(on ? s : R(0));
      const V t2 = T::bc(on ? (x1 ? t : -t) : R(0)), s2 = T::bc(on ? (x1 ? s : -s) : R(0));
#pragma unroll
      for (int z = 0; z < N; ++z) {
        if (z & (M1 | M2)) continue;
        zz_quad<V>(hv[z], hv[z | M2], hv[z | M1], hv[z | M1 | M2], tl, sl, t2, s2);
      }
    } else {
      // one of the bits is amplitude bit 0, whose x bit is the packed component xr: scalar per component
      constexpr int BL = B1 >= PB ? B1 : B2;          // the lane bit
      const bool xl = xlane<BL>(m);
      // packed over xr with per-component coefficients (the two components differ in x1 or x2)
      R tl[XR], sl[XR], t2[XR], s2[XR];
#pragma unroll
      for (int xr = 0; xr < XR; ++xr) {
        const bool x1 = B1 >= PB ? xl : xr != 0, x2 = B2 >= PB ? xl : xr != 0, on = x1 != x2;
        tl[xr] = on ? t : R(0); sl[xr] = on ? s : R(0);
        t2[xr] = on ? (x1 ? t : -t) : R(0); s2[xr] = on ? (x1 ? s : -s) : R(0);
      }
      const V vtl = T::make(tl[0], tl[XR - 1]), vsl = T::make(sl[0], sl[XR - 1]);
      const V vt2 = T::make(t2[0], t2[XR - 1]), vs2 = T::make(s2[0], s2[XR - 1]);
#pragma unroll
      for (int z = 0; z < N; ++z) {
        if (z & (M1 | M2)) continue;
        zz_quad<V>(hv[z], hv[z | M2], hv[z | M1], hv[z | M1 | M2], vtl, vsl, vt2, vs2);
      }
    }
  }

  // one block of the backward sweep; st: staged rows of the block's two gates (lower, higher), cl: slot of the
  // lower-qubit gate, cph: the entangler's words
  template <int PA, int PC>
  static __device__ __forceinline__ void block_bwd(V (&h)[N], const R* st, R* cl, R* cph, int m) {
    su2_bwd<PC>(h, st + STW, cl + SW, m);
    su2_bwd<PA>(h, st, cl, m);
    phase_bwd<PA, PC>(h, cph, m);
  }
  template <int J, bool CHECKED>
  static __device__ __forceinline__ void blocks_bwd(int k0, int K, R* cs, const R* stage, R* cph, int m, V (&h)[N]) {
    if constexpr (J >= 0) {
      if (!CHECKED || k0 + J < K)
        block_bwd<NQ - 1 - lo_q(J), NQ - 1 - hi_q(J)>(h, stage + STW * (2 * J), cs + 2 * SW * J, cph + CW * J, m);
      blocks_bwd<J - 1, CHECKED>(k0, K, cs, stage, cph, m, h);
    }
  }
  template <int Q>
  static __device__ __forceinline__ void surface_bwd(R* coef, const R* stage, int m, V (&h)[N]) {
    if constexpr (Q >= 0) {
      su2_bwd<NQ - 1 - Q>(h, stage + STW * Q, coef + SW * Q, m);
      surface_bwd<Q - 1>(coef, stage, m, h);
    }
  }
  // Staged rows of one gate: Rx angle from the forward data (cos phi = 1 + ty sy, theta = 2 phi), Rz angle zeta.
  static __device__ __forceinline__ void stage_gate(R* st, R ty, R sy, R cz, R sz) {
    const R cy = R(1) + ty * sy;   // 1 - tan(phi/2) sin phi = cos phi
    const R ct = cy * cy - sy * sy, sth = R(2) * cy * sy;
    Vec4Load<R>::st(st, ct, -sth, R(1), R(0));
    Vec4Load<R>::st(st + 4, ct, sth, cz, sz);
  }
  // Staging of one layer (blocks k0 .. k0 + NBL - 1): the sample's lanes split the layer's 2 NBL fused gates.
  // e^{i zeta} = d e^{i a/2}, d = A (lower-qubit gate) / B (higher-qubit gate) of the forward sweep's merged diagonal.
  static __device__ __forceinline__ void stage_layer(int k0, int K, const R* coef, const R* cph0, R* stage, int m,
                                                     int group = NBL) {
    const int nb = K - k0 < group ? K - k0 : group;
#pragma unroll 1
    for (int j = m; j < 2 * nb; j += TPS) {
      const int k = k0 + (j >> 1), hi = j & 1;
      const R* cl = coef + SW * (NQ + 2 * k);
      const R* cf = cl + SW * hi;
      const R* cc = cph0 + CW * k;
      const R dr = cl[4 + 2 * hi], di = cl[5 + 2 * hi];
      const R ch = cc[0], sh = cc[1];
      stage_gate(stage + STW * j, cf[0], cf[1], dr * ch - di * sh, dr * sh + di * ch);
    }
  }
  // surface gates: zeta = phi_in - pi/2
  static __device__ __forceinline__ void stage_surface(const R* coef, R* stage, int m) {
#pragma unroll 1
    for (int q = m; q < NQ; q += TPS) {
      const R* cf = coef + SW * q;
      stage_gate(stage + STW * q, cf[0], cf[1], cf[5], -cf[4]);
    }
  }
  template <int Q>
  static __device__ __forceinline__ void tail_bwd(const KParams<R>& p, const R* coef, int m, V (&h)[N]) {
    if constexpr (Q < NQ) {
      const R* cf = coef + SW * p.last_slot[Q];
      rz_bwd<NQ - 1 - Q>(h, -cf[3], cf[2], m);     // Rz(phi_out + pi/2): e^{i w} = i u_out
      tail_bwd<Q + 1>(p, coef, m, h);
    }
  }
  static __device__ __forceinline__ void backward(const KParams<R>& p, const LayerBar lb, const HCp*, R* coef, R* stage,
                                                  R* cph0, int m, V (&h)[N]) {
    const int K = p.n_cp;
    if (lb.bwd) __syncthreads();
    tail_bwd<0>(p, coef, m, h);
    int k0 = (K / NBL) * NBL;          // first block of the partial layer, if there is one
    if (k0 < K) {
      stage_layer(k0, K, coef, cph0, stage, m);
      __syncwarp();
      blocks_bwd<NBL - 1, true>(k0, K, coef + SW * NQ + 2 * SW * k0, stage, cph0 + CW * k0, m, h);
      __syncwarp();
    }
#pragma unroll 1
    for (k0 -= NBL; k0 >= 0; k0 -= NBL) {
      stage_layer(k0, K, coef, cph0, stage, m);
      __syncwarp();
      blocks_bwd<NBL - 1, false>(k0, K, coef + SW * NQ + 2 * SW * k0, stage, cph0 + CW * k0, m, h);
      __syncwarp();
    }
    stage_surface(coef, stage, m);
    __syncwarp();
    surface_bwd<NQ - 1>(coef, stage, m, h);
  }
};

// The same sweeps for ANY block-structured template (topology.py:7-20 allows every `layer`; the paper's kite and
// square Toffoli-4 layers, twisted placements, non-periodic free blocks): the qubit pair of a block is read from the
// shared-memory gate metadata and dispatched by one uniform switch per block into the compile-time-pair code above
// (n (n - 1) / 2 variants).  All warps of a CTA take the same case, so the instruction-cache footprint per layer is
// what the compile-time-layer kernels have; the cost is the branch and the lost scheduling across block boundaries.
#define CPF_PAIR_LIST(X) X(0, 1) X(0, 2) X(0, 3) X(0, 4) X(1, 2) X(1, 3) X(1, 4) X(2, 3) X(2, 4) X(3, 4)
template <typename R, int NQ, int CPT>
struct HeisSweepAny : HeisSweep<R, NQ, CPT, 1, 0x0ull, 0x1ull> {
  using Base = HeisSweep<R, NQ, CPT, 1, 0x0ull, 0x1ull>;
  using V = typename Base::V;
  static constexpr int N = Base::N, SW = Base::SW, CW = Base::CW, STW = Base::STW, TPS = Base::TPS;
  static constexpr int GROUP = 4;                                   // blocks staged at a time (backward sweep)
  static constexpr int NSTAGE = 2 * GROUP > NQ ? 2 * GROUP : NQ;
  static __device__ __forceinline__ int pair_code(const HCp& md) { return ((md.flags >> 4) & 7) * 8 + ((md.flags >> 8) & 7); }

  static __device__ __forceinline__ void forward(const KParams<R>& p, const LayerBar lb, const HCp* s_cp, const R* coef,
                                                 V (&yr)[N], V (&yi)[N]) {
    Base::template surface_fwd<0>(yr, yi, coef);
    const int K = p.n_cp;
    const R* cs = coef + SW * NQ;
    if (lb.fwd) __syncthreads();
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
      switch (pair_code(s_cp[k])) {
#define CPF_X(LO, HI)                                                                                        \
        case LO * 8 + HI:                                                                                    \
          if constexpr (HI < NQ) Base::template block_fwd<NQ - 1 - LO, NQ - 1 - HI>(cs, yr, yi);             \
          break;
        CPF_PAIR_LIST(CPF_X)
#undef CPF_X
        default: break;
      }
      cs += 2 * SW;
    }
    Base::template tail_fwd<0>(p, yr, yi, coef);
  }

  static __device__ __forceinline__ void backward(const KParams<R>& p, const LayerBar lb, const HCp* s_cp, R* coef,
                                                  R* stage, R* cph0, int m, V (&h)[N]) {
    const int K = p.n_cp;
    if (lb.bwd) __syncthreads();
    Base::template tail_bwd<0>(p, coef, m, h);
#pragma unroll 1
    for (int k0 = K > 0 ? ((K - 1) / GROUP) * GROUP : -1; k0 >= 0; k0 -= GROUP) {
      Base::stage_layer(k0, K, coef, cph0, stage, m, GROUP);
      __syncwarp();
      const int k1 = k0 + GROUP < K ? k0 + GROUP : K;
#pragma unroll 1
      for (int k = k1 - 1; k >= k0; --k) {
        const R* st = stage + STW * 2 * (k - k0);
        R* cl = coef + SW * (NQ + 2 * k);
        R* cph = cph0 + CW * k;
        switch (pair_code(s_cp[k])) {
#define CPF_X(LO, HI)                                                                                        \
          case LO * 8 + HI:                                                                                  \
            if constexpr (HI < NQ) Base::template block_bwd<NQ - 1 - LO, NQ - 1 - HI>(h, st, cl, cph, m);    \
            break;
          CPF_PAIR_LIST(CPF_X)
#undef CPF_X
          default: break;
        }
      }
      __syncwarp();
    }
    Base::stage_surface(coef, stage, m);
    __syncwarp();
    Base::template surface_bwd<NQ - 1>(coef, stage, m, h);
  }
};

// The multi-target variant (engine_impl.cuh: IsMultiTarget): the same sweeps; the forward sweep starts from the sample's
// own V^dag, read from the target table in global memory instead of the TMA-staged copy in shared memory.
template <typename R, int NQ, int CPT>
struct HeisSweepAnyMT : HeisSweepAny<R, NQ, CPT> {
  static constexpr bool MULTI_TARGET = true;
};

// ------------------------------------------------------------------------------------------
// update / coefficient phase helpers (per gate, executed by the gate's owner thread)
// ------------------------------------------------------------------------------------------
// Per-sample arrays are addressed as array[off + index] with a 32-bit element offset off = b * P (the
// host checks B * P < 2^32): one IMAD.WIDE per access instead of a 64-bit multiply chain.
template <typename R>
struct UpdCtx {
  int phase;            // PH_COEF / PH_ADAM / PH_GRAD
  bool active;          // this thread's sample exists
  bool store_best;      // the step being finished improved on the best regloss: keep its parameters
  bool skip_coef;       // last pass: no new coefficients
  bool hist;            // parameter history is recorded for this step
  unsigned off;         // b * P
  size_t hist_off;      // (b * hist_len + gu + 1) * P
  R bc1, bc2, ibc1, ibc2;
};

// Optimiser state {theta, m, v, best} of a sample in the kernel's scratch, LANE-INTERLEAVED: with one 16-byte record
// per parameter the update phase was bound by the L1 -> L2 request port (one 32-byte sector per cycle and SM; every
// access of a warp touched 16-32 half-used sectors), so the layout makes every access of a warp cover whole sectors.  A parameter has a POSITION q (heis_pk_pos_*) chosen so that the parameters the lanes of a sample
// touch in the same instruction are neighbours; positions are stored in blocks of 16: word (q >> 4) * 64 + f * 16 +
// (q & 15) holds field f (0 theta, 1 m, 2 v, 3 best-regloss parameter) of position q.  A fused gate g, rotation j:
//   surface gates (g < n):      q = (j TPS + g) 2                                  (lane g, one gate per lane)
//   block gates (gb = g - n):   q = 6 TPS + (((i >> 1) 3 + j) TPS + m) 2 + (i & 1),  m = gb % TPS, i = gb / TPS
// i.e. the two gates (i even, i odd) a lane updates side by side (heis_pair_update) are the two halves of an aligned
// 8-byte pair and the 8 lanes of a 4-qubit sample read one contiguous 64-byte row per field.  The entanglers follow
// at cp_base in the same pair-interleaved order (heis_pk_pos_cp).  The kernel packs the caller's separate arrays (include/cpflow_b200.h: cpf_adam_buffers) into this
// scratch at launch and unpacks at the end; `best` is only ever written (when a step improved), never read back
// before the unpack.
__host__ __device__ inline int heis_pk_pos_su2(int g, int j, int nq, int tps) {
  if (g < nq) return (j * tps + g) * 2;
  const int gb = g - nq, m = gb % tps, i = gb / tps;
  return 6 * tps + (((i >> 1) * 3 + j) * tps + m) * 2 + (i & 1);
}
__host__ __device__ inline int heis_pk_pair_iters(int nq, int tps, int n_su2) {
  const int nb = n_su2 > nq ? n_su2 - nq : 0;
  return (nb + 2 * tps - 1) / (2 * tps);
}
__host__ __device__ inline int heis_pk_cp_base(int nq, int tps, int n_su2) {
  return 6 * tps + heis_pk_pair_iters(nq, tps, n_su2) * 6 * tps;
}
// entangler k = m + TPS i (lane m, i-th entangler of the lane): pairs (i even, i odd) side by side like the fused gates
__host__ __device__ inline int heis_pk_pos_cp(int k, int cp_base, int tps) {
  const int m = k % tps, i = k / tps;
  return cp_base + ((i >> 1) * tps + m) * 2 + (i & 1);
}
__host__ __device__ inline int heis_pk_cp_pair_iters(int tps, int n_cp) { return (n_cp + 2 * tps - 1) / (2 * tps); }
// words (of R) per sample
__host__ __device__ inline int heis_pk_stride(int nq, int tps, int n_su2, int n_cp) {
  return ((heis_pk_cp_base(nq, tps, n_su2) + heis_pk_cp_pair_iters(tps, n_cp) * 2 * tps + 15) & ~15) * 4;
}
template <typename R> struct Pk4 { R th, mu, nu, best; };
template <typename R> __device__ __forceinline__ R* pk_at(R* pk, int q) { return pk + ((q >> 4) << 6) + (q & 15); }
template <typename R> __device__ __forceinline__ const R* pk_at(const R* pk, int q) { return pk + ((q >> 4) << 6) + (q & 15); }
template <typename R> __device__ __forceinline__ Pk4<R> pk_load(const R* pk, int q) {
  const R* b = pk_at(pk, q);
  return {b[0], b[16], b[32], R(0)};
}
template <typename R> __device__ __forceinline__ void pk_store(R* pk, int q, const Pk4<R>& v) {
  R* b = pk_at(pk, q);
  b[0] = v.th; b[16] = v.mu; b[32] = v.nu;
}

// MUFU approximations (rsqrt: 2^-22.4, rcp: 1 ulp) refined by one Newton step: the unit phases of the ZYZ data are
// built from these, and a modulus error of 2e-7 per phase accumulates over the ~3 K diagonal factors of a sweep
// (measured: worst gradient error of 4096 samples on C3 1.46e-5 with the raw approximations; profiles/grad_accuracy_r2.txt).
__device__ __forceinline__ float rsqrt_fast(float a) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
  const float h = 0.5f * a * r;
  return fmaf(r, fmaf(-h, r, 0.5f), r);          // r (1.5 - 0.5 a r^2)
}
__device__ __forceinline__ double rsqrt_fast(double a) { return rsqrt_r(a); }
__device__ __forceinline__ float rcp_fast(float a) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
  return fmaf(r, fmaf(-a, r, 1.0f), r);          // r (2 - a r)
}
__device__ __forceinline__ double rcp_fast(double a) { return 1.0 / a; }
static __device__ __noinline__ SinCos<float> sincos_slow_v(float x) { float s, c; sincosf(x, &s, &c); return {s, c}; }
// sin/cos for the parameter phase, inlined so the three evaluations of a fused gate interleave
__device__ __forceinline__ void sincos_core(float x, float& s, float& c) {
  const float j = rintf(x * 0.636619747f);
  float r = fmaf(j, -1.57079601e+00f, x);
  r = fmaf(j, -3.13916473e-07f, r);
  r = fmaf(j, -5.39030253e-15f, r);
  const int q = __float2int_rn(j);
  const float r2 = r * r;
  float sp = fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f);
  sp = fmaf(sp, r2, -1.6666654611e-1f);
  sp = fmaf(sp * r2, r, r);
  float cp = fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f);
  cp = fmaf(cp, r2, 4.166664568298827e-2f);
  cp = fmaf(cp * r2, r2, fmaf(r2, -0.5f, 1.0f));
  const float ss = (q & 1) ? cp : sp;
  const float cc = (q & 1) ? sp : cp;
  s = (q & 2) ? -ss : ss;
  c = ((q + 1) & 2) ? -cc : cc;
}
__device__ __forceinline__ void sincos_inl(float x, float& s, float& c) {
  sincos_core(x, s, c);
  if (fabsf(x) > 48000.f) { const SinCos<float> t = sincos_slow_v(x); s = t.s; c = t.c; }
}
__device__ __forceinline__ void sincos_inl(double x, double& s, double& c) { sincos_r(x, s, c); }
// the three half angles of a fused gate: one (never taken in practice) large-argument test for all of them
__device__ __forceinline__ void sincos3(bool on0, bool on1, bool on2, float x0, float x1, float x2, float& s0, float& c0,
                                        float& s1, float& c1, float& s2, float& c2) {
  if (on0) sincos_core(x0, s0, c0);
  if (on1) sincos_core(x1, s1, c1);
  if (on2) sincos_core(x2, s2, c2);
  if (fmaxf(fmaxf(on0 ? fabsf(x0) : 0.f, on1 ? fabsf(x1) : 0.f), on2 ? fabsf(x2) : 0.f) > 48000.f) {
    if (on0) sincos_inl(x0, s0, c0);
    if (on1) sincos_inl(x1, s1, c1);
    if (on2) sincos_inl(x2, s2, c2);
  }
}
__device__ __forceinline__ void sincos3(bool on0, bool on1, bool on2, double x0, double x1, double x2, double& s0,
                                        double& c0, double& s1, double& c1, double& s2, double& c2) {
  if (on0) sincos_r(x0, s0, c0);
  if (on1) sincos_r(x1, s1, c1);
  if (on2) sincos_r(x2, s2, c2);
}

// optax scale_by_adam + scale(-lr) (optimization.py:22-23).  double: exact IEEE sequence of the oracle.
// float: reciprocal bias corrections, approximate sqrt and division (<= 2 ulp each; the reference's XLA
// arithmetic is not bit-reproducible either, the Adam parity tests bound the drift).
__device__ __forceinline__ void adam_inl(const KParams<double>& p, const UpdCtx<double>& u, double g, double& th,
                                         double& mu, double& nu) {
  mu = add_rn(mul_rn(p.omb1, g), mul_rn(p.b1, mu));
  nu = add_rn(mul_rn(p.omb2, mul_rn(g, g)), mul_rn(p.b2, nu));
  const double mu_hat = mu / u.bc1, nu_hat = nu / u.bc2;
  th = add_rn(th, mul_rn(-p.lr, mu_hat / add_rn(sqrt(nu_hat), p.eps)));
}
__device__ __forceinline__ void adam_inl(const KParams<float>& p, const UpdCtx<float>& u, float g, float& th,
                                         float& mu, float& nu) {
  mu = add_rn(mul_rn(p.omb1, g), mul_rn(p.b1, mu));
  nu = add_rn(mul_rn(p.omb2, mul_rn(g, g)), mul_rn(p.b2, nu));
  const float mu_hat = mu * u.ibc1, nu_hat = nu * u.ibc2;
  // .ftz forms: without them ptxas wraps each MUFU in a denormal rescue (4 extra instructions); a denormal
  // nu_hat is far below eps^2 either way
  float rt, iv;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rt) : "f"(nu_hat));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iv) : "f"(add_rn(rt, p.eps)));
  th = add_rn(th, mul_rn(-p.lr, mul_rn(mu_hat, iv)));
}

// one parameter: gradient sink (loss_grad mode) or best-parameter bookkeeping + Adam step on the packed state
// PLAIN: Adam pass of a launch without freeze mask and parameter history (the stage-1 runs of Synthesize.static()):
// the per-parameter tests on those pointers disappear from the gate loops.
// pi: parameter index (the caller's arrays), q: its position in the packed state
template <typename R, bool PLAIN>
__device__ __forceinline__ void heis_apply(const KParams<R>& p, const UpdCtx<R>& u, R* pk, int pi, int q, R g, Pk4<R>& v) {
  if (!PLAIN && u.phase == PH_GRAD) {
    if (u.active) p.grad_out[u.off + (unsigned)pi] = g;
    return;
  }
  // v.th is still the pre-update parameter of the step being finished (optimization.py:70-73)
  if (u.store_best && u.active) pk_at(pk, q)[48] = v.th;
  if (PLAIN || !(p.freeze && p.freeze[u.off + (unsigned)pi])) adam_inl(p, u, g, v.th, v.mu, v.nu);
  if (u.active) {
    pk_store(pk, q, v);
    if (!PLAIN && u.hist) p.hist_params[u.hist_off + pi] = v.th;
  }
}

// (alpha, beta) <- R_a(c, s) * (alpha, beta) for a rotation about a compile-time-foldable axis: 8 FMA
template <typename R>
__device__ __forceinline__ void su2_lmul_axis(int a, R c, R s, R& ar, R& ai, R& br, R& bi) {
  if (a == 0) {        // Rx = [[c, -is], [-is, c]]
    const R nar = c * ar + s * bi, nai = c * ai - s * br, nbr = c * br + s * ai, nbi = c * bi - s * ar;
    ar = nar; ai = nai; br = nbr; bi = nbi;
  } else if (a == 1) { // Ry = [[c, -s], [s, c]]
    const R nar = c * ar - s * br, nai = c * ai - s * bi, nbr = c * br + s * ar, nbi = c * bi + s * ai;
    ar = nar; ai = nai; br = nbr; bi = nbi;
  } else if (a == 2) { // Rz = diag(c - is, c + is)
    const R nar = c * ar + s * ai, nai = c * ai - s * ar, nbr = c * br - s * bi, nbi = c * bi + s * br;
    ar = nar; ai = nai; br = nbr; bi = nbi;
  }
}

// Everything the update of one fused gate reads from global / shared memory.  The gate loops below are
// software pipelined: the loads of the next gate are issued before the current gate is processed, so the
// L2 round trips (theta, Adam moments, half-angle cos/sin of the fused rotations) overlap the arithmetic.
template <typename R>
struct GateIn {
  int pi0, pi1, pi2, axes;
  int q0;                 // position of the first rotation's parameter in the packed state; the others: + 2 TPS each
  Pk4<R> v0, v1, v2;
  R sx, sy, sz, c2, s2, c3, s3;
};
template <typename R, int NQ, int TPS>
__device__ __forceinline__ GateIn<R> heis_gate_load(const KParams<R>& p, const UpdCtx<R>& u, const R* pk, bool valid, int g,
                                                    const Su2Meta* md, const HSu2* ms, const R* cf, const R* ax) {
  GateIn<R> in;
  in.pi0 = in.pi1 = in.pi2 = -1; in.axes = 0xfff; in.q0 = 0;
  in.v0 = in.v1 = in.v2 = Pk4<R>{R(0), R(0), R(0), R(0)};
  in.sx = in.sy = in.sz = in.c2 = in.s2 = in.c3 = in.s3 = R(0);
  if (!valid) return in;
  const HSu2 hm = *ms;
  in.pi0 = hm.pidx[0]; in.pi1 = hm.pidx[1]; in.pi2 = hm.pidx[2];
  in.axes = hm.axes;
  in.q0 = heis_pk_pos_su2(g, 0, NQ, TPS);
  if (in.pi0 >= 0) in.v0 = pk_load(pk, in.q0); else in.v0.th = R(md->cangle[0]);
  if (in.pi1 >= 0) in.v1 = pk_load(pk, in.q0 + 2 * TPS); else in.v1.th = R(md->cangle[1]);
  if (in.pi2 >= 0) in.v2 = pk_load(pk, in.q0 + 4 * TPS); else in.v2.th = R(md->cangle[2]);
  if (u.phase != PH_COEF) {
    // gradient sums of the backward sweep, back to the gate's output frame: the sweep reads them after the gate's
    // own Rz(phi_out + pi/2) is undone, e^{i w} = i u_out (u_out is still in words 2, 3 from the last update)
    const R px = cf[0], py = cf[1], wr = -cf[3], wi = cf[2];
    in.sx = wr * px - wi * py; in.sy = wi * px + wr * py; in.sz = cf[4];
    Vec4Load<R>::ld(ax, in.c2, in.s2, in.c3, in.s3);
  }
  return in;
}

// Fused one-qubit gate: finish the step (chain rule through the fusion, Adam), then the new ZYZ data of the gate.
// AX* >= 0: compile-time rotation axes (the selects fold away); AX0 == -2: axes from the gate metadata.
template <typename R, int TPS, int AX0, int AX1, int AX2, bool PLAIN>
__device__ __forceinline__ void heis_su2_update(const KParams<R>& p, const UpdCtx<R>& u, R* pk, const Su2Meta* md,
                                                GateIn<R> in, R* cf, R* ax) {
  const int a0 = in.axes & 15, a1 = (in.axes >> 4) & 15, a2 = (in.axes >> 8) & 15;   // 15 = unused slot
  const int ax0 = AX0 == -2 ? (a0 == 15 ? -1 : a0) : AX0;
  const int ax1 = AX0 == -2 ? (a1 == 15 ? -1 : a1) : AX1;
  const int ax2 = AX0 == -2 ? (a2 == 15 ? -1 : a2) : AX2;
  if (u.phase != PH_COEF) {
    // chain rule through G = R_2 R_1 R_0: g_2 = S . e_2, g_1 = S . (R_2 e_1) = (R_2^T S) . e_1,
    // g_0 = (R_1^T R_2^T S) . e_0: rotate S backwards (no products with the zero entries of unit vectors)
    const R C2 = in.c2 * in.c2 - in.s2 * in.s2, S2 = R(2) * in.c2 * in.s2;
    const R C3 = in.c3 * in.c3 - in.s3 * in.s3, S3 = R(2) * in.c3 * in.s3;
    R sx = in.sx, sy = in.sy, sz = in.sz;
    const R g2 = sel3(ax2, sx, sy, sz);
    rot_axis(ax2, C3, -S3, sx, sy, sz);
    const R g1 = sel3(ax1, sx, sy, sz);
    rot_axis(ax1, C2, -S2, sx, sy, sz);
    const R g0 = sel3(ax0, sx, sy, sz);
    if (in.pi2 >= 0) heis_apply<R, PLAIN>(p, u, pk, in.pi2, in.q0 + 4 * TPS, g2, in.v2);
    if (in.pi1 >= 0) heis_apply<R, PLAIN>(p, u, pk, in.pi1, in.q0 + 2 * TPS, g1, in.v1);
    if (in.pi0 >= 0) heis_apply<R, PLAIN>(p, u, pk, in.pi0, in.q0, g0, in.v0);
  }
  if (!u.skip_coef) {
    R c0 = R(1), s0 = R(0), c1 = R(1), s1 = R(0), c2 = R(1), s2 = R(0);
    sincos3(ax0 >= 0, ax1 >= 0, ax2 >= 0, in.v0.th * R(0.5), in.v1.th * R(0.5), in.v2.th * R(0.5), s0, c0, s1, c1, s2, c2);
    R ar, ai, br, bi;
    su2_of(ax0, c0, s0, ar, ai, br, bi);
    su2_lmul_axis(ax1, c1, s1, ar, ai, br, bi);
    su2_lmul_axis(ax2, c2, s2, ar, ai, br, bi);
    if (u.active) { ax[0] = c1; ax[1] = s1; ax[2] = c2; ax[3] = s2; }
    // ZYZ form for the forward sweep: alpha = cy p_a, beta = sy p_b, u_out = p_b conj(p_a), u_in = conj(p_a p_b)
    const R na = ar * ar + ai * ai, nb = br * br + bi * bi;
    const bool oka = na > R(1e-30), okb = nb > R(1e-30);
    const R ia = oka ? rsqrt_fast(na) : R(0), ib = okb ? rsqrt_fast(nb) : R(0);
    const R par = oka ? ar * ia : R(1), pai = ai * ia, pbr = okb ? br * ib : R(1), pbi = bi * ib;
    // Ry by phi with cos phi = cy = |alpha| >= 0, sin phi = sy = |beta| >= 0, in lifting form (Cols::ry_lift)
    const R cyv = na * ia, syv = nb * ib;
    cf[0] = -syv * rcp_fast(R(1) + cyv); cf[1] = syv;
    cf[2] = pbr * par + pbi * pai; cf[3] = pbi * par - pbr * pai;
    cf[4] = par * pbr - pai * pbi; cf[5] = -(par * pbi + pai * pbr);
  }
}
// ------------------------------------------------------------------------------------------
// Packed update of TWO fused gates per thread (float, PLAIN runs, compile-time axes): component .x is gate g, .y is
// gate g + stride of the same lane.  The parameter phase is latency bound (dependent FMA / MUFU chains, two warps per
// scheduler and CTA): two gates side by side in FFMA2 / FMUL2 / FADD2 halve its instruction count and double the
// work in flight per thread.  Every component follows the arithmetic of the scalar float path operation by operation
// (same roundings: Adam as separate multiplies and adds), so a gate's result does not depend on its partner.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 p2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 bc2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 sel2(bool kx, bool ky, float2 a, float2 b) { return make_float2(kx ? a.x : b.x, ky ? a.y : b.y); }

// x' = C x - S y; y' = S x + C y on the two coordinates the axis does not fix (rot_axis, packed)
template <int A>
__device__ __forceinline__ void rot_axis2(float2 C, float2 S, float2 nS, float2& x, float2& y, float2& z) {
  if constexpr (A == 0) { const float2 ny = fma2(nS, z, mul2(C, y)), nz = fma2(S, y, mul2(C, z)); y = ny; z = nz; }
  else if constexpr (A == 1) { const float2 nz = fma2(nS, x, mul2(C, z)), nx = fma2(S, z, mul2(C, x)); z = nz; x = nx; }
  else if constexpr (A == 2) { const float2 nx = fma2(nS, y, mul2(C, x)), ny = fma2(S, x, mul2(C, y)); x = nx; y = ny; }
}
template <int A> __device__ __forceinline__ float2 sel3c(float2 x, float2 y, float2 z) { return A == 0 ? x : (A == 1 ? y : z); }
// (alpha, beta) <- R_A(c, s) (alpha, beta)   (su2_lmul_axis, packed)
template <int A>
__device__ __forceinline__ void su2_lmul_axis2(float2 c, float2 s, float2& ar, float2& ai, float2& br, float2& bi) {
  const float2 ns = neg2(s);
  if constexpr (A == 0) {
    const float2 nar = fma2(s, bi, mul2(c, ar)), nai = fma2(ns, br, mul2(c, ai)), nbr = fma2(s, ai, mul2(c, br)),
                 nbi = fma2(ns, ar, mul2(c, bi));
    ar = nar; ai = nai; br = nbr; bi = nbi;
  } else if constexpr (A == 1) {
    const float2 nar = fma2(ns, br, mul2(c, ar)), nai = fma2(ns, bi, mul2(c, ai)), nbr = fma2(s, ar, mul2(c, br)),
                 nbi = fma2(s, ai, mul2(c, bi));
    ar = nar; ai = nai; br = nbr; bi = nbi;
  } else if constexpr (A == 2) {
    const float2 nar = fma2(s, ai, mul2(c, ar)), nai = fma2(ns, ar, mul2(c, ai)), nbr = fma2(ns, bi, mul2(c, br)),
                 nbi = fma2(s, br, mul2(c, bi));
    ar = nar; ai = nai; br = nbr; bi = nbi;
  }
}
// R_A1(c1, s1) R_A0(c0, s0) as (alpha, beta): every component is one product (the zeros of su2_of folded by hand)
template <int A0, int A1>
__device__ __forceinline__ void su2_two2(float2 c0, float2 s0, float2 c1, float2 s1, float2& ar, float2& ai, float2& br,
                                         float2& bi) {
  const float2 z = bc2(0.f);
  ar = c0; ai = z; br = z; bi = z;
  if constexpr (A0 == 0) bi = neg2(s0); else if constexpr (A0 == 1) br = s0; else ai = neg2(s0);
  su2_lmul_axis2<A1>(c1, s1, ar, ai, br, bi);
}
__device__ __forceinline__ float2 rsqrt_fast2(float2 a) {
  float rx, ry;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rx) : "f"(a.x));
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(ry) : "f"(a.y));
  const float2 r = p2(rx, ry);
  const float2 nh = mul2(mul2(bc2(-0.5f), a), r);              // -(0.5 a) r, rounded like the scalar 0.5f * a * r
  return fma2(r, fma2(nh, r, bc2(0.5f)), r);
}
__device__ __forceinline__ float2 rcp_fast2(float2 a) {
  float rx, ry;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rx) : "f"(a.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ry) : "f"(a.y));
  const float2 r = p2(rx, ry);
  return fma2(r, fma2(neg2(a), r, bc2(1.0f)), r);
}
// sincos_core on both components
__device__ __forceinline__ void sincos_core2(float2 x, float2& s, float2& c) {
  const float2 t = mul2(x, bc2(0.636619747f));
  const float2 j = p2(rintf(t.x), rintf(t.y));
  float2 r = fma2(j, bc2(-1.57079601e+00f), x);
  r = fma2(j, bc2(-3.13916473e-07f), r);
  r = fma2(j, bc2(-5.39030253e-15f), r);
  const int qx = __float2int_rn(j.x), qy = __float2int_rn(j.y);
  const float2 r2 = mul2(r, r);
  float2 sp = fma2(r2, bc2(-1.9515295891e-4f), bc2(8.3321608736e-3f));
  sp = fma2(sp, r2, bc2(-1.6666654611e-1f));
  sp = fma2(mul2(sp, r2), r, r);
  float2 cp = fma2(r2, bc2(2.443315711809948e-5f), bc2(-1.388731625493765e-3f));
  cp = fma2(cp, r2, bc2(4.166664568298827e-2f));
  cp = fma2(mul2(cp, r2), r2, fma2(r2, bc2(-0.5f), bc2(1.0f)));
  const float ssx = (qx & 1) ? cp.x : sp.x, ccx = (qx & 1) ? sp.x : cp.x;
  const float ssy = (qy & 1) ? cp.y : sp.y, ccy = (qy & 1) ? sp.y : cp.y;
  s = p2((qx & 2) ? -ssx : ssx, (qy & 2) ? -ssy : ssy);
  c = p2(((qx + 1) & 2) ? -ccx : ccx, ((qy + 1) & 2) ? -ccy : ccy);
}

// What the update of a gate pair reads from global memory (requested one pair ahead): theta, m, v of the three
// rotations, .x = gate a, .y = gate b (one aligned 8-byte pair per field in the lane-interleaved state).
struct PairGlob { float2 th0, mu0, nu0, th1, mu1, nu1, th2, mu2, nu2; };
template <int TPS>
__device__ __forceinline__ PairGlob heis_pair_load(const float* pk, int q0, bool valid) {
  PairGlob q;
  const float2 z = make_float2(0.f, 0.f);
  q.th0 = q.mu0 = q.nu0 = q.th1 = q.mu1 = q.nu1 = q.th2 = q.mu2 = q.nu2 = z;
  if (valid) {
    const float* b0 = pk_at(pk, q0);
    const float* b1 = pk_at(pk, q0 + 2 * TPS);
    const float* b2 = pk_at(pk, q0 + 4 * TPS);
    q.th0 = *reinterpret_cast<const float2*>(b0); q.mu0 = *reinterpret_cast<const float2*>(b0 + 16);
    q.nu0 = *reinterpret_cast<const float2*>(b0 + 32);
    q.th1 = *reinterpret_cast<const float2*>(b1); q.mu1 = *reinterpret_cast<const float2*>(b1 + 16);
    q.nu1 = *reinterpret_cast<const float2*>(b1 + 32);
    q.th2 = *reinterpret_cast<const float2*>(b2); q.mu2 = *reinterpret_cast<const float2*>(b2 + 16);
    q.nu2 = *reinterpret_cast<const float2*>(b2 + 32);
  }
  return q;
}
// Adam on a parameter pair (adam_inl, float, packed) and the stores of the pair's fields (on: the pair exists and the
// sample is a real one)
__device__ __forceinline__ void heis_apply2(const KParams<float>& p, const UpdCtx<float>& u, float* pk, int q, bool on,
                                            float2 g, float2& th, float2& mu, float2& nu) {
  float* b = pk_at(pk, q);
  // th is still the pre-update parameter of the step being finished (optimization.py:70-73)
  if (u.store_best && on) *reinterpret_cast<float2*>(b + 48) = th;
  mu = add2(mul2(bc2(p.omb1), g), mul2(bc2(p.b1), mu));
  nu = add2(mul2(bc2(p.omb2), mul2(g, g)), mul2(bc2(p.b2), nu));
  const float2 mh = mul2(mu, bc2(u.ibc1)), nh = mul2(nu, bc2(u.ibc2));
  float rx, ry, ix, iy;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rx) : "f"(nh.x));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(ry) : "f"(nh.y));
  const float2 den = add2(p2(rx, ry), bc2(p.eps));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(ix) : "f"(den.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iy) : "f"(den.y));
  th = add2(th, mul2(bc2(-p.lr), mul2(mh, p2(ix, iy))));
  if (on) {
    *reinterpret_cast<float2*>(b) = th;
    *reinterpret_cast<float2*>(b + 16) = mu;
    *reinterpret_cast<float2*>(b + 32) = nu;
  }
}
// NP gate pairs of one lane, side by side in ONE basic block (no branch between the pairs: the parameter phase is a
// long dependent chain per pair - load, chain rule, MUFU, sin/cos, SU(2) products, rsqrt, rcp - and the instruction
// scheduler interleaves the independent chains).  Pair k: gates ga[k] and ga[k] + TPS (has_b[k]), q0[k] the position
// of rotation 0 of its first gate; the fields of a missing gate are zero (heis_kernel zeroes unused positions when it
// packs the state).  Returns the largest |half angle| seen: arguments beyond the fast range reduction are handled
// by the caller (heis_kernel), out of line, so that the hot path has no branch.
template <int TPS, int AX0, int AX1, int AX2, int NP>
__device__ __forceinline__ float heis_pairs_update(const KParams<float>& p, const UpdCtx<float>& u, float* pk,
                                                   PairGlob (&q)[NP], const int (&q0)[NP], const int (&ga)[NP],
                                                   const bool (&has_b)[NP], float* coef) {
  constexpr int SW = HEIS_SU2_WORDS;
  float big = 0.f;
  if (u.phase != PH_COEF) {
    float2 g0[NP], g1[NP], g2[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) {
      const float* cfa = coef + SW * ga[k];
      const float* cfb = coef + SW * (has_b[k] ? ga[k] + TPS : ga[k]);
      // gradient sums of the backward sweep, back to the gates' output frames (heis_gate_load)
      const float4 la = *reinterpret_cast<const float4*>(cfa), lb = *reinterpret_cast<const float4*>(cfb);
      const float2 px = p2(la.x, lb.x), py = p2(la.y, lb.y), wi = p2(la.z, lb.z), wr = p2(-la.w, -lb.w);
      float2 sx = fma2(neg2(wi), py, mul2(wr, px)), sy = fma2(wr, py, mul2(wi, px)), sz = p2(cfa[4], cfb[4]);
      // half-angle cos / sin of the second and third rotation at the parameters of the step being finished:
      // recomputed (the scalar path keeps them in global memory: 32 bytes of L2 traffic per gate and step)
      const float2 y1 = mul2(q[k].th1, bc2(0.5f)), y2 = mul2(q[k].th2, bc2(0.5f));
      float2 c2, s2, c3, s3;
      sincos_core2(y1, s2, c2); sincos_core2(y2, s3, c3);
      // chain rule through G = R_2 R_1 R_0 (heis_su2_update); rotations by -theta: (C, -S) with S = 2 c s
      const float2 C2 = fma2(c2, c2, neg2(mul2(s2, s2))), t2 = mul2(bc2(2.f), c2), S2 = mul2(t2, s2), nS2 = mul2(neg2(t2), s2);
      const float2 C3 = fma2(c3, c3, neg2(mul2(s3, s3))), t3 = mul2(bc2(2.f), c3), S3 = mul2(t3, s3), nS3 = mul2(neg2(t3), s3);
      g2[k] = sel3c<AX2>(sx, sy, sz);
      rot_axis2<AX2>(C3, nS3, S3, sx, sy, sz);
      g1[k] = sel3c<AX1>(sx, sy, sz);
      rot_axis2<AX1>(C2, nS2, S2, sx, sy, sz);
      g0[k] = sel3c<AX0>(sx, sy, sz);
    }
#pragma unroll
    for (int k = 0; k < NP; ++k) {
      heis_apply2(p, u, pk, q0[k] + 4 * TPS, u.active, g2[k], q[k].th2, q[k].mu2, q[k].nu2);
      heis_apply2(p, u, pk, q0[k] + 2 * TPS, u.active, g1[k], q[k].th1, q[k].mu1, q[k].nu1);
      heis_apply2(p, u, pk, q0[k], u.active, g0[k], q[k].th0, q[k].mu0, q[k].nu0);
    }
  }
  if (!u.skip_coef) {
#pragma unroll
    for (int k = 0; k < NP; ++k) {
      float* cfa = coef + SW * ga[k];
      float* cfb = coef + SW * (has_b[k] ? ga[k] + TPS : ga[k]);
      const float2 x0 = mul2(q[k].th0, bc2(0.5f)), x1 = mul2(q[k].th1, bc2(0.5f)), x2 = mul2(q[k].th2, bc2(0.5f));
      float2 s0, c0, s1, c1, s2, c2;
      sincos_core2(x0, s0, c0); sincos_core2(x1, s1, c1); sincos_core2(x2, s2, c2);
      big = fmaxf(big, fmaxf(fmaxf(fmaxf(fabsf(x0.x), fabsf(x0.y)), fmaxf(fabsf(x1.x), fabsf(x1.y))),
                             fmaxf(fabsf(x2.x), fabsf(x2.y))));
      float2 ar, ai, br, bi;
      su2_two2<AX0, AX1>(c0, s0, c1, s1, ar, ai, br, bi);
      su2_lmul_axis2<AX2>(c2, s2, ar, ai, br, bi);
      // ZYZ form for the forward sweep (heis_su2_update)
      const float2 na = fma2(ar, ar, mul2(ai, ai)), nb = fma2(br, br, mul2(bi, bi));
      const bool oax = na.x > 1e-30f, oay = na.y > 1e-30f, obx = nb.x > 1e-30f, oby = nb.y > 1e-30f;
      const float2 zero = bc2(0.f), one = bc2(1.f);
      const float2 ia = sel2(oax, oay, rsqrt_fast2(na), zero), ib = sel2(obx, oby, rsqrt_fast2(nb), zero);
      const float2 par = sel2(oax, oay, mul2(ar, ia), one), pai = mul2(ai, ia);
      const float2 pbr = sel2(obx, oby, mul2(br, ib), one), pbi = mul2(bi, ib);
      const float2 cyv = mul2(na, ia), syv = mul2(nb, ib);
      const float2 ty = mul2(neg2(syv), rcp_fast2(add2(one, cyv)));
      const float2 uor = fma2(pbr, par, mul2(pbi, pai)), uoi = fma2(pbi, par, neg2(mul2(pbr, pai)));
      const float2 uir = fma2(par, pbr, neg2(mul2(pai, pbi))), uii = neg2(fma2(par, pbi, mul2(pai, pbr)));
      *reinterpret_cast<float4*>(cfa) = make_float4(ty.x, syv.x, uor.x, uoi.x);
      *reinterpret_cast<float2*>(cfa + 4) = make_float2(uir.x, uii.x);
      if (has_b[k]) {
        *reinterpret_cast<float4*>(cfb) = make_float4(ty.y, syv.y, uor.y, uoi.y);
        *reinterpret_cast<float2*>(cfb + 4) = make_float2(uir.y, uii.y);
      }
    }
  }
  return big;
}
// gates g0, g0 + TPS, ... < g_end of one class: four at a time (two pairs), then the remaining one or two (g0 is the
// lane's first gate of the class, so the pair (g, g + TPS) shares one 8-byte slot per field).  Returns the largest
// |half angle| of the new parameters.
template <int NQ, int TPS, int AX0, int AX1, int AX2>
__device__ __forceinline__ float heis_su2_loop_pair(const KParams<float>& p, const UpdCtx<float>& u, float* pk, int g0,
                                                    int g_end, float* coef) {
  int q0 = heis_pk_pos_su2(g0, 0, NQ, TPS);
  float big = 0.f;
  int g = g0;
#pragma unroll 1
  for (; g + 2 * TPS < g_end; g += 4 * TPS) {
    // consecutive pairs of a lane are 6 TPS positions apart (three rotations x TPS lanes x 2).  (Requesting the angles
    // of the next four gates one iteration ahead was measured: no gain, 143.7 vs 143.2 ms on the C3 shape.)
    PairGlob q[2] = {heis_pair_load<TPS>(pk, q0, true), heis_pair_load<TPS>(pk, q0 + 6 * TPS, true)};
    const int qs[2] = {q0, q0 + 6 * TPS}, gs[2] = {g, g + 2 * TPS};
    const bool hb[2] = {true, g + 3 * TPS < g_end};
    big = fmaxf(big, heis_pairs_update<TPS, AX0, AX1, AX2, 2>(p, u, pk, q, qs, gs, hb, coef));
    q0 += 12 * TPS;
  }
  if (g < g_end) {
    PairGlob q[1] = {heis_pair_load<TPS>(pk, q0, true)};
    const int qs[1] = {q0}, gs[1] = {g};
    const bool hb[1] = {g + TPS < g_end};
    big = fmaxf(big, heis_pairs_update<TPS, AX0, AX1, AX2, 1>(p, u, pk, q, qs, gs, hb, coef));
  }
  return big;
}

// packed axes of a gate class: a0 | a1 << 4 | a2 << 8 (15 = unused slot); 0xffff = not uniform
constexpr int AXP_ZXZ = 2 | (0 << 4) | (2 << 8);
constexpr int AXP_XYZ = 0 | (1 << 4) | (2 << 8);
constexpr int AXP_XZ = 0 | (2 << 4) | (15 << 8);

// gates g0, g0 + stride, ... < g_end of one class (compile-time axes), software pipelined.  (Issuing the first loads of
// all three gate classes together at the top of the parameter phase was measured: no gain in float - 121.6 vs 121.3 M
// evals/s on C3 - and 1.5 KB of spills in the double kernels; each loop keeps its own prologue.)
template <typename R, int NQ, int TPS, int AX0, int AX1, int AX2, bool PLAIN>
__device__ __forceinline__ void heis_su2_loop(const KParams<R>& p, const HSu2* ms, const UpdCtx<R>& u, R* pk, int g0,
                                              int g_end, R* coef, R* aux) {
  constexpr int stride = TPS;
  constexpr int SW = HEIS_SU2_WORDS;
  // Two gates in flight, loop unrolled by two so that the buffers keep their registers (no copies at the back
  // edge): the state of gate g + 2 stride is requested as soon as gate g is done and has the whole update of
  // gate g + stride to arrive (the L2 round trip is about as long as one gate's update).
  GateIn<R> ga = heis_gate_load<R, NQ, TPS>(p, u, pk, g0 < g_end, g0, p.su2 + g0, ms + g0, coef + SW * g0, aux + 4 * g0);
  GateIn<R> gb = heis_gate_load<R, NQ, TPS>(p, u, pk, g0 + stride < g_end, g0 + stride, p.su2 + g0 + stride, ms + g0 + stride,
                                            coef + SW * (g0 + stride), aux + 4 * (g0 + stride));
#pragma unroll 1
  for (int g = g0; g < g_end; g += 2 * stride) {
    heis_su2_update<R, TPS, AX0, AX1, AX2, PLAIN>(p, u, pk, p.su2 + g, ga, coef + SW * g, aux + 4 * g);
    const int g2 = g + 2 * stride;
    ga = heis_gate_load<R, NQ, TPS>(p, u, pk, g2 < g_end, g2, p.su2 + g2, ms + g2, coef + SW * g2, aux + 4 * g2);
    const int g1 = g + stride;
    if (g1 < g_end) heis_su2_update<R, TPS, AX0, AX1, AX2, PLAIN>(p, u, pk, p.su2 + g1, gb, coef + SW * g1, aux + 4 * g1);
    const int g3 = g + 3 * stride;
    gb = heis_gate_load<R, NQ, TPS>(p, u, pk, g3 < g_end, g3, p.su2 + g3, ms + g3, coef + SW * g3, aux + 4 * g3);
  }
}
// Entanglers two at a time (float, PLAIN runs, every entangler a CP gate with a parameter): .x is entangler k, .y is
// k + TPS; same arithmetic per component as the scalar loop in heis_kernel.
template <int NQ, int TPS>
__device__ __forceinline__ float heis_cp_loop_pair(const KParams<float>& p, const UpdCtx<float>& u, const HCp* s_cp, float* pk,
                                                   int cp_base, int m, float* coef, float* coef_cp, float& reg_part) {
  constexpr int SW = HEIS_SU2_WORDS, CW = HEIS_CP_WORDS;
  const float2 z = make_float2(0.f, 0.f);
  float big = 0.f;
  int q = cp_base + 2 * m;
  float2 th_n = z, mu_n = z, nu_n = z;
  if (m < p.n_cp) {
    const float* b = pk_at(pk, q);
    th_n = *reinterpret_cast<const float2*>(b); mu_n = *reinterpret_cast<const float2*>(b + 16);
    nu_n = *reinterpret_cast<const float2*>(b + 32);
  }
#pragma unroll 1
  for (int k = m; k < p.n_cp; k += 2 * TPS) {
    float2 th = th_n, mu = mu_n, nu = nu_n;
    const int kb = k + TPS, kn = k + 2 * TPS;
    const bool has_b = kb < p.n_cp;
    if (kn < p.n_cp) {
      const float* b = pk_at(pk, q + 2 * TPS);
      th_n = *reinterpret_cast<const float2*>(b); mu_n = *reinterpret_cast<const float2*>(b + 16);
      nu_n = *reinterpret_cast<const float2*>(b + 32);
    }
    const bool pen_a = p.pen.kind != CPF_PEN_NONE && (s_cp[k].flags & 1) != 0;
    const bool pen_b = p.pen.kind != CPF_PEN_NONE && has_b && (s_cp[has_b ? kb : k].flags & 1) != 0;
    float* cfa = coef_cp + CW * k;
    float* cfb = coef_cp + CW * (has_b ? kb : k);
    // word 6 of the block's higher-qubit gate slot: r * penalty slope at this angle
    float* rsa = coef + SW * (NQ + 2 * k + 1) + 6;
    float* rsb = coef + SW * (NQ + 2 * (has_b ? kb : k) + 1) + 6;
    if (u.phase != PH_COEF) {
      const float2 g = add2(p2(cfa[0], cfb[0]), p2(*rsa, *rsb));
      heis_apply2(p, u, pk, q, u.active, g, th, mu, nu);
    }
    if (!u.skip_coef) {
      const float2 x = mul2(th, bc2(0.5f));
      float2 s, c;
      sincos_core2(x, s, c);
      big = fmaxf(big, fmaxf(fabsf(x.x), fabsf(x.y)));       // beyond the fast reduction: redone by the caller
      float rs_a = 0.f, rs_b = 0.f;
      if (pen_a) {
        float val, slope;
        penalty_eval_fast(p.pen, th.x, val, slope);
        reg_part += val;
        rs_a = mul_rn(p.pen.r, slope);
      }
      if (pen_b) {
        float val, slope;
        penalty_eval_fast(p.pen, th.y, val, slope);
        reg_part += val;
        rs_b = mul_rn(p.pen.r, slope);
      }
      // CP(a) = CP(a - 2 pi): keep cos(a/2) >= 0 (phase_bwd)
      const bool na = c.x < 0.f, nb = c.y < 0.f;
      c = p2(na ? -c.x : c.x, nb ? -c.y : c.y);
      s = p2(na ? -s.x : s.x, nb ? -s.y : s.y);
      const float2 t = mul2(neg2(s), rcp_fast2(add2(bc2(1.f), c)));
      cfa[0] = c.x; cfa[1] = s.x; cfa[2] = t.x; *rsa = rs_a;
      if (has_b) { cfb[0] = c.y; cfb[1] = s.y; cfb[2] = t.y; *rsb = rs_b; }
    }
    q += 2 * TPS;
  }
  return big;
}

// pairs: the packed two-gates-per-thread path may be used (float Adam runs without freeze mask / history whose fused
// gates are all-parameter); returns the largest |half angle| it met (0 from the scalar loops, which reduce large
// arguments themselves)
template <typename R, int NQ, int TPS>
__device__ __forceinline__ R heis_su2_loop_any(int axp, bool plain, bool pairs, const KParams<R>& p, const HSu2* ms,
                                               const UpdCtx<R>& u, R* pk, int g0, int g_end, R* coef, R* aux) {
  if constexpr (sizeof(R) == 4) {
    if (pairs) {
      if (axp == AXP_XYZ) return heis_su2_loop_pair<NQ, TPS, 0, 1, 2>(p, u, pk, g0, g_end, coef);
      if (axp == AXP_ZXZ) return heis_su2_loop_pair<NQ, TPS, 2, 0, 2>(p, u, pk, g0, g_end, coef);
    }
  }
  if (axp == AXP_XYZ) {
    if (plain) heis_su2_loop<R, NQ, TPS, 0, 1, 2, true>(p, ms, u, pk, g0, g_end, coef, aux);
    else heis_su2_loop<R, NQ, TPS, 0, 1, 2, false>(p, ms, u, pk, g0, g_end, coef, aux);
  } else if (axp == AXP_ZXZ) {
    if (plain) heis_su2_loop<R, NQ, TPS, 2, 0, 2, true>(p, ms, u, pk, g0, g_end, coef, aux);
    else heis_su2_loop<R, NQ, TPS, 2, 0, 2, false>(p, ms, u, pk, g0, g_end, coef, aux);
  } else if (axp == AXP_XZ) heis_su2_loop<R, NQ, TPS, 0, 2, -1, false>(p, ms, u, pk, g0, g_end, coef, aux);
  else heis_su2_loop<R, NQ, TPS, -2, -2, -2, false>(p, ms, u, pk, g0, g_end, coef, aux);
  return R(0);
}

// f(parameter index or -1, position) for every position of the packed state that lane m of a sample owns: the slots of
// its fused gates in both update loops (present or not) and its entanglers
template <int NQ, int TPS, typename F>
__device__ __forceinline__ void heis_pk_visit(int n_su2, int n_cp, const HSu2* s_su2, const HCp* s_cp, int m, F f) {
  for (int j = 0; j < 3; ++j) {
    const int q = (j * TPS + m) * 2;
    f(m < NQ && m < n_su2 ? (int)s_su2[m].pidx[j] : -1, q);
    f(-1, q + 1);
  }
  const int iters = 2 * heis_pk_pair_iters(NQ, TPS, n_su2);
  for (int i = 0; i < iters; ++i) {
    const int g = NQ + m + i * TPS;
    for (int j = 0; j < 3; ++j) f(g < n_su2 ? (int)s_su2[g].pidx[j] : -1, heis_pk_pos_su2(g, j, NQ, TPS));
  }
  const int cp_base = heis_pk_cp_base(NQ, TPS, n_su2), cp_iters = 2 * heis_pk_cp_pair_iters(TPS, n_cp);
  for (int i = 0; i < cp_iters; ++i) {
    const int k = m + i * TPS;
    f(k < n_cp ? (int)s_cp[k].pidx : -1, heis_pk_pos_cp(k, cp_base, TPS));
  }
}

// The block size is a launch parameter (a multiple of 32 up to HCfg::MAXT); p.spb of its blockDim.x / TPS
// sample slots are used (heis_geometry spreads the batch evenly over SMs and rounds).
template <typename R, int NQ, int CPT, typename SWP>
__global__ void __launch_bounds__(HCfg<R, NQ, CPT>::MAXT, 1)
heis_kernel(const KParams<R> p) {
  using C = HCfg<R, NQ, CPT>;
  using T = VT<R, CPT>;
  using V = typename T::V;
  constexpr int N = C::N, TPS = C::TPS, PB = C::PB, XR = C::XR;
  constexpr int SW = HEIS_SU2_WORDS, CW = HEIS_CP_WORDS;
  constexpr bool MT = IsMultiTarget<SWP>::value;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  R* s_target = reinterpret_cast<R*>(smem_raw);
  HSu2* s_su2 = reinterpret_cast<HSu2*>(smem_raw + p.target_bytes);
  HCp* s_cp = reinterpret_cast<HCp*>(s_su2 + p.n_su2);
  R* s_coef = reinterpret_cast<R*>(smem_raw + p.target_bytes + heis_meta_bytes(p.n_su2, p.n_cp));

  const int tid = threadIdx.x;
  // ---- prologue: TMA-stage V^dag (packed by pack_target_heis_kernel) ----
  if (!MT && tid == 0) {
    mbar_init(&s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (!MT && tid == 0) {
    mbar_expect_tx(&s_bar, (uint32_t)p.target_bytes);
    tma_bulk_g2s(s_target, p.target_packed, (uint32_t)p.target_bytes, &s_bar);
  }
  // gate metadata -> shared memory (compact records)
  for (int g = tid; g < p.n_su2; g += blockDim.x) {
    const Su2Meta* md = p.su2 + g;
    HSu2 hm;
    unsigned axes = 0;
    for (int j = 0; j < 3; ++j) {
      hm.pidx[j] = (int16_t)md->pidx[j];
      axes |= (unsigned)(md->axis[j] < 0 ? 15 : md->axis[j]) << (4 * j);
    }
    hm.axes = (uint16_t)axes;
    s_su2[g] = hm;
  }
  for (int k = tid; k < p.n_cp; k += blockDim.x) {
    const CpMeta* md = p.cp + k;
    HCp hm;
    hm.pidx = (int16_t)md->pidx;
    hm.flags = (uint16_t)(((p.cp_pen ? p.cp_pen[k] != 0 : md->penalised != 0) ? 1 : 0) | (md->is_cz ? 2 : 0) |
                          ((md->lo_q & 7) << 4) | ((md->hi_q & 7) << 8));
    hm.prev_lo = md->prev_lo; hm.prev_hi = md->prev_hi;
    s_cp[k] = hm;
  }
  __syncthreads();
  if constexpr (!MT) mbar_wait(&s_bar, 0);

  const int sl = tid / TPS;   // sample within the block
  const int m = tid % TPS;    // lane within the sample: column group (forward), x >> PB (backward)
  // ring position -> (sample, visit); an unsliced launch has ring_start = 0, ring_end = B (visit 0 for everybody)
  const long long c_raw = p.ring_start + (long long)blockIdx.x * p.spb + sl;
  const bool active = sl < p.spb && c_raw < p.ring_end;
  const long long c_pos = active ? c_raw : p.ring_end - 1;
  const long long b = c_pos % p.B;
  const long long step0 = p.step0 + (c_pos / p.B) * (long long)p.nsteps;
  const int P = p.P;
  // idle sample slots (block size rounded up to whole warps) replay the launch's last sample in one spare store
  R* coef = s_coef + (size_t)(sl < p.spb ? sl : p.spb) * p.coef_stride;
  R* stage = coef + SW * p.n_su2;                          // staged rows of one layer of the backward sweep
  R* coef_cp = stage + HEIS_STAGE_WORDS * SWP::NSTAGE;
  const R* tgt = s_target;
  if constexpr (MT) tgt = p.target_packed + (size_t)p.target_index[b] * (size_t)(2 * N * (N + 1));   // heis_target_words
  const V* tv = reinterpret_cast<const V*>(tgt) + 2 * (size_t)m * (N + 1);

  const unsigned off = (unsigned)(b * P);   // host: B * P < 2^32
  R* aux = p.aux + (size_t)b * p.n_su2 * 4;
  R* pk = reinterpret_cast<R*>(p.pk) + (size_t)b * p.pk_stride;
  const int cp_base = heis_pk_cp_base(NQ, TPS, p.n_su2);
  {
    // pack this sample's optimiser state (a resumed run, step0 > 0, carries its moments and best parameters);
    // positions no gate owns are zeroed (the pair path computes on them)
    const bool resume = p.mode == M_ADAM && step0 > 0;
    heis_pk_visit<NQ, TPS>(p.n_su2, p.n_cp, s_su2, s_cp, m, [&](int pi, int q) {
      R th = R(0), mu = R(0), nu = R(0), be = R(0);
      if (pi >= 0) {
        th = p.angles[off + pi]; be = th;
        if (resume) { mu = p.m[off + pi]; nu = p.v[off + pi]; be = p.best_params[off + pi]; }
      }
      if (active) { R* d = pk_at(pk, q); d[0] = th; d[16] = mu; d[32] = nu; d[48] = be; }
    });
    // parameters that feed no gate never reach the packed state: their outputs are written here
    if (p.unreferenced_params && p.mode == M_ADAM && !resume && active)
      for (int i = m; i < P; i += TPS) { p.m[off + i] = R(0); p.v[off + i] = R(0); p.best_params[off + i] = p.angles[off + i]; }
    __syncwarp();
  }
  const R NN = R(N) * R(N);

  LayerBar lb;
  lb.fwd = (p.sync_sweeps & 1) != 0; lb.bwd = (p.sync_sweeps & 2) != 0;

  R best = R(0), best_reg_v = R(0);
  bool improved_prev = false;
  if (p.mode == M_ADAM && step0 > 0) { best = p.best_regloss[b]; best_reg_v = p.best_reg[b]; }

  for (int it = 0; it <= p.nsteps; ++it) {
    const long long gi = step0 + it;
    const int phase = it == 0 ? PH_COEF : (p.mode == M_ADAM ? PH_ADAM : PH_GRAD);
    // ---------------- parameter phase (a sample's threads split the gates) ----------------
    R reg_part = R(0);
#ifdef CPF_EXP_SKIP_UPDATE      // timing experiment only (tools/build_variant.py): sweeps without the parameter phase
    if (it == 0 || it == p.nsteps)
#endif
    {
      UpdCtx<R> u;
      u.phase = phase; u.active = active; u.off = off;
      const long long gu = gi - 1;
      u.store_best = improved_prev && p.mode == M_ADAM && phase == PH_ADAM;
      u.skip_coef = it == p.nsteps;
      u.hist = p.hist_params != nullptr && gu + 1 < p.hist_len;
      u.hist_off = u.hist ? (size_t)(b * p.hist_len + gu + 1) * (size_t)P : 0;
      u.bc1 = u.bc2 = u.ibc1 = u.ibc2 = R(1);
      if (phase == PH_ADAM) {
        u.bc1 = bias_corr(p.b1, R(gu + 1));
        u.bc2 = bias_corr(p.b2, R(gu + 1));
        u.ibc1 = R(1) / u.bc1; u.ibc2 = R(1) / u.bc2;
      }
      // surface gates (slots < NQ) and block gates (the rest) each share one axis pattern in the templates
      // plain: an Adam RUN without freeze mask and parameter history.  Every pass of such a run, the first
      // (coefficient-only) one of a launch included, goes through the same PLAIN instantiation of the gate loops:
      // split and time-sliced runs are bit-identical to one launch by construction, not by the compiler's choice of
      // identical FMA contractions in two instantiations
      const bool plain = p.mode == M_ADAM && p.freeze == nullptr && p.hist_params == nullptr;
      const int n_surf = NQ < p.n_su2 ? NQ : p.n_su2;
      const bool pairs = sizeof(R) == 4 && plain && p.su2_all_params;
      R big = heis_su2_loop_any<R, NQ, TPS>(p.axp_surface, plain, pairs, p, s_su2, u, pk, m, n_surf, coef, aux);
      big = fmax(big, heis_su2_loop_any<R, NQ, TPS>(p.axp_block, plain, pairs, p, s_su2, u, pk, NQ + m, p.n_su2, coef, aux));
      // entangler angles, software pipelined like the fused-gate loops: the packed state of the next gate is
      // requested before the current one is processed
      const bool cp_pairs = sizeof(R) == 4 && plain && p.cp_all_params;
      auto cp_scalar = [&](const UpdCtx<R>& u) {
        const int phase = u.phase;
        int k = m;
        int pi_n = -1;
        Pk4<R> v_n = Pk4<R>{R(0), R(0), R(0), R(0)};
        HCp md_n = HCp{-1, 0, 0, 0};
        if (k < p.n_cp) { md_n = s_cp[k]; pi_n = md_n.pidx; if (pi_n >= 0) v_n = pk_load(pk, heis_pk_pos_cp(k, cp_base, TPS)); }
#pragma unroll 1
        for (; k < p.n_cp; k += TPS) {
          const HCp md = md_n;
          R* cf = coef_cp + CW * k;
          const int pi = pi_n;
          Pk4<R> v = v_n;
          const int kn = k + TPS;
          if (kn < p.n_cp) { md_n = s_cp[kn]; pi_n = md_n.pidx; if (pi_n >= 0) v_n = pk_load(pk, heis_pk_pos_cp(kn, cp_base, TPS)); }
          const bool pen_on = p.pen.kind != CPF_PEN_NONE && pi >= 0 && (md.flags & 1) != 0;
          if (pi < 0) v.th = R(p.cp[k].cangle);
          // cf[0]: dL/da from the sweep; word 6 of the block's higher-qubit gate slot: r * penalty slope at this angle
          R* rsw = coef + SW * (NQ + 2 * k + 1) + 6;
          if (phase != PH_COEF && pi >= 0) {
            const R g = add_rn(cf[0], *rsw);
            if (plain) heis_apply<R, true>(p, u, pk, pi, heis_pk_pos_cp(k, cp_base, TPS), g, v);
            else heis_apply<R, false>(p, u, pk, pi, heis_pk_pos_cp(k, cp_base, TPS), g, v);
          }
          const R th = v.th;
          if (!u.skip_coef) {
            R s = R(1), c = R(0);                  // half angle; CZ = CP(pi): cos(pi/2) = 0 exactly
            if (!(md.flags & 2)) sincos_inl(th * R(0.5), s, c);
            R rs = R(0);
            if (pen_on) {
              R val, slope;
              penalty_eval_fast(p.pen, th, val, slope);
              reg_part += val;
              rs = mul_rn(p.pen.r, slope);
            }
            // CP(a) = CP(a - 2 pi): keep cos(a/2) >= 0, so the ZZ pair rotation of the backward sweep is a rotation
            // by at most pi/2 and its lifting coefficient t = -tan(a/4) is bounded (phase_bwd)
            if (c < R(0)) { c = -c; s = -s; }
            cf[0] = c; cf[1] = s; cf[2] = -s * rcp_fast(R(1) + c); *rsw = rs;
          }
        }
      };
      if constexpr (sizeof(R) == 4) {
        if (cp_pairs) big = fmax(big, heis_cp_loop_pair<NQ, TPS>(p, u, s_cp, pk, cp_base, m, coef, coef_cp, reg_part));
      }
      if (!cp_pairs) cp_scalar(u);
      if constexpr (sizeof(R) == 4) {
        // The packed paths reduce sin / cos arguments with the three-constant scheme only; a half angle beyond its
        // range (never seen in an optimisation: |theta| > 96000) sends the whole warp once more through the scalar
        // loops, coefficients only, whose sin / cos fall back to the library reduction.
        if ((pairs || cp_pairs) && !u.skip_coef && __any_sync(0xffffffffu, big > R(48000))) {
          UpdCtx<R> u2 = u;
          u2.phase = PH_COEF;
          if (pairs) {
            heis_su2_loop_any<R, NQ, TPS>(p.axp_surface, false, false, p, s_su2, u2, pk, m, n_surf, coef, aux);
            heis_su2_loop_any<R, NQ, TPS>(p.axp_block, false, false, p, s_su2, u2, pk, NQ + m, p.n_su2, coef, aux);
          }
          if (cp_pairs) { reg_part = R(0); cp_scalar(u2); }
        }
      }
    }
    __syncwarp();
    if (it == p.nsteps) break;
    // merged diagonals of the forward sweep: A = pending(lo) u_in(lo), B = pending(hi) u_in(hi), A B e^{ia}
    for (int k = m; k < p.n_cp; k += TPS) {
      const HCp md = s_cp[k];
      R* cl = coef + SW * (NQ + 2 * k);
      R* ch = cl + SW;
      const R* pl = coef + SW * md.prev_lo;
      const R* ph = coef + SW * md.prev_hi;
      const R* cc = coef_cp + CW * k;
      const R plr = pl[2], pli = pl[3], phr = ph[2], phi = ph[3];
      const R ar = plr * cl[4] - pli * cl[5], ai = plr * cl[5] + pli * cl[4];
      const R br = phr * ch[4] - phi * ch[5], bi = phr * ch[5] + phi * ch[4];
      const R abr = ar * br - ai * bi, abi = ar * bi + ai * br;
      const R c = cc[0] * cc[0] - cc[1] * cc[1], s = R(2) * cc[0] * cc[1];   // e^{ia} from the half angle
      cl[4] = ar; cl[5] = ai; cl[6] = br; cl[7] = bi;
      ch[4] = abr * c - abi * s; ch[5] = abr * s + abi * c;
    }
    __syncwarp();

#ifdef CPF_EXP_SKIP_SWEEPS      // timing experiment only: parameter phase without the sweeps
    if (it > 0) { improved_prev = true; continue; }
#endif
    // ---------------- forward sweep: Y = U V^dag ----------------
    V yr[N], yi[N];
#pragma unroll
    for (int r = 0; r < N; ++r) { yr[r] = tv[2 * r]; yi[r] = tv[2 * r + 1]; }
    SWP::forward(p, lb, s_cp, coef, yr, yi);

    // ---------------- pivot to the Pauli basis ----------------
    SWP::gather_wht(yr, yi);
    const R tr = __shfl_sync(0xffffffffu, T::get(yr[0], 0), 0, TPS);
    const R ti = __shfl_sync(0xffffffffu, T::get(yi[0], 0), 0, TPS);
    R reg = sample_sum<TPS>(reg_part);
    const R ab = sqrt_r(tr * tr + ti * ti);
    const R loss = R(1) - mul_rn(ab, ab) / NN;
    reg = mul_rn(p.pen.r, reg);

    if (p.mode == M_LOSSGRAD) {
      if (active && m == 0) {
        p.loss_out[b] = loss;
        if (p.reg_out) p.reg_out[b] = reg;
      }
      if (!p.grad_out) return;
    } else {
      const R regloss = add_rn(loss, reg);
      bool improved;
      if (gi == 0) {
        improved = true;
        if (active && m == 0) { p.init_regloss[b] = regloss; p.init_reg[b] = reg; }
      } else {
        improved = regloss < best;
      }
      // the parameters of an improving step are saved by the next update phase, which has them in registers
      improved_prev = improved;
      if (improved) { best = regloss; best_reg_v = reg; }
      if (active && p.hist_regloss && m == 0 && gi < p.hist_len)
        p.hist_regloss[b * p.hist_len + gi] = regloss;
      if (active && p.hist_params && gi == 0)
        for (int i = m; i < P; i += TPS) p.hist_params[b * p.hist_len * P + i] = p.angles[off + i];
    }

    // h[xr][z] = Re(i^{|x&z|} s W[x,z]),  s = i conj(t)/N^2 = (ti + i tr)/N^2,  x = (m << PB) | xr
    V h[N];
    {
      const R sr = ti / NN, si = tr / NN;
#pragma unroll
      for (int z = 0; z < N; ++z) {
        R hc[XR];
#pragma unroll
        for (int xr = 0; xr < XR; ++xr) {
          const R wr = T::get(yr[z], xr), wi = T::get(yi[z], xr);
          const R pq = sr * wr - si * wi, qq = sr * wi + si * wr;
          const int k = __popc(m & (z >> PB)) + (PB ? (xr & z & 1) : 0);
          const R val = (k & 1) ? -qq : pq;
          hc[xr] = (k & 2) ? -val : val;
        }
        h[z] = T::make(hc[0], hc[XR - 1]);
      }
    }
    __syncwarp();

    // ---------------- Heisenberg sweep ----------------
    SWP::backward(p, lb, s_cp, coef, stage, coef_cp, m, h);
    __syncwarp();
  }

  if (p.mode == M_ADAM && active) {
    // unpack the optimiser state into the caller's arrays
    // (every lane reads back the positions it wrote itself)
    heis_pk_visit<NQ, TPS>(p.n_su2, p.n_cp, s_su2, s_cp, m, [&](int pi, int q) {
      if (pi < 0) return;
      const R* d = pk_at(pk, q);
      p.angles[off + pi] = d[0]; p.m[off + pi] = d[16]; p.v[off + pi] = d[32]; p.best_params[off + pi] = d[48];
    });
    if (m == 0) { p.best_regloss[b] = best; p.best_reg[b] = best_reg_v; }
  }
}

// ---- target packing for heis_kernel: Y0 = V^dag, lane l = column group, all rows per lane ----
// dst index ((l * (N + 1) + r) * 2 + part) * CPT + k :  part 0 = Re, 1 = Im of conj(V[l*CPT + k][r])
template <typename R>
__global__ void pack_target_heis_kernel(const R* __restrict__ src, R* __restrict__ dst, int N, int cpt) {
  const int total = (N / cpt) * (N + 1) * 2 * cpt;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int k = i % cpt, t = i / cpt;
    int part = t % 2; t /= 2;
    int r = t % (N + 1), l = t / (N + 1);
    R val = R(0);
    if (r < N) {
      const R v = src[((size_t)(l * cpt + k) * N + r) * 2 + part];
      val = part ? -v : v;
    }
    dst[i] = val;
  }
}

// All targets of a multi-target table in one launch (blockIdx.y = target): the layout of pack_target_heis_kernel,
// target t at dst + t * heis_target_words.  src: n_targets row-major N x N complex matrices.
template <typename R>
__global__ void pack_targets_heis_kernel(const R* __restrict__ src, R* __restrict__ dst, int N, int cpt) {
  const int total = (N / cpt) * (N + 1) * 2 * cpt;
  src += (size_t)blockIdx.y * N * N * 2;
  dst += (size_t)blockIdx.y * total;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int k = i % cpt, t = i / cpt;
    int part = t % 2; t /= 2;
    int r = t % (N + 1), l = t / (N + 1);
    R val = R(0);
    if (r < N) {
      const R v = src[((size_t)(l * cpt + k) * N + r) * 2 + part];
      val = part ? -v : v;
    }
    dst[i] = val;
  }
}

// Launch geometry: spread the batch evenly over SMs and rounds so that the last wave is as full as the
// first (every CTA runs all the Adam steps of its samples, so a ragged last wave costs a whole wave).
//   ctas  resident CTAs per SM.  Each CTA is one synchronised instruction stream (its warps share the instruction
//         cache); two streams per SM overlap their phases (+4 % on C3 when both hold 8 warps) as long as the SM
//         keeps as many samples resident as with one: chosen automatically, env CPF_HEIS_CTAS overrides.
//   cap   samples per CTA allowed by shared memory, the register file, the thread limit and CPF_HEIS_WARPS
struct HeisGeometry { int block, spb, ctas; long long grid; size_t smem; };
inline long long heis_cap(int ctas, size_t fixed_bytes, size_t per_sample, int tps, int maxt, int regs, int warps_env) {
  // registers: allocated per warp in units of 256, 64 K per SM
  const int regs_warp = ((regs > 0 ? regs : 128) * 32 + 255) / 256 * 256;
  int warps = 65536 / regs_warp / ctas;
  if (warps > maxt / 32) warps = maxt / 32;
  if (warps_env > 0 && warps > warps_env) warps = warps_env;
  const long long cap_thr = (long long)warps * 32 / tps;
  const long long smem_cta = (long long)(227 * 1024) / ctas - 1024 - (long long)fixed_bytes;
  long long cap = smem_cta > 0 ? smem_cta / (long long)per_sample : 0;
  // a block whose last warp is only partly used parks the idle lanes on one spare slot
  if (cap > 0 && (cap * tps) % 32 != 0 && cap <= cap_thr) cap -= 1;
  if (cap > cap_thr) cap = cap_thr;
  return cap < 1 ? 1 : cap;
}
inline HeisGeometry heis_geometry(long long B, size_t fixed_bytes, size_t per_sample, int tps, int maxt, int regs,
                                  int n_sm = 0) {
  if (n_sm <= 0) {          // the current device (cpf_launch_plan passes a number to plan without one)
    int dev = 0;
    n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  }
  int ctas = 0, warps_env = 0;
  if (const char* e = getenv("CPF_HEIS_CTAS")) { int v = atoi(e); if (v >= 1 && v <= 16) ctas = v; }
  if (const char* e = getenv("CPF_HEIS_WARPS")) { int v = atoi(e); if (v >= 1) warps_env = v; }
  const long long slots1 = n_sm;
  auto spread = [&](int nc, long long& spb_out) {
    const long long cap = heis_cap(nc, fixed_bytes, per_sample, tps, maxt, regs, warps_env);
    const long long slots = slots1 * nc;
    long long rounds = (B + slots * cap - 1) / (slots * cap);
    if (rounds < 1) rounds = 1;               // empty batch
    long long spb = (B + slots * rounds - 1) / (slots * rounds);
    if (spb > cap) spb = cap;
    if (spb < 1) spb = 1;
    spb_out = spb;
    return cap;
  };
  long long spb = 1;
  if (ctas == 0) {
    // measured on B200: two streams of 8 warps beat one of 16 (+4 % C3, +29 % 5 qubits), two of 6 lose to one of 11
    long long spb1, spb2;
    const long long c1 = spread(1, spb1), c2 = spread(2, spb2);
    ctas = 2 * c2 >= c1 && (spb2 * tps + 31) / 32 >= 8 ? 2 : 1;
    spb = ctas == 2 ? spb2 : spb1;
  } else {
    spread(ctas, spb);
  }
  HeisGeometry g;
  g.spb = (int)spb;
  g.ctas = ctas;
  g.block = (int)((spb * tps + 31) / 32 * 32);
  g.grid = (B + spb - 1) / spb;
  g.smem = fixed_bytes + (size_t)(spb + (g.block > spb * tps ? 1 : 0)) * per_sample;
  // CPF_HEIS_SOLO=1 (measurements): pad the request so that the hardware cannot co-schedule a second CTA on the SM
  if (const char* e = getenv("CPF_HEIS_SOLO")) if (e[0] == '1' && g.smem < 120 * 1024) g.smem = 120 * 1024;
  return g;
}

// Time slicing of an Adam run whose batch is not a whole number of full waves (DESIGN.md: "ring slicing").  Every CTA
// keeps its samples for all the steps of a launch, so a batch of 1.3 waves either runs as 2 rounds of 2/3-full CTAs
// (the even spread of heis_geometry) or, sliced, as a ring: the T steps are cut into k chunks of T / k, the B k
// (sample, chunk) items are laid on a ring in sample-major order, and consecutive launches of `slots` items each walk
// along it.  All launches but the last run at full residency; stream order guarantees that chunk v + 1 of a sample
// starts after its chunk v has been written back (the run is resumable by construction: split runs are bit-identical
// to one run).
// The choice is an empirical throughput model fitted to B200 measurements of the C3 kernel (profiles/r2_*perf*):
//   one launch      relative rate (s / s_full)^0.7 for s resident samples per SM, times a tail factor
//                   1 - 0.05 min(1, 3 / rounds) (a CTA runs all T steps, so with few rounds the SMs that finish first
//                   idle: 10^5 samples in 11 rounds 121 M evals/s, 5 x 10^4 in 6 rounds 111 M, 2.5 x 10^4 in 3: 109 M,
//                   1.25 x 10^4 in 2 rounds of 43: 102 M)
//   sliced          1 / (1.035 + 3 / C) for chunks of C steps (drift between CTAs exposed at every launch boundary,
//                   state pack / unpack and the coefficient pass), times the fill of the last launch
//                   (116-118 M evals/s at every batch size measured).
struct HeisSlicing { int k; long long slots; };
inline HeisSlicing heis_slicing(long long B, int nsteps, size_t fixed_bytes, size_t per_sample, int tps, int maxt, int regs,
                                int n_sm, bool allowed) {
  HeisSlicing best{1, 0};
  const HeisGeometry full = heis_geometry((long long)1 << 40, fixed_bytes, per_sample, tps, maxt, regs, n_sm);
  const long long slots = (long long)full.spb * full.ctas * n_sm;
  best.slots = slots;
  int forced = -1;
  if (const char* e = getenv("CPF_HEIS_SLICES")) forced = atoi(e);
  if (!allowed || forced == 0 || forced == 1 || B <= 0 || nsteps < 2) return best;
  // a ring shorter than one launch would put two visits of a sample into the same launch: never sliced
  if (B <= slots) return best;
  if (forced > 1) {
    if (nsteps % forced == 0) best.k = forced;
    return best;
  }
  const HeisGeometry g1 = heis_geometry(B, fixed_bytes, per_sample, tps, maxt, regs, n_sm);
  const long long rounds = (g1.grid + (long long)g1.ctas * n_sm - 1) / ((long long)g1.ctas * n_sm);
  const double occ = (double)g1.spb * g1.ctas / ((double)full.spb * full.ctas);
  double rate_best = pow(occ < 1.0 ? occ : 1.0, 0.7) * (1.0 - 0.05 * (rounds >= 3 ? 3.0 / (double)rounds : 1.0));
  for (int k = 2; k <= 64 && nsteps / k >= 20; ++k) {
    if (nsteps % k) continue;
    const double launches = (double)(B * k) / (double)slots;
    const double rate = 1.0 / (1.035 + 3.0 / (nsteps / k)) * launches / ceil(launches);
    if (rate > rate_best * 1.01) { rate_best = rate; best.k = k; }
  }
  return best;
}

template <typename R, int NQ, int CPT, typename SWP>
int launch_heis_sized(KParams<R> p, cudaStream_t st, std::string& err) {
  using C = HCfg<R, NQ, CPT>;
  p.n_sched = 0; p.n_red = 0;
  p.coef_stride = heis_coef_stride(p.n_su2, p.n_cp, SWP::NSTAGE);
  if (p.P > 32767) { err = "heis kernel: more than 32767 parameters"; return CPF_ERR_UNSUPPORTED; }
  auto kern = heis_kernel<R, NQ, CPT, SWP>;
  static std::atomic<int> regs_cached{0};      // per instantiation
  int regs = regs_cached.load(std::memory_order_relaxed);
  if (regs == 0) {
    cudaFuncAttributes fa;
    regs = cudaFuncGetAttributes(&fa, kern) == cudaSuccess ? fa.numRegs : 128;
    regs_cached.store(regs, std::memory_order_relaxed);
  }
  int dev = 0, n_sm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  const size_t fixed = (size_t)p.target_bytes + heis_meta_bytes(p.n_su2, p.n_cp);
  const size_t per_sample = (size_t)p.coef_stride * sizeof(R);
  // CTA barrier at the start of the forward (bit 0) / backward (bit 1) sweep; env CPF_HEIS_SYNC overrides (tests)
  p.sync_sweeps = 3;
  if (const char* e = getenv("CPF_HEIS_SYNC")) { int v = atoi(e); if (v >= 0 && v <= 3) p.sync_sweeps = v; }
  const bool sliceable = p.mode == M_ADAM && p.hist_params == nullptr && p.hist_regloss == nullptr;
  const HeisSlicing sl = heis_slicing(p.B, p.nsteps, fixed, per_sample, C::TPS, C::MAXT, regs, n_sm, sliceable);
  const long long ring_total = p.B * sl.k;
  p.nsteps /= sl.k;
  long long smem_attr = 0;      // per call: cudaFuncSetAttribute is cheap, the limit is re-asserted for this device
  const long long per_launch = sl.k > 1 ? sl.slots : ring_total;      // unsliced: one launch over the whole batch
  for (long long c0 = 0; c0 < ring_total; c0 += per_launch) {
    const long long count = ring_total - c0 < per_launch ? ring_total - c0 : per_launch;
    const HeisGeometry g = heis_geometry(count, fixed, per_sample, C::TPS, C::MAXT, regs, n_sm);
    p.spb = g.spb;
    p.ring_start = c0; p.ring_end = c0 + count;
    if (g.smem > 227 * 1024) {
      err = "program too large for the shared-memory coefficient store (" + std::to_string(g.smem) + " bytes)";
      return CPF_ERR_UNSUPPORTED;
    }
    if ((long long)g.smem > smem_attr) {
      // the opt-in limit only ever grows (per instantiation and device; a smaller launch runs under a larger limit)
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
      if (e != cudaSuccess) { err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); return CPF_ERR_CUDA; }
      cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      smem_attr = (long long)g.smem;
    }
    if (g.grid <= 0 || count <= 0) return CPF_OK;
    if (g.grid > 2147483647LL) { err = "batch too large for one launch"; return CPF_ERR_UNSUPPORTED; }
    kern<<<(unsigned)g.grid, g.block, g.smem, st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { err = std::string("kernel launch: ") + cudaGetErrorString(e); return CPF_ERR_CUDA; }
  }
  return CPF_OK;
}

// Returns true and sets `rc` when a Heisenberg kernel compiled for this layered program exists.
// `dry` only answers the question (used before the target is staged in the heis layout).
template <typename R> bool launch_heis(const KParams<R>& p, const Program& prog, cudaStream_t st,
                                       std::string& err, int& rc, bool dry, int* n_stage = nullptr);
// columns per thread of the heis kernels for (dtype, n): selects the target packing
template <typename R> int heis_cpt(int n_qubits);
template <typename R> int launch_pack_target_heis(const R* src, R* dst, int n_qubits, int cpt, cudaStream_t st);

// Multi-target kernels (inst_multi_*.cu).  launch_heis_multi: HeisSweepAnyMT, returns false when none exists for the
// program's qubit count; launch_engine_multi: InterpSweepMT over the decoded schedule of engine_rb<R>(n, single).
// The pack functions fill a table of n_targets packed targets (heis / engine layout) in one launch.
template <typename R> bool launch_heis_multi(const KParams<R>& p, const Program& prog, cudaStream_t st, std::string& err,
                                             int& rc);
template <typename R> int launch_engine_multi(const KParams<R>& p, int n_qubits, bool single, cudaStream_t st,
                                              std::string& err);
template <typename R> int launch_pack_targets_heis(const R* src, R* dst, int n_qubits, int cpt, int n_targets,
                                                   cudaStream_t st);
template <typename R> int launch_pack_targets(const R* src, R* dst, int n_qubits, int cpt, bool single, int n_targets,
                                              cudaStream_t st);

}  // namespace cpf
