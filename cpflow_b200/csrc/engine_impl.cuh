// Kernel body of the cpflow_b200 engine (see engine.cuh for the design notes).
#pragma once
#include <type_traits>

#include "engine.cuh"

namespace cpf {

// ---- TMA (bulk async copy) + mbarrier helpers: stage the packed target into shared memory ---
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

template <typename R> struct Vec4Load;
template <> struct Vec4Load<float> {
  static __device__ __forceinline__ void ld(const float* p, float& a, float& b, float& c, float& d) {
    float4 t = *reinterpret_cast<const float4*>(p); a = t.x; b = t.y; c = t.z; d = t.w;
  }
  static __device__ __forceinline__ void st(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
  }
};
template <> struct Vec4Load<double> {
  static __device__ __forceinline__ void ld(const double* p, double& a, double& b, double& c, double& d) {
    double2 t = *reinterpret_cast<const double2*>(p), u = *reinterpret_cast<const double2*>(p + 2);
    a = t.x; b = t.y; c = u.x; d = u.y;
  }
  static __device__ __forceinline__ void st(double* p, double a, double b, double c, double d) {
    *reinterpret_cast<double2*>(p) = make_double2(a, b);
    *reinterpret_cast<double2*>(p + 2) = make_double2(c, d);
  }
};

template <typename R>
__device__ __forceinline__ R sel3(int a, R x, R y, R z) { return a == 0 ? x : (a == 1 ? y : z); }

enum Phase : int { PH_COEF = 0, PH_ADAM = 1, PH_GRAD = 2 };

// Gradient sink of the update phase: either store the gradient (loss_grad / cotangent modes) or run
// one optax-Adam step on the parameter (skipped for frozen parameters: cp_utils.py:100-108).
template <typename R>
__device__ __forceinline__ void apply_grad(const KParams<R>& p, bool active, long long b, int phase,
                                           long long gi, R bc1, R bc2, R ibc1, R ibc2, R* ang, R* mom, R* vel,
                                           const uint8_t* frz, int pi, R g, R& th, R mu0, R nu0) {
  const int P = p.P;
  if (phase == PH_GRAD) {
    if (active) p.grad_out[b * P + pi] = g;
    return;
  }
  // a frozen parameter skips the Adam update only: its (unchanged) value still goes into the history row
  if (!(frz && frz[pi])) {
    // (mu0, nu0: the moments before the step, loaded by the caller one gate ahead; zero for the first step)
    const AdamOut<R> o = adam_step_fused(g, th, mu0, nu0, p.b1, p.omb1, p.b2, p.omb2, bc1, bc2, ibc1, ibc2, p.eps, -p.lr);
    th = o.th;
    if (active) { mom[pi] = o.mu; vel[pi] = o.nu; ang[pi] = th; }
  }
  if (active && p.hist_params && gi + 1 < p.hist_len)
    p.hist_params[(b * p.hist_len + gi + 1) * P + pi] = th;
}

// resident CTAs per SM the register allocator is asked to allow for (state registers per thread
// = 4 * 2^RB * CPT * sizeof(R)/4 for phi and lambda together)
template <typename R, int RB, int CPT, int BLOCK = 128>
__host__ __device__ constexpr int min_blocks() {
  constexpr int state = 4 * (1 << RB) * CPT * (int)(sizeof(R) / 4);
  constexpr int mb = state <= 32 ? 5 : (state <= 64 ? 4 : (state <= 128 ? 2 : 1));
  return mb * BLOCK > 640 ? (640 / BLOCK > 0 ? 640 / BLOCK : 1) : mb;      // the same threads per SM for every block size
}

// ---- compile-time dispatch of the decoded ops -------------------------------------------------
#define CPF_SU2_CASE(I, ...) \
  case DC_SU2_REG0 + I: if constexpr (RB > I) { constexpr int BP = I; __VA_ARGS__; } break;
#define CPF_PH_CASE(I, ...) \
  case DC_PHASE0 + I: if constexpr (I < (1 << RB)) { constexpr int RM = I; __VA_ARGS__; } break;
// register masks with at most two bits set (a two-qubit gate)
#define CPF_PH_CASES(...)                                                                          \
  CPF_PH_CASE(0, __VA_ARGS__) CPF_PH_CASE(1, __VA_ARGS__) CPF_PH_CASE(2, __VA_ARGS__)               \
  CPF_PH_CASE(3, __VA_ARGS__) CPF_PH_CASE(4, __VA_ARGS__) CPF_PH_CASE(5, __VA_ARGS__)               \
  CPF_PH_CASE(6, __VA_ARGS__) CPF_PH_CASE(8, __VA_ARGS__) CPF_PH_CASE(9, __VA_ARGS__)               \
  CPF_PH_CASE(10, __VA_ARGS__) CPF_PH_CASE(12, __VA_ARGS__) CPF_PH_CASE(16, __VA_ARGS__)            \
  CPF_PH_CASE(17, __VA_ARGS__) CPF_PH_CASE(18, __VA_ARGS__) CPF_PH_CASE(20, __VA_ARGS__)            \
  CPF_PH_CASE(24, __VA_ARGS__)

// Multi-target (MT) kernels are the instantiations whose sweep type declares MULTI_TARGET = true (InterpSweepMT,
// heis_impl.cuh: HeisSweepAnyMT).  Sample b then reads its packed target, through L1 / L2, from the table at
// p.target_packed (targets back to back, each in the single-target packed layout) at entry p.target_index[b]; nothing
// is staged in shared memory.  Carrying the switch in the sweep type keeps the single-target kernels' names and code.
template <typename S, typename = void>
struct IsMultiTarget { static constexpr bool value = false; };
template <typename S>
struct IsMultiTarget<S, std::void_t<decltype(S::MULTI_TARGET)>> { static constexpr bool value = S::MULTI_TARGET; };

// ------------------------------------------------------------------------------------------
// Sweepers: how the forward and the adjoint sweep walk the gate schedule.
//   InterpSweep  — general programs: one dispatch per decoded op (program.hpp: DecodedSchedule).
//   LayerSweep   — layered templates (the CP / CZ ansatz of main.py:106-146): the blocks of one layer
//                  are compile-time constants, so the sweeps are straight-line code with immediate
//                  lane masks and coefficient offsets and no per-gate dispatch at all.
// ------------------------------------------------------------------------------------------
template <typename R, int NQ, int RB, int CPT, bool SINGLE>
struct InterpSweep {
  using C = Cfg<R, NQ, RB, CPT, SINGLE>;
  using CO = Cols<R, RB, CPT>;
  using T = VT<R, CPT>;
  using V = typename T::V;
  static constexpr int NA = C::NA, LB = C::LB, TPS = C::TPS;
  static constexpr bool USES_SCHED = true;

  static __device__ __forceinline__ void forward(const KParams<R>& p, R* coef, const uint2* s_dec, int la,
                                                 V (&pr)[NA], V (&pi)[NA]) {
#pragma unroll 1
  for (int i = 0; i < p.n_sched; ++i) {
    const uint2 d = s_dec[i];
    R c0, c1, c2, c3;
    Vec4Load<R>::ld(coef + (d.y & 0xffffu), c0, c1, c2, c3);
    const int lm = (d.x >> 8) & 0xff;
    switch (d.x & 0xffu) {
      CPF_SU2_CASE(0, (CO::template su2_reg<BP>(pr, pi, c0, c1, c2, c3)))
      CPF_SU2_CASE(1, (CO::template su2_reg<BP>(pr, pi, c0, c1, c2, c3)))
      CPF_SU2_CASE(2, (CO::template su2_reg<BP>(pr, pi, c0, c1, c2, c3)))
      CPF_SU2_CASE(3, (CO::template su2_reg<BP>(pr, pi, c0, c1, c2, c3)))
      CPF_SU2_CASE(4, (CO::template su2_reg<BP>(pr, pi, c0, c1, c2, c3)))
      case DC_SU2_LANE:
        if constexpr (LB > 0) CO::su2_lane(pr, pi, lm, (la & lm) != 0, c0, c1, c2, c3);
        break;
      CPF_PH_CASES({
        const bool on = (la & lm) == lm;
        CO::template phase<RM>(pr, pi, on ? c0 : R(1), on ? c1 : R(0));
      })
      case DC_CX: {
        const int cpos = lm & 15, tpos = lm >> 4;
        if (tpos < RB) {
          CPF_BP_SWITCH(RB, tpos, (CO::template cnot_reg<BP>(pr, pi, cpos, la)));
        } else {
          CO::cnot_lane(pr, pi, cpos, 1 << (tpos - RB), la);
        }
      } break;
      default: break;
    }
  }

  }

  static __device__ __forceinline__ void backward(const KParams<R>& p, R* coef, const uint2* s_dec,
                                                  const uint16_t* s_red, int la, int ls, V (&pr)[NA],
                                                  V (&pi)[NA], V (&lr)[NA], V (&li)[NA]) {
  // Per-thread partial gradient sums wait in `acc` (SU2: slots {0,1,2} or {3,4,5}; phase: 6 or 7)
  // until the schedule says "reduce": one transposing butterfly then sums up to 8 of them.
  R acc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = R(0);
#pragma unroll 1
  for (int i = p.n_sched - 1; i >= 0; --i) {
    const uint2 d = s_dec[i];
    R c0, c1, c2, c3;
    Vec4Load<R>::ld(coef + (d.y & 0xffffu), c0, c1, c2, c3);
    const int lm = (d.x >> 8) & 0xff;
    const bool hp = (d.x & (DF_PARAM << 16)) != 0;
    const bool second = (d.x & (1u << 20)) != 0;   // acc base 3 (SU2) / 7 (phase)
    R sx = R(0), sy = R(0), sz = R(0);
    switch (d.x & 0xffu) {
#define CPF_BWD_REG                                                              \
{                                                                              \
  if (hp) CO::template pauli_reg<BP>(pr, pi, lr, li, sx, sy, sz);              \
  CO::template su2_reg<BP>(pr, pi, c0, -c1, -c2, -c3);                         \
  CO::template su2_reg<BP>(lr, li, c0, -c1, -c2, -c3);                         \
}
      CPF_SU2_CASE(0, CPF_BWD_REG)
      CPF_SU2_CASE(1, CPF_BWD_REG)
      CPF_SU2_CASE(2, CPF_BWD_REG)
      CPF_SU2_CASE(3, CPF_BWD_REG)
      CPF_SU2_CASE(4, CPF_BWD_REG)
#undef CPF_BWD_REG
      case DC_SU2_LANE:
        if constexpr (LB > 0)
          CO::bwd_lane(pr, pi, lr, li, lm, (la & lm) != 0, hp, c0, c1, c2, c3, sx, sy, sz);
        break;
      CPF_PH_CASES({
        const bool on = (la & lm) == lm;
        if (hp) { sx = CO::template phase_sum<RM>(pr, pi, lr, li); sx = on ? sx : R(0); }
        const R c = on ? c0 : R(1), s = on ? -c1 : R(0);
        CO::template phase<RM>(pr, pi, c, s);
        CO::template phase<RM>(lr, li, c, s);
      })
      case DC_CX: {
        const int cpos = lm & 15, tpos = lm >> 4;
        if (tpos < RB) {
          CPF_BP_SWITCH(RB, tpos, {
            CO::template cnot_reg<BP>(pr, pi, cpos, la);
            CO::template cnot_reg<BP>(lr, li, cpos, la);
          });
        } else {
          CO::cnot_lane(pr, pi, cpos, 1 << (tpos - RB), la);
          CO::cnot_lane(lr, li, cpos, 1 << (tpos - RB), la);
        }
      } break;
      default: break;
    }
    if (hp) {
      if ((d.x & 0xffu) >= DC_PHASE0) {
        if (second) acc[7] = sx; else acc[6] = sx;
      } else if (second) {
        acc[3] = sx; acc[4] = sy; acc[5] = sz;
      } else {
        acc[0] = sx; acc[1] = sy; acc[2] = sz;
      }
      if (d.x & (DF_REDUCE << 16)) {
        __syncwarp();
        reduce8_store<TPS>(acc, s_red + 8 * (d.y >> 16), coef, ls);
      }
    }
  }
  }
};

template <typename R, int NQ, int RB, int CPT, bool SINGLE>
struct InterpSweepMT : InterpSweep<R, NQ, RB, CPT, SINGLE> {
  static constexpr bool MULTI_TARGET = true;
};

// Layered template: surface SU2 gate on every qubit (slot q), then K blocks; block k acts on the
// qubit pair of position k % NBL of the layer: phase gate (slot k), then SU2 on the pair's lower
// qubit (slot NQ + 2k) and on its higher qubit (slot NQ + 2k + 1).  LOQ / HIQ pack the layer's qubit
// pairs, 4 bits per block.  program.cpp (detect_layered) renumbers the slots into this order.
template <typename R, int NQ, int RB, int CPT, bool SINGLE, int NBL, unsigned long long LOQ,
          unsigned long long HIQ>
struct LayerSweep {
  using C = Cfg<R, NQ, RB, CPT, SINGLE>;
  using CO = Cols<R, RB, CPT>;
  using T = VT<R, CPT>;
  using V = typename T::V;
  static constexpr int NA = C::NA, LB = C::LB, TPS = C::TPS;
  static constexpr bool USES_SCHED = false;
  static __host__ __device__ constexpr int lo_q(int j) { return (int)((LOQ >> (4 * j)) & 15); }
  static __host__ __device__ constexpr int hi_q(int j) { return (int)((HIQ >> (4 * j)) & 15); }

  // ---- single gates at a compile-time amplitude-bit position ----
  template <int BP>
  static __device__ __forceinline__ void su2_fwd(V (&re)[NA], V (&im)[NA], const R* cf, int la) {
    R c0, c1, c2, c3;
    Vec4Load<R>::ld(cf, c0, c1, c2, c3);
    if constexpr (BP < RB) {
      CO::template su2_reg<BP>(re, im, c0, c1, c2, c3);
    } else {
      constexpr int lm = 1 << (BP - RB);
      CO::su2_lane(re, im, lm, (la & lm) != 0, c0, c1, c2, c3);
    }
  }
  template <int BP>
  static __device__ __forceinline__ void su2_bwd(V (&pr)[NA], V (&pi)[NA], V (&lr)[NA], V (&li)[NA],
                                                 const R* cf, int la, R& sx, R& sy, R& sz) {
    R c0, c1, c2, c3;
    Vec4Load<R>::ld(cf, c0, c1, c2, c3);
    if constexpr (BP < RB) {
      CO::template pauli_reg<BP>(pr, pi, lr, li, sx, sy, sz);
      CO::template su2_reg<BP>(pr, pi, c0, -c1, -c2, -c3);
      CO::template su2_reg<BP>(lr, li, c0, -c1, -c2, -c3);
    } else {
      constexpr int lm = 1 << (BP - RB);
      CO::bwd_lane(pr, pi, lr, li, lm, (la & lm) != 0, true, c0, c1, c2, c3, sx, sy, sz);
    }
  }
  template <int PA, int PB> struct Ph {
    static constexpr int RM = (PA < RB ? 1 << PA : 0) | (PB < RB ? 1 << PB : 0);
    static constexpr int LM = (PA >= RB ? 1 << (PA - RB) : 0) | (PB >= RB ? 1 << (PB - RB) : 0);
  };
  template <int PA, int PB>
  static __device__ __forceinline__ void phase_fwd(V (&re)[NA], V (&im)[NA], const R* cf, int la) {
    using H = Ph<PA, PB>;
    R c = cf[0], s = cf[1];
    if constexpr (H::LM != 0) {
      const bool on = (la & H::LM) == H::LM;
      c = on ? c : R(1); s = on ? s : R(0);
    }
    CO::template phase<H::RM>(re, im, c, s);
  }
  template <int PA, int PB>
  static __device__ __forceinline__ void phase_bwd(V (&pr)[NA], V (&pi)[NA], V (&lr)[NA], V (&li)[NA],
                                                   const R* cf, int la, R& s11) {
    using H = Ph<PA, PB>;
    R c = cf[0], s = -cf[1];
    s11 = CO::template phase_sum<H::RM>(pr, pi, lr, li);
    if constexpr (H::LM != 0) {
      const bool on = (la & H::LM) == H::LM;
      c = on ? c : R(1); s = on ? s : R(0); s11 = on ? s11 : R(0);
    }
    CO::template phase<H::RM>(pr, pi, c, s);
    CO::template phase<H::RM>(lr, li, c, s);
  }

  // ---- forward ----
  template <int Q>
  static __device__ __forceinline__ void surface_fwd(V (&pr)[NA], V (&pi)[NA], const R* coef, int la) {
    if constexpr (Q < NQ) {
      su2_fwd<NQ - 1 - Q>(pr, pi, coef + 8 * Q, la);
      surface_fwd<Q + 1>(pr, pi, coef, la);
    }
  }
  template <int J>
  static __device__ __forceinline__ void blocks_fwd(int k0, int K, const R* cs, const R* cph, int la,
                                                    V (&pr)[NA], V (&pi)[NA]) {
    if constexpr (J < NBL) {
      if (k0 + J >= K) return;
      constexpr int PA = NQ - 1 - lo_q(J), PB = NQ - 1 - hi_q(J);
      phase_fwd<PA, PB>(pr, pi, cph + 4 * J, la);
      su2_fwd<PA>(pr, pi, cs + 16 * J, la);
      su2_fwd<PB>(pr, pi, cs + 16 * J + 8, la);
      blocks_fwd<J + 1>(k0, K, cs, cph, la, pr, pi);
    }
  }
  static __device__ __forceinline__ void forward(const KParams<R>& p, R* coef, const uint2*, int la,
                                                 V (&pr)[NA], V (&pi)[NA]) {
    surface_fwd<0>(pr, pi, coef, la);
    const int K = p.n_cp;
    const R* cs = coef + 8 * NQ;
    const R* cph = coef + 8 * p.n_su2;
#pragma unroll 1
    for (int k0 = 0; k0 < K; k0 += NBL) {
      blocks_fwd<0>(k0, K, cs, cph, la, pr, pi);
      cs += 16 * NBL; cph += 4 * NBL;
    }
  }

  // ---- adjoint ----
  // 7 sums of a block (or 6 of two surface gates) -> one transposing butterfly; the lane holding
  // slot s stores it: slots 0-2 -> cfA[0..2], 3-5 -> cfB[0..2], 6 -> cph[0].
  static __device__ __forceinline__ void reduce_store(R (&acc)[8], int ls, R* cfA, R* cfB, R* cph) {
    int slot0; bool writer;
    reduce8<TPS>(acc, ls, slot0, writer);
    if (writer) {
#pragma unroll
      for (int k = 0; k < Red8<TPS>::CNT; ++k) {
        const int s = slot0 + k;
        R* dst = s < 3 ? cfA + s : (s < 6 ? cfB + (s - 3) : cph);
        if (s < 3 || (s < 6 && cfB != nullptr) || (s == 6 && cph != nullptr)) *dst = acc[k];
      }
    }
  }
  template <int J>
  static __device__ __forceinline__ void blocks_bwd(int k0, int K, R* cs, R* cph, int la, int ls,
                                                    V (&pr)[NA], V (&pi)[NA], V (&lr)[NA], V (&li)[NA]) {
    if constexpr (J >= 0) {
      if (k0 + J < K) {
        constexpr int PA = NQ - 1 - lo_q(J), PB = NQ - 1 - hi_q(J);
        R acc[8];
        acc[7] = R(0);
        su2_bwd<PB>(pr, pi, lr, li, cs + 16 * J + 8, la, acc[3], acc[4], acc[5]);
        su2_bwd<PA>(pr, pi, lr, li, cs + 16 * J, la, acc[0], acc[1], acc[2]);
        phase_bwd<PA, PB>(pr, pi, lr, li, cph + 4 * J, la, acc[6]);
        __syncwarp();
        reduce_store(acc, ls, cs + 16 * J, cs + 16 * J + 8, cph + 4 * J);
      }
      blocks_bwd<J - 1>(k0, K, cs, cph, la, ls, pr, pi, lr, li);
    }
  }
  template <int Q>
  static __device__ __forceinline__ void surface_bwd(R* coef, int la, int ls, V (&pr)[NA], V (&pi)[NA],
                                                     V (&lr)[NA], V (&li)[NA]) {
    if constexpr (Q >= 0) {
      R acc[8];
      acc[3] = acc[4] = acc[5] = acc[6] = acc[7] = R(0);
      su2_bwd<NQ - 1 - Q>(pr, pi, lr, li, coef + 8 * Q, la, acc[0], acc[1], acc[2]);
      if constexpr (Q >= 1) su2_bwd<NQ - Q>(pr, pi, lr, li, coef + 8 * (Q - 1), la, acc[3], acc[4], acc[5]);
      __syncwarp();
      reduce_store(acc, ls, coef + 8 * Q, Q >= 1 ? coef + 8 * (Q - 1) : nullptr, nullptr);
      surface_bwd<Q - 2>(coef, la, ls, pr, pi, lr, li);
    }
  }
  static __device__ __forceinline__ void backward(const KParams<R>& p, R* coef, const uint2*, const uint16_t*,
                                                  int la, int ls, V (&pr)[NA], V (&pi)[NA], V (&lr)[NA],
                                                  V (&li)[NA]) {
    const int K = p.n_cp;
    R* cph0 = coef + 8 * p.n_su2;
#pragma unroll 1
    for (int k0 = K > 0 ? ((K - 1) / NBL) * NBL : -1; k0 >= 0; k0 -= NBL)
      blocks_bwd<NBL - 1>(k0, K, coef + 8 * NQ + 16 * k0, cph0 + 4 * k0, la, ls, pr, pi, lr, li);
    surface_bwd<NQ - 1>(coef, la, ls, pr, pi, lr, li);
  }
};

template <typename R, int NQ, int RB, int CPT, bool SINGLE, typename SW>
__global__ void __launch_bounds__(Cfg<R, NQ, RB, CPT, SINGLE>::BLOCK, min_blocks<R, RB, CPT, Cfg<R, NQ, RB, CPT, SINGLE>::BLOCK>())
engine_kernel(const KParams<R> p) {
  using C = Cfg<R, NQ, RB, CPT, SINGLE>;
  using CO = Cols<R, RB, CPT>;
  using T = VT<R, CPT>;
  using V = typename T::V;
  constexpr int N = C::N, TPS = C::TPS, SPB = C::SPB, LB = C::LB, NA = C::NA;
  constexpr bool MT = IsMultiTarget<SW>::value;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t s_bar;
  R* s_target = reinterpret_cast<R*>(smem_raw);
  uint2* s_dec = reinterpret_cast<uint2*>(smem_raw + p.target_bytes);
  uint16_t* s_red = reinterpret_cast<uint16_t*>(s_dec + ((p.n_sched + 1) & ~1));
  R* s_coef = reinterpret_cast<R*>(s_red + 8 * p.n_red);

  const int tid = threadIdx.x;
  const bool need_target = !MT && (p.mode == M_ADAM || p.mode == M_LOSSGRAD);

  // ---- prologue: TMA-stage the target, copy the decoded schedule and the reduce tables ----
  if (need_target) {
    if (tid == 0) {
      mbar_init(&s_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      mbar_expect_tx(&s_bar, (uint32_t)p.target_bytes);
      tma_bulk_g2s(s_target, p.target_packed, (uint32_t)p.target_bytes, &s_bar);
    }
  }
  if constexpr (SW::USES_SCHED) {
    for (int i = tid; i < p.n_sched; i += C::BLOCK) s_dec[i] = reinterpret_cast<const uint2*>(p.dec)[i];
    for (int i = tid; i < 8 * p.n_red; i += C::BLOCK) s_red[i] = p.red[i];
  }
  __syncthreads();
  if (need_target) mbar_wait(&s_bar, 0);

  const int sl = tid / TPS;   // sample within the block
  const int ls = tid % TPS;   // lane within the sample
  const long long b_raw = (long long)blockIdx.x * SPB + sl;
  const bool active = b_raw < p.B;
  const long long b = active ? b_raw : p.B - 1;
  const int cg = ls >> LB;                 // column group
  const int la = ls & ((1 << LB) - 1);     // lane part of the amplitude index
  // column mode (n >= 6 unitaries): the batch is B * N single-column problems, b = sample * N + column
  const long long bs = (SINGLE && p.colmode) ? b / N : b;
  const int col0 = (SINGLE && p.colmode) ? (int)(b % N) : cg * CPT;
  const int P = p.P;
  R* coef = s_coef + (size_t)sl * p.coef_stride;
  R* coef_cp = coef + 8 * p.n_su2;
  const R* tgt = s_target;
  if constexpr (MT) tgt = p.target_packed + (size_t)p.target_index[b] * (size_t)((SINGLE ? 1 : N / CPT) * (N + 1) * 2 * CPT);
  const V* tv = reinterpret_cast<const V*>(tgt) + 2 * ((SINGLE ? 0 : cg * (N + 1)) + (la << RB));

  R* ang = p.angles + bs * P;   // M_LOSSGRAD/UNITARY/COTANGENT: read-only use
  R* mom = p.m ? p.m + b * P : nullptr;
  R* vel = p.v ? p.v + b * P : nullptr;
  const uint8_t* frz = p.freeze ? p.freeze + b * P : nullptr;
  const R NN = SINGLE ? R(1) : R(N) * R(N);

  R best = R(0), best_reg_v = R(0);
  if (p.mode == M_ADAM && p.step0 > 0) { best = p.best_regloss[b]; best_reg_v = p.best_reg[b]; }

  // iteration `it` first finishes step it-1 (gradients from the stored Pauli sums, Adam update),
  // then evaluates step it; one call site keeps the parameter-phase code in the binary once.
  for (int it = 0; it <= p.nsteps; ++it) {
    const long long gi = p.step0 + it;
    const int phase = it == 0 ? PH_COEF : (p.mode == M_ADAM ? PH_ADAM : PH_GRAD);
    // ---------------- parameter phase (a sample's threads split the gates) ----------------
    R reg_part = R(0);
    {
      const long long gu = gi - 1;            // the step being finished
      const bool skip_coef = it == p.nsteps;
      R bc1 = R(1), bc2 = R(1), ibc1 = R(1), ibc2 = R(1);
      if (phase == PH_ADAM) {
        bc1 = bias_corr(p.b1, R(gu + 1));
        bc2 = bias_corr(p.b2, R(gu + 1));
        ibc1 = R(1) / bc1; ibc2 = R(1) / bc2;
      }
      // Software pipeline: the metadata, angles and Adam moments of the lane's NEXT gate are requested before the
      // current one is processed (the loop was bound by these L2 round trips: long_scoreboard was the top stall).
      struct PGate { int ax0, ax1, ax2, pi0, pi1, pi2; R th0, th1, th2, mu0, mu1, mu2, nu0, nu1, nu2; };
      const bool want_mom = phase == PH_ADAM && gu != 0;
      auto gate_load = [&](int g) {
        PGate q{-1, -1, -1, -1, -1, -1, R(0), R(0), R(0), R(0), R(0), R(0), R(0), R(0), R(0)};
        if (g < p.n_su2) {
          const Su2Meta* md = p.su2 + g;
          q.ax0 = md->axis[0]; q.ax1 = md->axis[1]; q.ax2 = md->axis[2];
          q.pi0 = md->pidx[0]; q.pi1 = md->pidx[1]; q.pi2 = md->pidx[2];
          q.th0 = q.pi0 >= 0 ? ang[q.pi0] : R(md->cangle[0]);
          q.th1 = q.pi1 >= 0 ? ang[q.pi1] : R(md->cangle[1]);
          q.th2 = q.pi2 >= 0 ? ang[q.pi2] : R(md->cangle[2]);
          if (want_mom) {
            if (q.pi0 >= 0) { q.mu0 = mom[q.pi0]; q.nu0 = vel[q.pi0]; }
            if (q.pi1 >= 0) { q.mu1 = mom[q.pi1]; q.nu1 = vel[q.pi1]; }
            if (q.pi2 >= 0) { q.mu2 = mom[q.pi2]; q.nu2 = vel[q.pi2]; }
          }
        }
        return q;
      };
      PGate nxt = gate_load(ls);
      for (int g = ls; g < p.n_su2; g += TPS) {
        const PGate q = nxt;
        nxt = gate_load(g + TPS);
        R* cf = coef + 8 * g;
        const int ax0 = q.ax0, ax1 = q.ax1, ax2 = q.ax2;
        const int pi0 = q.pi0, pi1 = q.pi1, pi2 = q.pi2;
        R th0 = q.th0, th1 = q.th1, th2 = q.th2;
        if (phase != PH_COEF) {
          const R sx = cf[0], sy = cf[1], sz = cf[2];
          const R c2 = cf[4], s2 = cf[5], c3 = cf[6], s3 = cf[7];
          const R C2 = c2 * c2 - s2 * s2, S2 = R(2) * c2 * s2;
          const R C3 = c3 * c3 - s3 * s3, S3 = R(2) * c3 * s3;
          if (pi2 >= 0)
            apply_grad(p, active, b, phase, gu, bc1, bc2, ibc1, ibc2, ang, mom, vel, frz, pi2, sel3(ax2, sx, sy, sz), th2, q.mu2, q.nu2);
          if (pi1 >= 0) {
            R x = ax1 == 0, y = ax1 == 1, z = ax1 == 2;
            rot_axis(ax2, C3, S3, x, y, z);
            apply_grad(p, active, b, phase, gu, bc1, bc2, ibc1, ibc2, ang, mom, vel, frz, pi1, x * sx + y * sy + z * sz, th1, q.mu1, q.nu1);
          }
          if (pi0 >= 0) {
            R x = ax0 == 0, y = ax0 == 1, z = ax0 == 2;
            rot_axis(ax1, C2, S2, x, y, z);
            rot_axis(ax2, C3, S3, x, y, z);
            apply_grad(p, active, b, phase, gu, bc1, bc2, ibc1, ibc2, ang, mom, vel, frz, pi0, x * sx + y * sy + z * sz, th0, q.mu0, q.nu0);
          }
        }
        if (!skip_coef) {
          R c0 = R(1), s0 = R(0), c1 = R(1), s1 = R(0), c2 = R(1), s2 = R(0);
          if (ax0 >= 0) sincos_r(th0 * R(0.5), s0, c0);
          if (ax1 >= 0) sincos_r(th1 * R(0.5), s1, c1);
          if (ax2 >= 0) sincos_r(th2 * R(0.5), s2, c2);
          R ar, ai, br, bi, a2r, a2i, b2r, b2i;
          su2_of(ax0, c0, s0, ar, ai, br, bi);
          su2_of(ax1, c1, s1, a2r, a2i, b2r, b2i);
          su2_mul(a2r, a2i, b2r, b2i, ar, ai, br, bi);
          su2_of(ax2, c2, s2, a2r, a2i, b2r, b2i);
          su2_mul(a2r, a2i, b2r, b2i, ar, ai, br, bi);
          cf[0] = ar; cf[1] = ai; cf[2] = br; cf[3] = bi;
          cf[4] = c1; cf[5] = s1; cf[6] = c2; cf[7] = s2;
        }
      }
      for (int k = ls; k < p.n_cp; k += TPS) {
        const CpMeta* md = p.cp + k;
        R* cf = coef_cp + 4 * k;
        const int pi = md->pidx;
        const bool pen_on = p.pen.kind != CPF_PEN_NONE && pi >= 0 &&
                            (p.cp_pen ? p.cp_pen[k] != 0 : md->penalised != 0);
        R th = pi >= 0 ? ang[pi] : R(md->cangle);
        if (phase != PH_COEF && pi >= 0) {
          R g = R(-2) * cf[0];
          if (pen_on) {
            R val, slope;
            penalty_eval_fast(p.pen, th, val, slope);
            g = add_rn(g, mul_rn(p.pen.r, slope));
          }
          apply_grad(p, active, b, phase, gu, bc1, bc2, ibc1, ibc2, ang, mom, vel, frz, pi, g, th,
                     want_mom ? mom[pi] : R(0), want_mom ? vel[pi] : R(0));
        }
        if (!skip_coef) {
          R s = R(0), c = R(-1);                 // CZ = diag(1,1,1,-1) exactly
          if (!md->is_cz) sincos_r(th, s, c);
          cf[0] = c; cf[1] = s;
          if (pen_on) {
            R val, slope;
            penalty_eval_fast(p.pen, th, val, slope);
            reg_part += val;
          }
        }
      }
    }
    __syncwarp();
    if (it == p.nsteps) break;
    V pr[NA], pi[NA];
    // ---------------- forward sweep: U e_col ----------------
#pragma unroll
    for (int r = 0; r < NA; ++r) { pr[r] = T::onehot((la << RB) | r, col0); pi[r] = T::bc(R(0)); }
    // (CTA barrier at the sweep starts: the warps of a CTA walk the straight-line sweeps together and share the
    // instruction cache, see heis_impl.cuh; set per launch by launch_one)
    if (p.sync_sweeps & 1) __syncthreads();
    SW::forward(p, coef, s_dec, la, pr, pi);

    if (p.mode == M_UNITARY) {
      if (active) {
#pragma unroll
        for (int r = 0; r < NA; ++r)
#pragma unroll
          for (int k = 0; k < CPT; ++k) {
            R* dst = p.u_out + ((bs * N + ((la << RB) | r)) * N + col0 + k) * 2;
            dst[0] = T::get(pr[r], k); dst[1] = T::get(pi[r], k);
          }
      }
      return;
    }

    // ---------------- loss and adjoint seed ----------------
    V lr[NA], li[NA];
    R loss = R(0), reg = R(0);
    if (p.mode == M_COTANGENT) {
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const R* src = p.cot + ((b * N + ((la << RB) | j)) * N + col0) * 2;
        lr[j] = T::make(src[0], CPT > 1 ? src[2] : R(0));
        li[j] = T::make(src[1], CPT > 1 ? src[3] : R(0));
      }
    } else if (p.loss_kind == CPF_LOSS_RELPHASE) {
      V acc = T::bc(R(0));
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const V vr = tv[2 * j], vi = tv[2 * j + 1];
        const V w = T::fma(vi, vi, T::mul(vr, vr));
        const V q = T::fma(pi[j], pi[j], T::mul(pr[j], pr[j]));
        acc = T::fma(w, q, acc);
        const V ws = T::mul(w, T::bc(R(-1) / R(N)));
        lr[j] = T::mul(ws, pr[j]); li[j] = T::mul(ws, pi[j]);
      }
      R a = sample_sum<TPS>(T::hsum(acc));
      reg = sample_sum<TPS>(reg_part);
      loss = R(1) - a / R(N);
    } else {
      V trp = T::bc(R(0)), tip = trp, tin = trp;
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const V vr = tv[2 * j], vi = tv[2 * j + 1];
        trp = T::fma(vr, pr[j], trp); trp = T::fma(vi, pi[j], trp);
        tip = T::fma(vr, pi[j], tip); tin = T::fma(vi, pr[j], tin);
      }
      const R tr = sample_sum<TPS>(T::hsum(trp));
      const R ti = sample_sum<TPS>(T::hsum(T::sub(tip, tin)));
      reg = sample_sum<TPS>(reg_part);
      const R ab = sqrt_r(tr * tr + ti * ti);
      loss = R(1) - mul_rn(ab, ab) / NN;
      const V a = T::bc(-tr / NN), bq = T::bc(ti / NN), nb = T::bc(-ti / NN);
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const V vr = tv[2 * j], vi = tv[2 * j + 1];
        lr[j] = T::fma(bq, vi, T::mul(a, vr));
        li[j] = T::fma(nb, vr, T::mul(a, vi));
      }
    }
    reg = mul_rn(p.pen.r, reg);

    if (p.mode == M_LOSSGRAD) {
      if (active && ls == 0) {
        p.loss_out[b] = loss;
        if (p.reg_out) p.reg_out[b] = reg;
      }
      if (!p.grad_out) return;
    } else if (p.mode == M_ADAM) {
      const R regloss = add_rn(loss, reg);
      bool improved;
      if (gi == 0) {
        improved = true;
        if (active && ls == 0) { p.init_regloss[b] = regloss; p.init_reg[b] = reg; }
      } else {
        improved = regloss < best;
      }
      if (improved) {
        best = regloss; best_reg_v = reg;
        if (active)
          for (int i = ls; i < P; i += TPS) p.best_params[b * P + i] = ang[i];
      }
      if (active && p.hist_regloss && ls == 0 && gi < p.hist_len)
        p.hist_regloss[b * p.hist_len + gi] = regloss;
      if (active && p.hist_params && gi == 0)
        for (int i = ls; i < P; i += TPS) p.hist_params[b * p.hist_len * P + i] = ang[i];
    }

    // ---------------- adjoint sweep ----------------
    if (p.sync_sweeps & 2) __syncthreads();
    SW::backward(p, coef, s_dec, s_red, la, ls, pr, pi, lr, li);
    __syncwarp();
  }

  if (p.mode == M_ADAM && active && ls == 0) {
    p.best_regloss[b] = best;
    p.best_reg[b] = best_reg_v;
  }
}

// ---- target packing: row-major complex target -> kernel layout (padded rows) ----------------
// dst index: ((cg * (N + 1) + j) * 2 + part) * CPT + k  with column = cg * CPT + k
template <typename R>
__global__ void pack_target_kernel(const R* __restrict__ src, R* __restrict__ dst, int N, int cpt,
                                   int single) {
  const int groups = single ? 1 : N / cpt;
  const int total = groups * (N + 1) * 2 * cpt;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int k = i % cpt, r = i / cpt;
    int part = r % 2; r /= 2;
    int j = r % (N + 1), cg = r / (N + 1);
    R val = R(0);
    if (j < N) {
      if (single) val = src[j * 2 + part];
      else val = src[(j * N + cg * cpt + k) * 2 + part];
    }
    dst[i] = val;
  }
}

// All targets of a multi-target table in one launch (blockIdx.y = target): the layout of pack_target_kernel, target t
// at dst + t * (packed words of one target).  src: n_targets row-major N x N (single: N) complex arrays.
template <typename R>
__global__ void pack_targets_kernel(const R* __restrict__ src, R* __restrict__ dst, int N, int cpt, int single) {
  const int groups = single ? 1 : N / cpt;
  const int total = groups * (N + 1) * 2 * cpt;
  src += (size_t)blockIdx.y * (single ? N : N * N) * 2;
  dst += (size_t)blockIdx.y * total;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int k = i % cpt, r = i / cpt;
    int part = r % 2; r /= 2;
    int j = r % (N + 1), cg = r / (N + 1);
    R val = R(0);
    if (j < N) {
      if (single) val = src[j * 2 + part];
      else val = src[(j * N + cg * cpt + k) * 2 + part];
    }
    dst[i] = val;
  }
}

}  // namespace cpf
