// Isometry loss on 6-8 qubits (DESIGN.md section 2.4): L = 1 - |sum_c <W e_c| U |s_c>|^2 / k^2, where the s_c are the
// k basis states whose ancilla bits are 0 and W is the N x k matrix of their wanted images.
//
// A variant of engine_kernel's single-column interpreter (RB register bits, 2^(n-RB) lanes per column, the split of
// the single-column kernels: RB = 2 on 6-7 qubits, 16 / 32 lanes; RB = 3 on 8 qubits, 32 lanes): one sample is k lane
// groups, one per input column s_c, so a sample spans up to 1024 threads and several warps.  The sample's
// threads build ONE shared coefficient store per step; each group runs the forward sweep from e_{s_c}; the groups'
// partial overlaps are summed in a fixed order through shared memory, and every group seeds its adjoint with the same
// t (the HS seed with NN = k^2 and its own column of W).  The backward sweep must not overwrite coefficients another
// group still reads, so each group stores its gradient sums in its own slots (3 per fused gate, 1 per phase gate);
// the parameter phase adds the k groups' sums in a fixed order.  No floating-point atomics: a sample's results do not
// depend on its batch position or on how a run is split.  Barriers are CTA-wide (__syncthreads): a sample is more than
// a warp, and the samples of a CTA run the same number of steps.
//
// The relative-phase isometry loss (InterpSweepIsoPhase, 2-8 qubits) runs the same kernel with one change: the loss is
// 1 - sum_c |t_c|^2 / k, and each group seeds its adjoint with its own partial t_c (the HS seed with NN = k).
//
// The subspace losses (InterpSweepSub on 6-8 qubits, InterpSweepSubPhase on 2-8) run it with arbitrary input states:
// group c starts its forward sweep from a_c (column c of the packed inputs) instead of e_{s_c}, and the target holds the
// wanted images b_c.  A sample has k' = the next power of two >= k groups, so a CTA stays a whole number of warps; the
// packed columns c >= k of both are zero, so those groups add exactly 0 to every sum, and the loss is normalised by k.
#pragma once
#include <string>

#include "launch.cuh"

namespace cpf {

// Register bits of the isometry kernel on NQ qubits: those of the single-column kernels (engine_rb(NQ, true)), whose
// decoded schedule it runs; a lane group (one column) stays within one warp.
template <int NQ> constexpr int iso_rb() { return NQ == 8 ? 3 : 2; }
// engine_rb(NQ, true) on 2-8 qubits (inst_f32.cu: single_rb_f32, the same in float64): the register bits of the
// relative-phase isometry kernel, which also runs 2-5 qubits
template <int NQ> constexpr int iso_phase_rb() { return NQ == 8 ? 3 : NQ == 4 || NQ == 5 ? 1 : 2; }

// The sweep of iso_kernel with RB_ register bits.  The kernels' sweep types derive from it; they only set RB_ and the
// mode flags: ISOMETRY (always), COTANGENT (InterpSweepIsoCot), PHASES (InterpSweepIsoPhase) and INPUTS
// (InterpSweepSub, InterpSweepSubPhase).
template <typename R, int NQ, int RB_>
struct InterpSweepIsoRB : InterpSweep<R, NQ, RB_, 1, true> {
  using Base = InterpSweep<R, NQ, RB_, 1, true>;
  using CO = typename Base::CO;
  using V = typename Base::V;
  static constexpr int NA = Base::NA, LB = Base::LB, TPS = Base::TPS, RB = RB_;
  static constexpr bool ISOMETRY = true;
  static constexpr bool COTANGENT = false;
  static constexpr bool PHASES = false;
  static constexpr bool INPUTS = false;   // forward sweeps start from p.inputs_packed, not from basis states
  // InterpSweep::backward with the reduced sums stored at `sums` (this group's slots, reduce table re-pointed) instead
  // of over the coefficients, which the other groups of the sample may still be reading.
  static __device__ __forceinline__ void backward_into(const KParams<R>& p, const R* coef, R* sums, const uint2* s_dec,
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
        reduce8_store<TPS>(acc, s_red + 8 * (d.y >> 16), sums, ls);
      }
    }
  }
  }
};

// The isometry loss (one global phase) on 6-8 qubits.
template <typename R, int NQ>
struct InterpSweepIso : InterpSweepIsoRB<R, NQ, iso_rb<NQ>()> {};

// The cotangent mode of iso_kernel (cpf_adjoint_from_cotangent on 6-8 qubits, DESIGN.md section 2.4): a launch item
// is (sample b / n_chunks, column chunk b % n_chunks) with n_chunks = N / k; group c runs input column
// (b % n_chunks) * k + c and seeds its adjoint with that column of the caller's cotangent instead of the loss seed.
// The item's gradient (its groups' sums added in group order) goes to row b of a scratch array that
// launch_cot_reduce sums over the chunks in increasing order.
template <typename R, int NQ>
struct InterpSweepIsoCot : InterpSweepIso<R, NQ> {
  static constexpr bool COTANGENT = true;
};

// The relative-phase isometry loss (CPF_LOSS_ISOMETRY_RELPHASE, DESIGN.md section 2.4), on 2-8 qubits:
// L = 1 - sum_c |t_c|^2 / k with t_c = <W e_c| U |s_c>, W up to a phase per input column.  Group c seeds its adjoint
// with its own t_c / k instead of the shared t / k^2.  The register bits are those of the single-column split on every
// n (iso_phase_rb), so on 4-5 qubits they differ from iso_rb.
template <typename R, int NQ>
struct InterpSweepIsoPhase : InterpSweepIsoRB<R, NQ, iso_phase_rb<NQ>()> {
  static constexpr bool PHASES = true;
};

// The subspace loss (CPF_LOSS_SUBSPACE, one global phase) on 6-8 qubits: L = 1 - |sum_c <b_c| U |a_c>|^2 / k^2.
template <typename R, int NQ>
struct InterpSweepSub : InterpSweepIso<R, NQ> {
  static constexpr bool INPUTS = true;
};

// The relative-phase subspace loss (CPF_LOSS_SUBSPACE_RELPHASE) on 2-8 qubits: L = 1 - sum_c |<b_c| U |a_c>|^2 / k.
template <typename R, int NQ>
struct InterpSweepSubPhase : InterpSweepIsoPhase<R, NQ> {
  static constexpr bool INPUTS = true;
};

// words per group of the per-group gradient sums (odd: the groups of a sample store the same slot in distinct banks)
__host__ __device__ inline int iso_sum_stride(int n_su2, int n_cp) { return (3 * n_su2 + n_cp) | 1; }

// Gradient sums of the k groups of a sample, added in group order.
template <typename R>
struct GroupSums {
  const R* sums;
  int stride, k, n_su2;
  __device__ __forceinline__ void su2(int g, R& sx, R& sy, R& sz) const {
    const R* s = sums + 3 * g;
    sx = s[0]; sy = s[1]; sz = s[2];
    for (int c = 1; c < k; ++c) {
      s += stride;
      sx += s[0]; sy += s[1]; sz += s[2];
    }
  }
  __device__ __forceinline__ R cp(int kk) const {
    const R* s = sums + 3 * n_su2 + kk;
    R x = s[0];
    for (int c = 1; c < k; ++c) x += s[(size_t)c * stride];
    return x;
  }
};

// engine_kernel's parameter phase (kept as a copy: factoring it out of engine_kernel changed the code generated for
// the existing kernels).  The `nthr` threads of a sample (this one is `ls`) split the gates; unless phase == PH_COEF
// each gate first finishes step gi - 1 from its gradient sums (read through `sums`: GroupSums), then, unless
// `skip_coef`, writes its coefficients for step gi into `coef`.  Returns this thread's share of the penalty value.
template <typename R, typename Sums>
__device__ __forceinline__ R iso_param_phase(const KParams<R>& p, R* coef, const Sums& sums, int ls, int nthr, int phase,
                                             long long gi, bool skip_coef, bool active, long long b, R* ang, R* mom,
                                             R* vel, const uint8_t* frz) {
  R reg_part = R(0);
    const long long gu = gi - 1;            // the step being finished
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
    for (int g = ls; g < p.n_su2; g += nthr) {
      const PGate q = nxt;
      nxt = gate_load(g + nthr);
      R* cf = coef + 8 * g;
      const int ax0 = q.ax0, ax1 = q.ax1, ax2 = q.ax2;
      const int pi0 = q.pi0, pi1 = q.pi1, pi2 = q.pi2;
      R th0 = q.th0, th1 = q.th1, th2 = q.th2;
      if (phase != PH_COEF) {
        R sx, sy, sz;
        sums.su2(g, sx, sy, sz);
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
    for (int k = ls; k < p.n_cp; k += nthr) {
      const CpMeta* md = p.cp + k;
      R* cf = coef + 8 * p.n_su2 + 4 * k;
      const int pi = md->pidx;
      const bool pen_on = p.pen.kind != CPF_PEN_NONE && pi >= 0 &&
                          (p.cp_pen ? p.cp_pen[k] != 0 : md->penalised != 0);
      R th = pi >= 0 ? ang[pi] : R(md->cangle);
      if (phase != PH_COEF && pi >= 0) {
        R g = R(-2) * sums.cp(k);
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
  return reg_part;
}

// basis index of input column c: the bits of c deposited, in order, on the amplitude-index bits that are not ancillas
__device__ __forceinline__ int iso_column(int c, int amask, int nq) {
  int s = 0;
  for (int bit = 0; bit < nq; ++bit)
    if (!((amask >> bit) & 1)) { s |= (c & 1) << bit; c >>= 1; }
  return s;
}

// Shared memory per sample (words of R): coefficient store, k groups of gradient sums, k x {Re t_c, Im t_c, reg_c}.
__host__ __device__ inline int iso_sample_words(int coef_stride, int k, int sum_stride) {
  return (coef_stride + k * sum_stride + 3 * k + 3) & ~3;
}

template <typename R, int NQ, typename SW>
__global__ void __launch_bounds__(NQ <= 6 ? 512 : 1024, 1) iso_kernel(const KParams<R> p) {
  constexpr int RB = SW::RB;
  using C = Cfg<R, NQ, RB, 1, true>;
  using T = VT<R, 1>;
  using V = typename T::V;
  constexpr int N = C::N, GT = C::TPS, NA = C::NA;
  static_assert(SW::ISOMETRY, "iso_kernel runs the isometry sweep type");

  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint2* s_dec = reinterpret_cast<uint2*>(smem_raw);
  uint16_t* s_red = reinterpret_cast<uint16_t*>(s_dec + ((p.n_sched + 1) & ~1));
  R* s_smp = reinterpret_cast<R*>(s_red + 8 * p.n_red);

  const int tid = threadIdx.x, k = p.iso_k, spt = k * GT;
  const int sum_stride = iso_sum_stride(p.n_su2, p.n_cp);
  // the schedule, with the reduce table re-pointed from the coefficient words to the per-group sum slots
  for (int i = tid; i < p.n_sched; i += blockDim.x) s_dec[i] = reinterpret_cast<const uint2*>(p.dec)[i];
  for (int i = tid; i < 8 * p.n_red; i += blockDim.x) {
    const int o = p.red[i];
    s_red[i] = o == 0xffff ? 0xffff
                           : (o < 8 * p.n_su2 ? 3 * (o >> 3) + (o & 7) : 3 * p.n_su2 + ((o - 8 * p.n_su2) >> 2));
  }
  __syncthreads();

  const int sl = tid / spt;          // sample within the block
  const int ls = tid % spt;          // thread within the sample
  const int grp = ls / GT;           // input column of this thread's group
  const int la = ls % GT;            // lane part of the amplitude index
  const long long b_raw = (long long)blockIdx.x * (blockDim.x / spt) + sl;
  const bool active = b_raw < p.B;
  const long long b = active ? b_raw : p.B - 1;
  const int P = p.P;
  R* coef = s_smp + (size_t)sl * iso_sample_words(p.coef_stride, k, sum_stride);
  R* sums = coef + p.coef_stride;
  R* part = sums + (size_t)k * sum_stride;         // [k][3]: Re t_c, Im t_c, penalty share of group c
  const R* tv = SW::COTANGENT ? nullptr : p.target_packed + 2 * ((size_t)grp * N + (la << RB));
  // cotangent mode: item b is column chunk b % (N / k) of sample b / (N / k)
  const long long bs = SW::COTANGENT ? b / (N / k) : b;
  const int col0 = SW::COTANGENT ? (int)(b % (N / k)) * k + grp : iso_column(grp, p.iso_amask, NQ);

  R* ang = p.angles + bs * P;
  R* mom = p.m ? p.m + b * P : nullptr;
  R* vel = p.v ? p.v + b * P : nullptr;
  const uint8_t* frz = p.freeze ? p.freeze + b * P : nullptr;
  const R kn = SW::INPUTS ? R(p.sub_k) : R(k);     // the loss's k: the caller's, not the padded group count
  const R NN = kn * kn;

  R best = R(0), best_reg_v = R(0);
  if (p.mode == M_ADAM && p.step0 > 0) { best = p.best_regloss[b]; best_reg_v = p.best_reg[b]; }

  for (int it = 0; it <= p.nsteps; ++it) {
    const long long gi = p.step0 + it;
    const int phase = it == 0 ? PH_COEF : (p.mode == M_ADAM ? PH_ADAM : PH_GRAD);
    const R reg_part = iso_param_phase(p, coef, GroupSums<R>{sums, sum_stride, k, p.n_su2}, ls, spt, phase, gi,
                                       it == p.nsteps, active, b, ang, mom, vel, frz);
    __syncthreads();
    if (it == p.nsteps) break;
    V pr[NA], pi[NA];
    if constexpr (SW::INPUTS) {
      // this group's amplitudes of a_grp (column-major packed, like the target)
      const R* av = p.inputs_packed + 2 * ((size_t)grp * N + (la << RB));
#pragma unroll
      for (int r = 0; r < NA; ++r) { pr[r] = T::bc(av[2 * r]); pi[r] = T::bc(av[2 * r + 1]); }
    } else {
#pragma unroll
      for (int r = 0; r < NA; ++r) { pr[r] = T::onehot((la << RB) | r, col0); pi[r] = T::bc(R(0)); }
    }
    SW::forward(p, coef, s_dec, la, pr, pi);

    if constexpr (SW::COTANGENT) {
      // the adjoint seed is column col0 of cot[bs] (row-major [N][N] complex), read directly
      V lr[NA], li[NA];
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const R* src = p.cot + ((bs * N + ((la << RB) | j)) * N + col0) * 2;
        lr[j] = src[0]; li[j] = src[1];
      }
      SW::backward_into(p, coef, sums + (size_t)grp * sum_stride, s_dec, s_red, la, la, pr, pi, lr, li);
      __syncthreads();
      continue;
    }

    // ---------------- overlap: group partials, then the same fixed-order sum in every thread ----------------
    {
      R trp = R(0), tip = R(0), tin = R(0);
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const R vr = tv[2 * j], vi = tv[2 * j + 1];
        trp = T::fma(vr, pr[j], trp); trp = T::fma(vi, pi[j], trp);
        tip = T::fma(vr, pi[j], tip); tin = T::fma(vi, pr[j], tin);
      }
      const R tr_c = sample_sum<GT>(trp), ti_c = sample_sum<GT>(tip - tin), reg_c = sample_sum<GT>(reg_part);
      if (la == 0) { part[3 * grp] = tr_c; part[3 * grp + 1] = ti_c; part[3 * grp + 2] = reg_c; }
    }
    __syncthreads();
    R tr = part[0], ti = part[1], reg = part[2], loss;
    V lr[NA], li[NA];
    if constexpr (SW::PHASES) {
      // a phase per column: every thread adds sum_c |t_c|^2 and the penalty shares in group order; group grp seeds
      // with its own t_c / k
      R s2 = tr * tr + ti * ti;
      for (int c = 1; c < k; ++c) {
        const R xr = part[3 * c], xi = part[3 * c + 1];
        s2 += xr * xr + xi * xi;
        reg += part[3 * c + 2];
      }
      const R kk = kn;
      loss = R(1) - s2 / kk;
      const R tr_c = part[3 * grp], ti_c = part[3 * grp + 1];
      const V a = T::bc(-tr_c / kk), bq = T::bc(ti_c / kk), nb = T::bc(-ti_c / kk);
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        const V vr = tv[2 * j], vi = tv[2 * j + 1];
        lr[j] = T::fma(bq, vi, T::mul(a, vr));
        li[j] = T::fma(nb, vr, T::mul(a, vi));
      }
    } else {
      for (int c = 1; c < k; ++c) { tr += part[3 * c]; ti += part[3 * c + 1]; reg += part[3 * c + 2]; }
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
          for (int i = ls; i < P; i += spt) p.best_params[b * P + i] = ang[i];
      }
      if (active && p.hist_regloss && ls == 0 && gi < p.hist_len)
        p.hist_regloss[b * p.hist_len + gi] = regloss;
      if (active && p.hist_params && gi == 0)
        for (int i = ls; i < P; i += spt) p.hist_params[b * p.hist_len * P + i] = ang[i];
    }

    // ---------------- adjoint sweep: this group's sums into its own slots ----------------
    SW::backward_into(p, coef, sums + (size_t)grp * sum_stride, s_dec, s_red, la, la, pr, pi, lr, li);
    __syncthreads();
  }

  if (p.mode == M_ADAM && active && ls == 0) {
    p.best_regloss[b] = best;
    p.best_reg[b] = best_reg_v;
  }
}

// Target packing for the 6-8 qubit kernel: W (N x k, row-major complex) -> column-major [k][N] complex, so a group
// reads its column's amplitudes contiguously.
template <typename R>
__global__ void pack_iso_kernel(const R* __restrict__ src, R* __restrict__ dst, int N, int k) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * k * 2; i += gridDim.x * blockDim.x) {
    const int part = i & 1, r = i >> 1, j = r % N, c = r / N;
    dst[i] = src[((size_t)j * k + c) * 2 + part];
  }
}

// The n <= 5 isometry loss as an HS loss: V = 2^a [W at the columns s_c, 0 elsewhere] (N x N) with N = 2^a k.  The HS
// kernels then compute 1 - |t|^2 / k^2 and its gradient (the power-of-two scaling is exact).
template <typename R>
__global__ void pack_iso_hs_kernel(const R* __restrict__ src, R* __restrict__ dst, int nq, int k, int amask) {
  const int N = 1 << nq;
  const R scale = R(N / k);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * N * 2; i += gridDim.x * blockDim.x) {
    const int part = i & 1, r = i >> 1, j = r / N, s = r % N;
    R val = R(0);
    if ((s & amask) == 0) {
      int c = 0, bitc = 0;                       // s -> its column index: gather the non-ancilla bits
      for (int bit = 0; bit < nq; ++bit)
        if (!((amask >> bit) & 1)) { c |= ((s >> bit) & 1) << bitc; ++bitc; }
      val = scale * src[((size_t)j * k + c) * 2 + part];
    }
    dst[i] = val;
  }
}

// The n <= 5 subspace loss as an HS loss: V = (N/k) B A^dag (N x N; src = B then A, each N x k row-major), so
// Tr(V^dag U) = (N/k) sum_c <b_c| U |a_c> and the HS kernels compute 1 - |sum_c t_c|^2 / k^2 and its gradient.  The sum
// over c starts from +0, so with A = the basis columns e_{s_c} and a power-of-two k every entry is bit for bit the one
// pack_iso_hs_kernel writes.
template <typename R>
__global__ void pack_subspace_hs_kernel(const R* __restrict__ src, R* __restrict__ dst, int N, int k) {
  const R scale = R(N) / R(k);
  const R* A = src + (size_t)2 * N * k;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N * N; i += gridDim.x * blockDim.x) {
    const int j = i / N, s = i % N;
    const R* b = src + (size_t)2 * j * k;
    const R* a = A + (size_t)2 * s * k;
    R re = R(0), im = R(0);
    for (int c = 0; c < k; ++c) {           // b_c[j] conj(a_c[s])
      re += b[2 * c] * a[2 * c] + b[2 * c + 1] * a[2 * c + 1];
      im += b[2 * c + 1] * a[2 * c] - b[2 * c] * a[2 * c + 1];
    }
    dst[2 * i] = scale * re;
    dst[2 * i + 1] = scale * im;
  }
}

// grad[b, i] = sum over h of partial[b * n_chunks + h, i], in increasing h (the cotangent mode's chunk sum)
template <typename R>
__global__ void cot_reduce_kernel(const R* __restrict__ partial, R* __restrict__ grad, long long B, int P,
                                  int n_chunks) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < B * P;
       i += (long long)gridDim.x * blockDim.x) {
    const R* s = partial + (i / P) * n_chunks * P + i % P;
    R x = s[0];
    for (int h = 1; h < n_chunks; ++h) x += s[(size_t)h * P];
    grad[i] = x;
  }
}

// host side: geometry of one launch (also reported by cpf_launch_plan)
struct IsoGeometry {
  int spt, spb, block;
  size_t smem;
};
inline IsoGeometry iso_geometry(int n, int rb, int k, int n_su2, int n_cp, int n_sched, int n_red, size_t real_bytes) {
  IsoGeometry g;
  g.spt = k << (n - rb);
  g.spb = g.spt >= 128 ? 1 : 128 / g.spt;
  g.block = g.spb * g.spt;
  const int words = iso_sample_words(coef_stride_words(n_su2, n_cp), k, iso_sum_stride(n_su2, n_cp));
  g.smem = (size_t)((n_sched + 1) & ~1) * 8 + (size_t)n_red * 16 + (size_t)g.spb * words * real_bytes;
  return g;
}

// Columns per launch item of the cotangent mode: 32 (the k = 32 isometry launch shape), halved until the item's
// shared memory fits; a function of the program and the precision only.  0: not even one column fits.
inline int iso_cot_columns(int n, int rb, int n_su2, int n_cp, int n_sched, int n_red, size_t real_bytes) {
  for (int k = 32; k >= 1; k >>= 1)
    if (iso_geometry(n, rb, k, n_su2, n_cp, n_sched, n_red, real_bytes).smem <= 227 * 1024) return k;
  return 0;
}

template <typename R, int NQ, typename SW = InterpSweepIso<R, NQ>>
int launch_iso_sized(KParams<R> p, cudaStream_t st, std::string& err) {
  p.coef_stride = coef_stride_words(p.n_su2, p.n_cp);
  p.sync_sweeps = 0;
  if (engine_rb<R>(NQ, true) != SW::RB) {        // the decoded schedule in p is the one of engine_rb's split
    err = "isometry kernel: register bits differ from the decoded schedule's";
    return CPF_ERR_UNSUPPORTED;
  }
  const IsoGeometry g = iso_geometry(NQ, SW::RB, p.iso_k, p.n_su2, p.n_cp, p.n_sched, p.n_red, sizeof(R));
  if (g.smem > 227 * 1024) {
    err = "program too large for the shared-memory store of the isometry kernel (" + std::to_string(g.smem) + " bytes)";
    return CPF_ERR_UNSUPPORTED;
  }
  auto kern = iso_kernel<R, NQ, SW>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
  if (e != cudaSuccess) { err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); return CPF_ERR_CUDA; }
  const long long grid = (p.B + g.spb - 1) / g.spb;
  if (grid <= 0) return CPF_OK;
  if (grid > 2147483647LL) { err = "batch too large for one launch"; return CPF_ERR_UNSUPPORTED; }
  kern<<<(unsigned)grid, g.block, g.smem, st>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) { err = std::string("kernel launch: ") + cudaGetErrorString(e); return CPF_ERR_CUDA; }
  return CPF_OK;
}

// inst_iso_f32.cu / inst_iso_f64.cu
template <typename R> int launch_iso(const KParams<R>& p, int n_qubits, cudaStream_t st, std::string& err);
// inst_iso_phase_f32.cu / inst_iso_phase_f64.cu: the relative-phase isometry loss on 2-8 qubits
template <typename R> int launch_iso_phase(const KParams<R>& p, int n_qubits, cudaStream_t st, std::string& err);
// cotangent mode: p.B launch items of p.iso_k columns (p.B = batch * N / p.iso_k), gradients to p.grad_out [p.B][P]
template <typename R> int launch_iso_cot(const KParams<R>& p, int n_qubits, cudaStream_t st, std::string& err);
template <typename R> int launch_cot_reduce(const R* partial, R* grad, long long batch, int P, int n_chunks,
                                            cudaStream_t st);
template <typename R> int launch_pack_iso(const R* src, R* dst, int n_qubits, int k, int amask, bool as_hs,
                                          cudaStream_t st);
// inst_sub_f32.cu / inst_sub_f64.cu: the subspace losses on the isometry kernel (p.iso_k = k' groups, p.sub_k = k),
// CPF_LOSS_SUBSPACE on 6-8 qubits and CPF_LOSS_SUBSPACE_RELPHASE on 2-8
template <typename R> int launch_sub(const KParams<R>& p, int n_qubits, cudaStream_t st, std::string& err);
template <typename R> int launch_sub_phase(const KParams<R>& p, int n_qubits, cudaStream_t st, std::string& err);
// V = (N/k) B A^dag into dst (N x N row-major) from src = B then A (pack_subspace_hs_kernel)
template <typename R> int launch_pack_subspace_hs(const R* src, R* dst, int n_qubits, int k, cudaStream_t st);

}  // namespace cpf
