// Per-row loss terms of the mean-field-control train step and their adjoints.
//
// Each function evaluates, for ONE sample row, every flow pass a loss term of
// /root/reference/cnf_ot/mfc/applications.py needs, adds the row's weighted
// contribution to the loss slots, and immediately back-propagates through the
// passes (re-computing conditioner activations), pushing weight gradients to
// the CTA context.  Nothing per-row is ever written to HBM.
//
//   row_nll            kl_loss_fn                    applications.py:11-86
//   row_sample_terms   reverse_kl_loss_fn            applications.py:129-163
//                      potential_loss_fn             applications.py:176-205
//   row_kinetic        kinetic_loss_fn               applications.py:220-242
//                      kinetic_with_score_loss_fn    applications.py:245-276
//                      flow_matching_loss_fn         applications.py:279-374
// The batch means become sums with the 1/B, 1/b, lambda, T/Tn, D/2 factors
// folded into the per-row weights (they are linear), so partial sums from
// different GPUs add up to the reference's loss and gradient.
#pragma once

#include "flow_math.cuh"

namespace cnfot {

enum ProblemType { kOT = 0, kRWPO = 1, kFP = 2 };
enum PotentialKind { kPotNone = -1, kPotQuadratic = 0, kPotDoubleWell = 1, kPotObstacle = 2 };
enum DriftKind { kDriftGradient = 0, kDriftNonGradient = 1, kDriftLorenz = 2 };
enum LossSlot { kSlotFit0 = 0, kSlotFitT = 1, kSlotPotential = 2, kSlotKinetic = 3, kNumSlots = 8 };

template <typename T>
struct StepConsts {
  int type;        // ProblemType
  int potential;   // PotentialKind used by the potential term (or kPotNone)
  int drift;       // DriftKind (fp only)
  T horizon;       // T
  T a;             // potential / drift coefficient
  T dt, dx;        // finite-difference steps
  T kappa;         // score multiplier: 1/beta (rwpo) or sigma (fp)
  T var_src;       // reverse-KL source variance 2 (T+1) / beta
  T var_tgt;       // reverse-KL target variance 2 / beta
  T w_fit;         // lambda / B               (per KL / reverse-KL row)
  T w_pot;         // 1 / B (rwpo)  or  1 / b  (ot obstacle)
  T w_kin;         // 1 / (2 b Tn) (ot)  or  T / (2 b Tn) (rwpo, fp)
};

// ---- potentials (applications.py:181-191): value and gradient ------------------
template <typename T>
CNFOT_HD T potential_value_grad(int kind, T a, const T* r, int D, T* grad) {
  if (kind == kPotQuadratic) {
    T acc = 0;
    for (int i = 0; i < D; ++i) { acc += r[i] * r[i]; grad[i] = r[i]; }
    return acc / (T)2;
  }
  if (kind == kPotDoubleWell) {
    // (|r - a 1| |r + a 1| / 2)^2 = A B / 4
    T A = 0, B = 0;
    for (int i = 0; i < D; ++i) {
      A += (r[i] - a) * (r[i] - a);
      B += (r[i] + a) * (r[i] + a);
    }
    for (int i = 0; i < D; ++i) grad[i] = ((r[i] - a) * B + (r[i] + a) * A) / (T)2;
    return A * B / (T)4;
  }
  // obstacle: 50 exp(-|r|^2 / 2)
  T acc = 0;
  for (int i = 0; i < D; ++i) acc += r[i] * r[i];
  T v = (T)50 * m_exp(-acc / (T)2);
  for (int i = 0; i < D; ++i) grad[i] = -r[i] * v;
  return v;
}

// ---- drift targets (applications.py:308-372) -----------------------------------
// truth[i] and, given gres[i] = dLoss/d(resid_i) with resid = v - truth, the
// pull-back  gr[j] -= sum_i gres[i] d truth_i / d r_j.
template <typename T>
CNFOT_HD void drift_value(int kind, T a, const T* r, int D, T* truth) {
  if (kind == kDriftGradient) {
    T q = r[0] * r[0] + r[1] * r[1] - (T)4;
    truth[0] = a * (-q * r[0]);
    truth[1] = a * (-q * r[1] - (T)2 * (r[1] - (T)1));
  } else if (kind == kDriftNonGradient) {
    // -a r + 0.5 r J, J = I (x) [[0,1],[-1,0]] (2-D in the reference, :358-363)
    for (int i = 0; i < D; i += 2) {
      truth[i] = -a * r[i] - (T)0.5 * r[i + 1];
      truth[i + 1] = -a * r[i + 1] + (T)0.5 * r[i];
    }
  } else {
    const T s = (T)9;
    truth[0] = (T)10 * (r[1] - r[0]);
    truth[1] = s * r[0] * ((T)28 / s - r[2]) - r[1];
    truth[2] = s * r[0] * r[1] - r[2] * (T)8 / (T)3;
  }
}

template <typename T>
CNFOT_HD void drift_pullback(int kind, T a, const T* r, int D, const T* gres, T* gr) {
  if (kind == kDriftGradient) {
    T x = r[0], y = r[1];
    T q = x * x + y * y - (T)4;
    // truth0 = -a q x ; truth1 = -a (q y + 2 (y - 1))
    T t0x = -a * (q + (T)2 * x * x), t0y = -a * (T)2 * x * y;
    T t1x = -a * (T)2 * x * y, t1y = -a * (q + (T)2 * y * y + (T)2);
    gr[0] -= gres[0] * t0x + gres[1] * t1x;
    gr[1] -= gres[0] * t0y + gres[1] * t1y;
  } else if (kind == kDriftNonGradient) {
    for (int i = 0; i < D; i += 2) {
      gr[i] -= gres[i] * (-a) + gres[i + 1] * (T)0.5;
      gr[i + 1] -= gres[i] * (T)(-0.5) + gres[i + 1] * (-a);
    }
  } else {
    const T s = (T)9;
    T x = r[0], y = r[1], z = r[2];
    gr[0] -= gres[0] * (T)(-10) + gres[1] * (s * ((T)28 / s - z)) + gres[2] * (s * y);
    gr[1] -= gres[0] * (T)10 + gres[1] * (T)(-1) + gres[2] * (s * x);
    gr[2] -= gres[1] * (-s * x) + gres[2] * (-(T)8 / (T)3);
  }
}

// ---- KL row: -w log p(data | t) --------------------------------------------------
template <typename T, class Net, class DimsT, class Ctx, class SC, class FG>
CNFOT_HD T row_nll(const DimsT& dm, const SC& sc, T t, const T* data, T weight,
                   FG& gfirst, const RowTiles<T, Net>& tl, Ctx& ctx) {
  const int D = dm.D(), L = dm.L();
  if constexpr (kFlow2dInline<DimsT, Ctx>) {
    const bool stash = ctx.stash_on();
    Pass2d<T> p;
    p.in0 = data[0];
    p.in1 = data[1];
    const T ld = flow_pass_2d<T, Net>(sc, t, p, ctx, stash);
    const T x[2] = {p.out0, p.out1};
    const T lp = base_log_prob<T>(x, 2) + ld;
    T g0 = weight * p.out0, g1 = weight * p.out1;
    flow_pass_bwd_2d<T, Net>(sc, t, p, g0, g1, -weight, gfirst, ctx, stash);
    return -weight * lp;
  } else {
    T st[kMaxStateFloats];
    for (int i = 0; i < D; ++i) st[i] = data[i];
    const bool stash = ctx.stash_on();   // forward and backward of the same rows, back to back: keep the activations
    T ld = flow_pass<1, T, Net, DimsT, Ctx>(dm, sc, t, st, tl, ctx, stash);
    const T* x = st + L * D;
    T lp = base_log_prob<T>(x, D) + ld;
    T g[kMaxDim];
    for (int i = 0; i < D; ++i) g[i] = weight * x[i];  // d(-w lp)/dx = w x
    flow_pass_bwd<1, T, Net, DimsT, Ctx>(dm, sc, t, st, g, -weight, gfirst, tl, ctx, stash);
    return -weight * lp;
  }
}

// ---- rows pushed through the sample direction at one time t ----------------------
// do_fit: reverse-KL term  w_fit (log p(y) - log q_t(y));  do_pot: w_pot V(y).
template <typename T, class Net, class DimsT, class Ctx, class SC, class FG>
CNFOT_HD void row_sample_terms(const DimsT& dm, const SC& sc, T t,
                               const T* latent, bool do_fit, bool do_pot,
                               const StepConsts<T>& pc, T* loss_fit, T* loss_pot, FG& gfirst,
                               const RowTiles<T, Net>& tl, Ctx& ctx) {
  const int D = dm.D(), L = dm.L();
  T st[kMaxStateFloats];
  for (int i = 0; i < D; ++i) st[i] = latent[i];
  const bool stash = ctx.stash_on();
  T fldj = flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t, st, tl, ctx, stash);
  const T* y = st + L * D;
  T g[kMaxDim];
  for (int i = 0; i < D; ++i) g[i] = (T)0;
  T gld = (T)0;
  if (do_fit) {
    T lp = base_log_prob<T>(latent, D) - fldj;
    T r2 = (T)0;
    for (int i = 0; i < D; ++i) r2 += y[i] * y[i];
    const T half_log_2pi = (T)0.91893853320467274178;
    // log of the time-interpolated reference density (applications.py:159-163)
    T w1 = (pc.horizon - t) / pc.horizon, w2 = t / pc.horizon;
    T l1 = -(T)0.5 * r2 / pc.var_src - (T)D * (half_log_2pi + (T)0.5 * m_log(pc.var_src));
    T l2 = -(T)0.5 * r2 / pc.var_tgt - (T)D * (half_log_2pi + (T)0.5 * m_log(pc.var_tgt));
    T logq, coef;  // coef = -d log q / d y_i / y_i
    if (w2 <= (T)0) {
      logq = l1 + m_log(w1);
      coef = (T)1 / pc.var_src;
    } else if (w1 <= (T)0) {
      logq = l2 + m_log(w2);
      coef = (T)1 / pc.var_tgt;
    } else {
      T a1 = l1 + m_log(w1), a2 = l2 + m_log(w2);
      T m = m_max(a1, a2);
      T e1 = m_exp(a1 - m), e2 = m_exp(a2 - m);
      logq = m + m_log(e1 + e2);
      coef = (e1 / pc.var_src + e2 / pc.var_tgt) / (e1 + e2);
    }
    *loss_fit += pc.w_fit * (lp - logq);
    for (int i = 0; i < D; ++i) g[i] += pc.w_fit * coef * y[i];
    gld -= pc.w_fit;
  }
  if (do_pot) {
    T gp[kMaxDim];
    T v = potential_value_grad<T>(pc.potential, pc.a, y, D, gp);
    *loss_pot += pc.w_pot * v;
    for (int i = 0; i < D; ++i) g[i] += pc.w_pot * gp[i];
  }
  flow_pass_bwd<0, T, Net, DimsT, Ctx>(dm, sc, t, st, g, gld, gfirst, tl, ctx, stash);
}

// ---- kinetic-energy rows ----------------------------------------------------------
// ot:       v = (r(t+dt/2) - r(t-dt/2)) / dt,  optional obstacle potential at r(t)
// rwpo/fp:  v += kappa * score,  score_i = (log p(r3 + e_i dx/2) - log p(r3 - e_i dx/2)) / dx
//           fp additionally subtracts the drift target.
// Every pass starts from the SAME latent row (the reference reuses one PRNG key).
template <typename T, class Net, class DimsT, class Ctx, class SC, class FG>
CNFOT_HD void row_kinetic(const DimsT& dm, const SC& sc, T t, const T* latent,
                          const StepConsts<T>& pc, T* loss_kin, T* loss_pot, FG& gfirst,
                          const RowTiles<T, Net>& tl, Ctx& ctx) {
  const int D = dm.D(), L = dm.L();
  const bool with_score = pc.type != kOT;
  const bool need_r3 = with_score || pc.potential == kPotObstacle;
  const T t1 = t - pc.dt / (T)2, t2 = t + pc.dt / (T)2;
  T s1[kMaxStateFloats], s2[kMaxStateFloats], s3[kMaxStateFloats];
  for (int i = 0; i < D; ++i) { s1[i] = latent[i]; s2[i] = latent[i]; s3[i] = latent[i]; }
  flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t1, s1, tl, ctx);
  flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t2, s2, tl, ctx);
  if (need_r3) flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t, s3, tl, ctx);
  const T* r1 = s1 + L * D;
  const T* r2 = s2 + L * D;
  const T* r3 = s3 + L * D;
  T g2[kMaxDim], g3[kMaxDim];
  for (int i = 0; i < D; ++i) g3[i] = (T)0;
  if (!with_score) {
    T acc = (T)0;
    for (int i = 0; i < D; ++i) {
      T v = (r2[i] - r1[i]) / pc.dt;
      acc += v * v;
      g2[i] = (T)2 * pc.w_kin * v / pc.dt;
    }
    *loss_kin += pc.w_kin * acc;
    if (pc.potential == kPotObstacle) {
      T gp[kMaxDim];
      T v = potential_value_grad<T>(kPotObstacle, (T)0, r3, D, gp);
      *loss_pot += pc.w_pot * v;
      for (int i = 0; i < D; ++i) g3[i] = pc.w_pot * gp[i];
    }
  } else {
    T truth[kMaxDim], gres[kMaxDim];
    for (int i = 0; i < D; ++i) truth[i] = (T)0;
    if (pc.type == kFP) drift_value<T>(pc.drift, pc.a, r3, D, truth);
    T acc = (T)0;
    for (int i = 0; i < D; ++i) {
      // the two log-prob passes of coordinate i: forward both, then back-propagate
      // both at once -- resid_i depends on no other score component.
      T sp[kMaxStateFloats], sm[kMaxStateFloats];
      for (int j = 0; j < D; ++j) { sp[j] = r3[j]; sm[j] = r3[j]; }
      sp[i] = r3[i] + pc.dx / (T)2;
      sm[i] = r3[i] - pc.dx / (T)2;
      T ldp = flow_pass<1, T, Net, DimsT, Ctx>(dm, sc, t, sp, tl, ctx);
      T ldm = flow_pass<1, T, Net, DimsT, Ctx>(dm, sc, t, sm, tl, ctx);
      T lpp = base_log_prob<T>(sp + L * D, D) + ldp;
      T lpm = base_log_prob<T>(sm + L * D, D) + ldm;
      T score = (lpp - lpm) / pc.dx;
      T resid = (r2[i] - r1[i]) / pc.dt + pc.kappa * score - truth[i];
      acc += resid * resid;
      gres[i] = (T)2 * pc.w_kin * resid;
      g2[i] = gres[i] / pc.dt;
      T glp = gres[i] * pc.kappa / pc.dx;
      T g[kMaxDim];
      for (int j = 0; j < D; ++j) g[j] = -glp * sp[L * D + j];  // d lp / d latent = -x
      flow_pass_bwd<1, T, Net, DimsT, Ctx>(dm, sc, t, sp, g, glp, gfirst, tl, ctx);
      for (int j = 0; j < D; ++j) g3[j] += g[j];
      for (int j = 0; j < D; ++j) g[j] = glp * sm[L * D + j];
      flow_pass_bwd<1, T, Net, DimsT, Ctx>(dm, sc, t, sm, g, -glp, gfirst, tl, ctx);
      for (int j = 0; j < D; ++j) g3[j] += g[j];
    }
    *loss_kin += pc.w_kin * acc;
    if (pc.type == kFP) drift_pullback<T>(pc.drift, pc.a, r3, D, gres, g3);
  }
  T g1[kMaxDim];
  for (int i = 0; i < D; ++i) g1[i] = -g2[i];
  flow_pass_bwd<0, T, Net, DimsT, Ctx>(dm, sc, t2, s2, g2, (T)0, gfirst, tl, ctx);
  flow_pass_bwd<0, T, Net, DimsT, Ctx>(dm, sc, t1, s1, g1, (T)0, gfirst, tl, ctx);
  if (need_r3) flow_pass_bwd<0, T, Net, DimsT, Ctx>(dm, sc, t, s3, g3, (T)0, gfirst, tl, ctx);
}

#if defined(__CUDACC__)
// ---- kinetic rows, the passes of ONE row spread over a group of G consecutive lanes ------------------------------
// A kinetic row is 2-3 sample passes, (rwpo / fp) 2D shifted log-prob passes forward and backward, and 2-3 backward
// sample passes: one thread walking through all of them is the latency of a whole train step when the sub-batch
// (B // 32 rows) does not fill the GPU -- the reference's own default sizes.  Here lane `sub` of a group does
//   phase 1  the sample pass at t - dt/2 (sub 0), t + dt/2 (sub 1), t (sub >= 2: every further lane gets its own r3)
//   phase 2  (score) the log-prob pass at r3 +- dx/2 e_i, i = sub / 2, side = sub % 2, forward and -- straight away, so
//            the activation stash applies -- backward; the score, the residual and the adjoints are exchanged with
//            shuffles inside the group
//   phase 3  the backward sample pass of phase 1's pass (sub 0: -g2, sub 1: +g2, sub 2: g3, others: zero adjoint)
// G = 2 (ot without r3), 4 (ot / obstacle; score terms at D = 2) or the power of two >= 2D (<= 32).  The same sums as
// row_kinetic in another order of additions; the host picks this form when the step is too small to fill the GPU.
template <class Net, class DimsT, class Ctx, class SC, class FG>
__device__ __forceinline__ void row_kinetic_split(const DimsT& dm, const SC& sc, float t, const float* latent,
                                                  const StepConsts<float>& pc, int G, float* loss_kin, float* loss_pot,
                                                  FG& gfirst, const RowTiles<float, Net>& tl, Ctx& ctx) {
  using T = float;
  constexpr unsigned kAll = 0xffffffffu;
  const int D = dm.D(), L = dm.L();
  const unsigned lane = threadIdx.x & 31u, sub = lane & (unsigned)(G - 1), base = lane & ~(unsigned)(G - 1);
  const bool with_score = pc.type != kOT;
  const bool need_r3 = with_score || pc.potential == kPotObstacle;
  const T tq = sub == 0 ? t - pc.dt / (T)2 : (sub == 1 ? t + pc.dt / (T)2 : t);
  T s[kMaxStateFloats];
  for (int i = 0; i < D; ++i) s[i] = latent[i];
  flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, tq, s, tl, ctx);
  T r1[kMaxDim], r2[kMaxDim], r3[kMaxDim], gq[kMaxDim];
  for (int i = 0; i < D; ++i) {
    const T mine = s[L * D + i];
    r1[i] = __shfl_sync(kAll, mine, base);
    r2[i] = __shfl_sync(kAll, mine, base | 1u);
    r3[i] = need_r3 ? __shfl_sync(kAll, mine, base | 2u) : (T)0;
    gq[i] = (T)0;
  }
  if (!with_score) {
    T acc = (T)0;
    for (int i = 0; i < D; ++i) {
      const T v = (r2[i] - r1[i]) / pc.dt;
      acc += v * v;
      const T g2 = (T)2 * pc.w_kin * v / pc.dt;
      gq[i] = sub == 0 ? -g2 : (sub == 1 ? g2 : (T)0);
    }
    if (sub == 0) *loss_kin += pc.w_kin * acc;
    if (pc.potential == kPotObstacle) {
      T gp[kMaxDim];
      const T v = potential_value_grad<T>(kPotObstacle, (T)0, r3, D, gp);
      if (sub == 2) {
        *loss_pot += pc.w_pot * v;
        for (int i = 0; i < D; ++i) gq[i] = pc.w_pot * gp[i];
      }
    }
  } else {
    T truth[kMaxDim];
    for (int i = 0; i < D; ++i) truth[i] = (T)0;
    if (pc.type == kFP) drift_value<T>(pc.drift, pc.a, r3, D, truth);
    const bool active = (int)sub < 2 * D;
    const int ci = active ? (int)(sub >> 1) : 0;
    const bool minus = (sub & 1u) != 0u;
    T sp[kMaxStateFloats];
    for (int j = 0; j < D; ++j) sp[j] = r3[j];
    sp[ci] = r3[ci] + (minus ? -pc.dx : pc.dx) / (T)2;
    const bool stash = ctx.stash_on();   // forward and backward of the same pass, back to back
    const T ld = flow_pass<1, T, Net, DimsT, Ctx>(dm, sc, t, sp, tl, ctx, stash);
    const T lp = base_log_prob<T>(sp + L * D, D) + ld;
    const T lpo = __shfl_xor_sync(kAll, lp, 1);
    const T score = (minus ? lpo - lp : lp - lpo) / pc.dx;
    const T resid = (r2[ci] - r1[ci]) / pc.dt + pc.kappa * score - truth[ci];
    const T gres_mine = active ? (T)2 * pc.w_kin * resid : (T)0;
    if (active && !minus) *loss_kin += pc.w_kin * resid * resid;
    const T glp = (minus ? -gres_mine : gres_mine) * pc.kappa / pc.dx;
    T g[kMaxDim], g3[kMaxDim], gres[kMaxDim];
    for (int j = 0; j < D; ++j) g[j] = -glp * sp[L * D + j];   // d lp / d latent = -x
    flow_pass_bwd<1, T, Net, DimsT, Ctx>(dm, sc, t, sp, g, glp, gfirst, tl, ctx, stash);
    for (int j = 0; j < D; ++j) {
      T v = g[j];
      for (int o = 1; o < G; o <<= 1) v += __shfl_xor_sync(kAll, v, o);
      g3[j] = v;
      gres[j] = __shfl_sync(kAll, gres_mine, base | (unsigned)(2 * j));
    }
    if (pc.type == kFP) drift_pullback<T>(pc.drift, pc.a, r3, D, gres, g3);
    for (int i = 0; i < D; ++i) {
      const T g2 = gres[i] / pc.dt;
      gq[i] = sub == 0 ? -g2 : (sub == 1 ? g2 : (sub == 2 ? g3[i] : (T)0));
    }
  }
  flow_pass_bwd<0, T, Net, DimsT, Ctx>(dm, sc, tq, s, gq, (T)0, gfirst, tl, ctx);
}
#endif

// ---- evaluation energies (forward only) --------------------------------------------------
// One row's  sum_i v_i^2  of utils.calc_kinetic_energy (with_score = false,
// /root/reference/cnf_ot/utils.py:311-340: v = (r(t+dt/2) - r(t-dt/2)) / dt) or of
// utils.calc_score_kinetic_energy (with_score, utils.py:343-389: v += kappa * score, the score by
// central differences of log_prob with step dx).  All passes start from the same latent row.
template <typename T, class Net, class DimsT, class Ctx, class SC>
CNFOT_HD T row_kinetic_value(const DimsT& dm, const SC& sc, T t, const T* latent, T dt,
                             bool with_score, T kappa, T dx, const RowTiles<T, Net>& tl, Ctx& ctx) {
  const int D = dm.D(), L = dm.L();
  T s1[kMaxStateFloats], s2[kMaxStateFloats];
  for (int i = 0; i < D; ++i) { s1[i] = latent[i]; s2[i] = latent[i]; }
  flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t - dt / (T)2, s1, tl, ctx);
  flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t + dt / (T)2, s2, tl, ctx);
  T v[kMaxDim];
  for (int i = 0; i < D; ++i) v[i] = (s2[L * D + i] - s1[L * D + i]) / dt;
  if (with_score) {
    T s3[kMaxStateFloats];
    for (int i = 0; i < D; ++i) s3[i] = latent[i];
    flow_pass<0, T, Net, DimsT, Ctx>(dm, sc, t, s3, tl, ctx);
    const T* r3 = s3 + L * D;
    for (int i = 0; i < D; ++i) {
      T sp[kMaxStateFloats];
      T lp[2];
      for (int side = 0; side < 2; ++side) {
        for (int j = 0; j < D; ++j) sp[j] = r3[j];
        sp[i] = r3[i] + (side == 0 ? dx : -dx) / (T)2;
        T ld = flow_pass<1, T, Net, DimsT, Ctx>(dm, sc, t, sp, tl, ctx);
        lp[side] = base_log_prob<T>(sp + L * D, D) + ld;
      }
      v[i] += kappa * (lp[0] - lp[1]) / dx;
    }
  }
  T acc = (T)0;
  for (int i = 0; i < D; ++i) acc += v[i] * v[i];
  return acc;
}

// ---- optax.adam (scale_by_adam + scale(-lr); cnf_ot/mfc/solvers.py:55,95-96) of the wide engine's device-resident update
// The arithmetic of the fused tail (step_tail / adam_one in flow_kernels.cuh, which keep their own copy: routing the
// fused kernels through these helpers changed their instruction schedule).  Bias corrections of update number `stepno`
// (0-based): 1 - b^(stepno + 1) without the cancellation, -expm1((stepno + 1) log b); float32 is accurate to ~2e-7
// relative here (optax itself evaluates 1 - b ** count in float32)
CNFOT_HD void adam_bias(uint32_t stepno, float b1, float b2, float& c1, float& c2) {
  const float n1 = (float)stepno + 1.f;
  c1 = -expm1f(n1 * logf(b1));
  c2 = -expm1f(n1 * logf(b2));
}
// one parameter: the old moments and parameter (m, v, w) in, the new ones out
CNFOT_HD void adam_elem(float lr, float b1, float b2, float eps, float c1, float c2, float g, float& m, float& v, float& w) {
  m = b1 * m + (1.f - b1) * g;
  v = b2 * v + (1.f - b2) * g * g;
  w = w - lr * (m / c1) / (sqrtf(v / c2) + eps);
}

}  // namespace cnfot
