// Per-row algorithms of the time-conditioned autoregressive RQS flow:
// conditioner MLP forward / backward, one flow pass in either direction with
// its log-det, and the reverse-mode pass that re-computes activations instead
// of storing them.  One "row" is one sample of the batch; on the device one
// thread owns one row and everything below lives in its registers / local
// memory, the conditioner weights are read (broadcast) from shared memory.
//
// Semantics follow the reference exactly (SURVEY.md Appendix A):
//   conditioner          /root/reference/cnf_ot/models/flows.py:46-86
//   per-layer algebra    /root/reference/cnf_ot/models/autoregressive.py:76-136
//   stacking, direction  /root/reference/cnf_ot/models/flows.py:138-175,
//                        /root/reference/cnf_ot/models/conditional.py:147-177,217-243
//
// Everything that is CTA-wide on the device is delegated to a context policy `Ctx`:
//   first_params()               the shared `first` spline parameters (Pp floats)
//   first_knots()                their normalised knots (FirstKnots, built once per kernel)
//   weights(w_off, count)        the weights of the conditioner at blob offset w_off
//                                (device: resident in, or staged into, shared memory)
//   begin()                      the row tiles may be overwritten (device: barrier)
//   commit(w_off, n_in, tiles)   add this row's rank-1 updates of every layer of that
//                                conditioner to the gradient (device: barrier + CTA-wide
//                                reduction of the staged tiles)
// The host test harness uses a plain context.  Control flow is uniform across rows,
// which the device context relies on (it contains CTA-wide barriers).
#pragma once

#include "rqs_math.cuh"

namespace cnfot {

constexpr int kMaxStateFloats = 64;  // (L+1)*D per pass kept in local memory
constexpr int kMaxDim = 32;          // rows wider than this use the GEMM path

// ---- parameter blob layout ---------------------------------------------------
// One flat fp32 buffer ("weights blob"); the gradient buffer has the same
// layout.  Pp = P rounded up to a multiple of 4 so every matrix row is 16-byte
// aligned (padding entries are zero and stay zero).
//   [ first (Pp) ]
//   for l in 0..L-1, for d in 1..D-1:          (d = position in the permutation)
//     W0 ((d+1) x H) b0 (H)  { Wm (H x H) bm (H) }_{m=1..M-1}  Wout (H x Pp) bout (Pp)
// Matrices are (in, out) row-major like haiku's `w`; each bias directly follows
// its matrix so [W; b] is one (in+1) x out matrix.
struct FlowLayout {
  int D, L, M, H, K, P, Pp;
  int mlp_const;     // floats of one MLP excluding the (d+1) x H input matrix
  int layer_stride;  // floats of one flow layer (all its MLPs)
  int total;         // floats of the whole blob
};

inline FlowLayout make_layout(int D, int L, int M, int H, int K) {
  FlowLayout f;
  f.D = D; f.L = L; f.M = M; f.H = H; f.K = K;
  f.P = 3 * K + 1;
  f.Pp = (f.P + 3) / 4 * 4;
  f.mlp_const = H + (M - 1) * (H * H + H) + H * f.Pp + f.Pp;
  // sum_{d=1}^{D-1} [(d+1) H + mlp_const]
  f.layer_stride = (D - 1) * f.mlp_const + H * ((D - 1) * (D + 2) / 2);
  f.total = f.Pp + L * f.layer_stride;
  return f;
}

template <int H, int K, int M>
struct NetCfg {
  static constexpr int kH = H, kK = K, kM = M;
  static constexpr int kP = 3 * K + 1;
  static constexpr int kPp = (kP + 3) / 4 * 4;
  static constexpr int kMlpConst = H + (M - 1) * (H * H + H) + H * kPp + kPp;
};

// Runtime (DC == 0) or compile-time (DC > 0) flow shape.
template <int DC, int LC>
struct Dims {
  static constexpr int kD = DC, kL = LC;   // > 0: compile-time
  int D_, L_;
  CNFOT_HD int D() const { return DC > 0 ? DC : D_; }
  CNFOT_HD int L() const { return LC > 0 ? LC : L_; }
};

template <class Net>
CNFOT_HD int mlp_offset(int D, int layer, int d) {
  int layer_stride = (D - 1) * Net::kMlpConst + Net::kH * ((D - 1) * (D + 2) / 2);
  return Net::kPp + layer * layer_stride + (d - 1) * Net::kMlpConst +
         Net::kH * ((d - 1) * (d + 2) / 2);
}

// coordinate handled at position d of layer l (alternating identity / reversed
// permutations: flows.py:141-143 with minimum_perm=True)
CNFOT_HD int perm_at(int layer, int d, int D) { return (layer & 1) ? (D - 1 - d) : d; }

// ---- 4-wide loads / stores ------------------------------------------------------
template <typename T>
CNFOT_HD void load4(const T* p, T (&v)[4]) {
  v[0] = p[0]; v[1] = p[1]; v[2] = p[2]; v[3] = p[3];
}
template <typename T>
CNFOT_HD void store4(T* p, T a, T b, T c, T d) {
  p[0] = a; p[1] = b; p[2] = c; p[3] = d;
}
#if defined(__CUDA_ARCH__)
template <>
__device__ __forceinline__ void load4<float>(const float* p, float (&v)[4]) {
  float4 q = *reinterpret_cast<const float4*>(p);
  v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
template <>
__device__ __forceinline__ void store4<float>(float* p, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
#endif

// out[0..N) += v * row[0..N)
template <typename T, int N>
CNFOT_HD void axpy_row(T v, const T* row, T* out) {
#pragma unroll
  for (int j = 0; j < N; j += 4) {
    T w[4];
    load4<T>(row + j, w);
#pragma unroll
    for (int q = 0; q < 4; ++q) out[j + q] += v * w[q];
  }
}

// sum_j g[j] * row[j]
template <typename T, int N>
CNFOT_HD T dot_row(const T* g, const T* row) {
  T acc0 = 0, acc1 = 0;
#pragma unroll
  for (int j = 0; j < N; j += 4) {
    T w[4];
    load4<T>(row + j, w);
    acc0 += g[j] * w[0];
    acc1 += g[j + 1] * w[1];
    acc0 += g[j + 2] * w[2];
    acc1 += g[j + 3] * w[3];
  }
  return acc0 + acc1;
}

// ---- per-row tiles ------------------------------------------------------------------
// The activations of one conditioner evaluation live in per-row tiles rather than in
// registers.  On the device every pointer addresses the calling thread's row of a
// CTA-wide shared-memory tile ([128 rows][padded width]): that is exactly the staging
// the CTA-wide weight-gradient reduction (DeviceSink) reads, so nothing is copied
// twice, and the layer loops below can stay rolled (small code: the fully unrolled
// register version overflowed the instruction cache).  On the host they are plain arrays.
// A row is stored as 16-byte chunks; chunk c lives at chunk position c ^ sw (sw_h for the
// H-wide tiles, sw_p for the Pp-wide one).  On the device sw is a per-row XOR swizzle that
// makes the strided 128-bit accesses of the reduction bank-conflict-free without padding
// (see tile_swizzle in device_common.cuh); on the host it is 0.
template <typename T, class Net>
struct RowTiles {
  T* in;                 // [roundup4(n_in)]  MLP input [t, conditioning coords...], zero padded
  T* hid[Net::kM];       // [H]   post-ReLU activations of hidden layer m
  T* gh[Net::kM];        // [H]   adjoint of the pre-activations of hidden layer m
  T* gth;                // [Pp]  adjoint of the raw spline params (the MLP output)
  int sw_h, sw_p;
};

// element offset of the 4-float chunk that starts at logical element j (j % 4 == 0)
CNFOT_HD int chunk_at(int j, int sw) { return ((j >> 2) ^ sw) << 2; }

// The two dense contractions of a hidden / output layer, CUDA-core flavour: the input
// vector is read back from its row tile four entries at a time (rolled loop, small code).
// A context may override them (DeviceCtx with tensor cores: tcgen05 over the same tiles).
//   forward   y[j] = sum_i x[i] W[i][j]          W: (K x N) row-major
//   backward  y[i] = sum_j g[j] W[i][j]          W: (N x K) row-major, g given in registers
template <typename T, int K, int N>
CNFOT_HD void dense_fwd_from_tile(const T* xt, int sw, const T* W, T* y) {
#pragma unroll 1
  for (int i = 0; i < K; i += 4) {
    T a[4];
    load4<T>(xt + chunk_at(i, sw), a);
#pragma unroll
    for (int q = 0; q < 4; ++q) axpy_row<T, N>(a[q], W + (i + q) * N, y);
  }
}
template <typename T, int K, int N>
CNFOT_HD void dense_bwd_from_regs(const T* g, const T* W, T* y) {
#pragma unroll 1
  for (int i = 0; i < N; i += 4) {
#pragma unroll
    for (int q = 0; q < 4; ++q) y[i + q] = dot_row<T, K>(g, W + (i + q) * K);
  }
}

// Conditioner forward: tiles.in -> tiles.hid[*] -> theta (registers).
// `mlp` is the running index of the conditioner, layer * (D-1) + (d-1).
template <typename T, class Net, class Ctx>
CNFOT_HD void mlp_forward(const T* W, int mlp, int n_in, const RowTiles<T, Net>& tl, T* theta,
                          Ctx& ctx) {
  constexpr int H = Net::kH, M = Net::kM, Pp = Net::kPp;
  const T* b0 = W + n_in * H;
  T acc[H];
#pragma unroll
  for (int j = 0; j < H; ++j) acc[j] = b0[j];
#pragma unroll 1
  for (int i = 0; i < n_in; ++i) axpy_row<T, H>(tl.in[i], W + i * H, acc);
#pragma unroll
  for (int j = 0; j < H; ++j) acc[j] = m_max(acc[j], (T)0);
#pragma unroll
  for (int j = 0; j < H; j += 4)
    store4<T>(tl.hid[0] + chunk_at(j, tl.sw_h), acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
  const T* Wm = b0 + H;
#pragma unroll
  for (int m = 1; m < M; ++m) {
    const T* bm = Wm + H * H;
    T y[H];
#pragma unroll
    for (int j = 0; j < H; ++j) y[j] = (T)0;
    ctx.template dense_fwd<H, H>(tl.hid[m - 1], tl.sw_h, acc, Wm, mlp * M + m - 1, y);
#pragma unroll
    for (int j = 0; j < H; ++j) acc[j] = m_max(y[j] + bm[j], (T)0);
#pragma unroll
    for (int j = 0; j < H; j += 4)
      store4<T>(tl.hid[m] + chunk_at(j, tl.sw_h), acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
    Wm = bm + H;
  }
  const T* bo = Wm + H * Pp;
#pragma unroll
  for (int j = 0; j < Pp; ++j) theta[j] = (T)0;
  ctx.template dense_fwd<H, Pp>(tl.hid[M - 1], tl.sw_h, acc, Wm, mlp * M + M - 1, theta);
#pragma unroll
  for (int j = 0; j < Pp; ++j) theta[j] += bo[j];
}

// Conditioner backward (data gradients): given gtheta (registers) fills tiles.gth and
// tiles.gh[*] and returns the adjoint of the inputs in gin[1..n_in) (gin[0], the adjoint
// of t, is not needed).  The weight gradients are taken from the tiles by Ctx::commit.
template <typename T, class Net, class Ctx>
CNFOT_HD void mlp_backward(const T* W, int mlp, int n_in, const RowTiles<T, Net>& tl,
                           const T* gtheta, T* gin, Ctx& ctx) {
  constexpr int H = Net::kH, M = Net::kM, Pp = Net::kPp;
#pragma unroll
  for (int j = 0; j < Pp; j += 4)
    store4<T>(tl.gth + chunk_at(j, tl.sw_p), gtheta[j], gtheta[j + 1], gtheta[j + 2], gtheta[j + 3]);
  const T* Wout = W + n_in * H + H + (M - 1) * (H * H + H);
  T g[H], y[H];
  ctx.template dense_bwd<Pp, H>(tl.gth, tl.sw_p, gtheta, Wout, mlp * M + M - 1, y);
#pragma unroll
  for (int i = 0; i < H; i += 4) {
    T a[4];
    load4<T>(tl.hid[M - 1] + chunk_at(i, tl.sw_h), a);
#pragma unroll
    for (int q = 0; q < 4; ++q) g[i + q] = a[q] > (T)0 ? y[i + q] : (T)0;
    store4<T>(tl.gh[M - 1] + chunk_at(i, tl.sw_h), g[i], g[i + 1], g[i + 2], g[i + 3]);
  }
#pragma unroll
  for (int m = M - 1; m >= 1; --m) {
    const T* Wm = W + n_in * H + H + (m - 1) * (H * H + H);
    ctx.template dense_bwd<H, H>(tl.gh[m], tl.sw_h, g, Wm, mlp * M + m - 1, y);
#pragma unroll
    for (int i = 0; i < H; i += 4) {
      T a[4];
      load4<T>(tl.hid[m - 1] + chunk_at(i, tl.sw_h), a);
#pragma unroll
      for (int q = 0; q < 4; ++q) g[i + q] = a[q] > (T)0 ? y[i + q] : (T)0;
      store4<T>(tl.gh[m - 1] + chunk_at(i, tl.sw_h), g[i], g[i + 1], g[i + 2], g[i + 3]);
    }
  }
#pragma unroll 1
  for (int i = 1; i < n_in; ++i) gin[i] = dot_row<T, H>(g, W + i * H);
}

template <typename T, class Net>
CNFOT_HD void assume_tiles_shared(const RowTiles<T, Net>& tl, bool with_grad) {
  CNFOT_ASSUME_SHARED(tl.in);
#pragma unroll
  for (int m = 0; m < Net::kM; ++m) CNFOT_ASSUME_SHARED(tl.hid[m]);
  if (with_grad) {
#pragma unroll
    for (int m = 0; m < Net::kM; ++m) CNFOT_ASSUME_SHARED(tl.gh[m]);
    CNFOT_ASSUME_SHARED(tl.gth);
  }
}

// Fill tiles.in with [t, cvec[perm(0)], ..., cvec[perm(d-1)]], zero padded to a multiple of 4.
template <typename T, class Net>
CNFOT_HD void fill_mlp_input(const RowTiles<T, Net>& tl, T t, const T* cvec, int layer, int d,
                             int D) {
  tl.in[0] = t;
  for (int j = 0; j < d; ++j) tl.in[1 + j] = cvec[perm_at(layer, j, D)];
  for (int j = d + 1; j < ((d + 4) & ~3); ++j) tl.in[j] = (T)0;
}

// ---- one pass through the flow -----------------------------------------------
// DIR 0: "sample direction", latent -> physical: layers 0..L-1, each applying
//        Autoregressive.inverse_and_log_det (conditioners read the layer INPUT,
//        spline inverse formula).
// DIR 1: "log-prob direction", physical -> latent: layers L-1..0, each applying
//        Autoregressive.forward_and_log_det (conditioners read the OUTPUT being
//        built, sequential in d, spline forward formula).
// states[0..D) is the input; states[(s+1)*D ..] the result of step s.
//
// Returns the summed log-det of the pass.
template <int DIR, typename T, class Net, class DimsT, class Ctx, class SC>
CNFOT_CALL T flow_pass(const DimsT& dm, const SC& sc, T t, T* states,
                       const RowTiles<T, Net>& tl, Ctx& ctx, bool stash = false) {
  constexpr int K = Net::kK, Pp = Net::kPp, H = Net::kH;
  const int D = dm.D(), L = dm.L();
  if constexpr (!Ctx::kWarpMlp) assume_tiles_shared<T, Net>(tl, false);
  CNFOT_ASSUME_LOCAL(states);
  CNFOT_ASSUME_LOCAL(&ctx);   // the callers' context, tiles and shape live in their local memory: LDL, not generic loads
  CNFOT_ASSUME_LOCAL(&tl);
  CNFOT_ASSUME_LOCAL(&dm);
  T ld_total = (T)0;
#pragma unroll 1
  for (int s = 0; s < L; ++s) {
    const int layer = DIR == 0 ? s : L - 1 - s;
    const T* v = states + s * D;
    T* u = states + (s + 1) * D;
    const T* cvec = DIR == 0 ? v : u;
#pragma unroll 1
    for (int d = 0; d < D; ++d) {
      const int i = perm_at(layer, d, D);
      SplineState<T, K> st;
      if (d == 0) {
        // the shared, unconditioned `first` spline: knots normalised once per kernel
        rqs_locate_first<DIR == 0, T, K>(v[i], ctx.first_knots(), sc, st);
      } else {
        T theta[Pp];
        if constexpr (Ctx::kWarpMlp) {
          ctx.cond_forward(D, layer, d, t, cvec, theta, false, stash);
        } else {
          const T* W = ctx.weights(mlp_offset<Net>(D, layer, d), (d + 1) * H + Net::kMlpConst);
          CNFOT_ASSUME_SHARED(W);
          fill_mlp_input<T, Net>(tl, t, cvec, layer, d, D);
          mlp_forward<T, Net, Ctx>(W, layer * (D - 1) + d - 1, d + 1, tl, theta, ctx);
        }
        rqs_locate_raw<DIR == 0, T, K>(v[i], theta, sc, st);
        if constexpr (Ctx::kWarpMlp) {
          if (stash) ctx.stash_state(D, layer, d, st);
        }
      }
      T out, ld;
      if (DIR == 0) rqs_inverse_map<T, K>(v[i], st, sc, out, ld);
      else rqs_forward_map<T, K>(v[i], st, sc, out, ld);
      u[i] = out;
      ld_total += ld;
    }
  }
  return ld_total;
}

// Reverse mode of flow_pass.  On entry g[0..D) is the adjoint of the pass
// output (states[L*D..]), gld the adjoint of the summed log-det; on exit g is
// the adjoint of the pass input.  gfirst accumulates the knot adjoints of the
// shared `first` spline (pulled back to its raw parameters and flushed to the sink
// once per kernel).  Conditioner activations are re-computed, not stored.
template <int DIR, typename T, class Net, class DimsT, class Ctx, class SC>
CNFOT_CALL void flow_pass_bwd(const DimsT& dm, const SC& sc, T t, const T* states,
                              T* g, T gld, FirstGrad<T, Net::kK>& gfirst, const RowTiles<T, Net>& tl, Ctx& ctx,
                              bool stash = false) {
  constexpr int K = Net::kK, Pp = Net::kPp, H = Net::kH;
  const int D = dm.D(), L = dm.L();
  if constexpr (!Ctx::kWarpMlp) assume_tiles_shared<T, Net>(tl, true);
  CNFOT_ASSUME_LOCAL(states);
  CNFOT_ASSUME_LOCAL(g);
  CNFOT_ASSUME_LOCAL(&gfirst);
  CNFOT_ASSUME_LOCAL(&ctx);
  CNFOT_ASSUME_LOCAL(&tl);
  CNFOT_ASSUME_LOCAL(&dm);
#pragma unroll 1
  for (int s = L - 1; s >= 0; --s) {
    const int layer = DIR == 0 ? s : L - 1 - s;
    const T* v = states + s * D;
    const T* u = states + (s + 1) * D;
    const T* cvec = DIR == 0 ? v : u;
    // DIR 0: any order works, ascending keeps the in-place update valid;
    // DIR 1: descending, so g[coordinate] is complete before it is consumed.
#pragma unroll 1
    for (int dd = 0; dd < D; ++dd) {
      const int d = DIR == 0 ? dd : D - 1 - dd;
      const int i = perm_at(layer, d, D);
      SplineState<T, K> st;
      int w_off = 0;
      const T* W = nullptr;
      if (d == 0) {
        rqs_locate_first<DIR == 0, T, K>(v[i], ctx.first_knots(), sc, st);
      } else if (Ctx::kWarpMlp && stash) {
        // the forward pass of the same rows left the activations and the located spline in the stash
        if constexpr (Ctx::kWarpMlp) ctx.cond_restore(D, layer, d, st, sc.min_slope);
      } else {
        T theta[Pp];
        if constexpr (Ctx::kWarpMlp) {
          ctx.cond_forward(D, layer, d, t, cvec, theta, true);
        } else {
          w_off = mlp_offset<Net>(D, layer, d);
          ctx.begin();  // the tiles of the previous conditioner are free again
          W = ctx.weights(w_off, (d + 1) * H + Net::kMlpConst);
          CNFOT_ASSUME_SHARED(W);
          fill_mlp_input<T, Net>(tl, t, cvec, layer, d, D);
          mlp_forward<T, Net, Ctx>(W, layer * (D - 1) + d - 1, d + 1, tl, theta, ctx);
        }
        rqs_locate_raw<DIR == 0, T, K>(v[i], theta, sc, st);
      }
      KnotAdjoints<T> ka;
      if (DIR == 0) g[i] = rqs_inverse_map_bwd<T, K>(v[i], st, sc, g[i], gld, ka);
      else g[i] = rqs_forward_map_bwd<T, K>(v[i], st, sc, g[i], gld, ka);
      if (d == 0) {
        first_grad_add<T, K>(gfirst, st, ka.gx0, ka.gx1, ka.gy0, ka.gy1, ka.gd0, ka.gd1, ka.gst);
      } else {
        T gtheta[Pp];
#pragma unroll
        for (int j = 0; j < Pp; ++j) gtheta[j] = (T)0;
        scatter_to_raw<T, K>(st, sc, ka.gx0, ka.gx1, ka.gy0, ka.gy1, ka.gd0, ka.gd1, ka.gst, gtheta);
        if constexpr (Ctx::kWarpMlp) {
          ctx.cond_backward(D, layer, d, t, cvec, gtheta, g);
        } else {
          T gin[kMaxDim + 1];
          mlp_backward<T, Net, Ctx>(W, layer * (D - 1) + d - 1, d + 1, tl, gtheta, gin, ctx);
          for (int j = 0; j < d; ++j) g[perm_at(layer, j, D)] += gin[1 + j];
          ctx.commit(w_off, d + 1, tl);
        }
      }
    }
  }
}

// log N(x; 0, I)
template <typename T>
CNFOT_HD T base_log_prob(const T* x, int D) {
  T acc = (T)0;
  for (int i = 0; i < D; ++i) acc += x[i] * x[i];
  return (T)-0.5 * acc - (T)0.91893853320467274178 * (T)D;
}

// p - ((1 - mix) N(y; 0, var0 I) + mix N(y; 0, var1 I)): the error of a density p at y against the reference density of
// the fp evaluation (solvers.py:238-252,270-276), for density_kernel (flow_kernels.cuh) and the wide engine's density head
// (wide.cu)
CNFOT_HD float ref_mixture_error(float p, const float* y, int D, float mix, float var0, float var1) {
  const float half_log_2pi = 0.91893853320467274178f;
  float r2 = 0.f;
  for (int i = 0; i < D; ++i) r2 += y[i] * y[i];
  const float p0 = m_exp(-0.5f * r2 / var0 - (float)D * (half_log_2pi + 0.5f * m_log(var0)));
  const float p1 = m_exp(-0.5f * r2 / var1 - (float)D * (half_log_2pi + 0.5f * m_log(var1)));
  // the contraction nvcc made of p0 * (1 - mix) + p1 * mix written inline in density_kernel: its code is unchanged
  return p - fmaf(p1, mix, p0 * (1.f - mix));
}

}  // namespace cnfot
