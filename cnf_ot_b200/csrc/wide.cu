// Wide-conditioner engine: the train step (and the flow passes under it) for flows whose conditioner
// MLPs are too large for the fused per-row kernels -- BASELINE config 5: D = 32, 16 layers, hidden 512,
// 139 M parameters.  Same semantics as flow_pass / flow_pass_bwd in flow_math.cuh
// (/root/reference/cnf_ot/models/autoregressive.py:76-136, flows.py:46-86,138-175), restructured
// around the batch instead of the row:
//
//   * the batch is cut into chunks of R rows (default 4 x 148 x 128 = 75 776: every hidden-layer GEMM is exactly
//     four waves of 128 x 256 tiles at two CTAs per SM, and the narrow layers (N = 16 / 48), whose grids are
//     one CTA per 128 rows, get four resident CTAs per SM to hide their load latency -- measured 1.7x faster
//     per row than single-wave chunks whose activations would stay in L2);
//   * a chunk's flow state is a matrix S (R x Kx), row = [x_0 .. x_{D-1} | t | 0 ..], one per flow
//     layer boundary.  The conditioner of (layer, d) reads it DIRECTLY as the A operand of its input
//     GEMM: its (d+1) x H input matrix is scattered once per step into a Kx x H matrix whose row k is
//     the weight row of state column k (zero where the conditioner does not look), so the
//     autoregressive masking and the alternating permutation cost nothing per row;
//   * every dense layer runs on tcgen05 (dense_tc.cu: 3xTF32, TMEM accumulators, TMA-staged prepared
//     weights), the spline + log-det is a per-row kernel on the 16 raw parameters the last GEMM wrote;
//   * backward re-computes a conditioner's activations, differentiates the spline, and runs
//     dgrad (prepared W^T, ReLU mask fused in the epilogue) and wgrad (K-major gathered A^T G,
//     red.global into the gradient blob) per layer; the input adjoints of the first layer are
//     accumulated straight into the chunk's adjoint state G (R x Kx) by the GEMM epilogue.
//
// Loss heads (kl_loss_fn, kinetic_loss_fn, potential_loss_fn; applications.py:11-86,176-242) are small
// per-row kernels between the forward and the backward sweep of a chunk.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "dense_tc.h"
#include "philox.cuh"
#include "wide.h"

namespace cnfot {

namespace {

constexpr int kMaxM = 4;
constexpr int kMaxPass = 5;   // flow passes alive at once: r(t-dt/2), r(t+dt/2), r(t), and the two shifted log-prob passes
constexpr int kThreads = 256;
constexpr int kInWgradSlice = 64;   // state columns per thread in wide_in_wgrad_kernel (KV4 <= 16 float4s)

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
inline int64_t round_up64(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

struct WideDims {
  int D, L, M, H, Pp, Kx;
  int64_t prep_mlp;   // prepared floats of one conditioner (one direction)
};

WideDims make_dims(const FlowLayout& lay) {
  WideDims w;
  w.D = lay.D; w.L = lay.L; w.M = lay.M; w.H = lay.H; w.Pp = lay.Pp;
  // D <= 63: one slice of <= 64 columns in steps of 16.  Wider rows: whole 64-column slices, so that the transposed
  // input GEMM (N = Kx) lands on the 64 / 128 / 256-wide dense_tc tiles and wide_in_wgrad_kernel walks 256-byte slices.
  w.Kx = lay.D + 1 <= kInWgradSlice ? round_up(lay.D + 1, 16) : round_up(lay.D + 1, kInWgradSlice);
  w.prep_mlp = 2 * ((int64_t)w.Kx * w.H + (int64_t)(w.M - 1) * w.H * w.H + (int64_t)w.H * w.Pp);
  return w;
}

__host__ __device__ inline int64_t mlp_blob_offset(const FlowLayout& lay, int layer, int d) {
  return lay.Pp + (int64_t)layer * lay.layer_stride + (int64_t)(d - 1) * lay.mlp_const +
         (int64_t)lay.H * ((d - 1) * (d + 2) / 2);
}

// ---- weight preparation: every matrix of every conditioner into tcgen05 tile order, hi / lo split ----
// blockIdx.y = conditioner (layer * (D-1) + d - 1).  `pf` serves X * W, `pt` (may be NULL) serves G * W^T.
__device__ __forceinline__ void put_split(float* tile_base, int64_t n_cols, int k, int n, float v) {
  // round-to-nearest 3xTF32 split, as dense_prep_kernel
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  const float hi = __uint_as_float(r);
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v - hi));
  float* t = tile_base + (int64_t)(k >> 4) * 2 * n_cols * 16;
  const int p = sw64_pos(n, k & 15);
  t[p] = hi;
  t[n_cols * 16 + p] = __uint_as_float(r);
}

__global__ void __launch_bounds__(kThreads)
wide_prep_kernel(const float* __restrict__ W, FlowLayout lay, WideDims wd, float* __restrict__ prep_fwd,
                 float* __restrict__ prep_T) {
  const int mlp = blockIdx.y;
  const int layer = mlp / (wd.D - 1), d = mlp % (wd.D - 1) + 1, rev = layer & 1;
  const int H = wd.H, Kx = wd.Kx, Pp = wd.Pp;
  const float* w = W + mlp_blob_offset(lay, layer, d);
  float* pf = prep_fwd + (int64_t)mlp * wd.prep_mlp;
  float* pt = prep_T ? prep_T + (int64_t)mlp * wd.prep_mlp : nullptr;
  const int stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  // input layer: state column k -> weight row w0_row(k)
  for (int e = t0; e < Kx * H; e += stride) {
    const int k = e / H, h = e - k * H;
    const int row = w0_row(k, wd.D, d, rev);
    const float v = row >= 0 ? w[(int64_t)row * H + h] : 0.f;
    put_split(pf, H, k, h, v);
    if (pt) put_split(pt, Kx, h, k, v);
  }
  pf += 2 * (int64_t)Kx * H;
  if (pt) pt += 2 * (int64_t)Kx * H;
  w += (int64_t)(d + 1) * H + H;
  for (int m = 1; m < wd.M; ++m) {
    for (int e = t0; e < H * H; e += stride) {
      const int i = e / H, j = e - i * H;
      const float v = w[e];
      put_split(pf, H, i, j, v);
      if (pt) put_split(pt, H, j, i, v);
    }
    pf += 2 * (int64_t)H * H;
    if (pt) pt += 2 * (int64_t)H * H;
    w += (int64_t)H * H + H;
  }
  for (int e = t0; e < H * Pp; e += stride) {
    const int i = e / Pp, j = e - i * Pp;
    const float v = w[e];
    put_split(pf, Pp, i, j, v);
    if (pt) put_split(pt, H, j, i, v);
  }
}

// ---- where a pass's rows and time come from -------------------------------------------------------------------
// Explicit: rows [r0, r0 + n) of an array and a time value.  Drawn: the rows of the step's Philox draw (philox.cuh, the
// numbers the fused step kernel and cnfot_philox_rows / _times_host produce), global row row0 + r, and, with
// t_index >= 0, the step's uniform time t_index plus `t` (the kinetic passes' -dt/2, +dt/2, 0).
struct PassSrc {
  const float* rows;   // (n x D) explicit rows, or NULL: drawn
  float t;
  int source;          // kRowsNormal / kRowsOtSource (drawn)
  int t_index;         // drawn time index, or -1: `t` alone
  uint64_t salt;       // key modifier of the normal draw: StepSalts::B or ::b
  int64_t row0;
};
inline PassSrc explicit_src(const float* rows, float t) {
  PassSrc p = {};
  p.rows = rows;
  p.t = t;
  p.t_index = -1;
  return p;
}
// key and step of the draws: by value, or read from the train state's words [key, step] (device-resident update)
struct DrawKey {
  uint64_t key;
  uint32_t step;
  const unsigned long long* state;
  uint64_t salt_c, salt_t;   // categorical (ot source modes) and uniform (times) key modifiers
  float horizon;
};
struct PassDraw {   // a DrawKey resolved inside a kernel
  uint64_t key;
  uint32_t step;
};
__device__ __forceinline__ PassDraw resolve(const DrawKey& dk) {
  PassDraw d{dk.key, dk.step};
  if (dk.state) {
    d.key = __ldcg(dk.state);
    d.step = (uint32_t)__ldcg(dk.state + 1);
  }
  return d;
}
__device__ __forceinline__ float pass_time(const PassSrc& ps, const DrawKey& dk, const PassDraw& d) {
  return ps.t_index >= 0 ? philox_time(d.key ^ dk.salt_t, d.step, ps.t_index, dk.horizon) + ps.t : ps.t;
}
// column c < D of row r of the pass (explicit rows: ld_rows floats apart)
__device__ __forceinline__ float pass_entry(const PassSrc& ps, const DrawKey& dk, const PassDraw& d, int64_t r, int ld_rows,
                                            int D, int c) {
  if (ps.rows) return ps.rows[r * ld_rows + c];
  return philox_entry(d.key ^ ps.salt, d.key ^ dk.salt_c, d.step, ps.source, (uint64_t)(ps.row0 + r), D, c);
}

// ---- chunk state initialisation: S[0] = [rows | t | 0], S[1..L] = [0 | t | 0] ---------------------------
__global__ void __launch_bounds__(kThreads)
wide_init_kernel(PassSrc ps, DrawKey dk, int ld_rows, int64_t n, int D, int Kx, int L, int64_t state_stride,
                 const float* __restrict__ cond, int64_t cond_stride, int shift_col, float shift, float* __restrict__ S) {
  const int64_t per = n * Kx;
  const int64_t total = per * (L + 1);
  const PassDraw d = !ps.rows || ps.t_index >= 0 ? resolve(dk) : PassDraw{0, 0};
  const float t = pass_time(ps, dk, d);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e / per);
    const int64_t q = e - (int64_t)s * per;
    const int64_t r = q / Kx;
    const int c = (int)(q - r * Kx);
    float v = 0.f;
    if (c < D) v = s == 0 ? pass_entry(ps, dk, d, r, ld_rows, D, c) + (c == shift_col ? shift : 0.f) : 0.f;
    else if (c == D) v = cond ? cond[r * cond_stride] : t;
    S[(int64_t)s * state_stride + q] = v;
  }
}

// ---- spline kernels: one row per thread, raw parameters from the last GEMM (or the shared `first`) ----
template <int K>
__device__ __forceinline__ void load_theta(const float* __restrict__ theta, int64_t r, int bcast, float* th) {
  constexpr int Pp = (3 * K + 1 + 3) / 4 * 4;
  const float4* p = reinterpret_cast<const float4*>(theta + (bcast ? 0 : r * Pp));
#pragma unroll
  for (int j = 0; j < Pp / 4; ++j) {
    const float4 v = __ldg(p + j);
    th[4 * j] = v.x; th[4 * j + 1] = v.y; th[4 * j + 2] = v.z; th[4 * j + 3] = v.w;
  }
}

// DIR 0: spline inverse formula (sample direction); DIR 1: forward formula (log-prob direction)
template <int K, int DIR>
__global__ void __launch_bounds__(kThreads)
wide_spline_kernel(const float* __restrict__ theta, int bcast, const float* __restrict__ Sin, float* __restrict__ Sout,
                   int Kx, int col, float* __restrict__ LD, int ld_accumulate, int64_t n, SplineConsts<float> sc) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  constexpr int Pp = (3 * K + 1 + 3) / 4 * 4;
  float th[Pp];
  load_theta<K>(theta, r, bcast, th);
  const float v = Sin[r * Kx + col];
  SplineState<float, K> st;
  float out, ld;
  if (DIR == 0) rqs_inverse<float, K>(v, th, sc, st, out, ld);
  else rqs_forward<float, K>(v, th, sc, st, out, ld);
  Sout[r * Kx + col] = out;
  LD[r] = ld_accumulate ? LD[r] + ld : ld;
}

// Reverse mode: G[r][col] (adjoint of the spline output) is replaced by the adjoint of its input;
// GTheta (n x Pp) receives the adjoint of the raw parameters.  gld = gld_scalar (+ gld_rows[r]).
template <int K, int DIR>
__global__ void __launch_bounds__(kThreads)
wide_spline_vjp_kernel(const float* __restrict__ theta, int bcast, const float* __restrict__ Sin, int Kx, int col,
                       float* __restrict__ G, float gld_scalar, const float* __restrict__ gld_rows,
                       float* __restrict__ GTheta, int64_t n, SplineConsts<float> sc) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  constexpr int Pp = (3 * K + 1 + 3) / 4 * 4;
  float th[Pp], gth[Pp];
  load_theta<K>(theta, r, bcast, th);
  const float v = Sin[r * Kx + col];
  const float go = G[r * Kx + col];
  const float gl = gld_scalar + (gld_rows ? gld_rows[r] : 0.f);
  SplineState<float, K> st;
  float out, ld, gi;
#pragma unroll
  for (int j = 0; j < Pp; ++j) gth[j] = 0.f;
  if (DIR == 0) {
    rqs_inverse<float, K>(v, th, sc, st, out, ld);
    gi = rqs_inverse_bwd<float, K>(v, st, sc, go, gl, gth);
  } else {
    rqs_forward<float, K>(v, th, sc, st, out, ld);
    gi = rqs_forward_bwd<float, K>(v, st, sc, go, gl, gth);
  }
  G[r * Kx + col] = gi;
  float4* q = reinterpret_cast<float4*>(GTheta + r * Pp);
#pragma unroll
  for (int j = 0; j < Pp / 4; ++j) q[j] = make_float4(gth[4 * j], gth[4 * j + 1], gth[4 * j + 2], gth[4 * j + 3]);
}

// ---- column sums (bias gradients, gradient of `first`): dst[c] += sum_r G[r][c] ------------------------
__global__ void __launch_bounds__(kThreads)
wide_colsum_kernel(const float* __restrict__ G, int ldg, int64_t rows, int N, float* __restrict__ dst) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int sub = threadIdx.x >> 5;
  const int64_t per = (rows + gridDim.y - 1) / gridDim.y;
  const int64_t lo = blockIdx.y * per, hi = lo + per < rows ? lo + per : rows;
  float a0 = 0.f, a1 = 0.f;
  if (c < N) {
    int64_t r = lo + sub;
    for (; r + 8 < hi; r += 16) {
      a0 += __ldg(G + r * ldg + c);
      a1 += __ldg(G + (r + 8) * ldg + c);
    }
    if (r < hi) a0 += __ldg(G + r * ldg + c);
  }
  __shared__ float part[8][32];
  part[sub][threadIdx.x & 31] = a0 + a1;
  __syncthreads();
  if (sub == 0 && c < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += part[k][threadIdx.x & 31];
    atomicAdd(dst + c, t);
  }
}

// ---- the narrow ends of a conditioner on CUDA cores -----------------------------------------------------------
// The output layer (H -> Pp = 16) and the input layer's weight gradient (<= 33 state columns) have one tiny GEMM
// dimension: as 128-row tensor-core tiles they were latency-bound one-CTA-per-128-rows pipelines (100-145 us per
// 75 776 rows, ncu launch list r01); as streaming FFMA kernels they run at the speed their one pass over the
// (rows x H) activation allows.  Exact fp32 FMAs, no split.

// Shared-memory operands are read as warp-wide broadcasts; a broadcast still costs the load unit one cycle per
// 128 bytes of REGISTERS written (32 lanes x 16 B = 4 cycles per LDS.128), so every kernel re-uses each broadcast
// value for several rows / hidden units held in registers.

// Theta (n x PP) = A (n x H) * Wout (H x PP) + bout.  A warp takes 16 rows as 4 row groups x 8 k-phases: a load
// instruction reads 32 contiguous bytes of 4 rows, the weights come from a padded shared tile (row stride 20
// floats: the 8 phases hit 8 distinct 16-byte bank groups) and serve 4 rows each, the 8 partial sums are folded
// with 3 butterfly steps.
template <int PP>
__global__ void __launch_bounds__(kThreads)
wide_out_fwd_kernel(const float* __restrict__ A, const float* __restrict__ Wout, const float* __restrict__ bout, int64_t n,
                    int H, float* __restrict__ Theta) {
  extern __shared__ __align__(16) float wsm[];   // [H][PP + 4]
  constexpr int WS = PP + 4;
  constexpr int RT = 4;                          // row groups per warp pass
  for (int e = threadIdx.x; e < H * (PP / 4); e += blockDim.x) {
    const int k = e / (PP / 4), q = e - k * (PP / 4);
    *reinterpret_cast<float4*>(wsm + k * WS + 4 * q) = __ldg(reinterpret_cast<const float4*>(Wout + (int64_t)k * PP) + q);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, sub = lane & 7, rg = lane >> 3;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t base = warp * (4 * RT); base < n; base += n_warps * (4 * RT)) {
    const float* arow[RT];
    bool live[RT];
#pragma unroll
    for (int t = 0; t < RT; ++t) {
      const int64_t r = base + 4 * t + rg;
      live[t] = r < n;
      arow[t] = A + (live[t] ? r : 0) * H + sub;
    }
    float acc[RT][PP];
#pragma unroll
    for (int t = 0; t < RT; ++t)
#pragma unroll
      for (int p = 0; p < PP; ++p) acc[t][p] = 0.f;
#pragma unroll 2
    for (int k = 0; k < H; k += 8) {
      float a[RT];
#pragma unroll
      for (int t = 0; t < RT; ++t) a[t] = live[t] ? __ldg(arow[t] + k) : 0.f;
      const float* w = wsm + (k + sub) * WS;
#pragma unroll
      for (int q = 0; q < PP / 4; ++q) {
        const float4 w4 = *reinterpret_cast<const float4*>(w + 4 * q);
#pragma unroll
        for (int t = 0; t < RT; ++t) {
          acc[t][4 * q] += a[t] * w4.x; acc[t][4 * q + 1] += a[t] * w4.y;
          acc[t][4 * q + 2] += a[t] * w4.z; acc[t][4 * q + 3] += a[t] * w4.w;
        }
      }
    }
#pragma unroll
    for (int t = 0; t < RT; ++t) {
#pragma unroll
      for (int p = 0; p < PP; ++p) {
        acc[t][p] += __shfl_xor_sync(0xffffffffu, acc[t][p], 1);
        acc[t][p] += __shfl_xor_sync(0xffffffffu, acc[t][p], 2);
        acc[t][p] += __shfl_xor_sync(0xffffffffu, acc[t][p], 4);
      }
      // phase `sub` writes outputs [2 sub, 2 sub + 2) (PP = 16)
      if (live[t] && 2 * sub < PP) {
        float o0 = 0.f, o1 = 0.f;
#pragma unroll
        for (int p = 0; p < PP; p += 2) {
          o0 = (p >> 1) == sub ? acc[t][p] : o0;
          o1 = (p >> 1) == sub ? acc[t][p + 1] : o1;
        }
        *reinterpret_cast<float2*>(Theta + (base + 4 * t + rg) * PP + 2 * sub) =
            make_float2(o0 + __ldg(bout + 2 * sub), o1 + __ldg(bout + 2 * sub + 1));
      }
    }
  }
}

// ---- bulk-copy ring shared by the two streaming kernels below ---------------------------------------------------
// A CTA walks its row range in tiles of kRingRows rows; one thread fetches the next tile with 1-D bulk copies
// (cp.async.bulk -> mbarrier complete_tx) while everybody computes the current one: 33 KB per CTA in flight without
// occupying registers.  Two stages, so that two CTAs (16 warps) fit an SM: ncu (profiles/r01_wide_out_bwd_ncu_full.txt)
// showed the 4-stage / one-CTA version issue-bound at 8 warps per SM (issue slots 52 % busy, 2 warps per scheduler).
constexpr int kRingStages = 2;
constexpr int kRingRows = 16;
__device__ __forceinline__ uint32_t ring_s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ring_init(uint64_t* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ring_s32(bar)), "r"(1));
}
__device__ __forceinline__ void ring_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok) : "r"(ring_s32(bar)), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void ring_expect(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ring_s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ring_copy(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(ring_s32(dst)), "l"(src), "r"(bytes), "r"(ring_s32(bar)) : "memory");
}

// Backward of the output layer in ONE pass over A (n x H): a thread owns TH hidden units h (256 apart),
//   G2[r][h]     = A[r][h] > 0 ? sum_p GTheta[r][p] Wout[h][p] : 0     (adjoint of the last hidden pre-activation)
//   dWout[h][p] += sum_r A[r][h] GTheta[r][p],   dbout[p] += sum_r GTheta[r][p]
// A rows (the CTA's 512 columns) and GTheta rows arrive through the bulk-copy ring.
constexpr int kOutBwdThreads = 256;
constexpr int kOutBwdTH = 2;
constexpr int kOutBwdCols = kOutBwdThreads * kOutBwdTH;
template <int PP>
__global__ void __launch_bounds__(kOutBwdThreads)
wide_out_bwd_kernel(const float* __restrict__ A, const float* __restrict__ GTheta, const float* __restrict__ Wout, int64_t n,
                    int H, float* __restrict__ G2, float* __restrict__ dWout, float* __restrict__ dbout) {
  constexpr int NT_ = kOutBwdThreads, TH = kOutBwdTH;
  extern __shared__ __align__(128) float ring[];   // [stage][kRingRows][kOutBwdCols] | [stage][kRingRows][PP]
  __shared__ __align__(8) uint64_t full[kRingStages];
  float* ringA = ring;
  float* ringG = ring + kRingStages * kRingRows * kOutBwdCols;
  const int tid = threadIdx.x;
  const int hbase = blockIdx.x * kOutBwdCols;
  const int hcount = H - hbase < kOutBwdCols ? H - hbase : kOutBwdCols;
  const int h0 = hbase + tid;
  const int64_t per = ((n + gridDim.y - 1) / gridDim.y + 63) / 64 * 64;
  const int64_t lo = blockIdx.y * per, hi = lo + per < n ? lo + per : n;
  const int n_tiles = hi > lo ? (int)((hi - lo + kRingRows - 1) / kRingRows) : 0;
  auto issue = [&](int t) {   // one thread
    const int sidx = t % kRingStages;
    const int64_t r0 = lo + (int64_t)t * kRingRows;
    const int cnt = hi - r0 < kRingRows ? (int)(hi - r0) : kRingRows;
    ring_expect(&full[sidx], (uint32_t)(cnt * (hcount + PP) * 4));
    for (int rr = 0; rr < cnt; ++rr)
      ring_copy(ringA + (sidx * kRingRows + rr) * kOutBwdCols, A + (r0 + rr) * H + hbase, (uint32_t)(hcount * 4), &full[sidx]);
    ring_copy(ringG + sidx * kRingRows * PP, GTheta + r0 * PP, (uint32_t)(cnt * PP * 4), &full[sidx]);
  };
  if (tid == 0) {
    for (int q = 0; q < kRingStages; ++q) ring_init(&full[q]);
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  __syncthreads();
  if (tid == 0)
    for (int t = 0; t < kRingStages && t < n_tiles; ++t) issue(t);
  float w[TH][PP], acc[TH][PP];
  bool hv[TH];
#pragma unroll
  for (int j = 0; j < TH; ++j) {
    hv[j] = h0 + NT_ * j < H;
#pragma unroll
    for (int q = 0; q < PP / 4; ++q) {
      const float4 v = hv[j] ? __ldg(reinterpret_cast<const float4*>(Wout + (int64_t)(h0 + NT_ * j) * PP) + q)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
      w[j][4 * q] = v.x; w[j][4 * q + 1] = v.y; w[j][4 * q + 2] = v.z; w[j][4 * q + 3] = v.w;
    }
#pragma unroll
    for (int p = 0; p < PP; ++p) acc[j][p] = 0.f;
  }
  float bsum = 0.f;   // thread p < PP of the blocks with blockIdx.x == 0: column p of this block's GTheta rows
  for (int t = 0; t < n_tiles; ++t) {
    const int sidx = t % kRingStages;
    const int64_t r0 = lo + (int64_t)t * kRingRows;
    const int cnt = hi - r0 < kRingRows ? (int)(hi - r0) : kRingRows;
    ring_wait(&full[sidx], (uint32_t)((t / kRingStages) & 1));
    const float* ta = ringA + sidx * kRingRows * kOutBwdCols + tid;
    const float* tg = ringG + sidx * kRingRows * PP;
    if (blockIdx.x == 0 && tid < PP)
      for (int rr = 0; rr < cnt; ++rr) bsum += tg[rr * PP + tid];
#pragma unroll 4
    for (int rr = 0; rr < cnt; ++rr) {
      float a[TH], sacc[TH];
#pragma unroll
      for (int j = 0; j < TH; ++j) {
        a[j] = hv[j] ? ta[rr * kOutBwdCols + NT_ * j] : 0.f;
        sacc[j] = 0.f;
      }
#pragma unroll
      for (int q = 0; q < PP / 4; ++q) {
        const float4 g = *reinterpret_cast<const float4*>(tg + rr * PP + 4 * q);
#pragma unroll
        for (int j = 0; j < TH; ++j) {
          sacc[j] += g.x * w[j][4 * q] + g.y * w[j][4 * q + 1] + g.z * w[j][4 * q + 2] + g.w * w[j][4 * q + 3];
          acc[j][4 * q] += a[j] * g.x; acc[j][4 * q + 1] += a[j] * g.y;
          acc[j][4 * q + 2] += a[j] * g.z; acc[j][4 * q + 3] += a[j] * g.w;
        }
      }
#pragma unroll
      for (int j = 0; j < TH; ++j)
        if (hv[j]) G2[(r0 + rr) * H + h0 + NT_ * j] = a[j] > 0.f ? sacc[j] : 0.f;
    }
    __syncthreads();   // everybody is done with the stage: refill it
    if (tid == 0 && t + kRingStages < n_tiles) issue(t + kRingStages);
  }
#pragma unroll
  for (int j = 0; j < TH; ++j)
    if (hv[j]) {
#pragma unroll
      for (int q = 0; q < PP / 4; ++q)
        asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(dWout + (int64_t)(h0 + NT_ * j) * PP + 4 * q),
                     "f"(acc[j][4 * q]), "f"(acc[j][4 * q + 1]), "f"(acc[j][4 * q + 2]), "f"(acc[j][4 * q + 3]) : "memory");
    }
  if (blockIdx.x == 0 && tid < PP) atomicAdd(dbout + tid, bsum);
}
template <int PP>
constexpr size_t out_bwd_smem() { return (size_t)kRingStages * kRingRows * (kOutBwdCols + PP) * sizeof(float); }

// Weight gradient of the input layer: dW0[w0_row(k)][h] += sum_r S[r][k] G1[r][h], db0[h] += sum_r G1[r][h];
// a thread owns 2 hidden units (256 apart), 4 KV4 state columns accumulated in registers for each; G1 rows (the
// CTA's 512 columns) and the state rows arrive through the bulk-copy ring.
// SLICED (Kx > 64, KV4 = 16): blockIdx.z takes the state columns [64 z, 64 z + 64); the ring holds that 256-byte slice of
// each row.  A slice the conditioner does not read at all (no column with a weight row) returns at once; db0 is summed
// by the slice that holds the time column D.
constexpr int kInWgradTH = 2;
constexpr int kInWgradCols = kThreads * kInWgradTH;
template <int KV4, bool SLICED = false>
__global__ void __launch_bounds__(kThreads)
wide_in_wgrad_kernel(const float* __restrict__ S, int Kx, const float* __restrict__ G1, int64_t n, int H, int D, int d, int rev,
                     float* __restrict__ dW0, float* __restrict__ db0) {
  constexpr int KV = 4 * KV4, TH = kInWgradTH;
  static_assert(!SLICED || KV == kInWgradSlice, "a sliced CTA owns one whole slice");
  const int c0 = SLICED ? (int)blockIdx.z * kInWgradSlice : 0;
  const int sw = SLICED ? kInWgradSlice : Kx;      // floats of a state row in the ring
  if (SLICED) {
    bool any = false;
    for (int k = 0; k < KV; ++k) any |= w0_row(c0 + k, D, d, rev) >= 0;
    if (!any) return;
  }
  extern __shared__ __align__(128) float ring[];   // [stage][kRingRows][kInWgradCols] | [stage][kRingRows][sw]
  __shared__ __align__(8) uint64_t full[kRingStages];
  float* ringG = ring;
  float* ringS = ring + kRingStages * kRingRows * kInWgradCols;
  const int tid = threadIdx.x;
  const int hbase = blockIdx.x * kInWgradCols;
  const int hcount = H - hbase < kInWgradCols ? H - hbase : kInWgradCols;
  const int h0 = hbase + tid;
  bool hv[TH];
#pragma unroll
  for (int j = 0; j < TH; ++j) hv[j] = h0 + kThreads * j < H;
  const int64_t per = ((n + gridDim.y - 1) / gridDim.y + 63) / 64 * 64;
  const int64_t lo = blockIdx.y * per, hi = lo + per < n ? lo + per : n;
  const int n_tiles = hi > lo ? (int)((hi - lo + kRingRows - 1) / kRingRows) : 0;
  auto issue = [&](int t) {   // one thread
    const int sidx = t % kRingStages;
    const int64_t r0 = lo + (int64_t)t * kRingRows;
    const int cnt = hi - r0 < kRingRows ? (int)(hi - r0) : kRingRows;
    ring_expect(&full[sidx], (uint32_t)(cnt * (hcount + sw) * 4));
    for (int rr = 0; rr < cnt; ++rr)
      ring_copy(ringG + (sidx * kRingRows + rr) * kInWgradCols, G1 + (r0 + rr) * H + hbase, (uint32_t)(hcount * 4), &full[sidx]);
    if (SLICED) {
      for (int rr = 0; rr < cnt; ++rr)
        ring_copy(ringS + (sidx * kRingRows + rr) * sw, S + (r0 + rr) * Kx + c0, (uint32_t)(sw * 4), &full[sidx]);
    } else {
      ring_copy(ringS + sidx * kRingRows * Kx, S + r0 * Kx, (uint32_t)(cnt * Kx * 4), &full[sidx]);
    }
  };
  if (tid == 0) {
    for (int q = 0; q < kRingStages; ++q) ring_init(&full[q]);
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  __syncthreads();
  if (tid == 0)
    for (int t = 0; t < kRingStages && t < n_tiles; ++t) issue(t);
  float acc[TH][KV], bsum[TH];
#pragma unroll
  for (int j = 0; j < TH; ++j) {
    bsum[j] = 0.f;
#pragma unroll
    for (int k = 0; k < KV; ++k) acc[j][k] = 0.f;
  }
  for (int t = 0; t < n_tiles; ++t) {
    const int sidx = t % kRingStages;
    const int64_t r0 = lo + (int64_t)t * kRingRows;
    const int cnt = hi - r0 < kRingRows ? (int)(hi - r0) : kRingRows;
    ring_wait(&full[sidx], (uint32_t)((t / kRingStages) & 1));
    const float* tg = ringG + sidx * kRingRows * kInWgradCols + tid;
    const float* ts = ringS + sidx * kRingRows * sw;
#pragma unroll 2
    for (int rr = 0; rr < cnt; ++rr) {
      float g[TH];
#pragma unroll
      for (int j = 0; j < TH; ++j) {
        g[j] = hv[j] ? tg[rr * kInWgradCols + kThreads * j] : 0.f;
        bsum[j] += g[j];
      }
#pragma unroll
      for (int q = 0; q < KV4; ++q) {
        const float4 sv = *reinterpret_cast<const float4*>(ts + rr * sw + 4 * q);
#pragma unroll
        for (int j = 0; j < TH; ++j) {
          acc[j][4 * q] += g[j] * sv.x; acc[j][4 * q + 1] += g[j] * sv.y;
          acc[j][4 * q + 2] += g[j] * sv.z; acc[j][4 * q + 3] += g[j] * sv.w;
        }
      }
    }
    __syncthreads();
    if (tid == 0 && t + kRingStages < n_tiles) issue(t + kRingStages);
  }
#pragma unroll
  for (int j = 0; j < TH; ++j)
    if (hv[j]) {
      const int h = h0 + kThreads * j;
#pragma unroll
      for (int k = 0; k < KV; ++k) {
        const int row = w0_row(c0 + k, D, d, rev);
        if (row >= 0) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(dW0 + (int64_t)row * H + h), "f"(acc[j][k]) : "memory");
      }
      if (!SLICED || (int)blockIdx.z == D / kInWgradSlice) atomicAdd(db0 + h, bsum[j]);
    }
}
// sw: floats of a state row in the ring (Kx, or one 64-column slice)
inline size_t in_wgrad_smem(int sw) { return (size_t)kRingStages * kRingRows * (kInWgradCols + sw) * sizeof(float); }

// ---- loss heads ------------------------------------------------------------------------------------------
__device__ __forceinline__ void block_add(double v, double* dst) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(dst, v);
}

// kl_loss_fn row: -w log p(data | t) = -w (log N(z) + ld); G = w z (applications.py:85)
__global__ void __launch_bounds__(kThreads)
wide_nll_head_kernel(const float* __restrict__ Z, const float* __restrict__ LD, int64_t n, int D, int Kx, float w,
                     float* __restrict__ G, double* __restrict__ slot) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double loss = 0.0;
  if (r < n) {
    float acc = 0.f;
    for (int c = 0; c < Kx; ++c) {
      const float z = c < D ? Z[r * Kx + c] : 0.f;
      acc += z * z;
      G[r * Kx + c] = w * z;
    }
    const float lp = -0.5f * acc - 0.91893853320467274178f * (float)D + LD[r];
    loss = -(double)w * (double)lp;
  }
  block_add(loss, slot);
}

// kinetic_loss_fn rows (applications.py:220-242) + the ot/obstacle potential at r(t) (:190-191, :398-401)
__global__ void __launch_bounds__(kThreads)
wide_kinetic_head_kernel(const float* __restrict__ R1, const float* __restrict__ R2, const float* __restrict__ R3,
                         int64_t n, int D, int Kx, float dt, float w_kin, float w_pot, float* __restrict__ G1,
                         float* __restrict__ G2, float* __restrict__ G3, double* __restrict__ slot_kin,
                         double* __restrict__ slot_pot) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double lk = 0.0, lp = 0.0;
  if (r < n) {
    const float idt = 1.f / dt;
    float acc = 0.f;
    for (int c = 0; c < Kx; ++c) {
      float g = 0.f;
      if (c < D) {
        const float v = (R2[r * Kx + c] - R1[r * Kx + c]) * idt;
        acc += v * v;
        g = 2.f * w_kin * v * idt;
      }
      G2[r * Kx + c] = g;
      G1[r * Kx + c] = -g;
    }
    lk = (double)w_kin * (double)acc;
    if (R3) {
      float q = 0.f;
      for (int c = 0; c < D; ++c) q += R3[r * Kx + c] * R3[r * Kx + c];
      const float pv = 50.f * __expf(-0.5f * q);
      for (int c = 0; c < Kx; ++c) G3[r * Kx + c] = c < D ? -w_pot * pv * R3[r * Kx + c] : 0.f;
      lp = (double)w_pot * (double)pv;
    }
  }
  block_add(lk, slot_kin);
  if (R3) block_add(lp, slot_pot);
}

// The per-row heads below hold D-float arrays in local memory; NX is their bound.  They are instantiated at 64 (every
// dim up to 64) and at 256 (up to kWideMaxDim): the driver reserves local memory per resident thread for the largest
// frame a launch needs, so the small dims keep their small frames.
constexpr int kHeadSmall = 64, kHeadLarge = 256;
static_assert(kWideMaxDim < kHeadLarge, "head arrays hold a whole row");

// Rows pushed through the sample direction at time t (row_sample_terms of step_math.cuh):
// do_fit: reverse_kl_loss_fn (applications.py:129-163)  w_fit (log p(y) - log q_t(y));  do_pot: potential_loss_fn (:176-205)
template <int NX>
__global__ void __launch_bounds__(kThreads)
wide_sample_head_kernel(const float* __restrict__ Z0, const float* __restrict__ Y, const float* __restrict__ LD, int64_t n,
                        int D, int Kx, float t, int do_fit, int do_pot, StepConsts<float> pc, float* __restrict__ G,
                        double* __restrict__ slot_fit, double* __restrict__ slot_pot) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double lf = 0.0, lpot = 0.0;
  if (r < n) {
    float y[NX], g[NX];
    float r2 = 0.f, z2 = 0.f;
    for (int c = 0; c < D; ++c) {
      y[c] = Y[r * Kx + c];
      g[c] = 0.f;
      r2 += y[c] * y[c];
      z2 += Z0[r * Kx + c] * Z0[r * Kx + c];
    }
    if (do_fit) {
      const float half_log_2pi = 0.91893853320467274178f;
      const float lp = -0.5f * z2 - half_log_2pi * (float)D - LD[r];
      const float w1 = (pc.horizon - t) / pc.horizon, w2 = t / pc.horizon;
      const float l1 = -0.5f * r2 / pc.var_src - (float)D * (half_log_2pi + 0.5f * logf(pc.var_src));
      const float l2 = -0.5f * r2 / pc.var_tgt - (float)D * (half_log_2pi + 0.5f * logf(pc.var_tgt));
      float logq, coef;   // coef = -d log q / d y_i / y_i
      if (w2 <= 0.f) { logq = l1 + logf(w1); coef = 1.f / pc.var_src; }
      else if (w1 <= 0.f) { logq = l2 + logf(w2); coef = 1.f / pc.var_tgt; }
      else {
        const float a1 = l1 + logf(w1), a2 = l2 + logf(w2);
        const float m = fmaxf(a1, a2);
        const float e1 = expf(a1 - m), e2 = expf(a2 - m);
        logq = m + logf(e1 + e2);
        coef = (e1 / pc.var_src + e2 / pc.var_tgt) / (e1 + e2);
      }
      lf = (double)pc.w_fit * (double)(lp - logq);
      for (int c = 0; c < D; ++c) g[c] += pc.w_fit * coef * y[c];
    }
    if (do_pot) {
      float gp[NX];
      const float v = potential_value_grad<float>(pc.potential, pc.a, y, D, gp);
      lpot = (double)pc.w_pot * (double)v;
      for (int c = 0; c < D; ++c) g[c] += pc.w_pot * gp[c];
    }
    for (int c = 0; c < Kx; ++c) G[r * Kx + c] = c < D ? g[c] : 0.f;
  }
  block_add(lf, slot_fit);
  block_add(lpot, slot_pot);
}

// Coordinate i of kinetic_with_score_loss_fn / flow_matching_loss_fn (applications.py:245-374; row_kinetic of
// step_math.cuh): score_i from the two shifted log-prob passes, resid_i = (r2_i - r1_i)/dt + kappa score_i - truth_i,
// loss += w_kin resid_i^2; seeds the adjoints of the five passes.
template <int NX>
__global__ void __launch_bounds__(kThreads)
wide_score_head_kernel(int i, const float* __restrict__ R1, const float* __restrict__ R2, const float* __restrict__ R3,
                       const float* __restrict__ Zp, const float* __restrict__ LDp, const float* __restrict__ Zm,
                       const float* __restrict__ LDm, int64_t n, int D, int Kx, StepConsts<float> pc, float* __restrict__ G1,
                       float* __restrict__ G2, float* __restrict__ Gp, float* __restrict__ Gm, float* __restrict__ GLp,
                       float* __restrict__ GLm, float* __restrict__ GRES, double* __restrict__ slot_kin) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double lk = 0.0;
  if (r < n) {
    float zp2 = 0.f, zm2 = 0.f;
    for (int c = 0; c < D; ++c) {
      zp2 += Zp[r * Kx + c] * Zp[r * Kx + c];
      zm2 += Zm[r * Kx + c] * Zm[r * Kx + c];
    }
    // base log-densities: the -D log(2 pi)/2 terms cancel in the difference
    const float score = ((-0.5f * zp2 + LDp[r]) - (-0.5f * zm2 + LDm[r])) / pc.dx;
    float truth_i = 0.f;
    if (pc.type == kFP) {
      float r3[NX], truth[NX];
      for (int c = 0; c < D; ++c) { r3[c] = R3[r * Kx + c]; truth[c] = 0.f; }
      drift_value<float>(pc.drift, pc.a, r3, D, truth);
      truth_i = truth[i];
    }
    const float resid = (R2[r * Kx + i] - R1[r * Kx + i]) / pc.dt + pc.kappa * score - truth_i;
    lk = (double)pc.w_kin * (double)resid * (double)resid;
    const float gres = 2.f * pc.w_kin * resid;
    GRES[r * Kx + i] = gres;
    G2[r * Kx + i] = gres / pc.dt;
    G1[r * Kx + i] = -gres / pc.dt;
    const float glp = gres * pc.kappa / pc.dx;
    for (int c = 0; c < Kx; ++c) {
      Gp[r * Kx + c] = c < D ? -glp * Zp[r * Kx + c] : 0.f;   // d log N(z) / dz = -z
      Gm[r * Kx + c] = c < D ? glp * Zm[r * Kx + c] : 0.f;
    }
    GLp[r] = glp;
    GLm[r] = -glp;
  }
  block_add(lk, slot_kin);
}

// G3 += Gp + Gm (the input adjoints of the two shifted passes are adjoints of r3)
__global__ void __launch_bounds__(kThreads)
wide_add2_kernel(float* __restrict__ G3, const float* __restrict__ Gp, const float* __restrict__ Gm, int64_t count) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
    G3[e] += Gp[e] + Gm[e];
}

// fp: resid = v - truth(r3): pull the residual adjoints back through the drift target (applications.py:308-372)
template <int NX>
__global__ void __launch_bounds__(kThreads)
wide_drift_pullback_kernel(const float* __restrict__ R3, const float* __restrict__ GRES, int64_t n, int D, int Kx,
                           StepConsts<float> pc, float* __restrict__ G3) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  float r3[NX], gres[NX], g3[NX];
  for (int c = 0; c < D; ++c) { r3[c] = R3[r * Kx + c]; gres[c] = GRES[r * Kx + c]; g3[c] = G3[r * Kx + c]; }
  drift_pullback<float>(pc.drift, pc.a, r3, D, gres, g3);
  for (int c = 0; c < D; ++c) G3[r * Kx + c] = g3[c];
}

// ---- evaluation energies (forward only; utils.calc_kinetic_energy / calc_score_kinetic_energy, cnf_ot/utils.py:311-389)
__global__ void __launch_bounds__(kThreads)
wide_velocity_kernel(const float* __restrict__ R1, const float* __restrict__ R2, int64_t n, int D, int Kx, float dt,
                     float* __restrict__ V) {
  const int64_t total = n * Kx;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % Kx);
    V[e] = c < D ? (R2[e] - R1[e]) / dt : 0.f;
  }
}
// V[r][i] += kappa * score_i, score_i by central differences of log_prob (the -D log(2 pi)/2 terms cancel)
__global__ void __launch_bounds__(kThreads)
wide_score_add_kernel(int i, const float* __restrict__ Zp, const float* __restrict__ LDp, const float* __restrict__ Zm,
                      const float* __restrict__ LDm, int64_t n, int D, int Kx, float kappa, float dx, float* __restrict__ V) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  float zp2 = 0.f, zm2 = 0.f;
  for (int c = 0; c < D; ++c) {
    zp2 += Zp[r * Kx + c] * Zp[r * Kx + c];
    zm2 += Zm[r * Kx + c] * Zm[r * Kx + c];
  }
  V[r * Kx + i] += kappa * ((-0.5f * zp2 + LDp[r]) - (-0.5f * zm2 + LDm[r])) / dx;
}
__global__ void __launch_bounds__(kThreads)
wide_sumsq_kernel(const float* __restrict__ V, int64_t count, double weight, double* __restrict__ slot) {
  double acc = 0.0;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
    acc += (double)V[e] * (double)V[e];
  block_add(acc * weight, slot);
}
__global__ void wide_energy_out_kernel(const double* __restrict__ slots, double* __restrict__ out) {
  if (threadIdx.x == 0) out[0] = slots[kSlotKinetic];
}

// ---- densities on a grid / at Monte-Carlo samples (density_kernel of flow_kernels.cuh on a chunk) -----------------
struct DensityPoints {
  int mode;                          // 0 grid, 1 Monte-Carlo
  int nx, ny;                        // grid: flat point r = (ti, iy, ix)
  double x_min, x_step, y_min, y_step;
  const float* t_dev;                // grid: (n_t) times
  uint64_t key_n;                    // Monte-Carlo: Philox key of the (n, D) normal draw
  uint32_t step;
  float cond;                        // Monte-Carlo: the time
};
// points [r0, r0 + n) into the chunk: S[0] = [point | t | 0 ..], S[1..L] = [0 | t | 0 ..] (wide_init_kernel's layout);
// a grid chunk may cross a time boundary, so t is per row
__global__ void __launch_bounds__(kThreads)
wide_density_init_kernel(DensityPoints dp, int64_t r0, int64_t n, int D, int Kx, int L, int64_t state_stride,
                         float* __restrict__ S) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int64_t g = r0 + r;
  float* s0 = S + r * Kx;
  float t;
  if (dp.mode == 0) {
    const int64_t per_t = (int64_t)dp.nx * dp.ny;
    const int ti = (int)(g / per_t);
    const int64_t q = g - (int64_t)ti * per_t;
    const int iy = (int)(q / dp.nx), ix = (int)(q - (int64_t)iy * dp.nx);
    s0[0] = (float)(dp.x_min + (double)ix * dp.x_step);
    s0[1] = (float)(dp.y_min + (double)iy * dp.y_step);
    t = dp.t_dev[ti];
  } else {
    philox_row(dp.key_n, dp.key_n, dp.step, kRowsNormal, (uint64_t)g, D, s0);
    t = dp.cond;
  }
  for (int s = 0; s <= L; ++s) {
    float* row = S + (int64_t)s * state_stride + r * Kx;
    for (int c = s == 0 ? D : 0; c < Kx; ++c) row[c] = c == D ? t : 0.f;
  }
}
// lp = log N(Z) + ld_sign LD (grid: Z = latent output, +ildj; Monte-Carlo: Z = latent input, -fldj); density = exp(lp) and,
// with_ref, the squared error at the points Y against the reference mixture, summed in double into `slot`
__global__ void __launch_bounds__(kThreads)
wide_density_head_kernel(const float* __restrict__ Z, const float* __restrict__ Y, const float* __restrict__ LD,
                         float ld_sign, int64_t n, int D, int Kx, float* __restrict__ density, int with_ref, float mix,
                         float var0, float var1, double* __restrict__ slot) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double sq = 0.0;
  if (r < n) {
    const float p = m_exp(base_log_prob<float>(Z + r * Kx, D) + ld_sign * LD[r]);
    if (density) density[r] = p;
    if (with_ref) {
      const float e = ref_mixture_error(p, Y + r * Kx, D, mix, var0, var1);
      sq = (double)e * (double)e;
    }
  }
  if (with_ref) block_add(sq, slot);
}

// ---- batched passes: several flow passes that start from the same rows share ONE chunk ---------------------------
// (rows [j n, (j + 1) n) of the chunk = pass j).  Fewer, larger launches: a small-batch step is launch-bound.
struct MultiSrc {
  PassSrc src[3];
};
// state 0 = [src_j rows | t_j | 0] for j < reps, states 1..L = [0 | t_j | 0]
__global__ void __launch_bounds__(kThreads)
wide_init_multi_kernel(MultiSrc ms, DrawKey dk, int64_t n, int reps, int D, int Kx, int L, int64_t state_stride,
                       float* __restrict__ S) {
  const int64_t per = n * reps * Kx;
  const int64_t total = per * (L + 1);
  // every source of one chunk is drawn or none is (unused entries: zeroed)
  const PassDraw d = !ms.src[0].rows ? resolve(dk) : PassDraw{0, 0};
  const float tj[3] = {pass_time(ms.src[0], dk, d), pass_time(ms.src[1], dk, d), pass_time(ms.src[2], dk, d)};
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e / per);
    const int64_t q = e - (int64_t)s * per;
    const int64_t row = q / Kx;
    const int c = (int)(q - row * Kx);
    const int j = (int)(row / n);
    const int64_t r = row - (int64_t)j * n;
    float v = 0.f;
    if (c < D) v = s == 0 ? pass_entry(ms.src[j], dk, d, r, D, D, c) : 0.f;
    else if (c == D) v = j == 0 ? tj[0] : (j == 1 ? tj[1] : tj[2]);
    S[(int64_t)s * state_stride + q] = v;
  }
}
// the 2 D shifted copies of the rows R3 (n x Kx): copy j = 2 i + side is R3 + (side ? -shift : +shift) e_i, all at the
// time of R3 (its column D)
__global__ void __launch_bounds__(kThreads)
wide_init_shift_kernel(const float* __restrict__ R3, int64_t n, int D, int Kx, int L, int64_t state_stride, float shift,
                       float* __restrict__ S) {
  const int64_t per = n * 2 * D * Kx;
  const int64_t total = per * (L + 1);
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e / per);
    const int64_t q = e - (int64_t)s * per;
    const int64_t row = q / Kx;
    const int c = (int)(q - row * Kx);
    const int j = (int)(row / n);
    const int64_t r = row - (int64_t)j * n;
    float v = 0.f;
    if (c < D) v = s == 0 ? R3[r * Kx + c] + (c == (j >> 1) ? ((j & 1) ? -shift : shift) : 0.f) : 0.f;
    else if (c == D) v = R3[r * Kx + D];
    S[(int64_t)s * state_stride + q] = v;
  }
}
// All coordinates of the score-kinetic term at once (wide_score_head_kernel for every i): Z / LD hold the 2 D n
// latent outputs / log-dets of the shifted log-prob passes; seeds Gs (2 D n rows), GLs, the adjoints of r1, r2
// (G1, G2; every column written), zeroes G3 and fills GRES.
template <int NX>
__global__ void __launch_bounds__(kThreads)
wide_score_head_all_kernel(const float* __restrict__ R1, const float* __restrict__ R2, const float* __restrict__ R3,
                           const float* __restrict__ Z, const float* __restrict__ LDs, int64_t n, int D, int Kx,
                           StepConsts<float> pc, float* __restrict__ G1, float* __restrict__ G2, float* __restrict__ G3,
                           float* __restrict__ Gs, float* __restrict__ GLs, float* __restrict__ GRES,
                           double* __restrict__ slot_kin) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  double lk = 0.0;
  if (r < n) {
    float truth[NX];
    for (int c = 0; c < D; ++c) truth[c] = 0.f;
    if (pc.type == kFP) {
      float r3[NX];
      for (int c = 0; c < D; ++c) r3[c] = R3[r * Kx + c];
      drift_value<float>(pc.drift, pc.a, r3, D, truth);
    }
    for (int c = D; c < Kx; ++c) { G1[r * Kx + c] = 0.f; G2[r * Kx + c] = 0.f; GRES[r * Kx + c] = 0.f; }
    for (int c = 0; c < Kx; ++c) G3[r * Kx + c] = 0.f;
    for (int i = 0; i < D; ++i) {
      const int64_t rp = (int64_t)(2 * i) * n + r, rm = rp + n;
      float zp2 = 0.f, zm2 = 0.f;
      for (int c = 0; c < D; ++c) {
        zp2 += Z[rp * Kx + c] * Z[rp * Kx + c];
        zm2 += Z[rm * Kx + c] * Z[rm * Kx + c];
      }
      const float score = ((-0.5f * zp2 + LDs[rp]) - (-0.5f * zm2 + LDs[rm])) / pc.dx;
      const float resid = (R2[r * Kx + i] - R1[r * Kx + i]) / pc.dt + pc.kappa * score - truth[i];
      lk += (double)pc.w_kin * (double)resid * (double)resid;
      const float gres = 2.f * pc.w_kin * resid;
      GRES[r * Kx + i] = gres;
      G2[r * Kx + i] = gres / pc.dt;
      G1[r * Kx + i] = -gres / pc.dt;
      const float glp = gres * pc.kappa / pc.dx;
      for (int c = 0; c < Kx; ++c) {
        Gs[rp * Kx + c] = c < D ? -glp * Z[rp * Kx + c] : 0.f;
        Gs[rm * Kx + c] = c < D ? glp * Z[rm * Kx + c] : 0.f;
      }
      GLs[rp] = glp;
      GLs[rm] = -glp;
    }
  }
  block_add(lk, slot_kin);
}
// G3[r][c] += sum_j Gs[j n + r][c], j < reps (the input adjoints of the shifted passes are adjoints of r3)
__global__ void __launch_bounds__(kThreads)
wide_fold_kernel(float* __restrict__ G3, const float* __restrict__ Gs, int64_t n, int reps, int Kx) {
  const int64_t count = n * Kx;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
    float acc = G3[e];
    for (int j = 0; j < reps; ++j) acc += Gs[(int64_t)j * count + e];
    G3[e] = acc;
  }
}
__global__ void __launch_bounds__(kThreads) wide_fill_kernel(float* __restrict__ p, int64_t count, float v) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) p[e] = v;
}

// out slots: 0 total, 1 fit(0), 2 fit(T), 3 potential, 4 kinetic, 5-7 zero
__global__ void wide_finalize_kernel(const double* __restrict__ slots, float* __restrict__ out_slots) {
  if (threadIdx.x == 0) {
    const double t = slots[kSlotFit0] + slots[kSlotFitT] + slots[kSlotPotential] + slots[kSlotKinetic];
    out_slots[0] = (float)t;
    out_slots[1] = (float)slots[kSlotFit0];
    out_slots[2] = (float)slots[kSlotFitT];
    out_slots[3] = (float)slots[kSlotPotential];
    out_slots[4] = (float)slots[kSlotKinetic];
    out_slots[5] = out_slots[6] = out_slots[7] = 0.f;
  }
}

// ---- the device-resident update's tail: optax.adam on the step's gradient (adam_elem, shared with the fused tail) ----
// out = [gradient (total) | loss slots]; update number state[1]; a NaN gradient entry leaves its parameter alone
__global__ void __launch_bounds__(kThreads)
wide_adam_kernel(const float* __restrict__ out, int64_t total, const unsigned long long* __restrict__ state, float lr, float b1,
                 float b2, float eps, float* __restrict__ W, float* __restrict__ m, float* __restrict__ v,
                 float* __restrict__ loss_hist, int64_t loss_hist_len) {
  const uint32_t stepno = (uint32_t)__ldcg(state + 1);
  float c1, c2;
  adam_bias(stepno, b1, b2, c1, c2);
  const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i0 == 0 && loss_hist && (int64_t)stepno < loss_hist_len) loss_hist[stepno] = out[total];
  for (int64_t i = i0; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float g = out[i];
    if (g != g) continue;
    float mi = m[i], vi = v[i], wi = W[i];
    adam_elem(lr, b1, b2, eps, c1, c2, g, mi, vi, wi);
    m[i] = mi;
    v[i] = vi;
    W[i] = wi;
  }
}
// after every block of wide_adam_kernel has read it: the next update's number (and epoch, as the fused tail keeps it)
__global__ void wide_advance_kernel(unsigned long long* __restrict__ state) {
  if (threadIdx.x == 0) {
    state[1] += 1ULL;
    state[2] += 1ULL;
  }
}

// copy the D coordinates of a state to a dense (n x D) buffer
__global__ void __launch_bounds__(kThreads)
wide_extract_kernel(const float* __restrict__ S, int64_t n, int D, int Kx, float* __restrict__ out) {
  const int64_t total = n * D;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / D;
    const int c = (int)(e - r * D);
    out[e] = S[r * Kx + c];
  }
}

// logdet output of the model API: ld, or the density ConditionalTransformed returns
// (conditional.py:316-321,382-402): forward: log N(in) - ld ; inverse: log N(out) + ld
__global__ void __launch_bounds__(kThreads)
wide_logdet_out_kernel(const float* __restrict__ LD, const float* __restrict__ base_rows, int ld_base, int64_t n, int D,
                       int add_base, float sign, float* __restrict__ out) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  float v = LD[r];
  if (add_base) {
    float acc = 0.f;
    for (int c = 0; c < D; ++c) acc += base_rows[r * ld_base + c] * base_rows[r * ld_base + c];
    v = -0.5f * acc - 0.91893853320467274178f * (float)D + sign * v;
  }
  out[r] = v;
}

// model-API VJP: seed the adjoint state from (g_out, g_logdet) -- see flow_vjp_kernel in flow_kernels.cuh
__global__ void __launch_bounds__(kThreads)
wide_vjp_seed_kernel(const float* __restrict__ g_out, const float* __restrict__ g_logdet, const float* __restrict__ Zout,
                     int64_t n, int D, int Kx, int dir, int add_base, float* __restrict__ G, float* __restrict__ GL) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float gl = g_logdet ? g_logdet[r] : 0.f;
  for (int c = 0; c < Kx; ++c) {
    float g = c < D ? g_out[r * D + c] : 0.f;
    if (add_base && dir == 1 && c < D) g -= gl * Zout[r * Kx + c];
    G[r * Kx + c] = g;
  }
  GL[r] = (add_base && dir == 0) ? -gl : gl;
}
__global__ void __launch_bounds__(kThreads)
wide_vjp_out_kernel(const float* __restrict__ G, const float* __restrict__ g_logdet, const float* __restrict__ Zin,
                    int64_t n, int D, int Kx, int dir, int add_base, float* __restrict__ g_in) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n) return;
  const float gl = g_logdet ? g_logdet[r] : 0.f;
  for (int c = 0; c < D; ++c) {
    float g = G[r * Kx + c];
    if (add_base && dir == 0) g -= gl * Zin[r * Kx + c];
    g_in[r * D + c] = g;
  }
}

// the instantiation of a per-row head for rows of D coordinates
template <typename F>
F head_for(int D, F small, F large) { return D <= kHeadSmall ? small : large; }

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) only when a (kernel, device) needs more than it was given before:
// the call costs microseconds, a small-batch step makes hundreds of launches
cudaError_t set_smem_max(const void* kern, size_t bytes, int (&cur)[64]) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev >= 0 && dev < 64 && (int)bytes <= cur[dev]) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && dev >= 0 && dev < 64) cur[dev] = (int)bytes;
  return e;
}

// ---- the engine --------------------------------------------------------------------------------------------
struct WideEngine {
  cudaStream_t s;
  FlowLayout lay;
  WideDims wd;
  SplineConsts<float> sc;
  const float* W;
  float* grad;            // blob layout, accumulated (may be NULL: forward only)
  float* prep_fwd;
  float* prep_T;
  int64_t R;              // chunk capacity (rows)
  float* S[kMaxPass];     // (L+1) x R x Kx each
  float* LD[kMaxPass];
  float* G[kMaxPass];     // R x Kx each
  float* A[kMaxM];        // R x H each
  float* Ga;
  float* Gb;
  float* Theta;           // R x Pp
  float* GTheta;
  float* GL;              // R: per-row adjoint of the log-det (model-API VJP; score passes: GL and GL2)
  float* GL2;
  float* GRES;            // R x Kx: d loss / d residual_i of the score-kinetic rows (drift pull-back)
  float* V;               // R x Kx: velocities of the evaluation energies
  float* stashA;          // n_mlp x R x H: last hidden activations of pass 0, kept for its backward sweep (or NULL)
  float* stashT;          // n_mlp x R x Pp: raw spline parameters of pass 0
  double* slots;
  DrawKey dk = {};        // the step's draws (passes whose rows are not explicit)
  cudaError_t err = cudaSuccess;
  const char* what = "";

  bool ok() const { return err == cudaSuccess; }
  void check(cudaError_t e, const char* w) {
    if (err == cudaSuccess && e != cudaSuccess) { err = e; what = w; }
  }
  void check_launch(const char* w) { check(cudaGetLastError(), w); }
  int64_t state_stride() const { return R * wd.Kx; }
  float* state(int p, int s_) const { return S[p] + (int64_t)s_ * state_stride(); }
  static unsigned blocks_for(int64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

  void dense(const float* X, int64_t n, int K, int ldx, const float* P, int N, const float* bias, const float* mask,
             int ldm, int epi, float* Y, int ldy) {
    if (!ok()) return;
    bool sup = false;
    check(dense_forward(s, X, n, K, ldx, P, N, bias, mask, ldm, epi, Y, ldy, &sup), "dense_tc_kernel launch");
    if (ok() && !sup) { err = cudaErrorInvalidValue; what = "no dense kernel for this layer width"; }
  }

  // conditioner (layer, d >= 1) on the state rows `cst`: hidden activations into A[0..M-2] and `a_last`, raw spline
  // parameters into `theta`; with skip_last only the layers below the last hidden one are evaluated (the rest is
  // taken from the stash by the caller)
  void mlp_forward(int layer, int d, const float* cst, int64_t n, float* a_last, float* theta, bool skip_last = false) {
    const int H = wd.H, Kx = wd.Kx, Pp = wd.Pp, M = wd.M;
    const int mlp = layer * (wd.D - 1) + d - 1;
    const float* pf = prep_fwd + (int64_t)mlp * wd.prep_mlp;
    const float* w = W + mlp_blob_offset(lay, layer, d);
    const float* bias = w + (int64_t)(d + 1) * H;
    if (!(skip_last && M == 1)) dense(cst, n, Kx, Kx, pf, H, bias, nullptr, 0, 1, M == 1 ? a_last : A[0], H);
    pf += 2 * (int64_t)Kx * H;
    w = bias + H;
    for (int m = 1; m < M; ++m) {
      bias = w + (int64_t)H * H;
      if (!(skip_last && m == M - 1)) dense(A[m - 1], n, H, H, pf, H, bias, nullptr, 0, 1, m == M - 1 ? a_last : A[m], H);
      pf += 2 * (int64_t)H * H;
      w = bias + H;
    }
    if (skip_last || !ok()) return;
    bias = w + (int64_t)H * Pp;
    int64_t nb = (n + 127) / 128;   // 8 warps x 16 rows per block pass
    if (nb > 148 * 4) nb = 148 * 4;
    const size_t smem = (size_t)H * (Pp + 4) * sizeof(float);
    if (smem > 48 * 1024) {
      static int cur[64] = {};
      check(set_smem_max((const void*)wide_out_fwd_kernel<16>, smem, cur), "cudaFuncSetAttribute");
    }
    if (!ok()) return;
    wide_out_fwd_kernel<16><<<(unsigned)nb, kThreads, smem, s>>>(a_last, w, bias, n, H, theta);
    check_launch("wide_out_fwd_kernel launch");
  }

  void colsum(const float* Gm, int ldg, int64_t n, int N, float* dst) {
    if (!ok()) return;
    int64_t zy = n / 2048 + 1;
    if (zy > 296) zy = 296;
    wide_colsum_kernel<<<dim3((unsigned)((N + 31) / 32), (unsigned)zy), kThreads, 0, s>>>(Gm, ldg, n, N, dst);
    check_launch("wide_colsum_kernel launch");
  }

  void wgrad(const float* Am, int lda, const float* Gm, int ldg, int64_t n, int Ka, int Nb, float* dW, int ldw,
             float* db, const WgradMap* map = nullptr) {
    if (!ok()) return;
    check(dense_wgrad(s, Am, lda, Gm, ldg, n, Ka, Nb, dW, ldw, db, map), "dense_wgrad_kernel launch");
  }

  // backward of a conditioner given its activations (A[0..M-2], a_last) and GTheta: adds the input adjoints into
  // Gst (R x Kx) and the weight gradients into grad
  void mlp_backward(int layer, int d, const float* cst, float* Gst, int64_t n, const float* a_last) {
    const int H = wd.H, Kx = wd.Kx, Pp = wd.Pp, M = wd.M;
    const int mlp = layer * (wd.D - 1) + d - 1;
    const int64_t off = mlp_blob_offset(lay, layer, d);
    const float* pt = prep_T + (int64_t)mlp * wd.prep_mlp;
    const int64_t off_w0 = off, off_b0 = off + (int64_t)(d + 1) * H;
    const int64_t off_out = off_b0 + H + (int64_t)(M - 1) * ((int64_t)H * H + H);
    if (!ok()) return;
    // output layer: G2, dWout, dbout in one pass over the last hidden activations
    float* gc = Ga;
    float* gn = Gb;
    {
      const int hb = (H + kOutBwdCols - 1) / kOutBwdCols;
      int64_t ny = (n + 63) / 64;   // >= 64 rows per block, two blocks per SM (the ring takes 66 KB)
      if (ny * hb > 296) ny = 296 / hb;
      if (ny < 1) ny = 1;
      static int cur[64] = {};
      check(set_smem_max((const void*)wide_out_bwd_kernel<16>, out_bwd_smem<16>(), cur), "cudaFuncSetAttribute");
      if (!ok()) return;
      wide_out_bwd_kernel<16><<<dim3((unsigned)hb, (unsigned)ny), kOutBwdThreads, out_bwd_smem<16>(), s>>>(
          a_last, GTheta, W + off_out, n, H, gc, grad + off_out, grad + off_out + (int64_t)H * Pp);
      check_launch("wide_out_bwd_kernel launch");
    }
    for (int m = M - 1; m >= 1; --m) {
      const int64_t off_m = off_b0 + H + (int64_t)(m - 1) * ((int64_t)H * H + H);
      wgrad(A[m - 1], H, gc, H, n, H, H, grad + off_m, H, grad + off_m + (int64_t)H * H);
      const float* pt_m = pt + 2 * (int64_t)Kx * H + (int64_t)(m - 1) * 2 * H * H;
      dense(gc, n, H, H, pt_m, H, nullptr, A[m - 1], H, 2, gn, H);
      float* tmp = gc; gc = gn; gn = tmp;
    }
    if (!ok()) return;
    // input layer: dW0 / db0 on CUDA cores, the input adjoints accumulated into the adjoint state by the GEMM epilogue
    const bool sliced = Kx > kInWgradSlice;
    const int kv4 = sliced ? kInWgradSlice / 4 : (wd.D + 1 + 3) / 4;
    const int nz = sliced ? Kx / kInWgradSlice : 1;
    const int hb = (H + kInWgradCols - 1) / kInWgradCols;
    int64_t ny = (n + 63) / 64;
    if (ny * hb * nz > 296) ny = 296 / (hb * nz);
    if (ny < 1) ny = 1;
    dim3 grid((unsigned)hb, (unsigned)ny, (unsigned)nz);
    const size_t ring_bytes = in_wgrad_smem(sliced ? kInWgradSlice : Kx);
    if (sliced) {
      static int cur[64] = {};
      check(set_smem_max((const void*)wide_in_wgrad_kernel<kInWgradSlice / 4, true>, ring_bytes, cur), "cudaFuncSetAttribute");
      if (!ok()) return;
      wide_in_wgrad_kernel<kInWgradSlice / 4, true><<<grid, kThreads, ring_bytes, s>>>(cst, Kx, gc, n, H, wd.D, d, layer & 1,
                                                                                     grad + off_w0, grad + off_b0);
    } else switch (kv4) {
#define CNFOT_IN_WGRAD(Q)                                                                                              \
  case Q: {                                                                                                            \
    static int cur[64] = {};                                                                                           \
    check(set_smem_max((const void*)wide_in_wgrad_kernel<Q>, ring_bytes, cur), "cudaFuncSetAttribute");                \
    if (!ok()) return;                                                                                                 \
    wide_in_wgrad_kernel<Q><<<grid, kThreads, ring_bytes, s>>>(cst, Kx, gc, n, H, wd.D, d, layer & 1, grad + off_w0,   \
                                                               grad + off_b0);                                         \
    break;                                                                                                             \
  }
      CNFOT_IN_WGRAD(1) CNFOT_IN_WGRAD(2) CNFOT_IN_WGRAD(3) CNFOT_IN_WGRAD(4) CNFOT_IN_WGRAD(5) CNFOT_IN_WGRAD(6)
      CNFOT_IN_WGRAD(7) CNFOT_IN_WGRAD(8) CNFOT_IN_WGRAD(9) CNFOT_IN_WGRAD(10) CNFOT_IN_WGRAD(11) CNFOT_IN_WGRAD(12)
      CNFOT_IN_WGRAD(13) CNFOT_IN_WGRAD(14) CNFOT_IN_WGRAD(15) CNFOT_IN_WGRAD(16)
#undef CNFOT_IN_WGRAD
    }
    check_launch("wide_in_wgrad_kernel launch");
    dense(gc, n, H, H, pt, Kx, nullptr, nullptr, 0, 4, Gst, Kx);
  }

  template <int K>
  void spline(int dir, const float* theta, int bcast, const float* Sin, float* Sout, int col, float* LDp, int accumulate,
              int64_t n) {
    if (!ok()) return;
    if (dir == 0)
      wide_spline_kernel<K, 0><<<blocks_for(n), kThreads, 0, s>>>(theta, bcast, Sin, Sout, wd.Kx, col, LDp, accumulate, n, sc);
    else
      wide_spline_kernel<K, 1><<<blocks_for(n), kThreads, 0, s>>>(theta, bcast, Sin, Sout, wd.Kx, col, LDp, accumulate, n, sc);
    check_launch("wide_spline_kernel launch");
  }
  template <int K>
  void spline_vjp(int dir, const float* theta, int bcast, const float* Sin, int col, float* Gst, float gld,
                  const float* gld_rows, int64_t n) {
    if (!ok()) return;
    if (dir == 0)
      wide_spline_vjp_kernel<K, 0><<<blocks_for(n), kThreads, 0, s>>>(theta, bcast, Sin, wd.Kx, col, Gst, gld, gld_rows,
                                                                      GTheta, n, sc);
    else
      wide_spline_vjp_kernel<K, 1><<<blocks_for(n), kThreads, 0, s>>>(theta, bcast, Sin, wd.Kx, col, Gst, gld, gld_rows,
                                                                      GTheta, n, sc);
    check_launch("wide_spline_vjp_kernel launch");
  }

  // state 0 of pass p = [rows (+ shift on one coordinate) | t | 0]; ld_rows = row stride of explicit rows (0: dense, D)
  void init_states(int p, const PassSrc& ps, int64_t n, const float* cond = nullptr, int64_t cond_stride = 0,
                   int ld_rows = 0, int shift_col = -1, float shift = 0.f) {
    if (!ok()) return;
    int64_t total = n * wd.Kx * (wd.L + 1);
    int64_t b = (total + kThreads - 1) / kThreads;
    if (b > 148 * 16) b = 148 * 16;
    wide_init_kernel<<<(unsigned)b, kThreads, 0, s>>>(ps, dk, ld_rows ? ld_rows : wd.D, n, wd.D, wd.Kx, wd.L, state_stride(),
                                                      cond, cond_stride, shift_col, shift, S[p]);
    check_launch("wide_init_kernel launch");
  }
  void init_states(int p, const float* rows, int64_t n, float t, const float* cond = nullptr, int64_t cond_stride = 0) {
    init_states(p, explicit_src(rows, t), n, cond, cond_stride);
  }

  static unsigned grid_for(int64_t count) {
    int64_t b = (count + kThreads - 1) / kThreads;
    return (unsigned)(b > 148 * 16 ? 148 * 16 : (b < 1 ? 1 : b));
  }
  // pass p = `reps` passes over the same n rows (sources / times per pass in ms), stacked in one chunk
  void init_multi(int p, const MultiSrc& ms, int64_t n, int reps) {
    if (!ok()) return;
    wide_init_multi_kernel<<<grid_for(n * reps * wd.Kx * (wd.L + 1)), kThreads, 0, s>>>(ms, dk, n, reps, wd.D, wd.Kx, wd.L,
                                                                                        state_stride(), S[p]);
    check_launch("wide_init_multi_kernel launch");
  }
  void init_shift(int p, const float* R3, int64_t n, float shift) {
    if (!ok()) return;
    wide_init_shift_kernel<<<grid_for(n * 2 * wd.D * wd.Kx * (wd.L + 1)), kThreads, 0, s>>>(R3, n, wd.D, wd.Kx, wd.L,
                                                                                            state_stride(), shift, S[p]);
    check_launch("wide_init_shift_kernel launch");
  }
  void fill(float* p, int64_t count, float v) {
    if (!ok()) return;
    wide_fill_kernel<<<grid_for(count), kThreads, 0, s>>>(p, count, v);
    check_launch("wide_fill_kernel launch");
  }

  bool stashing(int p) const { return p == 0 && stashA != nullptr; }
  float* stash_a(int st, int d) const { return stashA + ((int64_t)st * (wd.D - 1) + d - 1) * R * wd.H; }
  float* stash_t(int st, int d) const { return stashT + ((int64_t)st * (wd.D - 1) + d - 1) * R * wd.Pp; }

  // one pass through the flow (flow_pass<DIR> of flow_math.cuh on a chunk); result in state(p, L), LD[p].
  // keep: pass 0 leaves every conditioner's last hidden activations and raw spline parameters in the stash
  // (when the workspace has one) so that flow_bwd does not re-run the hidden GEMMs.
  template <int K>
  void flow_pass(int dir, int p, int64_t n, bool keep = false) {
    const int D = wd.D, L = wd.L;
    keep = keep && stashing(p);
    for (int st = 0; st < L && ok(); ++st) {
      const int layer = dir == 0 ? st : L - 1 - st;
      const float* Sin = state(p, st);
      float* Sout = state(p, st + 1);
      const float* cst = dir == 0 ? Sin : Sout;
      for (int d = 0; d < D && ok(); ++d) {
        const int col = perm_at(layer, d, D);
        float* th = keep && d > 0 ? stash_t(st, d) : Theta;
        if (d > 0) mlp_forward(layer, d, cst, n, keep ? stash_a(st, d) : A[wd.M - 1], th);
        spline<K>(dir, d == 0 ? W : th, d == 0, Sin, Sout, col, LD[p], !(st == 0 && d == 0), n);
      }
    }
  }

  // reverse mode of flow_pass: G[p] holds the adjoint of state(p, L) on entry, of state(p, 0) on exit
  template <int K>
  void flow_bwd(int dir, int p, int64_t n, float gld, const float* gld_rows, bool kept = false) {
    const int D = wd.D, L = wd.L;
    kept = kept && stashing(p);
    for (int st = L - 1; st >= 0 && ok(); --st) {
      const int layer = dir == 0 ? st : L - 1 - st;
      const float* Sin = state(p, st);
      const float* cst = dir == 0 ? Sin : state(p, st + 1);
      for (int dd = 0; dd < D && ok(); ++dd) {
        const int d = dir == 0 ? dd : D - 1 - dd;
        const int col = perm_at(layer, d, D);
        const float* a_last = kept && d > 0 ? stash_a(st, d) : A[wd.M - 1];
        const float* th = kept && d > 0 ? stash_t(st, d) : Theta;
        if (d > 0) mlp_forward(layer, d, cst, n, A[wd.M - 1], Theta, kept);
        spline_vjp<K>(dir, d == 0 ? W : th, d == 0, Sin, col, G[p], gld, gld_rows, n);
        if (d == 0) colsum(GTheta, wd.Pp, n, wd.Pp, grad);
        else mlp_backward(layer, d, cst, G[p], n, a_last);
      }
    }
  }
};

int64_t chunk_rows() {
  int64_t r = 4 * 148 * 128;
  if (const char* e = getenv("CNFOT_WIDE_CHUNK")) {
    const long v = atol(e);
    if (v >= 128 && v <= (1 << 20)) r = round_up64(v, 128);
  }
  return r;
}

struct Carve {
  char* p;
  int64_t used = 0;
  explicit Carve(void* base) : p((char*)base) {}
  template <typename T>
  T* take(int64_t count) {
    T* out = p ? (T*)(p + used) : nullptr;
    used += round_up64(count * (int64_t)sizeof(T), 256);
    return out;
  }
};

// carve (or, with base == NULL, just size) the workspace
int64_t carve(void* base, const FlowLayout& lay, int64_t max_rows, bool with_grad, int n_pass, WideEngine* e) {
  WideDims wd = make_dims(lay);
  int64_t R = chunk_rows();
  if (max_rows < R) R = round_up64(max_rows > 0 ? max_rows : 1, 128);
  Carve c(base);
  const int64_t n_mlp = (int64_t)lay.L * (lay.D - 1);
  double* slots = c.take<double>(kNumSlots);
  float* pf = c.take<float>(n_mlp * wd.prep_mlp);
  float* pt = with_grad ? c.take<float>(n_mlp * wd.prep_mlp) : nullptr;
  float *S[kMaxPass] = {}, *LDp[kMaxPass] = {}, *G[kMaxPass] = {};
  for (int p = 0; p < n_pass; ++p) {
    S[p] = c.take<float>((int64_t)(lay.L + 1) * R * wd.Kx);
    LDp[p] = c.take<float>(R);
    if (with_grad) G[p] = c.take<float>(R * wd.Kx);
  }
  float* A[kMaxM];
  for (int m = 0; m < kMaxM; ++m) A[m] = m < lay.M ? c.take<float>(R * lay.H) : nullptr;
  float* Ga = with_grad ? c.take<float>(R * lay.H) : nullptr;
  float* Gb = with_grad && lay.M > 1 ? c.take<float>(R * lay.H) : nullptr;
  float* Theta = c.take<float>(R * lay.Pp);
  float* GTheta = with_grad ? c.take<float>(R * lay.Pp) : nullptr;
  float* GL = with_grad ? c.take<float>(R) : nullptr;
  float* GL2 = with_grad && n_pass > 3 ? c.take<float>(R) : nullptr;
  float* GRES = with_grad && n_pass > 3 ? c.take<float>(R * wd.Kx) : nullptr;
  float* V = !with_grad && n_pass > 3 ? c.take<float>(R * wd.Kx) : nullptr;
  // stash of pass 0 (last hidden activations + raw spline parameters of every conditioner): skips the re-computation
  // of the hidden GEMMs in the backward sweep.  Taken when it fits the budget (CNFOT_WIDE_STASH_GB, default 96;
  // 0 disables): BASELINE config 5 needs 79 GB at the default chunk -- this is what 180 GB of HBM3e are for.
  const int64_t stash_floats = with_grad ? n_mlp * R * (int64_t)(lay.H + lay.Pp) : 0;
  double budget_gb = 96.0;
  if (const char* ev = getenv("CNFOT_WIDE_STASH_GB")) budget_gb = atof(ev);
  const bool stash = stash_floats > 0 && (double)stash_floats * 4.0 <= budget_gb * 1e9;
  float* stashA = stash ? c.take<float>(n_mlp * R * (int64_t)lay.H) : nullptr;
  float* stashT = stash ? c.take<float>(n_mlp * R * (int64_t)lay.Pp) : nullptr;
  if (e) {
    e->lay = lay; e->wd = wd; e->R = R; e->slots = slots; e->prep_fwd = pf; e->prep_T = pt;
    for (int p = 0; p < kMaxPass; ++p) { e->S[p] = S[p]; e->LD[p] = LDp[p]; e->G[p] = G[p]; }
    for (int m = 0; m < kMaxM; ++m) e->A[m] = A[m];
    e->Ga = Ga; e->Gb = Gb; e->Theta = Theta; e->GTheta = GTheta; e->GL = GL; e->GL2 = GL2; e->GRES = GRES; e->V = V; e->stashA = stashA; e->stashT = stashT;
  }
  return c.used;
}

void launch_prep(WideEngine& e, bool with_T) {
  if (!e.ok()) return;
  const int n_mlp = e.lay.L * (e.lay.D - 1);
  if (n_mlp == 0) return;
  int bx = (e.wd.H * e.wd.H + kThreads - 1) / kThreads;
  if (bx > 64) bx = 64;
  wide_prep_kernel<<<dim3((unsigned)bx, (unsigned)n_mlp), kThreads, 0, e.s>>>(e.W, e.lay, e.wd, e.prep_fwd,
                                                                               with_T ? e.prep_T : nullptr);
  e.check_launch("wide_prep_kernel launch");
}

// the same rows at time t + dt (t - dt / 2 == t + (-dt / 2) exactly: the times of row_kinetic in step_math.cuh)
inline PassSrc at_time(PassSrc ps, float dt) {
  ps.t = ps.t + dt;
  return ps;
}

// kinetic terms of one chunk of the b-row sub-batch: `rt` = its rows at time t (row_kinetic of step_math.cuh)
template <int K>
void kinetic_chunk(WideEngine& e, const StepConsts<float>& pc, const PassSrc& rt, int64_t n) {
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  const bool with_score = pc.type != kOT;
  const bool obstacle = pc.potential == kPotObstacle && !with_score;
  e.init_states(0, at_time(rt, -pc.dt / 2.f), n);
  e.init_states(1, at_time(rt, pc.dt / 2.f), n);
  e.flow_pass<K>(0, 0, n);
  e.flow_pass<K>(0, 1, n);
  if (obstacle || with_score) {
    e.init_states(2, rt, n);
    e.flow_pass<K>(0, 2, n);
  }
  if (!e.ok()) return;
  if (!with_score) {
    wide_kinetic_head_kernel<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
        e.state(0, L), e.state(1, L), obstacle ? e.state(2, L) : nullptr, n, D, Kx, pc.dt, pc.w_kin, pc.w_pot, e.G[0], e.G[1],
        e.G[2], e.slots + kSlotKinetic, e.slots + kSlotPotential);
    e.check_launch("wide_kinetic_head_kernel launch");
  } else {
    const size_t gbytes = (size_t)n * Kx * sizeof(float);
    e.check(cudaMemsetAsync(e.G[0], 0, gbytes, e.s), "cudaMemsetAsync");
    e.check(cudaMemsetAsync(e.G[1], 0, gbytes, e.s), "cudaMemsetAsync");
    e.check(cudaMemsetAsync(e.G[2], 0, gbytes, e.s), "cudaMemsetAsync");
    e.check(cudaMemsetAsync(e.GRES, 0, gbytes, e.s), "cudaMemsetAsync");
    int64_t ab = (n * Kx + kThreads - 1) / kThreads;
    if (ab > 148 * 16) ab = 148 * 16;
    for (int i = 0; i < D && e.ok(); ++i) {
      // the two log-prob passes of coordinate i start from r3 -+ e_i dx/2 at the time of r3: forward both, then
      // back-propagate both
      const float* r3 = e.state(2, L);
      e.init_states(3, explicit_src(r3, 0.f), n, r3 + D, Kx, Kx, i, pc.dx / 2.f);
      e.init_states(4, explicit_src(r3, 0.f), n, r3 + D, Kx, Kx, i, -pc.dx / 2.f);
      e.flow_pass<K>(1, 3, n);
      e.flow_pass<K>(1, 4, n);
      if (!e.ok()) return;
      const auto score_head = head_for(D, wide_score_head_kernel<kHeadSmall>, wide_score_head_kernel<kHeadLarge>);
      score_head<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
          i, e.state(0, L), e.state(1, L), e.state(2, L), e.state(3, L), e.LD[3], e.state(4, L), e.LD[4], n, D, Kx, pc, e.G[0],
          e.G[1], e.G[3], e.G[4], e.GL, e.GL2, e.GRES, e.slots + kSlotKinetic);
      e.check_launch("wide_score_head_kernel launch");
      e.flow_bwd<K>(1, 3, n, 0.f, e.GL);
      e.flow_bwd<K>(1, 4, n, 0.f, e.GL2);
      if (!e.ok()) return;
      wide_add2_kernel<<<(unsigned)ab, kThreads, 0, e.s>>>(e.G[2], e.G[3], e.G[4], n * Kx);
      e.check_launch("wide_add2_kernel launch");
    }
    if (pc.type == kFP && e.ok()) {
      const auto pullback = head_for(D, wide_drift_pullback_kernel<kHeadSmall>, wide_drift_pullback_kernel<kHeadLarge>);
      pullback<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(e.state(2, L), e.GRES, n, D, Kx, pc, e.G[2]);
      e.check_launch("wide_drift_pullback_kernel launch");
    }
  }
  e.flow_bwd<K>(0, 1, n, 0.f, nullptr);
  e.flow_bwd<K>(0, 0, n, 0.f, nullptr);
  if (obstacle || with_score) e.flow_bwd<K>(0, 2, n, 0.f, nullptr);
}

// CNFOT_WIDE_BATCH=0 keeps one flow pass per chunk (the path large batches take anyway)
bool batching_enabled() {
  const char* ev = getenv("CNFOT_WIDE_BATCH");
  return !(ev && ev[0] == '0');
}

// kinetic_chunk with the passes of a row stacked in shared chunks: [r(t-dt/2); r(t+dt/2); r(t)] is ONE sample-
// direction pass of 2-3 n rows and the 2 D shifted log-prob passes of the score are ONE pass of 2 D n rows.
// Requires 3 n <= R and (score) 2 D n <= R.
template <int K>
void kinetic_chunk_batched(WideEngine& e, const StepConsts<float>& pc, const PassSrc& rt, int64_t n) {
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  const bool with_score = pc.type != kOT;
  const bool obstacle = pc.potential == kPotObstacle && !with_score;
  const int reps = (obstacle || with_score) ? 3 : 2;
  MultiSrc ms;
  ms.src[0] = at_time(rt, -pc.dt / 2.f); ms.src[1] = at_time(rt, pc.dt / 2.f); ms.src[2] = rt;
  e.init_multi(0, ms, n, reps);
  e.flow_pass<K>(0, 0, n * reps);
  if (!e.ok()) return;
  const int64_t blk = n * Kx;
  float* r1 = e.state(0, L);
  float* g1 = e.G[0];
  if (!with_score) {
    wide_kinetic_head_kernel<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
        r1, r1 + blk, obstacle ? r1 + 2 * blk : nullptr, n, D, Kx, pc.dt, pc.w_kin, pc.w_pot, g1, g1 + blk, g1 + 2 * blk,
        e.slots + kSlotKinetic, e.slots + kSlotPotential);
    e.check_launch("wide_kinetic_head_kernel launch");
  } else {
    e.init_shift(1, r1 + 2 * blk, n, pc.dx / 2.f);
    e.flow_pass<K>(1, 1, n * 2 * D);
    if (!e.ok()) return;
    const auto score_head_all = head_for(D, wide_score_head_all_kernel<kHeadSmall>, wide_score_head_all_kernel<kHeadLarge>);
    score_head_all<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
        r1, r1 + blk, r1 + 2 * blk, e.state(1, L), e.LD[1], n, D, Kx, pc, g1, g1 + blk, g1 + 2 * blk, e.G[1], e.GL, e.GRES,
        e.slots + kSlotKinetic);
    e.check_launch("wide_score_head_all_kernel launch");
    e.flow_bwd<K>(1, 1, n * 2 * D, 0.f, e.GL);
    if (!e.ok()) return;
    wide_fold_kernel<<<WideEngine::grid_for(blk), kThreads, 0, e.s>>>(g1 + 2 * blk, e.G[1], n, 2 * D, Kx);
    e.check_launch("wide_fold_kernel launch");
    if (pc.type == kFP) {
      const auto pullback = head_for(D, wide_drift_pullback_kernel<kHeadSmall>, wide_drift_pullback_kernel<kHeadLarge>);
      pullback<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(r1 + 2 * blk, e.GRES, n, D, Kx, pc, g1 + 2 * blk);
      e.check_launch("wide_drift_pullback_kernel launch");
    }
  }
  e.flow_bwd<K>(0, 0, n * reps, 0.f, nullptr);
}

// the step's row sets: the caller's arrays and host times, or (draws != NULL) the Philox draws of the step
struct StepRows {
  const float *latent, *latent_sub, *src, *tgt, *t_batch_host;
  const WideDraws* draws;
  int D;
  // rows [r0, r0 + n) of a row set of the B-row terms (sub = false) or of the b-row kinetic terms (sub = true) at time t,
  // plus, with t_index >= 0, the step's time t_index
  PassSrc at(const float* rows, int source, bool sub, int64_t r0, float t, int t_index = -1) const {
    if (!draws) return explicit_src(rows + r0 * D, t_index >= 0 ? t_batch_host[t_index] + t : t);
    PassSrc p = {};
    p.t = t;
    p.source = source;
    p.t_index = t_index;
    p.salt = sub ? draws->salts.b : draws->salts.B;
    p.row0 = (sub ? draws->row0_b : draws->row0_B) + r0;
    return p;
  }
};

template <int K>
void run_step(WideEngine& e, const StepConsts<float>& pc, const StepRows& in, int n_t, int64_t rows_B, int64_t rows_b) {
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  const bool batch = batching_enabled();
  // kinetic terms: the b-row sub-batch at every sampled time
  const bool with_score = pc.type != kOT;
  for (int it = 0; it < n_t && e.ok(); ++it) {
    // rows per chunk such that the stacked passes fit: 3 n <= R and, with the score, 2 D n <= R
    int64_t cap = e.R / (with_score && 2 * D > 3 ? 2 * D : 3);
    const bool stacked = batch && cap >= 1 && rows_b <= cap * 4;   // large sub-batches: plain chunks fill the GPU anyway
    if (!stacked) cap = e.R;
    for (int64_t r0 = 0; r0 < rows_b && e.ok(); r0 += cap) {
      const int64_t n = rows_b - r0 < cap ? rows_b - r0 : cap;
      const PassSrc rt = in.at(in.latent_sub, kRowsNormal, true, r0, 0.f, it);
      if (stacked) kinetic_chunk_batched<K>(e, pc, rt, n);
      else kinetic_chunk<K>(e, pc, rt, n);
    }
  }
  const int64_t half = e.R / 2;
  if (pc.type == kOT) {
    // density-fit terms: -lambda mean log p(data | t) at t = 0 (source) and t = T (target)
    if (batch && half >= 1) {
      // source rows at t = 0 and the same number of target rows at t = T share a chunk
      for (int64_t r0 = 0; r0 < rows_B && e.ok(); r0 += half) {
        const int64_t n = rows_B - r0 < half ? rows_B - r0 : half;
        MultiSrc ms;
        ms.src[0] = in.at(in.src, kRowsOtSource, false, r0, 0.f);
        ms.src[1] = ms.src[2] = in.at(in.tgt, kRowsNormal, false, r0, pc.horizon);
        e.init_multi(0, ms, n, 2);
        e.flow_pass<K>(1, 0, 2 * n, true);
        if (!e.ok()) break;
        for (int side = 0; side < 2; ++side) {
          wide_nll_head_kernel<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
              e.state(0, L) + side * n * Kx, e.LD[0] + side * n, n, D, Kx, pc.w_fit, e.G[0] + side * n * Kx,
              e.slots + (side == 0 ? kSlotFit0 : kSlotFitT));
          e.check_launch("wide_nll_head_kernel launch");
        }
        e.flow_bwd<K>(1, 0, 2 * n, -pc.w_fit, nullptr, true);
      }
      return;
    }
    for (int side = 0; side < 2 && e.ok(); ++side) {
      const float t = side == 0 ? 0.f : pc.horizon;
      double* slot = e.slots + (side == 0 ? kSlotFit0 : kSlotFitT);
      for (int64_t r0 = 0; r0 < rows_B && e.ok(); r0 += e.R) {
        const int64_t n = rows_B - r0 < e.R ? rows_B - r0 : e.R;
        e.init_states(0, side == 0 ? in.at(in.src, kRowsOtSource, false, r0, t) : in.at(in.tgt, kRowsNormal, false, r0, t), n);
        e.flow_pass<K>(1, 0, n, true);
        if (!e.ok()) break;
        wide_nll_head_kernel<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(e.state(0, L), e.LD[0], n, D, Kx, pc.w_fit,
                                                                          e.G[0], slot);
        e.check_launch("wide_nll_head_kernel launch");
        e.flow_bwd<K>(1, 0, n, -pc.w_fit, nullptr, true);
      }
    }
    return;
  }
  // rwpo / fp: reverse-KL fit at t = 0 on the B latent rows; rwpo adds the terminal potential at t = T
  const int n_seg = pc.type == kRWPO ? 2 : 1;
  if (batch && n_seg == 2 && half >= 1) {
    // the fit rows at t = 0 and the same latent rows at t = T (potential) share a chunk; the log-det adjoint is
    // -w_fit on the first half and 0 on the second: per-row
    for (int64_t r0 = 0; r0 < rows_B && e.ok(); r0 += half) {
      const int64_t n = rows_B - r0 < half ? rows_B - r0 : half;
      MultiSrc ms;
      ms.src[0] = in.at(in.latent, kRowsNormal, false, r0, 0.f);
      ms.src[1] = ms.src[2] = in.at(in.latent, kRowsNormal, false, r0, pc.horizon);
      e.init_multi(0, ms, n, 2);
      e.flow_pass<K>(0, 0, 2 * n, true);
      if (!e.ok()) break;
      for (int seg = 0; seg < 2; ++seg) {
        const auto sample_head = head_for(D, wide_sample_head_kernel<kHeadSmall>, wide_sample_head_kernel<kHeadLarge>);
        sample_head<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
            e.state(0, 0) + seg * n * Kx, e.state(0, L) + seg * n * Kx, e.LD[0] + seg * n, n, D, Kx, seg == 0 ? 0.f : pc.horizon, seg == 0,
            seg == 1, pc, e.G[0] + seg * n * Kx, e.slots + kSlotFit0, e.slots + kSlotPotential);
        e.check_launch("wide_sample_head_kernel launch");
      }
      e.fill(e.GL, n, -pc.w_fit);
      e.fill(e.GL + n, n, 0.f);
      e.flow_bwd<K>(0, 0, 2 * n, 0.f, e.GL, true);
    }
    return;
  }
  for (int seg = 0; seg < n_seg && e.ok(); ++seg) {
    const int do_fit = seg == 0, do_pot = seg == 1;
    const float t = seg == 0 ? 0.f : pc.horizon;
    for (int64_t r0 = 0; r0 < rows_B && e.ok(); r0 += e.R) {
      const int64_t n = rows_B - r0 < e.R ? rows_B - r0 : e.R;
      e.init_states(0, in.at(in.latent, kRowsNormal, false, r0, t), n);
      e.flow_pass<K>(0, 0, n, true);
      if (!e.ok()) break;
      const auto sample_head = head_for(D, wide_sample_head_kernel<kHeadSmall>, wide_sample_head_kernel<kHeadLarge>);
      sample_head<<<WideEngine::blocks_for(n), kThreads, 0, e.s>>>(
          e.state(0, 0), e.state(0, L), e.LD[0], n, D, Kx, t, do_fit, do_pot, pc, e.G[0], e.slots + kSlotFit0,
          e.slots + kSlotPotential);
      e.check_launch("wide_sample_head_kernel launch");
      e.flow_bwd<K>(0, 0, n, do_fit ? -pc.w_fit : 0.f, nullptr, true);
    }
  }
}

}  // namespace

static_assert(kWideMaxDim == 255, "wide_supported's message names the bound");
bool wide_supported(const FlowLayout& lay, const char** why) {
  const char* w = nullptr;
  if (lay.D < 2) w = "wide engine needs dim >= 2";
  else if (lay.H < 16 || lay.H % 16 || (lay.H > 64 && lay.H % 64)) w = "wide engine needs hidden in {16, 32, 48} or a multiple of 64";
  else if (lay.M < 1 || lay.M > kMaxM) w = "wide engine supports 1..4 hidden layers";
  else if (lay.K != 5) w = "wide engine is instantiated for num_bins == 5";
  else if (lay.D > kWideMaxDim) w = "wide engine supports dim <= 255";
  else if ((int64_t)lay.L * (lay.D - 1) > 65535) w = "wide engine needs num_layers * (dim - 1) <= 65535";
  if (!w) {
    // FlowLayout offsets are int: the whole blob must stay below 2^31 floats (make_layout's sums, in 64 bits)
    const int64_t H = lay.H, mlp_const = H + (lay.M - 1) * (H * H + H) + H * lay.Pp + lay.Pp;
    const int64_t layer_stride = (int64_t)(lay.D - 1) * mlp_const + H * ((int64_t)(lay.D - 1) * (lay.D + 2) / 2);
    if (lay.Pp + lay.L * layer_stride > INT32_MAX) w = "wide engine needs a parameter blob below 2^31 floats";
  }
  if (why) *why = w;
  return w == nullptr;
}

int64_t wide_step_workspace_bytes(const FlowLayout& lay, int64_t rows_B, int64_t rows_b) {
  return carve(nullptr, lay, rows_B > rows_b ? rows_B : rows_b, true, kMaxPass, nullptr);
}

int64_t wide_flow_workspace_bytes(const FlowLayout& lay, int64_t rows, bool with_grad) {
  return carve(nullptr, lay, rows, with_grad, 1, nullptr);
}

cudaError_t wide_mfc_step(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const StepConsts<float>& pc,
                          const float* weights, const float* latent, const float* latent_sub, const float* src,
                          const float* tgt, const float* t_batch_host, const WideDraws* draws, int n_t, int64_t rows_B,
                          int64_t rows_b, float* out, const WideAdam* adam, void* workspace, const char** what) {
  WideEngine e;
  e.s = s; e.sc = sc; e.W = weights; e.grad = out;
  carve(workspace, lay, rows_B > rows_b ? rows_B : rows_b, true, kMaxPass, &e);
  if (draws) {
    e.dk.key = draws->key; e.dk.step = draws->step; e.dk.state = draws->state;
    e.dk.salt_c = draws->salts.Bc; e.dk.salt_t = draws->salts.t; e.dk.horizon = pc.horizon;
  }
  e.check(cudaMemsetAsync(out, 0, ((size_t)lay.total + kNumSlots) * sizeof(float), s), "cudaMemsetAsync");
  e.check(cudaMemsetAsync(e.slots, 0, kNumSlots * sizeof(double), s), "cudaMemsetAsync");
  launch_prep(e, true);
  StepRows in = {latent, latent_sub, src, tgt, t_batch_host, draws, lay.D};
  run_step<5>(e, pc, in, n_t, rows_B, rows_b);
  if (e.ok()) {
    wide_finalize_kernel<<<1, 32, 0, s>>>(e.slots, out + lay.total);
    e.check_launch("wide_finalize_kernel launch");
  }
  if (adam && e.ok()) {
    wide_adam_kernel<<<WideEngine::grid_for(lay.total), kThreads, 0, s>>>(out, lay.total, adam->state, adam->lr, adam->b1,
                                                                          adam->b2, adam->eps, adam->weights, adam->m,
                                                                          adam->v, adam->loss_hist, adam->loss_hist_len);
    e.check_launch("wide_adam_kernel launch");
    if (e.ok()) {
      wide_advance_kernel<<<1, 32, 0, s>>>(adam->state);
      e.check_launch("wide_advance_kernel launch");
    }
  }
  if (what) *what = e.what;
  return e.err;
}

cudaError_t wide_flow_eval(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                           int dir, const float* in, const float* cond, int64_t cond_stride, int64_t rows, float* out,
                           float* logdet, int add_base, void* workspace, const char** what) {
  WideEngine e;
  e.s = s; e.sc = sc; e.W = weights; e.grad = nullptr;
  carve(workspace, lay, rows, false, 1, &e);
  launch_prep(e, false);
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  for (int64_t r0 = 0; r0 < rows && e.ok(); r0 += e.R) {
    const int64_t n = rows - r0 < e.R ? rows - r0 : e.R;
    e.init_states(0, in + r0 * D, n, 0.f, cond + r0 * cond_stride, cond_stride);
    e.flow_pass<5>(dir, 0, n);
    if (!e.ok()) break;
    int64_t b = (n * D + kThreads - 1) / kThreads;
    if (b > 148 * 16) b = 148 * 16;
    wide_extract_kernel<<<(unsigned)b, kThreads, 0, s>>>(e.state(0, L), n, D, Kx, out + r0 * D);
    e.check_launch("wide_extract_kernel launch");
    if (logdet) {
      // forward: log N(latent input) - fldj ; inverse: log N(latent output) + ildj
      const float* base = dir == 0 ? e.state(0, 0) : e.state(0, L);
      wide_logdet_out_kernel<<<WideEngine::blocks_for(n), kThreads, 0, s>>>(e.LD[0], base, Kx, n, D, add_base,
                                                                        dir == 0 ? -1.f : 1.f, logdet + r0);
      e.check_launch("wide_logdet_out_kernel launch");
    }
  }
  if (what) *what = e.what;
  return e.err;
}

cudaError_t wide_flow_vjp(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                          int dir, const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                          const float* g_out, const float* g_logdet, int add_base, float* g_in, float* g_weights,
                          void* workspace, const char** what) {
  WideEngine e;
  e.s = s; e.sc = sc; e.W = weights; e.grad = g_weights;
  carve(workspace, lay, rows, true, 1, &e);
  e.check(cudaMemsetAsync(g_weights, 0, (size_t)lay.total * sizeof(float), s), "cudaMemsetAsync");
  launch_prep(e, true);
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  for (int64_t r0 = 0; r0 < rows && e.ok(); r0 += e.R) {
    const int64_t n = rows - r0 < e.R ? rows - r0 : e.R;
    e.init_states(0, in + r0 * D, n, 0.f, cond + r0 * cond_stride, cond_stride);
    e.flow_pass<5>(dir, 0, n, true);
    if (!e.ok()) break;
    wide_vjp_seed_kernel<<<WideEngine::blocks_for(n), kThreads, 0, s>>>(g_out + r0 * D, g_logdet ? g_logdet + r0 : nullptr,
                                                                    e.state(0, L), n, D, Kx, dir, add_base, e.G[0], e.GL);
    e.check_launch("wide_vjp_seed_kernel launch");
    e.flow_bwd<5>(dir, 0, n, 0.f, e.GL, true);
    if (g_in && e.ok()) {
      wide_vjp_out_kernel<<<WideEngine::blocks_for(n), kThreads, 0, s>>>(e.G[0], g_logdet ? g_logdet + r0 : nullptr,
                                                                     e.state(0, 0), n, D, Kx, dir, add_base, g_in + r0 * D);
      e.check_launch("wide_vjp_out_kernel launch");
    }
  }
  if (what) *what = e.what;
  return e.err;
}

int64_t wide_energy_workspace_bytes(const FlowLayout& lay) {
  return carve(nullptr, lay, chunk_rows(), false, kMaxPass, nullptr);
}

cudaError_t wide_kinetic_energy(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                                const float* latent, int64_t batch, int latent_blocks, const float* t_host, int n_t, float dt,
                                int with_score, float kappa, float dx, double* out, void* workspace, const char** what) {
  WideEngine e;
  e.s = s; e.sc = sc; e.W = weights; e.grad = nullptr;
  carve(workspace, lay, chunk_rows(), false, kMaxPass, &e);
  e.check(cudaMemsetAsync(e.slots, 0, kNumSlots * sizeof(double), s), "cudaMemsetAsync");
  launch_prep(e, false);
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  const double weight = 1.0 / (2.0 * (double)batch * (double)n_t);
  for (int it = 0; it < n_t && e.ok(); ++it) {
    const float t = t_host[it];
    const float* block = latent + (int64_t)(it % latent_blocks) * batch * D;
    for (int64_t r0 = 0; r0 < batch && e.ok(); r0 += e.R) {
      const int64_t n = batch - r0 < e.R ? batch - r0 : e.R;
      const float* rows = block + r0 * D;
      int64_t ab = (n * Kx + kThreads - 1) / kThreads;
      if (ab > 148 * 16) ab = 148 * 16;
      e.init_states(0, rows, n, t - dt / 2.f);
      e.init_states(1, rows, n, t + dt / 2.f);
      e.flow_pass<5>(0, 0, n);
      e.flow_pass<5>(0, 1, n);
      if (!e.ok()) break;
      wide_velocity_kernel<<<(unsigned)ab, kThreads, 0, s>>>(e.state(0, L), e.state(1, L), n, D, Kx, dt, e.V);
      e.check_launch("wide_velocity_kernel launch");
      if (with_score) {
        e.init_states(2, rows, n, t);
        e.flow_pass<5>(0, 2, n);
        for (int i = 0; i < D && e.ok(); ++i) {
          e.init_states(3, explicit_src(e.state(2, L), t), n, nullptr, 0, Kx, i, dx / 2.f);
          e.init_states(4, explicit_src(e.state(2, L), t), n, nullptr, 0, Kx, i, -dx / 2.f);
          e.flow_pass<5>(1, 3, n);
          e.flow_pass<5>(1, 4, n);
          if (!e.ok()) break;
          wide_score_add_kernel<<<WideEngine::blocks_for(n), kThreads, 0, s>>>(i, e.state(3, L), e.LD[3], e.state(4, L), e.LD[4],
                                                                           n, D, Kx, kappa, dx, e.V);
          e.check_launch("wide_score_add_kernel launch");
        }
      }
      if (!e.ok()) break;
      wide_sumsq_kernel<<<(unsigned)(ab > 592 ? 592 : ab), kThreads, 0, s>>>(e.V, n * Kx, weight, e.slots + kSlotKinetic);
      e.check_launch("wide_sumsq_kernel launch");
    }
  }
  if (e.ok()) {
    wide_energy_out_kernel<<<1, 32, 0, s>>>(e.slots, out);
    e.check_launch("wide_energy_out_kernel launch");
  }
  if (what) *what = e.what;
  return e.err;
}

int64_t wide_density_workspace_bytes(const FlowLayout& lay, int n_t) {
  return carve(nullptr, lay, chunk_rows(), false, 1, nullptr) + round_up64((int64_t)(n_t > 0 ? n_t : 0) * (int64_t)sizeof(float), 256);
}

namespace {

// the chunk loop of both density modes: one flow pass per chunk (grid: log-prob direction from the points; Monte-Carlo:
// sample direction from the latent draw), then the head
cudaError_t run_density(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                        const DensityPoints& dp, int64_t n, float* samples, float* density, int with_ref, float mix,
                        float var0, float var1, double* sq_err, void* workspace, const char** what) {
  WideEngine e;
  e.s = s; e.sc = sc; e.W = weights; e.grad = nullptr;
  carve(workspace, lay, chunk_rows(), false, 1, &e);
  if (with_ref) e.check(cudaMemsetAsync(e.slots, 0, kNumSlots * sizeof(double), s), "cudaMemsetAsync");
  launch_prep(e, false);
  const int D = e.wd.D, Kx = e.wd.Kx, L = e.wd.L;
  const int dir = dp.mode == 0 ? 1 : 0;
  for (int64_t r0 = 0; r0 < n && e.ok(); r0 += e.R) {
    const int64_t m = n - r0 < e.R ? n - r0 : e.R;
    wide_density_init_kernel<<<WideEngine::blocks_for(m), kThreads, 0, s>>>(dp, r0, m, D, Kx, L, e.state_stride(), e.S[0]);
    e.check_launch("wide_density_init_kernel launch");
    e.flow_pass<5>(dir, 0, m);
    if (!e.ok()) break;
    if (samples) {
      wide_extract_kernel<<<WideEngine::grid_for(m * D), kThreads, 0, s>>>(e.state(0, L), m, D, Kx, samples + r0 * D);
      e.check_launch("wide_extract_kernel launch");
    }
    if (density || with_ref) {
      const float* Z = dir == 1 ? e.state(0, L) : e.state(0, 0);
      const float* Y = dir == 1 ? e.state(0, 0) : e.state(0, L);
      wide_density_head_kernel<<<WideEngine::blocks_for(m), kThreads, 0, s>>>(
          Z, Y, e.LD[0], dir == 1 ? 1.f : -1.f, m, D, Kx, density ? density + r0 : nullptr, with_ref, mix, var0, var1,
          e.slots + kSlotKinetic);
      e.check_launch("wide_density_head_kernel launch");
    }
  }
  if (with_ref && e.ok()) {
    wide_energy_out_kernel<<<1, 32, 0, s>>>(e.slots, sq_err);
    e.check_launch("wide_energy_out_kernel launch");
  }
  if (what) *what = e.what;
  return e.err;
}

}  // namespace

cudaError_t wide_density_grid(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                              const float* t_host, int n_t, double x_min, double x_step, double y_min, double y_step, int nx,
                              int ny, float* density, int with_ref, float mix, float var0, float var1, double* sq_err,
                              void* workspace, const char** what) {
  DensityPoints dp = {};
  dp.mode = 0; dp.nx = nx; dp.ny = ny;
  dp.x_min = x_min; dp.x_step = x_step; dp.y_min = y_min; dp.y_step = y_step;
  // the times follow the chunk buffers in the workspace
  float* t_dev = (float*)((char*)workspace + carve(nullptr, lay, chunk_rows(), false, 1, nullptr));
  cudaError_t err = cudaMemcpyAsync(t_dev, t_host, (size_t)n_t * sizeof(float), cudaMemcpyHostToDevice, s);
  if (err != cudaSuccess) {
    if (what) *what = "H2D times";
    return err;
  }
  dp.t_dev = t_dev;
  return run_density(s, lay, sc, weights, dp, (int64_t)nx * ny * n_t, nullptr, density, with_ref, mix, var0, var1, sq_err,
                     workspace, what);
}

cudaError_t wide_density_mc(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                            float cond, uint64_t key_n, uint32_t step, int64_t n, float* samples, float* density,
                            int with_ref, float mix, float var0, float var1, double* sq_err, void* workspace,
                            const char** what) {
  DensityPoints dp = {};
  dp.mode = 1; dp.key_n = key_n; dp.step = step; dp.cond = cond;
  return run_density(s, lay, sc, weights, dp, n, samples, density, with_ref, mix, var0, var1, sq_err, workspace, what);
}

}  // namespace cnfot
