// Device-side plumbing shared by the fused flow / train-step kernels:
// shared-memory carving, the per-row activation tiles, the CTA-wide
// weight-gradient sink, loss reductions.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "flow_math.cuh"

namespace cnfot {

constexpr int kTile = 128;       // rows per CTA tile == threads per CTA (one row per thread)
constexpr int kWarps = kTile / 32;

// Staged [kTile][n] tiles (n a multiple of 4) are read 128 bits at a time by 8
// consecutive rows at once; those 8 accesses must fall into 8 distinct 16-byte bank
// groups.  With C = n/4 chunks per row:
//   C odd            dense rows already do (row stride is an odd number of groups)
//   C = 2, 4, 8k     dense rows + XOR swizzle of the chunk index with tile_swizzle(row)
//   other even C     pad the row to an odd number of groups (no swizzle)
__host__ __device__ inline bool tile_uses_swizzle(int n) {
  const int c = (n + 3) / 4;
  return c == 2 || c == 4 || (c >= 8 && c % 8 == 0);
}
__host__ __device__ inline int staged_stride(int n) {
  int q = (n + 3) / 4;
  if ((q & 1) == 0 && !tile_uses_swizzle(n)) q += 1;
  return q * 4;
}
__host__ __device__ inline int tile_swizzle(int n, int row) {
  if (!tile_uses_swizzle(n)) return 0;
  const int c = (n + 3) / 4;
  if (c == 2) return (row >> 2) & 1;
  if (c == 4) return (row >> 1) & 3;
  return row & 7;
}

// Shared-memory layout of one CTA (offsets in floats).
struct SmemPlan {
  int total;            // blob floats
  int w_in_smem;        // 1: whole blob resident in shared memory; 0: `first` resident and one
                        //    conditioner at a time staged at off_w (weights stream from L2)
  int off_w;            // resident blob, or [first (Pp) | staging buffer] when not resident
  int w_stage;          // floats of the staging buffer (largest conditioner), 0 if resident
  int off_acc;          // gradient accumulators (same layout as the blob); -1 if none
  int off_in, ld_in;    // [kTile][ld_in]  conditioner inputs
  int off_hid, ld_h;    // M tiles [kTile][ld_h] hidden activations
  int off_gh;           // M tiles [kTile][ld_h] hidden adjoints; -1 if none
  int off_gth, ld_p;    // [kTile][ld_p] spline-parameter adjoints; -1 if none
  int off_lo;           // tcgen05 engine: [kTile][16] scratch tile for the low tf32 halves; -1 if unused
  int off_wmma;         // tcgen05 engine: weights in MMA layout (4 tiles of 16x16 per dense layer)
  int off_frag;         // warp-MMA engine: hi/lo weight fragments (warp_mlp.cuh); -1 if unused
  int off_wt, wt_stride;  // warp-MMA engine: per-warp [32 x 16] tiles, floats per warp
  int off_fk;             // normalised knots of the shared `first` spline (FirstKnots, kFirstKnotFloats floats)
  int floats;
};

constexpr int kFirstKnotFloats = 128;   // room for FirstKnots<float, K> up to K = 20
constexpr int kTileAlign = 128;  // tiles start on 512-byte boundaries (hardware swizzle = address bits)
inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

inline SmemPlan plan_smem(const FlowLayout& f, bool with_grad, bool w_in_smem = true,
                          bool tensor_cores = false) {
  SmemPlan p;
  p.total = f.total;
  p.w_in_smem = w_in_smem ? 1 : 0;
  const int tot4 = (f.total + 3) / 4 * 4;
  p.ld_in = staged_stride((f.D + 3) / 4 * 4);
  p.ld_h = staged_stride(f.H);
  p.ld_p = staged_stride(f.Pp);
  p.off_w = 0;
  p.w_stage = w_in_smem ? 0 : (f.D * f.H + f.mlp_const + 3) / 4 * 4;
  int o = w_in_smem ? tot4 : f.Pp + p.w_stage;
  p.off_acc = with_grad ? o : -1;
  if (with_grad) o += tot4;
  o = align_up(o, kTileAlign);
  p.off_in = o; o += kTile * p.ld_in;
  o = align_up(o, kTileAlign);
  p.off_hid = o; o += f.M * kTile * p.ld_h;
  p.off_gh = with_grad ? o : -1;
  if (with_grad) o += f.M * kTile * p.ld_h;
  p.off_gth = with_grad ? o : -1;
  if (with_grad) o += kTile * p.ld_p;
  p.off_lo = -1;
  p.off_wmma = -1;
  p.off_frag = -1;
  p.off_wt = -1;
  p.wt_stride = 0;
  if (tensor_cores) {
    o = align_up(o, kTileAlign);
    p.off_lo = o; o += kTile * 16;
    p.off_wmma = o; o += f.L * (f.D - 1) * f.M * 4 * 256;
  }
  o = align_up(o, 4);
  p.off_fk = o; o += kFirstKnotFloats;
  p.floats = o;
  return p;
}

// Cooperative copy of the weight blob into shared memory (float4, coalesced).
__device__ inline void load_weights(float* sW, const float* __restrict__ gW, int total) {
  const int n4 = total >> 2;
  const float4* src = reinterpret_cast<const float4*>(gW);
  float4* dst = reinterpret_cast<float4*>(sW);
  for (int i = threadIdx.x; i < n4; i += blockDim.x) dst[i] = __ldg(src + i);
  for (int i = (n4 << 2) + threadIdx.x; i < total; i += blockDim.x) sW[i] = __ldg(gW + i);
}

// The normalised knots of the shared `first` spline (rqs_math.cuh: first_knots_build) by ONE WARP: lane k owns bin k and
// knot k; maxima, sums and the cumulative sums of the bin sizes travel with shuffles.  (One thread doing it serially was
// a ~400-instruction dependent chain, 1.7 us, on the critical path of every CTA's set-up.)  All 32 lanes must call.
template <int K, class SC>
__device__ __forceinline__ void first_knots_build_warp(const float* theta, const SC& c, FirstKnots<float, K>& fk) {
  static_assert(K + 1 <= 32, "one lane per knot");
  constexpr unsigned kAll = 0xffffffffu;
  const int k = threadIdx.x & 31;
  const bool bin = k < K;
  float pos[2], prob[2];
#pragma unroll
  for (int axis = 0; axis < 2; ++axis) {
    const float u = bin ? theta[axis * K + k] : -INFINITY;
    float m = u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kAll, m, o));
    const float e = bin ? m_exp_shifted(u, m_exp_shift_prep(m)) : 0.f;
    float sum = e;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(kAll, sum, o);
    const float inv = m_rcp(sum);
    const float size = bin ? e * (inv * c.bin_scale) + c.min_bin : 0.f;
    prob[axis] = e * inv;
    float acc = size;   // inclusive scan: lane k ends with size[0] + ... + size[k]
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float v = __shfl_up_sync(kAll, acc, o);
      if (k >= o) acc += v;
    }
    pos[axis] = c.lo + acc;   // position of knot k + 1
  }
  if (bin) {
    fk.pw[k] = prob[0];
    fk.ph[k] = prob[1];
    if (k + 1 <= K - 1) { fk.xp[k + 1] = pos[0]; fk.yp[k + 1] = pos[1]; }
  }
  if (k == 0) { fk.xp[0] = c.lo; fk.yp[0] = c.lo; fk.xp[K] = c.hi; fk.yp[K] = c.hi; }
  if (k <= K) {
    const float u = theta[2 * K + k] + c.slope_offset;
    fk.dk[k] = softplus(u) + c.min_slope;
    fk.sg[k] = sigmoid(u);
  }
}

// once per CTA: the normalised knots of the shared `first` spline, by warp 0
template <class Net>
__device__ inline void build_first_knots(const float* first_smem, float* fk_smem) {
  static_assert(sizeof(FirstKnots<float, Net::kK>) <= kFirstKnotFloats * sizeof(float), "FirstKnots does not fit its slot");
  if (threadIdx.x < 32)
    first_knots_build_warp<Net::kK>(first_smem, FixedSplineConsts<float, Net::kK>(),
                                    *reinterpret_cast<FirstKnots<float, Net::kK>*>(fk_smem));
}

template <class Net>
__device__ inline RowTiles<float, Net> make_row_tiles(float* smem, const SmemPlan& p) {
  RowTiles<float, Net> tl;
  const int r = threadIdx.x;
  tl.in = smem + p.off_in + r * p.ld_in;
#pragma unroll
  for (int m = 0; m < Net::kM; ++m) {
    tl.hid[m] = smem + p.off_hid + (m * kTile + r) * p.ld_h;
    tl.gh[m] = p.off_gh >= 0 ? smem + p.off_gh + (m * kTile + r) * p.ld_h : nullptr;
  }
  tl.gth = p.off_gth >= 0 ? smem + p.off_gth + r * p.ld_p : nullptr;
  tl.sw_h = tile_swizzle(Net::kH, r);
  tl.sw_p = tile_swizzle(Net::kPp, r);
  return tl;
}

// The CTA-wide context of the fused kernels (the `Ctx` policy of flow_math.cuh):
// weights in shared memory and the weight-gradient reduction over the staged row tiles.
//
// commit(): after every thread (= row) has written its conditioner input, hidden
// activations and adjoints into the tiles, the CTA re-partitions GEMM-style: the
// gradient of each layer, dW = A^T G over the tile's 128 rows, is cut into 4x4
// blocks; a lane owns one block for one eighth of the rows (8 row groups x 4 blocks
// per warp, 16 FMAs per pair of float4 loads), the 8 row groups are folded with a
// reduce-scatter butterfly (14 shuffles) and each lane adds its 2 results to the
// CTA's shared-memory accumulator.  Bias gradients (column sums of G) take a second,
// cheap phase.  Every accumulator element has exactly one owner lane per call, so no
// atomics are needed; the accumulators are flushed once per CTA at kernel end.
template <class Net>
struct DeviceCtx {
  using NetT = Net;
  static constexpr bool kWarpMlp = false;
  static constexpr bool kAccInGlobal = false;
  __device__ __forceinline__ void bind_partials(float*, bool = true) {}
  __device__ __forceinline__ void bind_frags(const float*) {}
  __device__ __forceinline__ void stash_acquire(int, int, uint32_t*) {}
  __device__ __forceinline__ void stash_release() {}
  __device__ __forceinline__ bool stash_on() const { return false; }   // the warp-level engines keep an activation stash
  static constexpr int H = Net::kH, M = Net::kM, Pp = Net::kPp;
  float* smem;
  const float* gW;   // the blob in global memory
  SmemPlan p;

  __device__ __forceinline__ int row_in_tile() const { return threadIdx.x; }
  __device__ __forceinline__ void setup(int, int, uint64_t*, uint32_t*) { load(); }
  __device__ __forceinline__ void teardown() {}

  // once per kernel: bring the blob (or just `first`) into shared memory
  __device__ __forceinline__ void load() {
    if (p.w_in_smem) load_weights(smem + p.off_w, gW, p.total);
    else load_weights(smem + p.off_w, gW, Pp);
    if (p.off_acc >= 0)
      for (int i = threadIdx.x; i < p.total; i += blockDim.x) smem[p.off_acc + i] = 0.f;
    __syncthreads();
    build_first_knots<Net>(smem + p.off_w, smem + p.off_fk);
    __syncthreads();
  }

  __device__ __forceinline__ const float* first_params() const { return smem + p.off_w; }
  __device__ __forceinline__ const FirstKnots<float, Net::kK>& first_knots() const {
    return *reinterpret_cast<const FirstKnots<float, Net::kK>*>(smem + p.off_fk);
  }

  __device__ __forceinline__ const float* weights(int w_off, int count) {
    if (p.w_in_smem) return smem + p.off_w + w_off;
    __syncthreads();  // previous conditioner's readers are done with the staging buffer
    float* dst = smem + p.off_w + Pp;
    const float4* src = reinterpret_cast<const float4*>(gW + w_off);
    for (int i = threadIdx.x; i < (count >> 2); i += blockDim.x)
      reinterpret_cast<float4*>(dst)[i] = __ldg(src + i);
    __syncthreads();
    return dst;
  }

  __device__ __forceinline__ void begin() { __syncthreads(); }

  // dense contractions of the hidden / output layers on the CUDA cores (see flow_math.cuh)
  template <int K, int N>
  __device__ __forceinline__ void dense_fwd(const float* xt, int sw, const float*, const float* Wm, int, float* y) {
    dense_fwd_from_tile<float, K, N>(xt, sw, Wm, y);
  }
  template <int K, int N>
  __device__ __forceinline__ void dense_bwd(const float*, int, const float* g, const float* Wm, int, float* y) {
    dense_bwd_from_regs<float, K, N>(g, Wm, y);
  }

  // one 4x4 block: rows rb*4.. of A (tile pa, stride lda) x cols cb*4.. of G
  __device__ __forceinline__ void block_accumulate(const float* pa, int lda, const float* pg,
                                                   int ldg, float* c) {
#pragma unroll 4
    for (int k = 0; k < kTile / 8; ++k) {
      const float4 g4 = *reinterpret_cast<const float4*>(pg + k * 8 * ldg);
      const float4 a4 = *reinterpret_cast<const float4*>(pa + k * 8 * lda);
      c[0] += a4.x * g4.x; c[1] += a4.x * g4.y; c[2] += a4.x * g4.z; c[3] += a4.x * g4.w;
      c[4] += a4.y * g4.x; c[5] += a4.y * g4.y; c[6] += a4.y * g4.z; c[7] += a4.y * g4.w;
      c[8] += a4.z * g4.x; c[9] += a4.z * g4.y; c[10] += a4.z * g4.z; c[11] += a4.z * g4.w;
      c[12] += a4.w * g4.x; c[13] += a4.w * g4.y; c[14] += a4.w * g4.z; c[15] += a4.w * g4.w;
    }
  }

  __device__ __noinline__ void reduce(int w_off, int n_in) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rg = lane & 7, slot = lane >> 3;
    constexpr int CH = H / 4, CP = Pp / 4;
    const int nb0 = ((n_in + 3) >> 2) * CH;          // input layer blocks
    constexpr int nbm = CH * CH;                       // each hidden layer
    constexpr int nbo = CH * CP;                       // output layer
    const int total = nb0 + (M - 1) * nbm + nbo;
    float* acc = smem + p.off_acc + w_off;
    const float* t_in = smem + p.off_in;
    const float* t_hid = smem + p.off_hid;
    const float* t_gh = smem + p.off_gh;
    const float* t_gth = smem + p.off_gth;
    const int off_hidden0 = n_in * H + H;             // first hidden (H x H) matrix
    for (int base = warp * 4; base < total; base += 4 * kWarps) {
      const int b = base + slot;
      const bool valid = b < total;
      const float *pa = t_in, *pg = t_gh;
      int lda = p.ld_in, ldg = p.ld_h, Na = n_in, ncol = H, rb = 0, cb = 0;
      float* dst = acc;
      if (valid) {
        if (b < nb0) {
          rb = b / CH; cb = b - rb * CH;
        } else if (b < nb0 + (M - 1) * nbm) {
          const int q = b - nb0;
          const int m = 1 + q / nbm;                  // hidden layer m: A = hid[m-1], G = gh[m]
          const int r = q - (m - 1) * nbm;
          rb = r / CH; cb = r - rb * CH;
          pa = t_hid + (m - 1) * kTile * p.ld_h; lda = p.ld_h; Na = H;
          pg = t_gh + m * kTile * p.ld_h;
          dst = acc + off_hidden0 + (m - 1) * (H * H + H);
        } else {
          const int r = b - nb0 - (M - 1) * nbm;     // output layer: A = hid[M-1], G = gth
          rb = r / CP; cb = r - rb * CP;
          pa = t_hid + (M - 1) * kTile * p.ld_h; lda = p.ld_h; Na = H;
          pg = t_gth; ldg = p.ld_p; ncol = Pp;
          dst = acc + off_hidden0 + (M - 1) * (H * H + H);
        }
      }
      float c[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) c[e] = 0.f;
      if (valid) {
        // rows rg, rg+8, ...: their swizzle depends on rg only (the +8k does not reach it)
        const int sa = pa == t_in ? 0 : tile_swizzle(H, rg);
        const int sg = ncol == H ? tile_swizzle(H, rg) : tile_swizzle(Pp, rg);
        block_accumulate(pa + rg * lda + ((rb ^ sa) << 2), lda, pg + rg * ldg + ((cb ^ sg) << 2), ldg, c);
      }
      // reduce-scatter over the 8 row groups (lane bits 0..2)
      const bool b2 = lane & 4, b1 = lane & 2, b0 = lane & 1;
      float v8[8], v4[4], v2[2];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float keep = b2 ? c[8 + q] : c[q], send = b2 ? c[q] : c[8 + q];
        v8[q] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float keep = b1 ? v8[4 + q] : v8[q], send = b1 ? v8[q] : v8[4 + q];
        v4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const float keep = b0 ? v4[2 + q] : v4[q], send = b0 ? v4[q] : v4[2 + q];
        v2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
      }
      const int row = rb * 4 + (b2 ? 2 : 0) + (b1 ? 1 : 0);
      if (valid && row < Na) {
        float2* q = reinterpret_cast<float2*>(dst + row * ncol + cb * 4 + (b0 ? 2 : 0));
        float2 cur = *q;
        cur.x += v2[0];
        cur.y += v2[1];
        *q = cur;
      }
    }
    // bias gradients: column sums of every G tile; one (tile, 4-column block) task per
    // warp iteration, the 32 lanes split the 128 rows
    constexpr int tasks = M * CH + CP;
    for (int task = warp; task < tasks; task += kWarps) {
      const float* pg;
      int ldg, cb;
      float* dst;
      if (task < M * CH) {
        const int m = task / CH;
        cb = task - m * CH;
        pg = t_gh + m * kTile * p.ld_h; ldg = p.ld_h;
        dst = m == 0 ? acc + n_in * H : acc + off_hidden0 + (m - 1) * (H * H + H) + H * H;
      } else {
        cb = task - M * CH;
        pg = t_gth; ldg = p.ld_p;
        dst = acc + off_hidden0 + (M - 1) * (H * H + H) + H * Pp;
      }
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      const int sg = task < M * CH ? tile_swizzle(H, lane) : tile_swizzle(Pp, lane);
#pragma unroll
      for (int k = 0; k < kTile / 32; ++k) {
        const float4 g4 = *reinterpret_cast<const float4*>(pg + (k * 32 + lane) * ldg + ((cb ^ sg) << 2));
        s.x += g4.x; s.y += g4.y; s.z += g4.z; s.w += g4.w;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
        s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
        s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
        s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
      }
      if (lane == 0) {
        float4* q = reinterpret_cast<float4*>(dst + cb * 4);
        float4 cur = *q;
        cur.x += s.x; cur.y += s.y; cur.z += s.z; cur.w += s.w;
        *q = cur;
      }
    }
  }

  __device__ __forceinline__ void commit(int w_off, int n_in, const RowTiles<float, Net>&) {
    __syncthreads();  // every row's tiles are written
    reduce(w_off, n_in);
  }

  // flush the per-thread adjoint of the shared `first` parameter (blob offset 0)
  __device__ __forceinline__ void flush_first(const float* gfirst, const RowTiles<float, Net>& tl) {
    __syncthreads();
#pragma unroll
    for (int j = 0; j < Pp; j += 4)
      *reinterpret_cast<float4*>(tl.gth + chunk_at(j, tl.sw_p)) =
          make_float4(gfirst[j], gfirst[j + 1], gfirst[j + 2], gfirst[j + 3]);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float* pg = smem + p.off_gth;
    for (int cb = warp; cb < Pp / 4; cb += kWarps) {
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      const int sg = tile_swizzle(Pp, lane);
#pragma unroll
      for (int k = 0; k < kTile / 32; ++k) {
        const float4 g4 = *reinterpret_cast<const float4*>(pg + (k * 32 + lane) * p.ld_p + ((cb ^ sg) << 2));
        s.x += g4.x; s.y += g4.y; s.z += g4.z; s.w += g4.w;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
        s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
        s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
        s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
      }
      if (lane == 0) {
        float4* q = reinterpret_cast<float4*>(smem + p.off_acc + cb * 4);
        float4 cur = *q;
        cur.x += s.x; cur.y += s.y; cur.z += s.z; cur.w += s.w;
        *q = cur;
      }
    }
    __syncthreads();
  }
};

// Sum a per-thread double over the CTA; result valid in thread 0.
__device__ inline double block_sum(double v, double* scratch /* kWarps doubles */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kWarps; ++w) t += scratch[w];
  return t;
}

}  // namespace cnfot
