// Warp-level tensor-core engine for the conditioner MLP of 16-wide networks
// (hidden == 16, padded spline-parameter count == 16: the mfc.yaml defaults).
//
// A warp owns 32 sample rows.  The per-row code (splines, loss terms, flow state) keeps its
// "one thread = one row" form; every conditioner evaluation inside it is done by the warp as
// a whole with mma.sync.m16n8k8 (tf32 inputs, fp32 accumulate), chained in registers:
//
//   * "C layout": thread (g = lane/4, t = lane%4) holds rows 8q+g (q = 0..3) x columns
//     {2t, 2t+1, 8+2t, 9+2t} of a [32 x 16] activation matrix -- the accumulator fragments of
//     2 m-tiles x 2 n-tiles.  An accumulator fragment is fed straight back as the A fragment
//     of the next layer by re-labelling the contraction index (logical k = t <-> feature 2t,
//     k = t+4 <-> feature 2t+1 inside each 8-wide k-step); the weight fragments are built with
//     the same re-labelling, so chaining layers costs no shuffles and no shared memory.
//   * fp32 fidelity: every product is split  x*w = x_hi*w_hi + x_lo*w_hi + x_hi*w_lo  with
//     x_hi = x rounded to tf32 and x_lo = x - x_hi (exact); the weights' hi/lo fragments are
//     built once per CTA.  24 MMAs replace the 256 FMAs per row of a 16x16 layer.
//   * row <-> C-layout changes (the spline needs all 16 parameters of its row in one thread) and
//     the transposed operands of the weight gradient  dW = A^T G  go through per-warp
//     [32 x 16] shared-memory tiles with an XOR swizzle that makes all four access patterns
//     (C-layout float2, row float4, transposed scalar A^T / G reads) bank-conflict-free.
//   * the thread <-> row map inside a warp is  row = 8t + g, so the quad (same g) that holds a
//     row's C-layout pieces also contains its owner: layer-0 inputs and the input gradients
//     move with quad-local shuffles only.
//   * weight gradients: per-warp MMA over its 32 rows, then added to the CTA's
//     partial-gradient row
//     in global memory with fire-and-forget red.global (L2); warps are otherwise independent --
//     no CTA barrier in the loop.
//
// Reference semantics: the conditioner of /root/reference/cnf_ot/models/flows.py:46-86
// (hk.nets.MLP([H]*M, activate_final=True) -> hk.Linear(P)), evaluated on [t, y[perm[:d]]]
// (/root/reference/cnf_ot/models/autoregressive.py:94-98,124-128).
#pragma once

#include "device_common.cuh"

namespace cnfot {

constexpr int kWtFloats = 32 * 16;   // one per-warp tile
constexpr int kFragFloats = 1024;    // per dense matrix: forward (512) + transposed (512) fragments

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// 3xTF32 split  v = hi + lo  with hi = v ROUNDED to tf32 (nearest, ties away: two integer instructions) and
// lo = v - hi (exact, |lo| <= 2^-12 |v|).  The tensor core truncates an operand register to its tf32 bits, so hi is
// passed explicitly; what the truncation then loses of lo is <= 2^-23 |v|.  Round 1 split by truncation
// (hi = the register itself, one instruction less per element): |lo| <= 2^-10 |v|, the truncated lo loses up to
// 2^-21 |v| and always towards zero -- a bias that does not average out over 10^5 rows and that the finite
// differences of the score terms (1 / dx = 100) amplify: 4.8e-5 of the largest gradient entry at 2^18 rows.
#if defined(CNFOT_TF32_TRUNC)   // the round-1 split, kept for A/B measurements (tools/diag_parity.py)
__device__ __forceinline__ uint32_t tf32_round(float v) { return __float_as_uint(v) & 0xFFFFE000u; }
#else
__device__ __forceinline__ uint32_t tf32_round(float v) { return (__float_as_uint(v) + 0x00001000u) & 0xFFFFE000u; }
#endif
__device__ __forceinline__ void split_tf32(float v, uint32_t& hi, uint32_t& lo) {
  hi = tf32_round(v);
  lo = __float_as_uint(v - __uint_as_float(hi));
}

// Shared-memory plan of the warp-MMA kernels (same struct as the CUDA-core plan; the row tiles
// of the latter are not used).
// resident: what the CUDA cores read of the blob (`first`, input layers, biases: compact copy, cw_floats) and the
// hi/lo fragments of the 16x16 matrices live in shared memory (measured on cfg 2: reading the input layers from global/L1 instead costs
// ~3 %, and a fifth CTA per SM at <= 102 registers is slower than four at 128).
// streamed (larger flows, e.g. dim 10): only `first` is resident; input layers / biases are read
// from the blob and the fragments from a buffer a prep kernel fills (build_frags_kernel), both in
// global memory through L1.
// Compact resident copy of the blob (resident plan): [first (Pp) | per conditioner: W0 ((d+1) x 16), b0, b1 .. b_{M-1}, bout].
// The 16 x 16 matrices themselves are only read as MMA fragments, so they are not copied.
__host__ __device__ inline int cw_layer_stride(int D, int M) { return 16 * ((D - 1) * (D + 2) / 2) + (D - 1) * (M + 1) * 16; }
__host__ __device__ inline int cw_offset(int D, int M, int Pp, int layer, int d) {
  return Pp + layer * cw_layer_stride(D, M) + 16 * ((d - 1) * (d + 2) / 2) + (d - 1) * (M + 1) * 16;
}
__host__ __device__ inline int cw_floats(int D, int L, int M, int Pp) { return Pp + L * cw_layer_stride(D, M); }

inline SmemPlan plan_smem_mma(const FlowLayout& f, bool with_grad, bool resident = true) {
  SmemPlan p;
  p.total = f.total;
  p.w_in_smem = resident ? 1 : 0;
  p.ld_in = p.ld_h = p.ld_p = 0;
  p.off_w = 0;
  p.w_stage = 0;
  int o = resident ? cw_floats(f.D, f.L, f.M, f.Pp) : f.Pp;
  p.off_acc = -1;   // weight gradients go straight to the CTA's partial row in global memory
  p.off_in = p.off_hid = p.off_gh = p.off_gth = p.off_lo = p.off_wmma = -1;
  o = align_up(o, 32);
  p.off_frag = o;
  if (resident) o += f.L * (f.D - 1) * f.M * kFragFloats;
  p.off_wt = o;
  p.wt_stride = (with_grad ? f.M + 1 : 1) * kWtFloats;
  o += kWarps * p.wt_stride;
  p.off_fk = o; o += kFirstKnotFloats;
  p.floats = o;
  return p;
}

// ---- shared-memory accessors on 32-bit shared-window addresses ------------------------------
// (the contexts are passed by reference through non-inlined per-row functions, so generic
// pointers kept in them would turn every access into a generic LD/ST with 64-bit address math)
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float2 lds64(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
// read-only data (weights, fragments): not volatile, the compiler may schedule / merge them
__device__ __forceinline__ float2 ldw64(uint32_t a) {
  float2 v;
  asm("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 ldw128(uint32_t a) {
  float4 v;
  asm("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts32(uint32_t a, float x) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(x) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, float x, float y) {
  asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(a), "f"(x), "f"(y) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
// fire-and-forget float adds into the CTA's partial-gradient row in global memory (resolved in L2;
// shared-memory float atomics would be compare-and-swap loops)
__device__ __forceinline__ void red_global(float* q, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(q), "f"(v) : "memory");
}
__device__ __forceinline__ void red_global2(float* q, float x, float y) {
  asm volatile("red.global.add.v2.f32 [%0], {%1,%2};" ::"l"(q), "f"(x), "f"(y) : "memory");
}

// A float-indexed reference to read-only weights: a shared-window address (resident plan) or a
// pointer into global memory (streamed plan).
template <bool RES>
struct WRef;
template <>
struct WRef<true> {
  uint32_t a;
  __device__ __forceinline__ WRef operator+(int floats) const { return WRef{a + (uint32_t)floats * 4u}; }
  __device__ __forceinline__ float2 ld2() const { return ldw64(a); }
  __device__ __forceinline__ float4 ld4() const { return ldw128(a); }
  __device__ __forceinline__ bool valid() const { return a != 0u; }
  __device__ __forceinline__ static WRef none() { return WRef{0u}; }
};
template <>
struct WRef<false> {
  const float* q;
  __device__ __forceinline__ WRef operator+(int floats) const { return WRef{q + floats}; }
  __device__ __forceinline__ float2 ld2() const { return __ldg(reinterpret_cast<const float2*>(q)); }
  __device__ __forceinline__ float4 ld4() const { return __ldg(reinterpret_cast<const float4*>(q)); }
  __device__ __forceinline__ bool valid() const { return q != nullptr; }
  __device__ __forceinline__ static WRef none() { return WRef{nullptr}; }
};

// One float4 of the hi/lo weight fragments of a 16-wide flow (hidden = Pp = 16):
//   element e = ((mat * 2 + dir) * 4 + ks * 2 + nt) * 32 + lane,  mat = mlp * M + slot
//   dir 0 (y = x W):    b0 = W[8ks+2t][8nt+g]   b1 = W[8ks+2t+1][8nt+g]
//   dir 1 (y = g W^T):  b0 = W[8nt+g][8ks+2t]   b1 = W[8nt+g][8ks+2t+1]
//   value = { b0_hi, b1_hi, b0_lo, b1_lo }
// LDG: the blob is in global memory (read-only path); false: a staged copy in shared memory
template <bool LDG = true>
__device__ __forceinline__ float4 frag_element(const float* __restrict__ blob, int D, int M, int e) {
  constexpr int H = 16, Pp = 16;
  const int ln = e & 31, ksnt = (e >> 5) & 3, dir = (e >> 7) & 1, mat = e >> 8;
  const int mlp = mat / M, slot = mat - mlp * M;
  const int layer = mlp / (D - 1), d = mlp - layer * (D - 1) + 1;
  const int mlp_const = H + (M - 1) * (H * H + H) + H * Pp + Pp;
  const int layer_stride = (D - 1) * mlp_const + H * ((D - 1) * (D + 2) / 2);
  const float* Ws = blob + Pp + layer * layer_stride + (d - 1) * mlp_const + H * ((d - 1) * (d + 2) / 2) +
                    (d + 1) * H + H + slot * (H * H + H);
  const int ks = ksnt >> 1, nt = ksnt & 1, gg = ln >> 2, tt = ln & 3;
  float b0, b1;
  const float* q0 = dir == 0 ? Ws + (8 * ks + 2 * tt) * 16 + 8 * nt + gg : Ws + (8 * nt + gg) * 16 + 8 * ks + 2 * tt;
  const float* q1 = q0 + (dir == 0 ? 16 : 1);
  if constexpr (LDG) { b0 = __ldg(q0); b1 = __ldg(q1); }
  else { b0 = *q0; b1 = *q1; }
  uint32_t h0, l0, h1, l1;
  split_tf32(b0, h0, l0);
  split_tf32(b1, h1, l1);
  return make_float4(__uint_as_float(h0), __uint_as_float(h1), __uint_as_float(l0), __uint_as_float(l1));
}

// streamed plan: fragments of every dense matrix into a global buffer (n_mat * kFragFloats floats)
static __global__ void build_frags_kernel(const float* __restrict__ blob, float* __restrict__ frags, int D, int M,
                                   int n_mat) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_mat * 256; e += gridDim.x * blockDim.x)
    reinterpret_cast<float4*>(frags)[e] = frag_element(blob, D, M, e);
}

// per-thread constants of the engine (recomputed from threadIdx.x where needed: cheaper than
// re-loading them from a context that lives in local memory)
struct MmaLane {
  uint32_t lane, g, t;
  uint32_t cbase;   // C-layout byte offset inside a tile, before the chunk term: (g*16 + 2*(t&1))*4
  uint32_t cu;      // C-layout chunk selector: chunk(q, nt) = cu ^ (2nt ^ q)
  uint32_t rbase;   // row-layout byte offset: (8t+g)*64
  uint32_t ru;      // row-layout chunk selector: chunk(c) = ru ^ c
  uint32_t tbase;   // transposed reads: (t*16 + (g&3))*4
  uint32_t tu;      // transposed reads: chunk selector (g>>2) ^ (t&2); chunk = tu ^ ks ^ {0,2} (^1 for rows +4)
  __device__ __forceinline__ MmaLane() {
    lane = threadIdx.x & 31;
    g = lane >> 2;
    t = lane & 3;
    const uint32_t fg = ((g >> 1) & 1) * 2 + ((g >> 2) & 1);
    cbase = (g * 16 + 2 * (t & 1)) * 4;
    cu = (t >> 1) ^ fg;
    rbase = (8 * t + g) * 64;
    ru = t ^ fg;
    tbase = (t * 16 + (g & 3)) * 4;
    tu = (g >> 2) ^ (t & 2);
  }
};

// Shared-window address of the CTA's dynamic shared memory: every `extern __shared__` array starts there, and the
// address is a link-time constant.
__device__ __forceinline__ uint32_t dyn_smem_base() {
  extern __shared__ __align__(1024) float cnfot_dyn_smem[];
  return (uint32_t)__cvta_generic_to_shared(cnfot_dyn_smem);
}
__device__ __forceinline__ float* dyn_smem_ptr() {
  extern __shared__ __align__(1024) float cnfot_dyn_smem[];
  return cnfot_dyn_smem;
}

// DC, LC > 0 (the train-step kernel specialised for the mfc.yaml flow, resident plan, with gradients): the shared-memory
// plan is a compile-time constant, so the tile / weight / fragment / knot addresses the engine needs all the time are
// immediates (+ the warp index) instead of members of a context that lives in the caller's local memory and has to be
// re-loaded after every asm memory clobber (a quarter of the kernel's long-scoreboard stalls, tools/ncu_stall_lines.py).
// STASH: the kernel keeps the activation stash (below) in tensor memory; false: no tcgen05 instruction is compiled in.
template <class Net, bool RES, int DC = 0, int LC = 0, bool STASH = false>
struct DeviceCtxMma {
  using NetT = Net;
  using Ref = WRef<RES>;
  static constexpr bool kConstPlan = RES && DC > 0 && LC > 0;
  // mirror of plan_smem_mma(f, with_grad = true, resident = true), in floats
  static constexpr int kcW = 0;
  static constexpr int kcCw = Net::kPp + LC * (16 * ((DC - 1) * (DC + 2) / 2) + (DC - 1) * (Net::kM + 1) * 16);
  static constexpr int kcFrag = (kcCw + 31) / 32 * 32;
  static constexpr int kcWt = kcFrag + LC * (DC - 1) * Net::kM * kFragFloats;
  static constexpr int kcWtStride = (Net::kM + 1) * kWtFloats;
  static constexpr int kcFk = kcWt + kWarps * kcWtStride;
  __device__ __forceinline__ Ref wref() const {
    if constexpr (kConstPlan) return Ref{dyn_smem_base() + (uint32_t)kcW * 4u};
    else return w_ref;
  }
  __device__ __forceinline__ Ref fref() const {
    if constexpr (kConstPlan) return Ref{dyn_smem_base() + (uint32_t)kcFrag * 4u};
    else return frag_ref;
  }
  __device__ __forceinline__ uint32_t swt() const {
    if constexpr (kConstPlan) return dyn_smem_base() + ((uint32_t)kcWt + (threadIdx.x >> 5) * (uint32_t)kcWtStride) * 4u;
    else return s_wt;
  }
  static constexpr bool kWarpMlp = true;
  static constexpr bool kStash = STASH;   // the activation stash is compiled in (kEngMmaStash)
  static constexpr bool kAccInGlobal = true;
  static constexpr int H = Net::kH, M = Net::kM, Pp = Net::kPp;
  static_assert(H == 16 && Pp == 16, "the warp-MMA engine is written for 16-wide layers");
  float* smem;
  const float* gW;
  SmemPlan p;
  float* gacc;   // this CTA's partial-gradient row (blob layout) in global memory; nullptr: forward only
  const float* gfrag;   // streamed plan: the fragment buffer in global memory
  Ref w_ref, frag_ref;  // blob and fragments (shared-window address or global pointer)
  uint32_t s_wt;        // shared-window address of this warp's tiles
  // Activation stash in tensor memory: the forward pass of a row that is differentiated right away (KL / reverse-KL /
  // potential rows: 97 % of a step) leaves every conditioner's hidden activations (as the warp holds them: MMA
  // fragments) and the located spline (SplineState of the thread's row: softmax probabilities, the gathered knots, slope
  // logits) here, and the backward pass reads them back instead of evaluating the conditioner and normalising the knots
  // a second time.  The stash is strictly per thread, which is the tcgen05.ld / tcgen05.st 32x32b shape: thread i of
  // warp w owns TMEM lane 32 w + i.  Columns of a thread (nc = L (D - 1) conditioners, c = layer (D - 1) + d - 1; every
  // 16-column access starts on a 16-column boundary):
  //   [16 (c M + m), +16)          hidden activations m of conditioner c (A order)
  //   [16 (nc M + c), +16)         located spline of conditioner c, floats 0..15
  //   [16 nc (M + 1) + 4 c, +4)    its floats 16..19
  // stash_nc == 0: no stash, the backward pass recomputes.
  static constexpr int kStateFloats = 2 * Net::kK + 10;
  static_assert(kStateFloats == 20, "the stash layout holds a located spline of 5 bins");
  uint32_t stash_t = 0;   // TMEM address of lane 32 w, column 0 (w: the calling thread's warp)
  int stash_nc = 0;
  int stash_cols = 0;     // columns allocated by this CTA
  __device__ __forceinline__ bool stash_on() const { return STASH && stash_nc != 0; }
  __device__ __forceinline__ int stash_ncond() const {
    if constexpr (kConstPlan) return LC * (DC - 1);
    else return stash_nc;
  }
  __device__ __forceinline__ static int stash_cond(int D, int layer, int d) { return layer * (D - 1) + d - 1; }
  // cols: a power of two >= 32 (the host launches a STASH kernel only with the stash on).  One warp allocates, every
  // thread leaves with the address.  A CTA allocates once, so it gives up its allocation permit right away.
  __device__ __forceinline__ void stash_acquire(int cols, int n_cond, uint32_t* slot) {
    if constexpr (STASH) {
      if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((uint32_t)__cvta_generic_to_shared(slot)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      stash_t = *slot + ((threadIdx.x & ~31u) << 16);
      stash_nc = n_cond;
      stash_cols = cols;
    }
  }
  // Every thread of the CTA calls this once it has no rows left: the columns go back to the SM at once (a kernel that
  // is launched behind this one may then allocate them while this CTA is still in its epilogue).
  __device__ __forceinline__ void stash_release() {
    if constexpr (STASH) {
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      if (threadIdx.x < 32) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(stash_t), "r"(stash_cols) : "memory");
      }
      stash_nc = 0;
      stash_cols = 0;
    }
  }
  __device__ __forceinline__ static void tmem_st16(uint32_t ta, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(ta), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]),
          "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
        : "memory");
  }
  __device__ __forceinline__ static void tmem_st4(uint32_t ta, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};"
                 ::"r"(ta), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
  }
  // load and wait in one statement: the outputs cannot be used before tcgen05.wait::ld has returned
  __device__ __forceinline__ static void tmem_ld16(uint32_t ta, float* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
          "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
        : "r"(ta) : "memory");
  }
  __device__ __forceinline__ static void tmem_ld16_4(uint32_t ta16, uint32_t ta4, float* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%20];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x4.b32 {%16,%17,%18,%19}, [%21];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]),
          "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]),
          "=f"(v[17]), "=f"(v[18]), "=f"(v[19])
        : "r"(ta16), "r"(ta4) : "memory");
  }
  __device__ __forceinline__ uint32_t stash_hidden(int c, int m) const { return stash_t + 16 * (c * M + m); }
  // the located spline of the calling thread's row (after rqs_locate_raw in the forward pass)
  __device__ __forceinline__ void stash_state(int D, int layer, int d, const SplineState<float, Net::kK>& st) const {
    if constexpr (STASH) {
      constexpr int K = Net::kK;
      float b[kStateFloats];
  #pragma unroll
      for (int k = 0; k < K; ++k) { b[k] = st.pw[k]; b[K + k] = st.ph[k]; }
      b[2 * K] = st.x0; b[2 * K + 1] = st.x1; b[2 * K + 2] = st.y0; b[2 * K + 3] = st.y1;
      b[2 * K + 4] = st.d0; b[2 * K + 5] = st.d1; b[2 * K + 6] = st.u0; b[2 * K + 7] = st.u1;
      b[2 * K + 8] = st.u_tail;
      b[2 * K + 9] = __int_as_float(st.idx | (st.tail << 8));
      const int c = stash_cond(D, layer, d), nc = stash_ncond();
      __syncwarp();   // the .aligned stores need the whole warp (the spline's search branches per row)
      tmem_st16(stash_t + 16 * (nc * M + c), b);
      tmem_st4(stash_t + 16 * nc * (M + 1) + 4 * c, b + 16);
    }
  }

  bool clear_acc;       // setup() zeroes the partial row (false: rows shared between CTAs, cleared by the caller)
  __device__ __forceinline__ void bind_partials(float* q, bool clear = true) { gacc = q; clear_acc = clear; }
  __device__ __forceinline__ void bind_frags(const float* q) { gfrag = q; }

  // row of the CTA tile owned by the calling thread
  __device__ __forceinline__ int row_in_tile() const {
    const int lane = threadIdx.x & 31;
    return (threadIdx.x & ~31) + 8 * (lane & 3) + (lane >> 2);
  }

  __device__ __forceinline__ void setup(int D, int L, uint64_t*, uint32_t*) {
    const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(smem);
    s_wt = s0 + (p.off_wt + (threadIdx.x >> 5) * p.wt_stride) * 4;
    if constexpr (kConstPlan) {   // the host's plan must be the one compiled in
      if (D != DC || L != LC || p.off_w != kcW || p.off_frag != kcFrag || p.off_wt != kcWt || p.wt_stride != kcWtStride ||
          p.off_fk != kcFk || smem != dyn_smem_ptr())
        __trap();
    }
    if (gacc && clear_acc)
      for (int i = threadIdx.x; i < p.total; i += blockDim.x) gacc[i] = 0.f;
    if constexpr (RES) {
      w_ref = Ref{s0 + (uint32_t)p.off_w * 4u};
      frag_ref = Ref{s0 + (uint32_t)p.off_frag * 4u};
      // The blob is staged in the warps' tiles (free until the first conditioner) with one coalesced copy; everything
      // below reads the staged copy.  (Building the fragments straight from global memory was 8 dependent L2 round
      // trips per thread: 4 of the 6 us a CTA spent here, tools/step_timeline.py.)
      float* stage = smem + p.off_wt;
      const bool staged = p.total <= kWarps * p.wt_stride;
      if (staged) {
        load_weights(stage, gW, p.total);
        __syncthreads();
      }
      const float* blob = staged ? stage : gW;
      for (int i = threadIdx.x; i < Pp; i += blockDim.x) smem[p.off_w + i] = blob[i];
      // compact copy: input layer + first bias are contiguous in the blob, the other biases follow their matrices
      for (int mlp = 0; mlp < L * (D - 1); ++mlp) {
        const int layer = mlp / (D - 1), d = mlp - layer * (D - 1) + 1;
        const float* src = blob + mlp_offset<Net>(D, layer, d);
        float* dst = smem + p.off_w + cw_offset(D, M, Pp, layer, d);
        const int n0 = (d + 2) * 16;
        for (int i = threadIdx.x; i < n0 + M * 16; i += blockDim.x) {
          int so = i;
          if (i >= n0) {
            const int m = (i - n0) >> 4, j = i & 15;   // bias of dense matrix m (hidden m + 1, or the output layer)
            so = n0 + m * (H * H + H) + H * H + j;
          }
          dst[i] = src[so];
        }
      }
      // The last warp normalises the knots of the shared `first` spline (device_common.cuh: first_knots_build_warp) while
      // the other warps build the weight fragments.
      const int n_mat = L * (D - 1) * M;
      const int nb = (int)blockDim.x - 32;
      if (staged) {
        if ((int)threadIdx.x >= nb) {
          first_knots_build_warp<Net::kK>(stage, FixedSplineConsts<float, Net::kK>(),
                                          *reinterpret_cast<FirstKnots<float, Net::kK>*>(smem + p.off_fk));
        } else {
          for (int e = threadIdx.x; e < n_mat * 256; e += nb)
            reinterpret_cast<float4*>(smem + p.off_frag)[e] = frag_element<false>(stage, D, M, e);
        }
        __syncthreads();
        return;
      }
      for (int e = threadIdx.x; e < n_mat * 256; e += blockDim.x)
        reinterpret_cast<float4*>(smem + p.off_frag)[e] = frag_element<true>(gW, D, M, e);
    } else {
      load_weights(smem + p.off_w, gW, Pp);
      w_ref = Ref{gW};
      frag_ref = Ref{gfrag};
    }
    __syncthreads();
    build_first_knots<Net>(smem + p.off_w, smem + p.off_fk);
    __syncthreads();
  }
  __device__ __forceinline__ void teardown() {}

  __device__ __forceinline__ const float* first_params() const { return smem + p.off_w; }
  __device__ __forceinline__ const FirstKnots<float, Net::kK>& first_knots() const {
    if constexpr (kConstPlan) return *reinterpret_cast<const FirstKnots<float, Net::kK>*>(dyn_smem_ptr() + kcFk);
    else return *reinterpret_cast<const FirstKnots<float, Net::kK>*>(smem + p.off_fk);
  }

  // ---- register layouts of a [32 x 16] matrix (thread (g, t); mt = m-tile, nt / ks = 8-column block)
  //   C order  c[mt][nt] = { (g, 2t), (g, 2t+1), (g+8, 2t), (g+8, 2t+1) }     MMA accumulator
  //   A order  a[mt][ks] = { (g, 2t), (g+8, 2t), (g, 2t+1), (g+8, 2t+1) }     MMA A operand
  // element (row 8q+g, column 8nt+2t+e):  c[q>>1][nt][2*(q&1)+e]  =  a[q>>1][nt][(q&1)+2e]
  // Every elementwise step between two layers (ReLU, ReLU mask) writes its result in A order, so the
  // accumulator -> operand permutation costs no instruction.
  //
  // ---- per-warp tiles: element (r, col) lives at r*16 + 4*((col>>2) ^ f(r)) + (col&3),
  //      f(r) = ((r>>3)&3) ^ (2*bit1(r) + bit2(r))
  __device__ __forceinline__ static void store_c(uint32_t tile, const MmaLane& ln, const float (&x)[2][2][4]) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
        sts64(tile + ln.cbase + q * 512 + 16 * (ln.cu ^ (2 * nt ^ q)), x[q >> 1][nt][2 * (q & 1)],
              x[q >> 1][nt][2 * (q & 1) + 1]);
  }
  __device__ __forceinline__ static void store_a(uint32_t tile, const MmaLane& ln, const float (&a)[2][2][4]) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const uint32_t ad = tile + ln.cbase + q * 512 + 16 * (ln.cu ^ (2 * nt ^ q));
        sts32(ad, a[q >> 1][nt][q & 1]);
        sts32(ad + 4, a[q >> 1][nt][(q & 1) + 2]);
      }
  }
  __device__ __forceinline__ static void load_c(uint32_t tile, const MmaLane& ln, float (&x)[2][2][4]) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const float2 v = lds64(tile + ln.cbase + q * 512 + 16 * (ln.cu ^ (2 * nt ^ q)));
        x[q >> 1][nt][2 * (q & 1)] = v.x;
        x[q >> 1][nt][2 * (q & 1) + 1] = v.y;
      }
  }
  __device__ __forceinline__ static void store_row(uint32_t tile, const MmaLane& ln, const float* v) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
      sts128(tile + ln.rbase + 16 * (ln.ru ^ c), v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
  }
  __device__ __forceinline__ static void load_row(uint32_t tile, const MmaLane& ln, float* v) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float4 q = lds128(tile + ln.rbase + 16 * (ln.ru ^ c));
      v[4 * c] = q.x; v[4 * c + 1] = q.y; v[4 * c + 2] = q.z; v[4 * c + 3] = q.w;
    }
  }

  // o (C order) = a (A order) * B (+ bias): 16 -> 16 for the warp's 32 rows; frag = the matrix'
  // 512-float fragment block, bias = the 16 biases (Ref::none(): no bias)
  __device__ __forceinline__ static void dense16(const float (&a)[2][2][4], Ref frag, Ref bias,
                                                 const MmaLane& ln, float (&o)[2][2][4]) {
    float2 c0 = make_float2(0.f, 0.f), c1 = c0;
    if (bias.valid()) {
      c0 = (bias + 2 * ln.t).ld2();
      c1 = (bias + 8 + 2 * ln.t).ld2();
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      o[mt][0][0] = c0.x; o[mt][0][1] = c0.y; o[mt][0][2] = c0.x; o[mt][0][3] = c0.y;
      o[mt][1][0] = c1.x; o[mt][1][1] = c1.y; o[mt][1][2] = c1.x; o[mt][1][3] = c1.y;
    }
    const Ref fr = frag + ln.lane * 4;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      uint32_t ahi[2][4], alo[2][4];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int e = 0; e < 4; ++e) split_tf32(a[mt][ks][e], ahi[mt][e], alo[mt][e]);
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const float4 f = (fr + (ks * 2 + nt) * 128).ld4();
        const uint32_t bh0 = __float_as_uint(f.x), bh1 = __float_as_uint(f.y);
        const uint32_t bl0 = __float_as_uint(f.z), bl1 = __float_as_uint(f.w);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          mma_tf32(o[mt][nt], alo[mt], bh0, bh1);
          mma_tf32(o[mt][nt], ahi[mt], bl0, bl1);
          mma_tf32(o[mt][nt], ahi[mt], bh0, bh1);
        }
      }
    }
  }

  // a (A order) = relu(c) (C order)
  __device__ __forceinline__ static void relu_to_a(const float (&c)[2][2][4], float (&a)[2][2][4]) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        a[mt][nt][0] = fmaxf(c[mt][nt][0], 0.f);
        a[mt][nt][1] = fmaxf(c[mt][nt][2], 0.f);
        a[mt][nt][2] = fmaxf(c[mt][nt][1], 0.f);
        a[mt][nt][3] = fmaxf(c[mt][nt][3], 0.f);
      }
  }

  // Conditioner forward for the warp's 32 rows: theta[0..16) of the calling thread's row.
  // keep: store the hidden activations in the warp's tiles for cond_backward.
  // put: also leave them in the activation stash for cond_restore (the caller adds the located spline: stash_state).
  __device__ __forceinline__ void cond_forward(int D, int layer, int d, float tval, const float* cvec,
                                               float* theta, bool keep, bool put = false) const {
    const int sc = stash_cond(D, layer, d);
    const MmaLane ln;
    const uint32_t wt = swt();
    const int n_in = d + 1, mlp = layer * (D - 1) + d - 1;
    const Ref W = wref() + (RES ? cw_offset(D, M, Pp, layer, d) : mlp_offset<Net>(D, layer, d));
    const Ref b0 = W + n_in * H;
    const Ref frag = fref() + mlp * M * kFragFloats;
    float x[2][2][4], a[2][2][4];
    {
      const float2 c0 = (b0 + 2 * ln.t).ld2();
      const float2 c1 = (b0 + 8 + 2 * ln.t).ld2();
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        x[mt][0][0] = c0.x; x[mt][0][1] = c0.y; x[mt][0][2] = c0.x; x[mt][0][3] = c0.y;
        x[mt][1][0] = c1.x; x[mt][1][1] = c1.y; x[mt][1][2] = c1.x; x[mt][1][3] = c1.y;
      }
    }
    // layer 0 on the CUDA cores (n_in is 2..D): inputs come from the row owners in the quad
#pragma unroll 1
    for (int i = 0; i < n_in; ++i) {
      const float xi = i == 0 ? tval : cvec[perm_at(layer, i - 1, D)];
      const float2 w0 = (W + i * 16 + 2 * ln.t).ld2();
      const float2 w1 = (W + i * 16 + 8 + 2 * ln.t).ld2();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float xq = __shfl_sync(0xffffffffu, xi, (ln.lane & ~3u) | q);
        float* a0 = x[q >> 1][0] + 2 * (q & 1);
        float* a1 = x[q >> 1][1] + 2 * (q & 1);
        a0[0] = fmaf(xq, w0.x, a0[0]); a0[1] = fmaf(xq, w0.y, a0[1]);
        a1[0] = fmaf(xq, w1.x, a1[0]); a1[1] = fmaf(xq, w1.y, a1[1]);
      }
    }
    relu_to_a(x, a);
    if (keep) {
      __syncwarp();   // the previous conditioner's readers are done with the tiles
      store_a(wt, ln, a);
    }
    if (STASH && put) tmem_st16(stash_hidden(sc, 0), &a[0][0][0]);
    // bias of dense matrix m: compact copy = right after b0; blob = after its matrix
    Ref bm = RES ? b0 + H : b0 + (H + H * H);
#pragma unroll
    for (int m = 1; m < M; ++m) {
      dense16(a, frag + (m - 1) * kFragFloats, bm, ln, x);
      relu_to_a(x, a);
      if (keep) store_a(wt + m * kWtFloats * 4, ln, a);
      if (STASH && put) tmem_st16(stash_hidden(sc, m), &a[0][0][0]);
      bm = bm + (RES ? H : H * H + H);
    }
    dense16(a, frag + (M - 1) * kFragFloats, bm, ln, x);
    const uint32_t scratch = wt + (keep ? M : 0) * kWtFloats * 4;
    __syncwarp();
    store_c(scratch, ln, x);
    __syncwarp();
    load_row(scratch, ln, theta);
  }

  // What cond_forward(keep = true) + rqs_locate_raw leave behind -- hidden activations in the warp's tiles, the located
  // spline of the calling thread's row -- read back from the activation stash the forward pass of the same rows filled
  // (cond_forward(put = true), stash_state).  One 16-column load per tile goes straight into the tile, so only 16 (20
  // for the spline) of the values are in registers at a time.
  __device__ __forceinline__ void cond_restore(int D, int layer, int d, SplineState<float, Net::kK>& st, float min_slope) const {
    if constexpr (STASH) {
      constexpr int K = Net::kK;
      const MmaLane ln;
      const uint32_t wt = swt();
      const int c = stash_cond(D, layer, d), nc = stash_ncond();
      __syncwarp();   // the previous conditioner's readers are done with the tiles; the warp is converged for .aligned
      // the stores of the forward pass have completed (they were issued a whole pass ago: this does not wait)
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  #pragma unroll
      for (int m = 0; m < M; ++m) {
        float a[2][2][4];
        tmem_ld16(stash_hidden(c, m), &a[0][0][0]);
        store_a(wt + m * kWtFloats * 4, ln, a);
      }
      float b[kStateFloats];
      tmem_ld16_4(stash_t + 16 * (nc * M + c), stash_t + 16 * nc * (M + 1) + 4 * c, b);
  #pragma unroll
      for (int k = 0; k < K; ++k) { st.pw[k] = b[k]; st.ph[k] = b[K + k]; }
      st.x0 = b[2 * K]; st.x1 = b[2 * K + 1]; st.y0 = b[2 * K + 2]; st.y1 = b[2 * K + 3];
      st.d0 = b[2 * K + 4]; st.d1 = b[2 * K + 5]; st.u0 = b[2 * K + 6]; st.u1 = b[2 * K + 7];
      st.u_tail = b[2 * K + 8];
      const int it = __float_as_int(b[2 * K + 9]);
      st.idx = it & 0xff;
      st.tail = it >> 8;
      st.s_tail = st.d0;
      if (st.tail == 2) st.s_tail = softplus(st.u_tail) + min_slope;
    }
  }

  // 4 per-thread partial sums (columns 2t, 2t+1, 8+2t, 9+2t of a 16-wide row) -> summed over the
  // 8 lanes with the same t, then added to dst[column]
  __device__ __forceinline__ static void colsum_add(const float (&v)[4], float* dst, const MmaLane& ln) {
    const bool hi = ln.lane & 16, b8 = ln.lane & 8;
    float k0 = hi ? v[2] : v[0], k1 = hi ? v[3] : v[1];
    const float s0 = hi ? v[0] : v[2], s1 = hi ? v[1] : v[3];
    k0 += __shfl_xor_sync(0xffffffffu, s0, 16);
    k1 += __shfl_xor_sync(0xffffffffu, s1, 16);
    float kk = b8 ? k1 : k0;
    const float ss = b8 ? k0 : k1;
    kk += __shfl_xor_sync(0xffffffffu, ss, 8);
    kk += __shfl_xor_sync(0xffffffffu, kk, 4);
    if (!(ln.lane & 4)) red_global(dst + (hi ? 8 : 0) + 2 * ln.t + (b8 ? 1 : 0), kk);
  }
  // column sums of an A-order matrix
  __device__ __forceinline__ static void colsum_a(const float (&a)[2][2][4], float* dst, const MmaLane& ln) {
    float s[4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      s[2 * nt] = (a[0][nt][0] + a[0][nt][1]) + (a[1][nt][0] + a[1][nt][1]);
      s[2 * nt + 1] = (a[0][nt][2] + a[0][nt][3]) + (a[1][nt][2] + a[1][nt][3]);
    }
    colsum_add(s, dst, ln);
  }

  // dst[i][j] += sum_r A[r][i] G[r][j] over the warp's 32 rows (A, G: swizzled tiles)
  __device__ __forceinline__ static void wgrad16(uint32_t TA, uint32_t TG, float* dst, const MmaLane& ln) {
    float dw[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) dw[nt][e] = 0.f;
    const uint32_t ta = TA + ln.tbase, tg = TG + ln.tbase;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      // rows 8ks+t (chunk selector tu^ks) and 8ks+t+4 (selector tu^ks^1)
      float av[4];
      av[0] = lds32(ta + ks * 512 + 16 * (ln.tu ^ ks));              // (m = g,   k = t)
      av[1] = lds32(ta + ks * 512 + 16 * (ln.tu ^ ks ^ 2));          // (m = g+8, k = t)
      av[2] = lds32(ta + ks * 512 + 256 + 16 * (ln.tu ^ ks ^ 1));    // (m = g,   k = t+4)
      av[3] = lds32(ta + ks * 512 + 256 + 16 * (ln.tu ^ ks ^ 3));    // (m = g+8, k = t+4)
      uint32_t ahi[4], alo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) split_tf32(av[e], ahi[e], alo[e]);
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const float b0 = lds32(tg + ks * 512 + 16 * (ln.tu ^ ks ^ (2 * nt)));            // (k = t,   n = g)
        const float b1 = lds32(tg + ks * 512 + 256 + 16 * (ln.tu ^ ks ^ (2 * nt) ^ 1));  // (k = t+4, n = g)
        uint32_t bh0, bh1, bl0, bl1;
        split_tf32(b0, bh0, bl0);
        split_tf32(b1, bh1, bl1);
        mma_tf32(dw[nt], alo, bh0, bh1);
        mma_tf32(dw[nt], ahi, bl0, bl1);
        mma_tf32(dw[nt], ahi, bh0, bh1);
      }
    }
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      float* q0 = dst + ln.g * 16 + 8 * nt + 2 * ln.t;
      red_global2(q0, dw[nt][0], dw[nt][1]);
      red_global2(q0 + 128, dw[nt][2], dw[nt][3]);
    }
  }

  // Conditioner backward for the warp's 32 rows.  cond_forward(..., keep = true) of the same
  // conditioner must have run just before.  gtheta: adjoint of the row's spline parameters;
  // gvec[coordinate] += adjoint of the conditioning coordinates; weight gradients -> gacc.
  __device__ __forceinline__ void cond_backward(int D, int layer, int d, float tval, const float* cvec,
                                                const float* gtheta, float* gvec) const {
    const MmaLane ln;
    const uint32_t wt = swt();
    const int n_in = d + 1, mlp = layer * (D - 1) + d - 1;
    const int w_off = mlp_offset<Net>(D, layer, d);
    const Ref W = wref() + (RES ? cw_offset(D, M, Pp, layer, d) : w_off);
    float* A = gacc + w_off;
    const Ref frag = fref() + (mlp * M * kFragFloats + 512);
    const uint32_t tg = wt + M * kWtFloats * 4;
    __syncwarp();
    store_row(tg, ln, gtheta);
    __syncwarp();
    float G[2][2][4];   // A order
    {
      float c[2][2][4];
      load_c(tg, ln, c);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          G[mt][nt][0] = c[mt][nt][0]; G[mt][nt][1] = c[mt][nt][2];
          G[mt][nt][2] = c[mt][nt][1]; G[mt][nt][3] = c[mt][nt][3];
        }
    }
#pragma unroll
    for (int slot = M - 1; slot >= 0; --slot) {
      // dense matrix `slot`: input = hidden activations `slot`, output adjoint = G
      const int moff = n_in * H + H + slot * (H * H + H);
      wgrad16(wt + slot * kWtFloats * 4, tg, A + moff, ln);
      colsum_a(G, A + moff + H * 16, ln);
      float dh[2][2][4], hm[2][2][4];
      dense16(G, frag + slot * kFragFloats, Ref::none(), ln, dh);
      load_c(wt + slot * kWtFloats * 4, ln, hm);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          G[mt][nt][0] = hm[mt][nt][0] > 0.f ? dh[mt][nt][0] : 0.f;
          G[mt][nt][1] = hm[mt][nt][2] > 0.f ? dh[mt][nt][2] : 0.f;
          G[mt][nt][2] = hm[mt][nt][1] > 0.f ? dh[mt][nt][1] : 0.f;
          G[mt][nt][3] = hm[mt][nt][3] > 0.f ? dh[mt][nt][3] : 0.f;
        }
      if (slot > 0) {
        __syncwarp();
        store_a(tg, ln, G);
        __syncwarp();
      }
    }
    // layer 0: bias, input matrix, input adjoints
    colsum_a(G, A + n_in * H, ln);
#pragma unroll 1
    for (int i = 0; i < n_in; ++i) {
      const float xi = i == 0 ? tval : cvec[perm_at(layer, i - 1, D)];
      const float2 w0 = (W + i * 16 + 2 * ln.t).ld2();
      const float2 w1 = (W + i * 16 + 8 + 2 * ln.t).ld2();
      float pw[4] = {0.f, 0.f, 0.f, 0.f}, pin[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float xq = __shfl_sync(0xffffffffu, xi, (ln.lane & ~3u) | q);
        // row 8q+g: columns 2t, 2t+1 (nt = 0) and 8+2t, 9+2t (nt = 1)
        const float g00 = G[q >> 1][0][q & 1], g01 = G[q >> 1][0][(q & 1) + 2];
        const float g10 = G[q >> 1][1][q & 1], g11 = G[q >> 1][1][(q & 1) + 2];
        pw[0] = fmaf(xq, g00, pw[0]); pw[1] = fmaf(xq, g01, pw[1]);
        pw[2] = fmaf(xq, g10, pw[2]); pw[3] = fmaf(xq, g11, pw[3]);
        pin[q] = g00 * w0.x + g01 * w0.y + g10 * w1.x + g11 * w1.y;
      }
      colsum_add(pw, A + i * 16, ln);
      if (i >= 1) {
        // sum over the quad; lane t ends up with the total of row 8t+g (its own row)
        const bool t2 = ln.lane & 2, t1 = ln.lane & 1;
        float k0 = t2 ? pin[2] : pin[0], k1 = t2 ? pin[3] : pin[1];
        const float s0 = t2 ? pin[0] : pin[2], s1 = t2 ? pin[1] : pin[3];
        k0 += __shfl_xor_sync(0xffffffffu, s0, 2);
        k1 += __shfl_xor_sync(0xffffffffu, s1, 2);
        float kk = t1 ? k1 : k0;
        const float ss = t1 ? k0 : k1;
        kk += __shfl_xor_sync(0xffffffffu, ss, 1);
        gvec[perm_at(layer, i - 1, D)] += kk;
      }
    }
  }

  // flush the per-thread adjoint of the shared `first` parameter (blob offset 0)
  __device__ __forceinline__ void flush_first(const float* gfirst, const RowTiles<float, Net>&) const {
    const uint32_t lane = threadIdx.x & 31;
#pragma unroll
    for (int j = 0; j < Pp; ++j) {
      float v = gfirst[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red_global(gacc + j, v);
    }
    __syncthreads();
  }
};

}  // namespace cnfot
