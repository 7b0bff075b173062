// C ABI of libcnfot.so (declared in include/cnfot.h): argument checking, kernel
// selection, launch configuration, workspace carving.  No torch types, no
// allocation, no stream synchronisation (except the *_host convenience entry).
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/cnfot.h"
#include "device_common.cuh"
#include "dense_tc.h"
#include "dispatch.h"
#include "flow_kernels.cuh"
#include "step_host.h"
#include "wide.h"

namespace cnfot {

// rqs_kernels.cu
cudaError_t rqs_eval_dispatch(int K, bool inverse, cudaStream_t s, const float* v,
                              const float* params, int64_t rows, const SplineConsts<float>& sc,
                              float* out, float* ld, int32_t* bin, int num_sms, bool* known);
cudaError_t rqs_vjp_dispatch(int K, bool inverse, cudaStream_t s, const float* v,
                             const float* params, const float* go, const float* gl, int64_t rows,
                             const SplineConsts<float>& sc, float* gi, float* gp, int num_sms,
                             bool* known);

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

static int cuda_fail(cudaError_t e, const char* what) {
  return fail(CNFOT_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

struct DeviceInfo {
  int device = -1;
  int num_sms = 0;
  int max_smem_optin = 0;
};

// Properties of the current device (cached per device id).
static int device_info(DeviceInfo* out) {
  static DeviceInfo cache[64];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice (no CUDA device? libcnfot has no CPU path)");
  if (dev < 0 || dev >= 64) return fail(CNFOT_ERR_CUDA, "device id %d out of range", dev);
  if (cache[dev].device != dev) {
    DeviceInfo d;
    d.device = dev;
    e = cudaDeviceGetAttribute(&d.num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
    e = cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
    cache[dev] = d;
  }
  *out = cache[dev];
  return 0;
}

constexpr int kMaxGrid = 148 * 8;   // upper bound on persistent CTAs (workspace sizing)
constexpr int64_t kCounterBytes = 256;

static int check_flow(const cnfot_flow_desc* f, FlowLayout* lay) {
  if (!f) return fail(CNFOT_ERR_ARG, "flow descriptor is NULL");
  if (f->dim < 1 || f->num_layers < 1 || f->mlp_layers < 1 || f->hidden < 1 || f->num_bins < 1)
    return fail(CNFOT_ERR_ARG, "flow descriptor has non-positive sizes");
  if (f->hidden % 4 != 0) return fail(CNFOT_ERR_ARG, "hidden size %d must be a multiple of 4", f->hidden);
  if (!(f->range_max > f->range_min) || f->num_bins * f->min_bin_size > f->range_max - f->range_min)
    return fail(CNFOT_ERR_ARG, "min_bin_size too large for the spline range");
  if (!(f->min_knot_slope < 1.f)) return fail(CNFOT_ERR_ARG, "min_knot_slope must be < 1");
  *lay = make_layout(f->dim, f->num_layers, f->mlp_layers, f->hidden, f->num_bins);
  return 0;
}

// The fused kernels hold the reference's spline constants (flows.py:124-132) as immediates.
static bool reference_spline_consts(const cnfot_flow_desc* f) {
  const SplineConsts<float> c = make_spline_consts<float>(f->num_bins, f->range_min, f->range_max, f->min_bin_size,
                                                          f->min_knot_slope);
  return c.lo == -10.f && c.hi == 10.f && c.min_bin == 1e-4f && c.min_slope == 1e-4f &&
         fabsf(c.slope_offset - 0.5411666523385311f) <= 1e-7f;
}

static int check_fused(const cnfot_flow_desc* f, const FlowLayout& lay) {
  if (!reference_spline_consts(f))
    return fail(CNFOT_ERR_ARG, "the fused flow kernels are compiled for the reference's spline constants (range -10..10, "
                               "min_bin_size = min_knot_slope = 1e-4; cnf_ot/models/flows.py:124-132)");
  if (f->dim > kMaxDim) return fail(CNFOT_ERR_ARG, "fused kernels support dim <= %d (got %d)", kMaxDim, f->dim);
  if ((f->num_layers + 1) * f->dim > kMaxStateFloats)
    return fail(CNFOT_ERR_ARG, "fused kernels need (num_layers+1)*dim <= %d (got %d)", kMaxStateFloats,
                (f->num_layers + 1) * f->dim);
  if (!find_flow_eval_kernel(lay))
    return fail(CNFOT_ERR_ARG,
                "no fused kernel instantiated for hidden=%d num_bins=%d mlp_layers=%d "
                "(see CNFOT_NET_LIST in cnf_ot_b200/csrc/dispatch.h)",
                f->hidden, f->num_bins, f->mlp_layers);
  return 0;
}

// shapes the fused per-row kernels cover (no error message: callers fall through to the wide engine)
static bool fused_ok(const cnfot_flow_desc* f, const FlowLayout& lay) {
  if (!(f->dim <= kMaxDim && (f->num_layers + 1) * f->dim <= kMaxStateFloats && find_flow_eval_kernel(lay) != nullptr))
    return false;
  if (!reference_spline_consts(f)) return false;
  if (tc_available(lay)) return true;   // 16-wide networks: the warp-MMA plans stream what does not fit
  // CUDA-core engine: even the staged plan (one conditioner at a time in shared memory) must fit a CTA
  DeviceInfo di;
  if (device_info(&di)) return true;    // no device: let the launch path report it
  return (int64_t)plan_smem(lay, true, false).floats * 4 <= di.max_smem_optin;
}
// the wide-conditioner engine (wide.cu) takes every shape the fused kernels do not, when it can
// (CNFOT_ENGINE=wide forces it for shapes both cover: used by the cross-engine parity tests)
static bool use_wide(const cnfot_flow_desc* f, const FlowLayout& lay) {
  if (!wide_supported(lay, nullptr)) return false;
  if (!fused_ok(f, lay)) return true;
  const char* e = getenv("CNFOT_ENGINE");
  return e && !strcmp(e, "wide");
}

static SplineConsts<float> spline_consts(const cnfot_flow_desc* f) {
  return make_spline_consts<float>(f->num_bins, f->range_min, f->range_max, f->min_bin_size,
                                   f->min_knot_slope);
}

struct LaunchCfg {
  int grid;
  size_t smem;
};
static thread_local int g_last_launch[4] = {0, 0, 0, 0};
// cnfot_last_launch_variant: {plan, stash TMEM columns, kinetic lane group, latency instantiation} of the most recent
// fused call.  The step and VJP entries reset it on entry and fill it in once their kernel is chosen; every other fused
// launch resets it (configure(), the wide-engine evaluation, energy and density paths).  Plan -1: not a step or VJP.
static thread_local int g_last_variant[4] = {-1, 0, 0, 0};
static void record_variant(int plan, int stash_cols, int kinetic_group, bool latency) {
  g_last_variant[0] = plan; g_last_variant[1] = stash_cols; g_last_variant[2] = kinetic_group;
  g_last_variant[3] = latency ? 1 : 0;
}

// Shared-memory plan and engine choice.
//   warp-MMA engine (warp_mlp.cuh)  16-wide networks: the default there.  Weights + hi/lo fragments resident
//                                   in shared memory when that leaves room for >= 2 CTAs per SM, otherwise
//                                   streamed from global memory (fragments built into the workspace)
//   CUDA-core engine                everything else; weights live in shared memory when weights +
//                                   accumulators + row tiles leave room for two CTAs per SM, otherwise
//                                   one conditioner at a time is staged from L2
//   tcgen05 engine (tc_engine.cuh)  16-wide networks, opt-in: its per-layer issue / commit / wait round
//                                   trips make it slower than both at hidden = 16 (DESIGN.md section 4.4)
// CNFOT_ENGINE=cuda|tc|mma in the environment overrides the choice (read on every call).
static int engine_override() {
  const char* e = getenv("CNFOT_ENGINE");
  if (!e) {
    const char* t = getenv("CNFOT_TC");
    return (t && t[0] == '1') ? kEngTc : -1;
  }
  if (!strcmp(e, "cuda")) return kEngCuda;
  if (!strcmp(e, "tc")) return kEngTc;
  if (!strcmp(e, "mma")) return kEngMma;
  return -1;
}

static int make_plan(const FlowLayout& lay, bool with_grad, SmemPlan* sp, int* engine, bool has_ws = true) {
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  const int want = engine_override();
  *engine = kEngCuda;
  if (want == kEngTc && tc_available(lay)) {
    SmemPlan t = plan_smem(lay, with_grad, true, true);
    if ((int64_t)t.floats * 4 * 2 <= di.max_smem_optin) {
      *sp = t;
      *engine = kEngTc;
      return 0;
    }
  }
  if ((want == kEngMma || want < 0) && tc_available(lay)) {
    SmemPlan m = plan_smem_mma(lay, with_grad);
    if ((int64_t)m.floats * 4 * 2 <= di.max_smem_optin) {
      *sp = m;
      *engine = kEngMma;
      return 0;
    }
    // larger flows: fragments in the caller's workspace (entry points that have one)
    if (has_ws) {
      *sp = plan_smem_mma(lay, with_grad, false);
      *engine = kEngMmaStream;
      return 0;
    }
  }
  SmemPlan p = plan_smem(lay, with_grad, true);
  if ((int64_t)p.floats * 4 * 2 > di.max_smem_optin) p = plan_smem(lay, with_grad, false);
  *sp = p;
  return 0;
}

// Persistent launch: as many CTAs as fit on the chip, capped by the tile count.
// tmem_cols: TMEM columns a CTA of this launch allocates (the tcgen05 engine: kTcTmemCols; the step and VJP kernels
// with the activation stash: stash_tmem_cols), 0 for kernels without tcgen05.alloc.
static int configure(const void* kernel, const SmemPlan& sp, int64_t tiles, LaunchCfg* cfg, int tmem_cols = 0) {
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  size_t smem = (size_t)sp.floats * sizeof(float);
  if ((int64_t)smem > di.max_smem_optin)
    return fail(CNFOT_ERR_ARG, "network too large for the fused kernels: needs %zu B of shared memory, device allows %d",
                smem, di.max_smem_optin);
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute");
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kTile, smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
  if (sp.off_wmma >= 0) tmem_cols = kTcTmemCols;
  if (tmem_cols > 0) {
    // The occupancy query answers 1 for any kernel that contains tcgen05.alloc (it cannot know how
    // many of the 512 TMEM columns a CTA takes).  Size the persistent grid from the real limits
    // instead: shared memory, registers and TMEM columns.
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, kernel);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncGetAttributes");
    int smem_sm = 0, regs_sm = 0;
    cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, di.device);
    cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, di.device);
    int by_smem = (int)(smem_sm / (smem + fa.sharedSizeBytes + 1024));
    int by_regs = regs_sm / (fa.numRegs * kTile > 0 ? fa.numRegs * kTile : 1);
    int by_tmem = 512 / tmem_cols;
    occ = by_smem < by_regs ? by_smem : by_regs;
    if (occ > by_tmem) occ = by_tmem;
  }
  if (getenv("CNFOT_DEBUG")) {
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, kernel);
    int o0 = 0, o1 = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o0, kernel, kTile, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o1, kernel, kTile, 60000);
    fprintf(stderr, "[cnfot] occ=%d (smem %zu) occ@0=%d occ@60000=%d regs=%d static_smem=%zu local=%zu maxdyn=%d carveout=%d\n",
            occ, smem, o0, o1, fa.numRegs, fa.sharedSizeBytes, fa.localSizeBytes, fa.maxDynamicSharedSizeBytes,
            fa.preferredShmemCarveout);
  }
  if (occ < 1) return fail(CNFOT_ERR_CUDA, "kernel does not fit on an SM");
  int64_t cap = (int64_t)di.num_sms * occ;
  if (cap > kMaxGrid) cap = kMaxGrid;
  int64_t g = tiles < cap ? tiles : cap;
  cfg->grid = (int)(g > 0 ? g : 1);
  cfg->smem = smem;
  g_last_launch[0] = cfg->grid;
  g_last_launch[1] = (int)smem;
  g_last_launch[2] = occ;
  g_last_launch[3] = sp.off_wmma >= 0 ? kEngTc : (sp.off_frag >= 0 ? kEngMma : kEngCuda);  // 2 also for the streamed plan
  record_variant(-1, 0, 0, false);
  return 0;
}

static int64_t frag_bytes(const FlowLayout& lay) {
  if (!tc_available(lay)) return 0;
  return (int64_t)lay.L * (lay.D - 1) * lay.M * kFragFloats * sizeof(float);
}
// [tile counter | per-CTA loss partials | per-CTA gradient partials | weight fragments (streamed warp-MMA plan)]
static int64_t partial_bytes(const FlowLayout& lay) {
  int64_t loss = (int64_t)kMaxGrid * kNumSlots * sizeof(double);
  int64_t grad = ((int64_t)kMaxGrid * lay.total * sizeof(float) + 255) / 256 * 256;
  return kCounterBytes + loss + grad + frag_bytes(lay);
}
// TMEM columns per CTA of the activation stash of the warp-MMA step and VJP kernels (warp_mlp.cuh: DeviceCtxMma): per
// thread and conditioner, M tiles of 16 hidden activations + the located spline (2 K + 10 floats), rounded up to the
// power of two tcgen05.alloc takes.  0 (recompute in the backward pass): other engines, flows over 128 columns (four
// CTAs per SM share an SM's 512; such flows are also the only ones on the streamed plan), or CNFOT_STEP_STASH=0.
// Non-zero selects the kernel instantiation with the stash (kEngMmaStash).
static int stash_tmem_cols(const FlowLayout& lay, int engine) {
  if (engine != kEngMma) return 0;
  const int per_thread = lay.L * (lay.D - 1) * (16 * lay.M + 2 * lay.K + 10);
  if (per_thread > 128) return 0;
  if (const char* e = getenv("CNFOT_STEP_STASH")) {   // tuning knob: 0 = always recompute
    if (e[0] == '0') return 0;
  }
  int cols = 32;
  while (cols < per_thread) cols <<= 1;
  return cols;
}
static float* carve_frags(void* ws, const FlowLayout& lay) {
  return (float*)((char*)ws + partial_bytes(lay) - frag_bytes(lay));
}
// streamed warp-MMA plan: fill the fragment buffer (stream-ordered before the main kernel)
static int launch_build_frags(cudaStream_t s, const FlowLayout& lay, const float* weights, float* frags) {
  const int n_mat = lay.L * (lay.D - 1) * lay.M;
  const int blocks = (n_mat * 256 + 255) / 256;
  build_frags_kernel<<<blocks < 1184 ? blocks : 1184, 256, 0, s>>>(weights, frags, lay.D, lay.M, n_mat);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "build_frags_kernel launch");
  return 0;
}

static PartialBuf carve_partials(void* ws, unsigned long long** counter) {
  char* p = (char*)ws;
  *counter = (unsigned long long*)p;
  PartialBuf pb;
  pb.loss = (double*)(p + kCounterBytes);
  pb.grad = (float*)(p + kCounterBytes + (int64_t)kMaxGrid * kNumSlots * sizeof(double));
  return pb;
}

// ---- finalize: sum per-CTA partials (double) into the output buffer ------------------
// out = [ grad (total) | loss slots: 0 total, 1 fit(0), 2 fit(T), 3 potential, 4 kinetic ]
// One block reduces 32 consecutive parameters: warp w sums partials w, w+8, ... (coalesced
// 128-byte reads), the 8 warps are folded through shared memory.  Fixed order => the
// result is bit-reproducible for a given grid size.
constexpr int kFinWarps = 32;  // 1024 threads: the per-CTA partials are read with many loads in flight
// sum over the CTAs c = warp, warp + kFinWarps, ... of pgrad[c][i], four independent loads in flight
__device__ __forceinline__ double column_partial(const float* __restrict__ pgrad, int n_cta, int total, int i,
                                                 int warp) {
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int c = warp;
  for (; c + 3 * kFinWarps < n_cta; c += 4 * kFinWarps) {
    const float v0 = __ldcg(pgrad + (int64_t)c * total + i);
    const float v1 = __ldcg(pgrad + (int64_t)(c + kFinWarps) * total + i);
    const float v2 = __ldcg(pgrad + (int64_t)(c + 2 * kFinWarps) * total + i);
    const float v3 = __ldcg(pgrad + (int64_t)(c + 3 * kFinWarps) * total + i);
    a0 += (double)v0; a1 += (double)v1; a2 += (double)v2; a3 += (double)v3;
  }
  for (; c < n_cta; c += kFinWarps) a0 += (double)__ldcg(pgrad + (int64_t)c * total + i);
  return (a0 + a1) + (a2 + a3);
}

__global__ void __launch_bounds__(32 * kFinWarps)
finalize_kernel(const float* __restrict__ pgrad, const double* __restrict__ ploss, int n_cta,
                int total, float* __restrict__ out_grad, float* __restrict__ out_slots,
                int accumulate) {
  __shared__ double part[kFinWarps][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  double acc = 0.0;
  if (i < total) acc = column_partial(pgrad, n_cta, total, i, warp);
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && i < total) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kFinWarps; ++w) t += part[w][lane];
    out_grad[i] = accumulate ? out_grad[i] + (float)t : (float)t;
  }
  if (out_slots && blockIdx.x == gridDim.x - 1) {
    // loss slots (the last block: it has the fewest gradient columns): 4 CTAs x 8 slots per warp pass
    __syncthreads();
    const int sl = lane & 7, sub = lane >> 3;
    double v = 0.0;
    for (int c = warp * 4 + sub; c < n_cta; c += 4 * kFinWarps) v += ploss[(int64_t)c * kNumSlots + sl];
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    part[warp][lane] = v;
    __syncthreads();
    if (warp == 0) {
      // lanes 0..7 <-> internal slots (fit0, fitT, potential, kinetic, unused...)
      double t = 0.0;
      if (lane < kNumSlots)
        for (int w = 0; w < kFinWarps; ++w) t += part[w][lane];
      double tot = t;
      tot += __shfl_xor_sync(0xffffffffu, tot, 1);
      tot += __shfl_xor_sync(0xffffffffu, tot, 2);  // lanes 0..3 now hold the sum of slots 0..3
      if (lane == 0) out_slots[0] = accumulate ? out_slots[0] + (float)tot : (float)tot;
      if (lane < 4) out_slots[1 + lane] = accumulate ? out_slots[1 + lane] + (float)t : (float)t;
      if (lane >= 5 && lane < kNumSlots) out_slots[lane] = 0.f;
    }
  }
}

static int launch_finalize(cudaStream_t s, const PartialBuf& pb, int n_cta, int total, float* out_grad,
                           float* out_slots, bool accumulate = false) {
  int blocks = (total + 31) / 32;
  finalize_kernel<<<blocks, 32 * kFinWarps, 0, s>>>(pb.grad, pb.loss, n_cta, total, out_grad, out_slots,
                                                   accumulate ? 1 : 0);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "finalize_kernel launch");
  return 0;
}

// ---- energy finalize: sum the CTAs' kinetic partials into one double ----------------------
__global__ void energy_finalize_kernel(const double* __restrict__ ploss, int n_cta, double* __restrict__ out) {
  double v = 0.0;
  for (int c = threadIdx.x; c < n_cta; c += 32) v += ploss[(int64_t)c * kNumSlots + kSlotKinetic];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (threadIdx.x == 0) out[0] = v;
}

// ---- Adam ----------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps,
                            float c1, float c2) {
  // optax.scale_by_adam + scale(-lr): m_hat = m / (1 - b1^t), v_hat = v / (1 - b2^t),
  // update = -lr * m_hat / (sqrt(v_hat) + eps)
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i];
    float mi = b1 * m[i] + (1.f - b1) * gi;
    float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= lr * (mi / c1) / (sqrtf(vi / c2) + eps);
  }
}

// ---- dimension-reduction loss head (cnf_ot/dr/trainers.py:91-111) -------------------------------------------
// loss += weight * sum (x - xr)^2 ; g_xr = -2 weight (x - xr)
__global__ void __launch_bounds__(256)
recon_head_kernel(const float* __restrict__ x, const float* __restrict__ xr, int64_t count, float weight,
                  float* __restrict__ g_xr, double* __restrict__ loss) {
  double acc = 0.0;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
    const float dlt = x[e] - xr[e];
    acc += (double)dlt * (double)dlt;
    g_xr[e] = -2.f * weight * dlt;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc != 0.0) atomicAdd(loss, acc * (double)weight);
}
// y[:, sub_dim:] = 0
__global__ void __launch_bounds__(256)
mask_tail_kernel(float* __restrict__ y, int64_t rows, int dim, int sub_dim) {
  const int64_t count = rows * dim;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
    if ((int)(e % dim) >= sub_dim) y[e] = 0.f;
}

}  // namespace cnfot

using namespace cnfot;

extern "C" {

int cnfot_abi_version(void) { return CNFOT_ABI_VERSION; }
static unsigned long long* g_step_timeline = nullptr;
void cnfot_debug_step_timeline(void* device_words) { g_step_timeline = (unsigned long long*)device_words; }

void cnfot_last_launch_info(int32_t* grid, int32_t* smem_bytes, int32_t* ctas_per_sm, int32_t* tensor_cores) {
  if (grid) *grid = g_last_launch[0];
  if (smem_bytes) *smem_bytes = g_last_launch[1];
  if (ctas_per_sm) *ctas_per_sm = g_last_launch[2];
  if (tensor_cores) *tensor_cores = g_last_launch[3];
}
void cnfot_last_launch_variant(int32_t* plan, int32_t* stash_tmem_cols, int32_t* kinetic_group, int32_t* latency) {
  if (plan) *plan = g_last_variant[0];
  if (stash_tmem_cols) *stash_tmem_cols = g_last_variant[1];
  if (kinetic_group) *kinetic_group = g_last_variant[2];
  if (latency) *latency = g_last_variant[3];
}
const char* cnfot_last_error(void) { return g_err; }

int64_t cnfot_param_count(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  return lay.total;
}

int64_t cnfot_spline_param_stride(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  return lay.Pp;
}

int64_t cnfot_offset_first(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  return 0;
}

int64_t cnfot_offset_linear(const cnfot_flow_desc* flow, int32_t layer, int32_t d, int32_t m, int32_t bias) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  if (layer < 0 || layer >= lay.L || d < 1 || d >= lay.D || m < 0 || m > lay.M) {
    fail(CNFOT_ERR_ARG, "offset_linear: index out of range");
    return -1;
  }
  const int H = lay.H;
  int64_t off = lay.Pp + (int64_t)layer * lay.layer_stride + (int64_t)(d - 1) * lay.mlp_const +
                (int64_t)H * ((d - 1) * (d + 2) / 2);
  const int n_in = d + 1;
  if (m == 0) return off + (bias ? n_in * H : 0);
  off += n_in * H + H + (int64_t)(m - 1) * (H * H + H);
  if (m < lay.M) return off + (bias ? H * H : 0);
  return off + (bias ? H * lay.Pp : 0);
}

int cnfot_flow_supported(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (use_wide(flow, lay)) return 0;
  return check_fused(flow, lay);
}

// ---- seam 2 ---------------------------------------------------------------------------
static int rqs_call(bool inverse, void* stream, const float* v, const float* params, int64_t rows,
                    int32_t K, float lo, float hi, float min_bin, float min_slope, float* out,
                    float* ld, int32_t* bin) {
  if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
  if (rows == 0) return 0;
  if (!v || !params || !out || !ld) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (K < 1 || !(hi > lo) || K * min_bin > hi - lo || !(min_slope < 1.f))
    return fail(CNFOT_ERR_ARG, "bad spline constants");
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  bool known = false;
  cudaError_t e = rqs_eval_dispatch(K, inverse, (cudaStream_t)stream, v, params, rows,
                                    make_spline_consts<float>(K, lo, hi, min_bin, min_slope), out, ld,
                                    bin, di.num_sms, &known);
  if (!known) return fail(CNFOT_ERR_ARG, "num_bins=%d not instantiated (see CNFOT_BINS_LIST)", K);
  if (e != cudaSuccess) return cuda_fail(e, "rqs kernel launch");
  return 0;
}

static int rqs_vjp_call(bool inverse, void* stream, const float* v, const float* params,
                        const float* go, const float* gl, int64_t rows, int32_t K, float lo, float hi,
                        float min_bin, float min_slope, float* gi, float* gp) {
  if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
  if (rows == 0) return 0;
  if (!v || !params || !go || !gl || !gi || !gp) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (K < 1 || !(hi > lo) || K * min_bin > hi - lo || !(min_slope < 1.f))
    return fail(CNFOT_ERR_ARG, "bad spline constants");
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  bool known = false;
  cudaError_t e = rqs_vjp_dispatch(K, inverse, (cudaStream_t)stream, v, params, go, gl, rows,
                                   make_spline_consts<float>(K, lo, hi, min_bin, min_slope), gi, gp,
                                   di.num_sms, &known);
  if (!known) return fail(CNFOT_ERR_ARG, "num_bins=%d not instantiated (see CNFOT_BINS_LIST)", K);
  if (e != cudaSuccess) return cuda_fail(e, "rqs vjp kernel launch");
  return 0;
}

int cnfot_rqs_forward(void* stream, const float* x, const float* params, int64_t rows, int32_t num_bins,
                      float range_min, float range_max, float min_bin_size, float min_knot_slope,
                      float* y, float* logdet, int32_t* bin_idx) {
  return rqs_call(false, stream, x, params, rows, num_bins, range_min, range_max, min_bin_size,
                  min_knot_slope, y, logdet, bin_idx);
}
int cnfot_rqs_inverse(void* stream, const float* y, const float* params, int64_t rows, int32_t num_bins,
                      float range_min, float range_max, float min_bin_size, float min_knot_slope,
                      float* x, float* logdet, int32_t* bin_idx) {
  return rqs_call(true, stream, y, params, rows, num_bins, range_min, range_max, min_bin_size,
                  min_knot_slope, x, logdet, bin_idx);
}
int cnfot_rqs_forward_vjp(void* stream, const float* x, const float* params, const float* g_y,
                          const float* g_logdet, int64_t rows, int32_t num_bins, float range_min,
                          float range_max, float min_bin_size, float min_knot_slope, float* g_x,
                          float* g_params) {
  return rqs_vjp_call(false, stream, x, params, g_y, g_logdet, rows, num_bins, range_min, range_max,
                      min_bin_size, min_knot_slope, g_x, g_params);
}
int cnfot_rqs_inverse_vjp(void* stream, const float* y, const float* params, const float* g_x,
                          const float* g_logdet, int64_t rows, int32_t num_bins, float range_min,
                          float range_max, float min_bin_size, float min_knot_slope, float* g_y,
                          float* g_params) {
  return rqs_vjp_call(true, stream, y, params, g_x, g_logdet, rows, num_bins, range_min, range_max,
                      min_bin_size, min_knot_slope, g_y, g_params);
}

// ---- seam 1 ---------------------------------------------------------------------------
static int flow_eval_call(int dir, void* stream, const cnfot_flow_desc* flow, const float* weights,
                          const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                          float* out, float* logdet, int32_t add_base, void* workspace = nullptr,
                          int64_t workspace_bytes = 0) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (use_wide(flow, lay)) {
    if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
    if (cond_stride != 0 && cond_stride != 1) return fail(CNFOT_ERR_ARG, "cond_stride must be 0 or 1");
    if (rows == 0) return 0;
    if (!weights || !in || !cond || !out) return fail(CNFOT_ERR_ARG, "NULL buffer");
    const int64_t need = wide_flow_workspace_bytes(lay, rows, false);
    if (!workspace)
      return fail(CNFOT_ERR_WORKSPACE, "this flow runs on the wide-conditioner engine, which needs a workspace: "
                                       "call cnfot_flow_forward_ws / cnfot_flow_inverse_ws");
    if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                            (long long)workspace_bytes, (long long)need);
    const char* what = "";
    cudaError_t e = wide_flow_eval((cudaStream_t)stream, lay, spline_consts(flow), weights, dir, in, cond, cond_stride,
                                   rows, out, logdet, add_base, workspace, &what);
    if (e != cudaSuccess) return cuda_fail(e, what);
    g_last_launch[0] = 0; g_last_launch[1] = 0; g_last_launch[2] = 0; g_last_launch[3] = kEngWide;
    record_variant(-1, 0, 0, false);
    return 0;
  }
  if (int rc = check_fused(flow, lay)) return rc;
  if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
  if (cond_stride != 0 && cond_stride != 1) return fail(CNFOT_ERR_ARG, "cond_stride must be 0 or 1");
  if (rows == 0) return 0;
  if (!weights || !in || !cond || !out) return fail(CNFOT_ERR_ARG, "NULL buffer");
  SmemPlan sp;
  int engine;
  if (int rc = make_plan(lay, false, &sp, &engine, false)) return rc;
  const void* kernel = find_flow_eval_kernel(lay, engine);
  LaunchCfg cfg;
  if (int rc = configure(kernel, sp, (rows + kTile - 1) / kTile, &cfg)) return rc;
  EvalArgs a;
  a.W = weights; a.frags = nullptr; a.in = in; a.cond = cond; a.cond_stride = cond_stride; a.rows = rows;
  a.out = out; a.logdet = logdet; a.dir = dir; a.add_base = add_base;
  a.D = lay.D; a.L = lay.L; a.plan = sp;
  void* args[] = {&a};
  cudaError_t e = cudaLaunchKernel(kernel, dim3(cfg.grid), dim3(kTile), args, cfg.smem, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "flow_eval_kernel launch");
  return 0;
}

int cnfot_flow_forward(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* in,
                       const float* cond, int64_t cond_stride, int64_t rows, float* out, float* logdet,
                       int32_t add_base) {
  return flow_eval_call(0, stream, flow, weights, in, cond, cond_stride, rows, out, logdet, add_base);
}
int cnfot_flow_inverse(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* in,
                       const float* cond, int64_t cond_stride, int64_t rows, float* out, float* logdet,
                       int32_t add_base) {
  return flow_eval_call(1, stream, flow, weights, in, cond, cond_stride, rows, out, logdet, add_base);
}

int64_t cnfot_flow_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  return use_wide(flow, lay) ? wide_flow_workspace_bytes(lay, rows, false) : 0;
}
int cnfot_flow_forward_ws(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* in,
                          const float* cond, int64_t cond_stride, int64_t rows, float* out, float* logdet,
                          int32_t add_base, void* workspace, int64_t workspace_bytes) {
  return flow_eval_call(0, stream, flow, weights, in, cond, cond_stride, rows, out, logdet, add_base, workspace,
                        workspace_bytes);
}
int cnfot_flow_inverse_ws(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* in,
                          const float* cond, int64_t cond_stride, int64_t rows, float* out, float* logdet,
                          int32_t add_base, void* workspace, int64_t workspace_bytes) {
  return flow_eval_call(1, stream, flow, weights, in, cond, cond_stride, rows, out, logdet, add_base, workspace,
                        workspace_bytes);
}

int64_t cnfot_flow_vjp_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  if (use_wide(flow, lay)) return wide_flow_workspace_bytes(lay, rows, true);
  return partial_bytes(lay);
}

static int flow_vjp_call(int dir, void* stream, const cnfot_flow_desc* flow, const float* weights,
                         const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                         const float* g_out, const float* g_logdet, int32_t add_base, float* g_in,
                         float* g_weights, void* workspace, int64_t workspace_bytes) {
  record_variant(-1, 0, 0, false);   // a call that launches no VJP kernel (rows == 0, errors) leaves no variant behind
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (use_wide(flow, lay)) {
    if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
    if (cond_stride != 0 && cond_stride != 1) return fail(CNFOT_ERR_ARG, "cond_stride must be 0 or 1");
    if (!weights || !g_weights || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
    if (rows > 0 && (!in || !cond || !g_out)) return fail(CNFOT_ERR_ARG, "NULL buffer");
    const int64_t need = wide_flow_workspace_bytes(lay, rows, true);
    if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                            (long long)workspace_bytes, (long long)need);
    const char* what = "";
    cudaError_t e = wide_flow_vjp((cudaStream_t)stream, lay, spline_consts(flow), weights, dir, in, cond, cond_stride,
                                  rows, g_out, g_logdet, add_base, g_in, g_weights, workspace, &what);
    if (e != cudaSuccess) return cuda_fail(e, what);
    g_last_launch[0] = 0; g_last_launch[1] = 0; g_last_launch[2] = 0; g_last_launch[3] = kEngWide;
    record_variant(kEngWide, 0, 0, false);
    return 0;
  }
  if (int rc = check_fused(flow, lay)) return rc;
  if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
  if (cond_stride != 0 && cond_stride != 1) return fail(CNFOT_ERR_ARG, "cond_stride must be 0 or 1");
  if (!weights || !g_weights || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (workspace_bytes < partial_bytes(lay)) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                                        (long long)workspace_bytes, (long long)partial_bytes(lay));
  cudaStream_t s = (cudaStream_t)stream;
  if (rows == 0) {
    cudaError_t e = cudaMemsetAsync(g_weights, 0, (size_t)lay.total * sizeof(float), s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    return 0;
  }
  if (!in || !cond || !g_out) return fail(CNFOT_ERR_ARG, "NULL buffer");
  SmemPlan sp;
  int engine;
  if (int rc = make_plan(lay, true, &sp, &engine)) return rc;
  const int stash_cols = stash_tmem_cols(lay, engine);   // seam 1 differentiates the rows it just evaluated
  const void* kernel = find_flow_vjp_kernel(lay, engine, stash_cols > 0);
  LaunchCfg cfg;
  if (int rc = configure(kernel, sp, (rows + kTile - 1) / kTile, &cfg, stash_cols)) return rc;
  record_variant(engine, stash_cols, 0, false);
  unsigned long long* counter;
  VjpArgs a;
  a.W = weights; a.frags = nullptr; a.in = in; a.cond = cond; a.cond_stride = cond_stride; a.rows = rows;
  if (engine == kEngMmaStream) {
    float* fr = carve_frags(workspace, lay);
    if (int rc = launch_build_frags(s, lay, weights, fr)) return rc;
    a.frags = fr;
  }
  a.g_out = g_out; a.g_logdet = g_logdet; a.g_in = g_in; a.dir = dir; a.add_base = add_base;
  a.D = lay.D; a.L = lay.L; a.plan = sp;
  a.pb = carve_partials(workspace, &counter);
  a.stash_cols = stash_cols;
  void* args[] = {&a};
  cudaError_t e = cudaLaunchKernel(kernel, dim3(cfg.grid), dim3(kTile), args, cfg.smem, s);
  if (e != cudaSuccess) return cuda_fail(e, "flow_vjp_kernel launch");
  return launch_finalize(s, a.pb, cfg.grid, lay.total, g_weights, nullptr);
}

int cnfot_flow_forward_vjp(void* stream, const cnfot_flow_desc* flow, const float* weights,
                           const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                           const float* g_out, const float* g_logdet, int32_t add_base, float* g_in,
                           float* g_weights, void* workspace, int64_t workspace_bytes) {
  return flow_vjp_call(0, stream, flow, weights, in, cond, cond_stride, rows, g_out, g_logdet, add_base,
                       g_in, g_weights, workspace, workspace_bytes);
}
int cnfot_flow_inverse_vjp(void* stream, const cnfot_flow_desc* flow, const float* weights,
                           const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                           const float* g_out, const float* g_logdet, int32_t add_base, float* g_in,
                           float* g_weights, void* workspace, int64_t workspace_bytes) {
  return flow_vjp_call(1, stream, flow, weights, in, cond, cond_stride, rows, g_out, g_logdet, add_base,
                       g_in, g_weights, workspace, workspace_bytes);
}

// ---- persistent step workspaces -------------------------------------------------------------------------
// A registered workspace is only ever touched by the step entries (stream-ordered): every step leaves its reduction
// buffers and counters clean for the next one (the kernel's tail zeroes what it read), so no memset sits between two
// consecutive step kernels -- which is also what lets the next launch overlap the previous kernel's end (below).
static std::mutex g_ws_mu;
static std::vector<std::pair<void*, int64_t>> g_ws_registered;
static bool ws_registered(const void* ws) {
  std::lock_guard<std::mutex> lk(g_ws_mu);
  for (const auto& e : g_ws_registered)
    if (e.first == ws) return true;
  return false;
}
int cnfot_workspace_release(void* workspace) {
  std::lock_guard<std::mutex> lk(g_ws_mu);
  for (size_t i = 0; i < g_ws_registered.size(); ++i)
    if (g_ws_registered[i].first == workspace) {
      g_ws_registered.erase(g_ws_registered.begin() + i);
      return 0;
    }
  return 0;
}

// Launch of the persistent flow kernels with programmatic stream serialisation: the kernel may be scheduled while the
// previous kernel of the stream is still in its tail; it executes griddepcontrol.wait before its first global access
// (flow_kernels.cuh), so only the launch latency and the CTA ramp-up overlap, never any data.  CNFOT_PDL=0: plain launch.
static bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("CNFOT_PDL");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on != 0;
}
static cudaError_t launch_step_kernel(const void* kernel, int grid, void** args, size_t smem, cudaStream_t s) {
  if (!pdl_enabled()) return cudaLaunchKernel(kernel, dim3(grid), dim3(kTile), args, smem, s);
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3(grid); lc.blockDim = dim3(kTile); lc.dynamicSmemBytes = smem; lc.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = at; lc.numAttrs = 1;
  return cudaLaunchKernelExC(&lc, kernel, args);
}

// ---- seam 3 ---------------------------------------------------------------------------
static int64_t step_ws_bytes(const cnfot_flow_desc* flow, const FlowLayout& lay, int64_t rows_B, int64_t rows_b) {
  return use_wide(flow, lay) ? wide_step_workspace_bytes(lay, rows_B, rows_b) : partial_bytes(lay);
}

int64_t cnfot_mfc_step_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows_B, int64_t rows_b,
                                       int32_t n_t) {
  (void)n_t;
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  return step_ws_bytes(flow, lay, rows_B, rows_b);
}

// The step on the wide-conditioner engine (wide.cu): hidden >= 64, e.g. BASELINE config 5.
static int mfc_step_wide(void* stream, const cnfot_flow_desc* flow, const FlowLayout& lay,
                         const cnfot_problem_desc* problem, const float* weights, const float* latent, const float* latent_sub,
                         const float* src, const float* tgt, const float* t_batch_host, int32_t n_t, int64_t rows_B,
                         int64_t rows_b, int64_t global_B, int64_t global_b, float lambda, float* out, void* workspace,
                         int64_t workspace_bytes, bool accumulate, const cnfot_peer_desc* peers) {
  if (!problem) return fail(CNFOT_ERR_ARG, "problem descriptor is NULL");
  if (peers)
    return fail(CNFOT_ERR_ARG, "the wide-conditioner engine has no fused all-reduce (its gradient is hundreds of MB): "
                               "call cnfot_mfc_step and all-reduce `out` with NCCL");
  if (accumulate) return fail(CNFOT_ERR_ARG, "the wide-conditioner engine does not take chunked host input");
  if (rows_B < 0 || rows_b < 0 || global_B < 1 || global_b < 1 || rows_B > global_B || rows_b > global_b)
    return fail(CNFOT_ERR_ARG, "bad row counts");
  if (n_t < 1) return fail(CNFOT_ERR_ARG, "t_batch_size must be >= 1");
  if (!weights || !out || !workspace || !t_batch_host) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (problem->type == CNFOT_OT) {
    if (rows_B > 0 && (!src || !tgt)) return fail(CNFOT_ERR_ARG, "ot needs src and tgt batches");
  } else if (rows_B > 0 && !latent) {
    return fail(CNFOT_ERR_ARG, "latent is NULL");
  }
  if (rows_b > 0 && !latent_sub) return fail(CNFOT_ERR_ARG, "latent_sub is NULL");
  const int64_t need = wide_step_workspace_bytes(lay, rows_B, rows_b);
  if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                          (long long)workspace_bytes, (long long)need);
  StepConsts<float> pc;
  const char* err = nullptr;
  if (make_step_consts<float>(*problem, lay.D, (double)lambda, global_B, global_b, n_t, &pc, &err))
    return fail(CNFOT_ERR_ARG, "%s", err);
  const char* what = "";
  cudaError_t e = wide_mfc_step((cudaStream_t)stream, lay, spline_consts(flow), pc, weights, latent, latent_sub, src, tgt,
                                t_batch_host, n_t, rows_B, rows_b, out, workspace, &what);
  if (e != cudaSuccess) return cuda_fail(e, what);
  g_last_launch[0] = 0; g_last_launch[1] = 0; g_last_launch[2] = 0; g_last_launch[3] = kEngWide;
  record_variant(kEngWide, 0, 0, false);
  return 0;
}

// Everything a step call can vary: where the rows come from, what the kernel's tail does with the result.
struct StepIo {
  // explicit inputs (rng == false)
  const float* latent = nullptr;
  const float* latent_sub = nullptr;
  const float* src = nullptr;
  const float* tgt = nullptr;
  const float* t_batch_host = nullptr;
  // on-chip draws (rng == true): philox.cuh streams of (key, step); row0_* = global index of the shard's first row
  bool rng = false;
  uint64_t key = 0;
  uint32_t step = 0;
  int64_t row0_B = 0, row0_b = 0;
  // result
  float* out = nullptr;
  bool accumulate = false;
  const cnfot_peer_desc* peers = nullptr;
  // device-resident update (state != nullptr): `workspace` is the train state, Adam runs in the kernel's tail
  bool stateful = false;
  float* weights_rw = nullptr;
  float* adam_m = nullptr;
  float* adam_v = nullptr;
  float lr = 0.f, b1 = 0.9f, b2 = 0.999f, eps = 1e-8f;
  float* loss_hist = nullptr;
  int64_t loss_hist_len = 0;
};

static unsigned long long dp_timeout_ns() {
  unsigned long long ms = 20000ULL;   // a rank that is this late is gone (CNFOT_DP_TIMEOUT_MS overrides)
  if (const char* e = getenv("CNFOT_DP_TIMEOUT_MS")) {
    const long long v = atoll(e);
    if (v > 0) ms = (unsigned long long)v;
  }
  return ms * 1000000ULL;
}

static int mfc_step_impl(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                         const float* weights, const StepIo& io, int32_t n_t,
                         int64_t rows_B, int64_t rows_b, int64_t global_B, int64_t global_b, float lambda,
                         void* workspace, int64_t workspace_bytes) {
  record_variant(-1, 0, 0, false);   // a call that launches no step kernel (no rows, errors) leaves no variant behind
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (use_wide(flow, lay)) {
    cnfot_workspace_release(workspace);   // the wide engine uses the memory as plain scratch: not clean afterwards
    if (io.rng || io.stateful)
      return fail(CNFOT_ERR_ARG, "the wide-conditioner engine takes explicit row arrays: fill them with cnfot_philox_rows "
                                 "and call cnfot_mfc_step (+ cnfot_adam_update)");
    return mfc_step_wide(stream, flow, lay, problem, weights, io.latent, io.latent_sub, io.src, io.tgt, io.t_batch_host, n_t,
                         rows_B, rows_b, global_B, global_b, lambda, io.out, workspace, workspace_bytes, io.accumulate, io.peers);
  }
  if (int rc = check_fused(flow, lay)) return rc;
  if (!problem) return fail(CNFOT_ERR_ARG, "problem descriptor is NULL");
  StepArgs a;
  memset(&a.tail, 0, sizeof(a.tail));
  PeerArgs& pa = a.tail.pa;
  const cnfot_peer_desc* peers = io.peers;
  if (peers) {
    if (peers->world < 1 || peers->world > 8 || peers->rank < 0 || peers->rank >= peers->world)
      return fail(CNFOT_ERR_ARG, "peer descriptor: need 1 <= world <= 8 and 0 <= rank < world");
    if (peers->epoch == 0 && !io.stateful) return fail(CNFOT_ERR_ARG, "peer descriptor: epoch starts at 1");
    pa.rank = peers->rank; pa.world = peers->world; pa.epoch = peers->epoch;
    pa.stride = (int)cnfot_dp_exchange_stride(flow);
    pa.timeout_ns = dp_timeout_ns();
    for (int k = 0; k < peers->world; ++k) {
      if (!peers->xbuf[k] || !peers->flags[k]) return fail(CNFOT_ERR_ARG, "peer descriptor: NULL peer buffer");
      if ((uintptr_t)peers->xbuf[k] & 7) return fail(CNFOT_ERR_ARG, "peer descriptor: exchange buffers must be 8-byte aligned");
      pa.xbuf[k] = (unsigned long long*)peers->xbuf[k]; pa.flags[k] = peers->flags[k];
    }
  }
  if (rows_B < 0 || rows_b < 0 || global_B < 1 || global_b < 1 || rows_B > global_B || rows_b > global_b)
    return fail(CNFOT_ERR_ARG, "bad row counts");
  if (n_t < 1 || n_t > kMaxSegments - 4) return fail(CNFOT_ERR_ARG, "t_batch_size must be in [1, %d]", kMaxSegments - 4);
  if (!weights || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (!io.out && !io.stateful) return fail(CNFOT_ERR_ARG, "out is NULL");
  if (!io.rng && !io.t_batch_host) return fail(CNFOT_ERR_ARG, "t_batch is NULL");
  if (workspace_bytes < partial_bytes(lay)) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                                        (long long)workspace_bytes, (long long)partial_bytes(lay));
  const char* err = nullptr;
  if (make_step_consts<float>(*problem, lay.D, (double)lambda, global_B, global_b, n_t, &a.pc, &err))
    return fail(CNFOT_ERR_ARG, "%s", err);
  if (!io.rng) {
    if (problem->type == CNFOT_OT) {
      if (rows_B > 0 && (!io.src || !io.tgt)) return fail(CNFOT_ERR_ARG, "ot needs src and tgt batches");
    } else {
      if (rows_B > 0 && !io.latent) return fail(CNFOT_ERR_ARG, "latent is NULL");
    }
    if (rows_b > 0 && !io.latent_sub) return fail(CNFOT_ERR_ARG, "latent_sub is NULL");
  } else if (io.row0_B < 0 || io.row0_b < 0 || io.row0_B + rows_B > global_B || io.row0_b + rows_b > global_b) {
    return fail(CNFOT_ERR_ARG, "shard [row0, row0 + rows) outside the global batch");
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (rows_B == 0 && rows_b == 0 && !peers && !io.stateful) {
    if (io.accumulate) return 0;
    cudaError_t e = cudaMemsetAsync(io.out, 0, (size_t)(lay.total + CNFOT_NUM_LOSS_SLOTS) * sizeof(float), s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
    return 0;
  }
  SmemPlan sp;
  int engine;
  if (int rc = make_plan(lay, true, &sp, &engine)) return rc;
  const int unit = kTile;

  // segments, most expensive first (kinetic rows run 3..3+4D passes each)
  int ns = 0;
  int64_t tiles = 0;
  auto add = [&](int kind, int slot, int do_fit, int do_pot, float t, int t_index, const float* rows, int source,
                 int64_t row0, int64_t n, int group) {
    if (n <= 0) return;
    Segment& sg = a.seg[ns++];
    sg.kind = kind; sg.slot = slot; sg.do_fit = do_fit; sg.do_pot = do_pot; sg.t = t; sg.t_index = t_index;
    sg.rows = rows; sg.source = io.rng ? source : (int)kRowsMemory; sg.row0 = row0;
    sg.n = n; sg.first_tile = tiles; sg.group = group;
    tiles += (n * group + unit - 1) / unit;
  };
  // Small steps (the reference's default batch sizes): one thread per kinetic row is the latency of the whole step, so
  // the passes of a row are spread over a group of lanes (row_kinetic_split) when the step would not fill the GPU twice.
  // CNFOT_KINETIC_SPLIT=0 / 1 forces the choice.
  int group = 1;
  {
    const bool with_score = problem->type != CNFOT_OT;
    const bool need_r3 = with_score || a.pc.potential == kPotObstacle;
    int g = with_score ? 4 : (need_r3 ? 4 : 2);
    while (with_score && g < 2 * lay.D) g <<= 1;
    const int64_t fit_tiles = (problem->type == CNFOT_FP ? 1 : 2) * ((rows_B + unit - 1) / unit);
    const int64_t serial_tiles = fit_tiles + (int64_t)n_t * ((rows_b + unit - 1) / unit);
    bool split = g <= 32 && serial_tiles <= kMaxGrid;
    if (const char* e = getenv("CNFOT_KINETIC_SPLIT")) split = g <= 32 && e[0] != '0';
    if (split) group = g;
  }
  // streamed plan: few rounds of tiles -> the long kinetic tiles set the time: the two-CTAs-per-SM instantiation
  bool latency = false;
  {
    const int64_t fit_tiles = (problem->type == CNFOT_FP ? 1 : 2) * ((rows_B + unit - 1) / unit);
    latency = fit_tiles + (int64_t)n_t * ((rows_b + unit - 1) / unit) < 8 * 4 * 148;
    if (const char* e = getenv("CNFOT_STEP_LATENCY")) latency = e[0] != '0';
  }
  const int stash_cols = stash_tmem_cols(lay, engine);
  const void* kernel = find_mfc_step_kernel(lay, engine, group > 1, latency, stash_cols > 0);
  for (int i = 0; i < n_t; ++i)
    add(group > 1 ? kSegKineticSplit : kSegKinetic, kSlotKinetic, 0, 0, io.rng ? 0.f : io.t_batch_host[i], io.rng ? i : -1,
        io.latent_sub, kRowsNormal, io.row0_b, rows_b, group);
  if (problem->type == CNFOT_OT) {
    add(kSegNll, kSlotFit0, 1, 0, 0.f, -1, io.src, kRowsOtSource, io.row0_B, rows_B, 1);
    add(kSegNll, kSlotFitT, 1, 0, (float)a.pc.horizon, -1, io.tgt, kRowsNormal, io.row0_B, rows_B, 1);
  } else {
    add(kSegSample, kSlotFit0, 1, 0, 0.f, -1, io.latent, kRowsNormal, io.row0_B, rows_B, 1);
    if (problem->type == CNFOT_RWPO) add(kSegSample, kSlotFit0, 0, 1, (float)a.pc.horizon, -1, io.latent, kRowsNormal, io.row0_B, rows_B, 1);
  }
  a.n_seg = ns;
  a.n_tiles = tiles;
  a.key = io.key;
  a.step = io.step;
  a.timeline = g_step_timeline;
  a.salt_B = philox_salt(kDrawNormal, (uint64_t)global_B);
  a.salt_Bc = philox_salt(kDrawCategorical, (uint64_t)global_B);
  a.salt_b = philox_salt(kDrawNormal, (uint64_t)global_b);
  a.salt_t = philox_salt(kDrawUniform, (uint64_t)n_t);
  LaunchCfg cfg;
  if (int rc = configure(kernel, sp, (tiles * unit + kTile - 1) / kTile, &cfg, stash_cols)) return rc;
  record_variant(engine, stash_cols, group, engine == kEngMmaStream && group == 1 && latency);
  a.W = weights;
  a.frags = nullptr;
  if (engine == kEngMmaStream) {
    float* fr = carve_frags(workspace, lay);
    if (int rc = launch_build_frags(s, lay, weights, fr)) return rc;
    a.frags = fr;
  }
  a.D = lay.D; a.L = lay.L; a.plan = sp;
  a.stash_cols = stash_cols;
  // workspace / train state: [header: sync words, state words, loss row | partial gradient rows]
  TailArgs& t = a.tail;
  char* wsb = (char*)workspace;
  t.sync = (uint32_t*)wsb;
  t.loss_row = (double*)(wsb) + kLossRowOffset;
  t.grad_rows = (float*)(wsb + kCounterBytes);
  const bool persistent = io.stateful || ws_registered(workspace);   // the previous step left the buffers clean
  t.n_rows = cfg.grid < kStepRows ? cfg.grid : kStepRows;
  if (const char* e = getenv("CNFOT_STEP_ROWS")) {   // tuning knob: partial gradient rows (<= 1184)
    const int v = atoi(e);
    if (v >= 1 && v <= (persistent ? kStepRows : kMaxGrid)) t.n_rows = v < cfg.grid ? v : cfg.grid;
  }
  // CTAs that stay for the reduction (the first to finish their tiles): four threads per output column
  // The waiting CTAs hold their SM slots until every CTA of the grid has arrived, so they must stay a fraction of
  // what is resident: at most half of a grid that spans more than one CTA per SM (a GPU shared with another kernel may
  // not hold all of it at once; the CTAs that exit make room for the rest), all of a smaller one.
  int n_tail = (lay.total + kNumSlots + kTile / 4 - 1) / (kTile / 4);
  if (n_tail > cfg.grid) n_tail = cfg.grid;
  if (cfg.grid > 148 && n_tail > cfg.grid / 2) n_tail = cfg.grid / 2;
  if (n_tail > 2 * 148) n_tail = 2 * 148;
  if (n_tail < 1) n_tail = 1;
  t.n_tail = n_tail;
  t.total = lay.total;
  t.n_tiles = tiles;
  t.accumulate = io.accumulate ? 1 : 0;
  t.out = io.out;
  if (io.stateful) {
    t.self_clean = 1;
    t.state = (unsigned long long*)wsb + kStateWordOffset;
    t.weights = io.weights_rw; t.adam_m = io.adam_m; t.adam_v = io.adam_v;
    t.lr = io.lr; t.b1 = io.b1; t.b2 = io.b2; t.eps = io.eps;
    t.loss_hist = io.loss_hist; t.loss_hist_len = io.loss_hist_len;
  } else if (persistent) {
    t.self_clean = 1;
  } else {
    cudaError_t e = cudaMemsetAsync(wsb, 0, (size_t)kCounterBytes + (size_t)t.n_rows * lay.total * sizeof(float), s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  }
  void* args[] = {&a};
  cudaError_t e = launch_step_kernel(kernel, cfg.grid, args, cfg.smem, s);
  if (e != cudaSuccess) return cuda_fail(e, "mfc_step_kernel launch");
  return 0;
}

int64_t cnfot_dp_exchange_stride(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  return (lay.total + kNumSlots + 31) / 32 * 32;
}
int64_t cnfot_dp_exchange_floats(const cnfot_flow_desc* flow, int32_t world) {
  const int64_t st = cnfot_dp_exchange_stride(flow);
  // [2 parities][world sources][stride] 64-bit words {value, epoch}
  return st < 0 ? -1 : 2 * 2 * (int64_t)world * st;
}
int64_t cnfot_dp_flag_count(const cnfot_flow_desc* flow, int32_t world) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  (void)world;
  return 32;   // word 0: abort; the arrival flags travel inside the data words
}

int cnfot_mfc_step_dp(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                      const float* weights, const float* latent, const float* latent_sub, const float* src,
                      const float* tgt, const float* t_batch_host, int32_t n_t, int64_t rows_B,
                      int64_t rows_b, int64_t global_B, int64_t global_b, float lambda, float* out,
                      void* workspace, int64_t workspace_bytes, const cnfot_peer_desc* peers) {
  if (!peers) return fail(CNFOT_ERR_ARG, "peer descriptor is NULL");
  StepIo io;
  io.latent = latent; io.latent_sub = latent_sub; io.src = src; io.tgt = tgt; io.t_batch_host = t_batch_host;
  io.out = out; io.peers = peers;
  return mfc_step_impl(stream, flow, problem, weights, io, n_t, rows_B, rows_b, global_B, global_b, lambda, workspace,
                       workspace_bytes);
}

int cnfot_workspace_register(void* stream, const cnfot_flow_desc* flow, void* workspace, int64_t workspace_bytes) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (use_wide(flow, lay)) return fail(CNFOT_ERR_ARG, "persistent workspaces serve the fused per-row step kernel, not the wide-conditioner engine");
  if (!workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (workspace_bytes < partial_bytes(lay)) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                                        (long long)workspace_bytes, (long long)partial_bytes(lay));
  cudaError_t e = cudaMemsetAsync(workspace, 0, (size_t)kCounterBytes + (size_t)kStepRows * lay.total * sizeof(float),
                                  (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  cnfot_workspace_release(workspace);
  std::lock_guard<std::mutex> lk(g_ws_mu);
  g_ws_registered.emplace_back(workspace, workspace_bytes);
  return 0;
}

int cnfot_mfc_step(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                   const float* weights, const float* latent, const float* latent_sub, const float* src,
                   const float* tgt, const float* t_batch_host, int32_t n_t, int64_t rows_B,
                   int64_t rows_b, int64_t global_B, int64_t global_b, float lambda, float* out,
                   void* workspace, int64_t workspace_bytes) {
  StepIo io;
  io.latent = latent; io.latent_sub = latent_sub; io.src = src; io.tgt = tgt; io.t_batch_host = t_batch_host;
  io.out = out;
  return mfc_step_impl(stream, flow, problem, weights, io, n_t, rows_B, rows_b, global_B, global_b, lambda, workspace,
                       workspace_bytes);
}

// ---- on-chip draws: the same numbers as arrays (explicit-input entries, the CPU oracle) ------------------
__global__ void __launch_bounds__(256)
philox_rows_kernel(unsigned long long key_n, unsigned long long key_c, uint32_t step, int source, int64_t row0, int64_t rows,
                   int dim, float* __restrict__ out) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
    float row[kMaxDim];
    philox_row(key_n, key_c, step, source, (uint64_t)(row0 + r), dim, row);
    for (int i = 0; i < dim; ++i) out[r * dim + i] = row[i];
  }
}

int cnfot_philox_rows(void* stream, uint64_t key, uint32_t step, int32_t source, int64_t global_rows, int64_t row0,
                      int64_t rows, int32_t dim, float* out) {
  if (rows < 0 || row0 < 0 || row0 + rows > global_rows || dim < 1 || dim > kMaxDim)
    return fail(CNFOT_ERR_ARG, "philox_rows: need 0 <= row0, row0 + rows <= global_rows, 1 <= dim <= %d", kMaxDim);
  if (source != CNFOT_ROWS_NORMAL && source != CNFOT_ROWS_OT_SOURCE) return fail(CNFOT_ERR_ARG, "philox_rows: unknown row source");
  if (rows == 0) return 0;
  if (!out) return fail(CNFOT_ERR_ARG, "NULL buffer");
  int64_t blocks = (rows + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  philox_rows_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(
      key ^ philox_salt(kDrawNormal, (uint64_t)global_rows), key ^ philox_salt(kDrawCategorical, (uint64_t)global_rows), step,
      source, row0, rows, dim, out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "philox_rows_kernel launch");
  return 0;
}

int cnfot_philox_times_host(uint64_t key, uint32_t step, int32_t n_t, float horizon, float* t_host) {
  if (n_t < 0 || (n_t > 0 && !t_host)) return fail(CNFOT_ERR_ARG, "philox_times: bad arguments");
  const uint64_t kt = key ^ philox_salt(kDrawUniform, (uint64_t)n_t);
  for (int i = 0; i < n_t; ++i) t_host[i] = philox_time(kt, step, i, horizon);
  return 0;
}

int cnfot_mfc_step_rng(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem, const float* weights,
                       uint64_t key, uint32_t step, int32_t n_t, int64_t row0_B, int64_t rows_B, int64_t row0_b,
                       int64_t rows_b, int64_t global_B, int64_t global_b, float lambda, float* out, void* workspace,
                       int64_t workspace_bytes, const cnfot_peer_desc* peers) {
  StepIo io;
  io.rng = true; io.key = key; io.step = step; io.row0_B = row0_B; io.row0_b = row0_b;
  io.out = out; io.peers = peers;
  return mfc_step_impl(stream, flow, problem, weights, io, n_t, rows_B, rows_b, global_B, global_b, lambda, workspace,
                       workspace_bytes);
}

// ---- device-resident update (solvers.py:90-97 as ONE kernel launch, CUDA-graph replayable) --------------------
int64_t cnfot_train_state_bytes(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  if (use_wide(flow, lay)) { fail(CNFOT_ERR_ARG, "no device-resident update for the wide-conditioner engine"); return -1; }
  return partial_bytes(lay);
}

int cnfot_train_state_init(void* stream, const cnfot_flow_desc* flow, void* state, int64_t state_bytes, uint64_t key,
                           uint64_t step, uint32_t epoch) {
  const int64_t need = cnfot_train_state_bytes(flow);
  if (need < 0) return CNFOT_ERR_ARG;
  if (!state) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (state_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "train state too small: %lld < %lld", (long long)state_bytes, (long long)need);
  FlowLayout lay;
  check_flow(flow, &lay);
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(state, 0, (size_t)kCounterBytes + (size_t)kStepRows * lay.total * sizeof(float), s);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  const unsigned long long words[3] = {key, step, (unsigned long long)epoch};
  e = cudaMemcpyAsync((unsigned long long*)state + kStateWordOffset, words, sizeof(words), cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) return cuda_fail(e, "H2D train state");
  e = cudaStreamSynchronize(s);   // `words` lives on this stack frame
  if (e != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
  return 0;
}

int cnfot_mfc_update(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem, void* state,
                     int64_t state_bytes, float* weights, float* adam_m, float* adam_v, const cnfot_adam_desc* adam,
                     int32_t n_t, int64_t row0_B, int64_t rows_B, int64_t row0_b, int64_t rows_b, int64_t global_B,
                     int64_t global_b, float lambda, float* out, float* loss_hist, int64_t loss_hist_len,
                     const cnfot_peer_desc* peers) {
  if (!state || !weights || !adam_m || !adam_v || !adam) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (loss_hist_len < 0 || (loss_hist_len > 0 && !loss_hist)) return fail(CNFOT_ERR_ARG, "bad loss history buffer");
  StepIo io;
  io.rng = true; io.row0_B = row0_B; io.row0_b = row0_b;
  io.out = out; io.peers = peers;
  io.stateful = true;
  io.weights_rw = weights; io.adam_m = adam_m; io.adam_v = adam_v;
  io.lr = adam->lr; io.b1 = adam->b1; io.b2 = adam->b2; io.eps = adam->eps;
  io.loss_hist = loss_hist; io.loss_hist_len = loss_hist_len;
  return mfc_step_impl(stream, flow, problem, weights, io, n_t, rows_B, rows_b, global_B, global_b, lambda, state,
                       state_bytes);
}

static int64_t align256(int64_t v) { return (v + 255) / 256 * 256; }

// Copy stream + events of the *_host entry (one set per device, created on first use).
struct HostPipe {
  bool ready_ = false;
  cudaStream_t copy;
  cudaEvent_t start;
  cudaEvent_t ready[4];
};
static int host_pipe(HostPipe** out) {
  static HostPipe pipes[64];
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  HostPipe& p = pipes[di.device];
  if (!p.ready_) {
    cudaError_t e = cudaStreamCreateWithFlags(&p.copy, cudaStreamNonBlocking);
    if (e != cudaSuccess) return cuda_fail(e, "cudaStreamCreateWithFlags");
    if ((e = cudaEventCreateWithFlags(&p.start, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "cudaEventCreate");
    for (int k = 0; k < 4; ++k)
      if ((e = cudaEventCreateWithFlags(&p.ready[k], cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "cudaEventCreate");
    p.ready_ = true;
  }
  *out = &p;
  return 0;
}

int64_t cnfot_mfc_step_host_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows_B, int64_t rows_b,
                                            int32_t n_t) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  (void)n_t;
  int64_t rowsB = align256(rows_B * lay.D * (int64_t)sizeof(float));
  int64_t rowsb = align256(rows_b * lay.D * (int64_t)sizeof(float));
  int64_t w = align256((int64_t)lay.total * sizeof(float));
  int64_t o = align256((int64_t)(lay.total + CNFOT_NUM_LOSS_SLOTS) * sizeof(float));
  return align256(step_ws_bytes(flow, lay, rows_B, rows_b)) + w + o + 3 * rowsB + rowsb;
}

int cnfot_mfc_step_host(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                        const float* weights_host, const float* latent_host,
                        const float* latent_sub_host, const float* src_host, const float* tgt_host,
                        const float* t_batch_host, int32_t n_t, int64_t rows_B, int64_t rows_b,
                        int64_t global_B, int64_t global_b, float lambda, float* out_host,
                        void* workspace, int64_t workspace_bytes) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (!weights_host || !out_host || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (rows_B < 0 || rows_b < 0) return fail(CNFOT_ERR_ARG, "bad row counts");
  int64_t need = cnfot_mfc_step_host_workspace_bytes(flow, rows_B, rows_b, n_t);
  if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                          (long long)workspace_bytes, (long long)need);
  cudaStream_t s = (cudaStream_t)stream;
  char* p = (char*)workspace;
  const int64_t ws_bytes = align256(step_ws_bytes(flow, lay, rows_B, rows_b));
  void* ws = p; p += ws_bytes;
  float* dW = (float*)p; p += align256((int64_t)lay.total * sizeof(float));
  float* dOut = (float*)p; p += align256((int64_t)(lay.total + CNFOT_NUM_LOSS_SLOTS) * sizeof(float));
  const int64_t bytesB = rows_B * lay.D * (int64_t)sizeof(float);
  float* dLat = (float*)p; p += align256(bytesB);
  float* dSrc = (float*)p; p += align256(bytesB);
  float* dTgt = (float*)p; p += align256(bytesB);
  float* dSub = (float*)p;
  cudaError_t e;
  // Zero-copy path: when every row buffer is pinned (page-locked and mapped: cudaHostAlloc /
  // cudaHostRegister / torch pin_memory), the kernel reads the rows straight from host memory.
  // Each row is read exactly once and the step is compute-bound (16 warps per SM hide the PCIe
  // latency), so the transfer overlaps the math tile by tile instead of preceding it.
  // CNFOT_HOST_ZEROCOPY=0 forces the staged copy.
  bool zero_copy = true;
  if (const char* ev = getenv("CNFOT_HOST_ZEROCOPY")) zero_copy = ev[0] != '0';
  const float* mapped[4] = {nullptr, nullptr, nullptr, nullptr};
  const float* hostp[4] = {latent_host, latent_sub_host, src_host, tgt_host};
  for (int k = 0; k < 4 && zero_copy; ++k) {
    if (!hostp[k]) continue;
    cudaPointerAttributes at;
    e = cudaPointerGetAttributes(&at, hostp[k]);
    if (e != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) {
      cudaGetLastError();  // pageable memory: not an error, use the staged path
      zero_copy = false;
      break;
    }
    mapped[k] = (const float*)at.devicePointer;
  }
  if ((e = cudaMemcpyAsync(dW, weights_host, (size_t)lay.total * sizeof(float), cudaMemcpyHostToDevice, s)) != cudaSuccess)
    return cuda_fail(e, "H2D weights");
  if (zero_copy) {
    StepIo io;
    io.latent = mapped[0]; io.latent_sub = mapped[1]; io.src = mapped[2]; io.tgt = mapped[3]; io.t_batch_host = t_batch_host;
    io.out = dOut;
    int rc = mfc_step_impl(stream, flow, problem, dW, io, n_t, rows_B, rows_b, global_B, global_b, lambda, ws, ws_bytes);
    if (rc) return rc;
  } else {
    // Staged path.  Row chunks: the H2D copy of chunk k+1 (internal copy stream) overlaps the kernels
    // of chunk k (caller's stream); every chunk adds into dOut.  The b-row sub-batch terms ride with
    // chunk 0.  Measured on B200 (tools/host_chunks.py, cfg 2): chunking does not pay, default 1.
    HostPipe* hp = nullptr;
    if (int rc = host_pipe(&hp)) return rc;
    int nchunk = 1;
    if (const char* ev = getenv("CNFOT_HOST_CHUNKS")) {  // tuning knob (1..4)
      const int v = atoi(ev);
      if (v >= 1 && v <= 4) nchunk = v;
    }
    if ((e = cudaEventRecord(hp->start, s)) != cudaSuccess) return cuda_fail(e, "cudaEventRecord");
    if ((e = cudaStreamWaitEvent(hp->copy, hp->start, 0)) != cudaSuccess) return cuda_fail(e, "cudaStreamWaitEvent");
    auto h2d = [&](cudaStream_t st, float* dst, const float* src, int64_t off_rows, int64_t n_rows) -> cudaError_t {
      if (!src || n_rows == 0) return cudaSuccess;
      return cudaMemcpyAsync(dst + off_rows * lay.D, src + off_rows * lay.D, (size_t)(n_rows * lay.D) * sizeof(float),
                             cudaMemcpyHostToDevice, st);
    };
    if ((e = h2d(s, dSub, latent_sub_host, 0, rows_b)) != cudaSuccess) return cuda_fail(e, "H2D latent_sub");
    for (int k = 0; k < nchunk; ++k) {
      const int64_t lo = rows_B * k / nchunk, hi = rows_B * (k + 1) / nchunk;
      if ((e = h2d(hp->copy, dLat, latent_host, lo, hi - lo)) != cudaSuccess) return cuda_fail(e, "H2D latent");
      if ((e = h2d(hp->copy, dSrc, src_host, lo, hi - lo)) != cudaSuccess) return cuda_fail(e, "H2D src");
      if ((e = h2d(hp->copy, dTgt, tgt_host, lo, hi - lo)) != cudaSuccess) return cuda_fail(e, "H2D tgt");
      if ((e = cudaEventRecord(hp->ready[k], hp->copy)) != cudaSuccess) return cuda_fail(e, "cudaEventRecord");
    }
    for (int k = 0; k < nchunk; ++k) {
      const int64_t lo = rows_B * k / nchunk, hi = rows_B * (k + 1) / nchunk;
      if ((e = cudaStreamWaitEvent(s, hp->ready[k], 0)) != cudaSuccess) return cuda_fail(e, "cudaStreamWaitEvent");
      StepIo io;
      io.latent = latent_host ? dLat + lo * lay.D : nullptr;
      io.latent_sub = latent_sub_host ? dSub : nullptr;
      io.src = src_host ? dSrc + lo * lay.D : nullptr;
      io.tgt = tgt_host ? dTgt + lo * lay.D : nullptr;
      io.t_batch_host = t_batch_host;
      io.out = dOut;
      io.accumulate = k > 0;
      int rc = mfc_step_impl(stream, flow, problem, dW, io, n_t, hi - lo, k == 0 ? rows_b : 0, global_B, global_b, lambda, ws,
                             ws_bytes);
      if (rc) return rc;
    }
  }
  e = cudaMemcpyAsync(out_host, dOut, (size_t)(lay.total + CNFOT_NUM_LOSS_SLOTS) * sizeof(float),
                      cudaMemcpyDeviceToHost, s);
  if (e != cudaSuccess) return cuda_fail(e, "D2H out");
  e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
  return 0;
}

int64_t cnfot_mfc_step_rng_host_workspace_bytes(const cnfot_flow_desc* flow) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  if (use_wide(flow, lay)) { fail(CNFOT_ERR_ARG, "on-chip draws are not available on the wide-conditioner engine"); return -1; }
  return align256(partial_bytes(lay)) + align256((int64_t)lay.total * sizeof(float)) +
         align256((int64_t)(lay.total + CNFOT_NUM_LOSS_SLOTS) * sizeof(float));
}

int cnfot_mfc_step_rng_host(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                            const float* weights_host, uint64_t key, uint32_t step, int32_t n_t, int64_t row0_B,
                            int64_t rows_B, int64_t row0_b, int64_t rows_b, int64_t global_B, int64_t global_b,
                            float lambda, float* out_host, void* workspace, int64_t workspace_bytes) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (!weights_host || !out_host || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  const int64_t need = cnfot_mfc_step_rng_host_workspace_bytes(flow);
  if (need < 0) return CNFOT_ERR_ARG;
  if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                          (long long)workspace_bytes, (long long)need);
  cudaStream_t s = (cudaStream_t)stream;
  char* p = (char*)workspace;
  const int64_t ws_bytes = align256(partial_bytes(lay));
  void* ws = p; p += ws_bytes;
  float* dW = (float*)p; p += align256((int64_t)lay.total * sizeof(float));
  float* dOut = (float*)p;
  cudaError_t e = cudaMemcpyAsync(dW, weights_host, (size_t)lay.total * sizeof(float), cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) return cuda_fail(e, "H2D weights");
  StepIo io;
  io.rng = true; io.key = key; io.step = step; io.row0_B = row0_B; io.row0_b = row0_b;
  // Pinned (mapped) out_host: the kernel's tail writes the 4.8 KB result straight into it (posted PCIe writes, visible
  // after the synchronisation below) -- one asynchronous copy and its latency less.  Pageable: staged.
  float* out_mapped = nullptr;
  {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, out_host) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
      out_mapped = (float*)at.devicePointer;
    else
      cudaGetLastError();   // an unregistered pointer is not an error here
  }
  io.out = out_mapped ? out_mapped : dOut;
  if (int rc = mfc_step_impl(stream, flow, problem, dW, io, n_t, rows_B, rows_b, global_B, global_b, lambda, ws, ws_bytes))
    return rc;
  if (!out_mapped) {
    e = cudaMemcpyAsync(out_host, dOut, (size_t)(lay.total + CNFOT_NUM_LOSS_SLOTS) * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) return cuda_fail(e, "D2H out");
  }
  e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
  return 0;
}

int64_t cnfot_kinetic_energy_workspace_bytes(const cnfot_flow_desc* flow, int32_t n_t) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  if (use_wide(flow, lay)) return wide_energy_workspace_bytes(lay);
  return partial_bytes(lay) + ((int64_t)(n_t > 0 ? n_t : 0) * (int64_t)sizeof(float) + 255) / 256 * 256;
}

int cnfot_kinetic_energy(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* latent,
                         int64_t batch, int32_t latent_blocks, const float* t_host, int32_t n_t, float dt,
                         int32_t with_score, float kappa, float dx, double* out, void* workspace,
                         int64_t workspace_bytes) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  if (!use_wide(flow, lay))
    if (int rc = check_fused(flow, lay)) return rc;
  if (batch < 1 || n_t < 1 || latent_blocks < 1) return fail(CNFOT_ERR_ARG, "batch, n_t and latent_blocks must be >= 1");
  if (!weights || !latent || !t_host || !out || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (!(dt > 0.f) || (with_score && !(dx > 0.f))) return fail(CNFOT_ERR_ARG, "dt and dx must be positive");
  const int64_t need = cnfot_kinetic_energy_workspace_bytes(flow, n_t);
  if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld",
                                          (long long)workspace_bytes, (long long)need);
  if (use_wide(flow, lay)) {
    const char* what = "";
    cudaError_t we = wide_kinetic_energy((cudaStream_t)stream, lay, spline_consts(flow), weights, latent, batch,
                                         latent_blocks, t_host, n_t, dt, with_score, kappa, dx, out, workspace, &what);
    if (we != cudaSuccess) return cuda_fail(we, what);
    g_last_launch[0] = 0; g_last_launch[1] = 0; g_last_launch[2] = 0; g_last_launch[3] = kEngWide;
    record_variant(-1, 0, 0, false);
    return 0;
  }
  cudaStream_t s = (cudaStream_t)stream;
  EnergyArgs a;
  float* t_dev = (float*)((char*)workspace + partial_bytes(lay));
  cudaError_t e = cudaMemcpyAsync(t_dev, t_host, (size_t)n_t * sizeof(float), cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) return cuda_fail(e, "H2D times");
  SmemPlan sp;
  int engine;
  if (int rc = make_plan(lay, false, &sp, &engine)) return rc;
  const void* kernel = find_energy_kernel(lay, engine);
  if (!kernel) return fail(CNFOT_ERR_ARG, "no energy kernel for this network shape");
  a.tiles_per_t = (batch + kTile - 1) / kTile;
  a.n_tiles = a.tiles_per_t * n_t;
  LaunchCfg cfg;
  if (int rc = configure(kernel, sp, a.n_tiles, &cfg)) return rc;
  a.W = weights;
  a.frags = nullptr;
  if (engine == kEngMmaStream) {
    float* fr = carve_frags(workspace, lay);
    if (int rc = launch_build_frags(s, lay, weights, fr)) return rc;
    a.frags = fr;
  }
  a.D = lay.D; a.L = lay.L; a.plan = sp;
  a.latent = latent; a.batch = batch; a.latent_blocks = latent_blocks;
  a.t_dev = t_dev; a.n_t = n_t; a.with_score = with_score;
  a.dt = dt; a.dx = dx; a.kappa = kappa;
  a.weight = 1.0 / (2.0 * (double)batch * (double)n_t);
  a.pb = carve_partials(workspace, &a.tile_counter);
  e = cudaMemsetAsync(a.tile_counter, 0, sizeof(unsigned long long), s);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync");
  void* args[] = {&a};
  e = cudaLaunchKernel(kernel, dim3(cfg.grid), dim3(kTile), args, cfg.smem, s);
  if (e != cudaSuccess) return cuda_fail(e, "energy_kernel launch");
  energy_finalize_kernel<<<1, 32, 0, s>>>(a.pb.loss, cfg.grid, out);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "energy_finalize_kernel launch");
  return 0;
}

// ---- densities on a grid / at Monte-Carlo samples (SURVEY.md section 8f row 3) ----------------------------
int64_t cnfot_density_workspace_bytes(const cnfot_flow_desc* flow, int32_t n_t) {
  FlowLayout lay;
  if (check_flow(flow, &lay)) return -1;
  if (use_wide(flow, lay)) return wide_density_workspace_bytes(lay, n_t);
  return partial_bytes(lay) + ((int64_t)(n_t > 0 ? n_t : 0) * (int64_t)sizeof(float) + 255) / 256 * 256 + 256;
}

static int density_call(void* stream, const cnfot_flow_desc* flow, const float* weights, DensityArgs& a, const float* t_host,
                        int32_t n_t, double* sq_err, void* workspace, int64_t workspace_bytes) {
  FlowLayout lay;
  if (int rc = check_flow(flow, &lay)) return rc;
  const bool wide = use_wide(flow, lay);
  if (!wide)
    if (int rc = check_fused(flow, lay)) return rc;
  if (!weights || !workspace) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (a.with_ref && (!sq_err || !(a.var0 > 0.f) || !(a.var1 > 0.f))) return fail(CNFOT_ERR_ARG, "reference density: need sq_err and positive variances");
  const int64_t need = cnfot_density_workspace_bytes(flow, n_t);
  if (workspace_bytes < need) return fail(CNFOT_ERR_WORKSPACE, "workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)need);
  cudaStream_t s = (cudaStream_t)stream;
  if (a.n == 0) {
    if (sq_err) { cudaError_t e = cudaMemsetAsync(sq_err, 0, sizeof(double), s); if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync"); }
    return 0;
  }
  if (wide) {
    const char* what = "";
    cudaError_t we = a.mode == 0
        ? wide_density_grid(s, lay, spline_consts(flow), weights, t_host, n_t, a.x_min, a.x_step, a.y_min, a.y_step, a.nx,
                            a.ny, a.density, a.with_ref, a.mix, a.var0, a.var1, sq_err, workspace, &what)
        : wide_density_mc(s, lay, spline_consts(flow), weights, a.cond, a.key_n, a.step, a.n, a.samples, a.density,
                          a.with_ref, a.mix, a.var0, a.var1, sq_err, workspace, &what);
    if (we != cudaSuccess) return cuda_fail(we, what);
    g_last_launch[0] = 0; g_last_launch[1] = 0; g_last_launch[2] = 0; g_last_launch[3] = kEngWide;
    record_variant(-1, 0, 0, false);
    return 0;
  }
  float* t_dev = (float*)((char*)workspace + partial_bytes(lay));
  if (n_t > 0) {
    cudaError_t e = cudaMemcpyAsync(t_dev, t_host, (size_t)n_t * sizeof(float), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return cuda_fail(e, "H2D times");
  }
  SmemPlan sp;
  int engine;
  if (int rc = make_plan(lay, false, &sp, &engine)) return rc;
  const void* kernel = find_density_kernel(lay, engine);
  if (!kernel) return fail(CNFOT_ERR_ARG, "no density kernel for this network shape");
  LaunchCfg cfg;
  if (int rc = configure(kernel, sp, (a.n + kTile - 1) / kTile, &cfg)) return rc;
  a.W = weights;
  a.frags = nullptr;
  if (engine == kEngMmaStream) {
    float* fr = carve_frags(workspace, lay);
    if (int rc = launch_build_frags(s, lay, weights, fr)) return rc;
    a.frags = fr;
  }
  a.D = lay.D; a.L = lay.L; a.plan = sp;
  a.t_dev = t_dev;
  unsigned long long* counter;
  a.pb = carve_partials(workspace, &counter);
  void* args[] = {&a};
  cudaError_t e = cudaLaunchKernel(kernel, dim3(cfg.grid), dim3(kTile), args, cfg.smem, s);
  if (e != cudaSuccess) return cuda_fail(e, "density_kernel launch");
  if (sq_err) {
    energy_finalize_kernel<<<1, 32, 0, s>>>(a.pb.loss, cfg.grid, sq_err);
    e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "energy_finalize_kernel launch");
  }
  return 0;
}

int cnfot_density_grid(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* t_host, int32_t n_t,
                       double x_min, double x_max, double y_min, double y_max, int32_t nx, int32_t ny, float* density,
                       int32_t with_ref, float mix, float var0, float var1, double* sq_err, void* workspace,
                       int64_t workspace_bytes) {
  if (!flow || flow->dim != 2) return fail(CNFOT_ERR_ARG, "density grids are two-dimensional (the reference's are): dim must be 2");
  if (n_t < 1 || nx < 2 || ny < 2 || !t_host) return fail(CNFOT_ERR_ARG, "density_grid: need n_t >= 1, nx, ny >= 2");
  if (!density && !with_ref) return fail(CNFOT_ERR_ARG, "density_grid: nothing to compute");
  DensityArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = 0; a.nx = nx; a.ny = ny; a.n_t = n_t;
  a.x_min = x_min; a.x_step = (x_max - x_min) / (nx - 1);   // np.linspace(x_min, x_max, nx)
  a.y_min = y_min; a.y_step = (y_max - y_min) / (ny - 1);
  a.n = (int64_t)nx * ny * n_t;
  a.density = density;
  a.with_ref = with_ref; a.mix = mix; a.var0 = var0; a.var1 = var1;
  return density_call(stream, flow, weights, a, t_host, n_t, with_ref ? sq_err : nullptr, workspace, workspace_bytes);
}

int cnfot_density_mc(void* stream, const cnfot_flow_desc* flow, const float* weights, float cond, uint64_t key, uint32_t step,
                     int64_t n, float* samples, float* density, int32_t with_ref, float mix, float var0, float var1,
                     double* sq_err, void* workspace, int64_t workspace_bytes) {
  if (n < 0) return fail(CNFOT_ERR_ARG, "density_mc: n < 0");
  if (!density && !with_ref && !samples) return fail(CNFOT_ERR_ARG, "density_mc: nothing to compute");
  DensityArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = 1; a.n = n; a.cond = cond;
  a.key_n = key ^ philox_salt(kDrawNormal, (uint64_t)n);
  a.step = step;
  a.samples = samples; a.density = density;
  a.with_ref = with_ref; a.mix = mix; a.var0 = var0; a.var1 = var1;
  return density_call(stream, flow, weights, a, nullptr, 0, with_ref ? sq_err : nullptr, workspace, workspace_bytes);
}

// ---- wide conditioner layers on tcgen05 (dense_tc.cu) ----------------------------------------
int64_t cnfot_dense_prepared_floats(int32_t K, int32_t N) {
  if (K < 16 || N < 16 || K % 16 || N % 16) return -1;
  return 2 * (int64_t)K * N;
}

int cnfot_dense_prepare(void* stream, const float* W, int32_t K, int32_t N, int32_t ldw, int32_t transpose,
                        float* prepared) {
  if (!W || !prepared) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (cnfot_dense_prepared_floats(K, N) < 0) return fail(CNFOT_ERR_ARG, "dense layers need K and N to be multiples of 16");
  cudaError_t e = dense_prep((cudaStream_t)stream, W, K, N, ldw, transpose != 0, prepared);
  if (e != cudaSuccess) return cuda_fail(e, "dense_prep_kernel launch");
  return 0;
}

int cnfot_dense_forward(void* stream, const float* X, int64_t rows, int32_t K, int32_t ldx, const float* prepared,
                        int32_t N, const float* bias, const float* mask_src, int32_t ldm, int32_t epilogue,
                        float* Y, int32_t ldy) {
  if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
  if (rows == 0) return 0;
  if (!X || !prepared || !Y) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (cnfot_dense_prepared_floats(K, N) < 0) return fail(CNFOT_ERR_ARG, "dense layers need K and N to be multiples of 16");
  if (epilogue < 0 || epilogue > 4) return fail(CNFOT_ERR_ARG, "unknown epilogue");
  if ((epilogue == 0 || epilogue == 1) && !bias) return fail(CNFOT_ERR_ARG, "bias is NULL");
  if (epilogue == 2 && !mask_src) return fail(CNFOT_ERR_ARG, "mask_src is NULL");
  if (ldx % 4 || ldy % 4 || (epilogue == 2 && ldm % 4)) return fail(CNFOT_ERR_ARG, "row strides must be multiples of 4 floats");
  bool ok = false;
  cudaError_t e = dense_forward((cudaStream_t)stream, X, rows, K, ldx, prepared, N, bias, mask_src, ldm, epilogue,
                                Y, ldy, &ok);
  if (!ok) return fail(CNFOT_ERR_ARG, "no dense kernel for N = %d", N);
  if (e != cudaSuccess) return cuda_fail(e, "dense_tc_kernel launch");
  return 0;
}

int cnfot_dense_wgrad(void* stream, const float* A, int32_t lda, const float* G, int32_t ldg, int64_t rows,
                      int32_t Ka, int32_t Nb, float* dW, int32_t ldw, float* db) {
  if (rows < 0) return fail(CNFOT_ERR_ARG, "rows < 0");
  if (rows == 0) return 0;
  if (!A || !G || !dW) return fail(CNFOT_ERR_ARG, "NULL buffer");
  if (Ka < 1 || Nb < 4 || Nb % 4 || ldw % 4 || ((uintptr_t)dW & 15))
    return fail(CNFOT_ERR_ARG, "dense_wgrad: Nb and ldw must be multiples of 4 and dW 16-byte aligned");
  cudaError_t e = dense_wgrad((cudaStream_t)stream, A, lda, G, ldg, rows, Ka, Nb, dW, ldw, db);
  if (e != cudaSuccess) return cuda_fail(e, "dense_wgrad_kernel launch");
  return 0;
}

int cnfot_recon_head(void* stream, const float* x, const float* xr, int64_t rows, int32_t dim, float weight,
                     float* g_xr, double* loss) {
  if (rows < 0 || dim < 1) return fail(CNFOT_ERR_ARG, "bad sizes");
  if (rows == 0) return 0;
  if (!x || !xr || !g_xr || !loss) return fail(CNFOT_ERR_ARG, "NULL buffer");
  const int64_t count = rows * dim;
  int64_t blocks = (count + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  recon_head_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(x, xr, count, weight, g_xr, loss);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "recon_head_kernel launch");
  return 0;
}

int cnfot_mask_tail(void* stream, float* y, int64_t rows, int32_t dim, int32_t sub_dim) {
  if (rows < 0 || dim < 1 || sub_dim < 0 || sub_dim > dim) return fail(CNFOT_ERR_ARG, "bad sizes");
  if (rows == 0 || sub_dim == dim) return 0;
  if (!y) return fail(CNFOT_ERR_ARG, "NULL buffer");
  int64_t blocks = (rows * dim + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  mask_tail_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(y, rows, dim, sub_dim);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "mask_tail_kernel launch");
  return 0;
}

int cnfot_adam_update(void* stream, float* params, const float* grads, float* m, float* v, int64_t count,
                      float lr, float b1, float b2, float eps, int64_t step) {
  if (count < 0 || step < 1) return fail(CNFOT_ERR_ARG, "bad count/step");
  if (count == 0) return 0;
  if (!params || !grads || !m || !v) return fail(CNFOT_ERR_ARG, "NULL buffer");
  DeviceInfo di;
  if (int rc = device_info(&di)) return rc;
  float c1 = (float)(1.0 - pow((double)b1, (double)step)), c2 = (float)(1.0 - pow((double)b2, (double)step));
  int threads = 256;
  int64_t blocks = (count + threads - 1) / threads;
  if (blocks > (int64_t)di.num_sms * 8) blocks = (int64_t)di.num_sms * 8;
  adam_kernel<<<(int)blocks, threads, 0, (cudaStream_t)stream>>>(params, grads, m, v, count, lr, b1, b2, eps, c1, c2);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "adam_kernel launch");
  return 0;
}

}  // extern "C"
