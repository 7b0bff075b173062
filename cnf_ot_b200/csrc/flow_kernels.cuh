// Fused whole-flow kernels (one thread = one sample row, weights in shared
// memory) behind cnfot_flow_* and cnfot_mfc_step.  Templated on the network
// shape (hidden, bins, mlp layers) and on a runtime / compile-time flow shape.
#pragma once

#include <type_traits>

#include "device_common.cuh"
#include "philox.cuh"
#include "step_math.cuh"
#include "tc_engine.cuh"
#include "warp_mlp.cuh"

namespace cnfot {

// CTA context by engine: 0 CUDA-core dense layers, 1 the tcgen05 engine (tc_engine.cuh),
// 2 the warp-level tensor-core engine (warp_mlp.cuh); 1 and 2 exist for 16-wide networks.
// kEngMmaStash: the warp-level engine with the activation stash in tensor memory -- a kernel instantiation of its own
// (step and VJP kernels only), so that no other kernel contains tcgen05 instructions.
enum Engine { kEngCuda = 0, kEngTc = 1, kEngMma = 2, kEngMmaStream = 3, kEngWide = 4, kEngMmaStash = 5 };
#ifndef CNFOT_MMA_MIN_CTAS
#define CNFOT_MMA_MIN_CTAS 4
#endif
constexpr int kMmaMinCtas = CNFOT_MMA_MIN_CTAS;   // register budget of the warp-MMA kernels: 65536 / (128 * n)
// The train-step kernel runs THREE CTAs (12 warps) per SM at up to 168 registers: measured on B200 against four at 128
// (round 1 and most of round 2) -- cfg 2 0.1467 vs 0.1501 ms, cfg 3 0.602 vs 0.655, cfg 4 (2^19 rows) 4.26 vs 4.70: the
// kernel is latency-bound and register-starved (spills, context members re-loaded from local memory after every asm
// memory clobber), and a warp with 168 registers is a third faster than one with 128.  Five CTAs at 102: 0.178 ms.
#ifndef CNFOT_STEP_MIN_CTAS
#define CNFOT_STEP_MIN_CTAS 3
#endif
constexpr int kStepMinCtas = CNFOT_STEP_MIN_CTAS;
// The streamed plan (flows too large for resident fragments, e.g. dim 10) has two instantiations: FOUR CTAs per SM for
// throughput and TWO (8 warps, up to 255 registers: the fastest single warp) for steps of few tile rounds, where the
// long kinetic tiles set the time -- cfg 4 (ms per step at 2^19 / 2^20 / 2^22 rows): two CTAs 3.93 / 7.76 / 30.8, three
// 4.28 / 5.98 / 23.7, four 4.75 / 5.55 / 21.5.  The host picks (api.cu: mfc_step_impl).
constexpr int kStepMinCtasStream = 4;
constexpr int kStepMinCtasStreamLatency = 2;
// DC, LC: compile-time flow shape (0 = runtime), passed by the train-step kernel only (warp_mlp.cuh: kConstPlan)
template <class Net, int ENG, int DC = 0, int LC = 0>
struct CtxSelect { using type = DeviceCtx<Net>; };
template <class Net, int DC, int LC>
struct CtxSelect<Net, kEngTc, DC, LC> { using type = DeviceCtxTC<Net>; };
template <class Net, int DC, int LC>
struct CtxSelect<Net, kEngMma, DC, LC> { using type = DeviceCtxMma<Net, true, DC, LC>; };
template <class Net, int DC, int LC>
struct CtxSelect<Net, kEngMmaStream, DC, LC> { using type = DeviceCtxMma<Net, false>; };
template <class Net, int DC, int LC>
struct CtxSelect<Net, kEngMmaStash, DC, LC> { using type = DeviceCtxMma<Net, true, DC, LC, true>; };

template <class Ctx>
__device__ __forceinline__ void ctx_setup(Ctx& ctx, int D, int L, uint64_t* mbar, uint32_t* slot) {
  ctx.setup(D, L, mbar, slot);
}
template <class Ctx>
__device__ __forceinline__ void ctx_teardown(Ctx& ctx) { ctx.teardown(); }

// ---- forward-only evaluation (model API: sample / forward / inverse / log_prob) ----
struct EvalArgs {
  const float* W;
  const float* frags;   // streamed warp-MMA plan: global fragment buffer (else nullptr)
  const float* in;
  const float* cond;
  int64_t cond_stride;
  int64_t rows;
  float* out;
  float* logdet;
  int dir;
  int add_base;
  int D, L;
  SmemPlan plan;
};

template <class Net, class DimsT, int ENG>
__global__ void __launch_bounds__(kTile, ENG >= kEngMma ? kMmaMinCtas : 1) flow_eval_kernel(EvalArgs a) {
  extern __shared__ __align__(1024) float smem[];
  __shared__ __align__(8) uint64_t tc_mbar;
  __shared__ uint32_t tc_slot;
  using Ctx = typename CtxSelect<Net, ENG>::type;
  Ctx ctx;
  ctx.smem = smem; ctx.gW = a.W; ctx.p = a.plan;
  ctx.bind_partials(nullptr);
  ctx.bind_frags(a.frags);
  ctx_setup(ctx, a.D, a.L, &tc_mbar, &tc_slot);
  const RowTiles<float, Net> tl = make_row_tiles<Net>(smem, a.plan);
  const DimsT dm{a.D, a.L};
  const int D = dm.D(), L = dm.L();
  for (int64_t tile = blockIdx.x; tile * kTile < a.rows; tile += gridDim.x) {
    const int64_t r = tile * kTile + ctx.row_in_tile();
    const bool live = r < a.rows;  // every thread runs the pass: the context has CTA barriers
    float st[kMaxStateFloats];
    for (int i = 0; i < D; ++i) st[i] = live ? a.in[r * D + i] : 0.f;
    const float t = live ? a.cond[r * a.cond_stride] : 0.f;
    float ld = a.dir == 0 ? flow_pass<0, float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), t, st, tl, ctx)
                          : flow_pass<1, float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), t, st, tl, ctx);
    if (!live) continue;
    for (int i = 0; i < D; ++i) a.out[r * D + i] = st[L * D + i];
    if (a.logdet) {
      if (a.add_base)
        ld = a.dir == 0 ? base_log_prob<float>(st, D) - ld
                        : base_log_prob<float>(st + L * D, D) + ld;
      a.logdet[r] = ld;
    }
  }
  ctx_teardown(ctx);
}

// ---- per-CTA partial results -------------------------------------------------------
struct PartialBuf {
  float* grad;     // [n_cta][total]
  double* loss;    // [n_cta][kNumSlots]
};

// sAcc: the CTA's shared-memory gradient accumulator, or nullptr when the context adds straight
// into the CTA's partial row (Ctx::kAccInGlobal)
__device__ inline void flush_partials(const PartialBuf& pb, const float* sAcc, int total,
                                      const double* loss /* kNumSlots, thread-local */,
                                      double* scratch) {
  __syncthreads();
  float* dst = pb.grad + (int64_t)blockIdx.x * total;
  if (sAcc)
    for (int i = threadIdx.x; i < total; i += blockDim.x) dst[i] = sAcc[i];
  for (int s = 0; s < kNumSlots; ++s) {
    double v = block_sum(loss[s], scratch);
    if (threadIdx.x == 0) pb.loss[(int64_t)blockIdx.x * kNumSlots + s] = v;
  }
}

// ---- generic VJP of one flow pass (what a custom_vjp backward rule calls) ----------
struct VjpArgs {
  const float* W;
  const float* frags;
  const float* in;
  const float* cond;
  int64_t cond_stride;
  int64_t rows;
  const float* g_out;
  const float* g_logdet;
  float* g_in;
  int dir;
  int add_base;
  int D, L;
  SmemPlan plan;
  PartialBuf pb;
  int stash_cols;               // TMEM columns of the activation stash per CTA (warp-level engines), or 0
};

template <class Net, class DimsT, int ENG>
__global__ void __launch_bounds__(kTile, ENG >= kEngMma ? kMmaMinCtas : 1) flow_vjp_kernel(VjpArgs a) {
  extern __shared__ __align__(1024) float smem[];
  __shared__ double scratch[kWarps];
  __shared__ __align__(8) uint64_t tc_mbar;
  __shared__ uint32_t tc_slot;
  using Ctx = typename CtxSelect<Net, ENG>::type;
  float* sAcc = Ctx::kAccInGlobal ? nullptr : smem + a.plan.off_acc;
  Ctx ctx;
  ctx.smem = smem; ctx.gW = a.W; ctx.p = a.plan;
  ctx.bind_partials(a.pb.grad + (int64_t)blockIdx.x * a.plan.total);
  ctx.bind_frags(a.frags);
  ctx.stash_acquire(a.stash_cols, a.L * (a.D - 1), &tc_slot);
  ctx_setup(ctx, a.D, a.L, &tc_mbar, &tc_slot);
  const RowTiles<float, Net> tl = make_row_tiles<Net>(smem, a.plan);
  const DimsT dm{a.D, a.L};
  const int D = dm.D(), L = dm.L();
  FirstGrad<float, Net::kK> gfirst;   // knot adjoints of the shared `first` spline (pulled back once, below)
#pragma unroll
  for (int j = 0; j <= Net::kK; ++j) { gfirst.gx[j] = 0.f; gfirst.gy[j] = 0.f; gfirst.gd[j] = 0.f; }
  for (int64_t tile = blockIdx.x; tile * kTile < a.rows; tile += gridDim.x) {
    const int64_t r = tile * kTile + ctx.row_in_tile();
    const bool live = r < a.rows;
    float st[kMaxStateFloats], g[kMaxDim];
    for (int i = 0; i < D; ++i) st[i] = live ? a.in[r * D + i] : 0.f;
    const float t = live ? a.cond[r * a.cond_stride] : 0.f;
    const bool stash = ctx.stash_on();   // forward and backward of the same rows, back to back: keep the activations
    if (a.dir == 0) flow_pass<0, float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), t, st, tl, ctx, stash);
    else flow_pass<1, float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), t, st, tl, ctx, stash);
    const float gl = (live && a.g_logdet) ? a.g_logdet[r] : 0.f;
    for (int i = 0; i < D; ++i) g[i] = live ? a.g_out[r * D + i] : 0.f;
    float gl_pass = gl;
    if (a.add_base) {
      if (a.dir == 0) gl_pass = -gl;
      else
        for (int i = 0; i < D; ++i) g[i] -= gl * st[L * D + i];
    }
    if (a.dir == 0)
      flow_pass_bwd<0, float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), t, st, g, gl_pass, gfirst, tl, ctx, stash);
    else
      flow_pass_bwd<1, float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), t, st, g, gl_pass, gfirst, tl, ctx, stash);
    if (a.add_base && a.dir == 0)
      for (int i = 0; i < D; ++i) g[i] -= gl * st[i];
    if (live && a.g_in)
      for (int i = 0; i < D; ++i) a.g_in[r * D + i] = g[i];
  }
  ctx.stash_release();
  {
    float graw[Net::kPp];
#pragma unroll
    for (int j = 0; j < Net::kPp; ++j) graw[j] = 0.f;
    first_grad_to_raw<float, Net::kK>(gfirst, ctx.first_knots(), FixedSplineConsts<float, Net::kK>(), graw);
    ctx.flush_first(graw, tl);
  }
  double zero[kNumSlots];
  for (int s = 0; s < kNumSlots; ++s) zero[s] = 0.0;
  flush_partials(a.pb, sAcc, a.plan.total, zero, scratch);
  ctx_teardown(ctx);
}

// ---- evaluation energies: kinetic energy over a time grid (forward only) --------------------
// tile = (time index, 128-row tile); latent block (ti % latent_blocks) feeds time ti.
struct EnergyArgs {
  const float* W;
  const float* frags;
  int D, L;
  SmemPlan plan;
  const float* latent;     // (latent_blocks * batch, D)
  int64_t batch;
  int latent_blocks;
  const float* t_dev;      // (n_t) times, device
  int n_t;
  int with_score;
  float dt, dx, kappa;
  double weight;           // 1 / (2 batch n_t)
  int64_t tiles_per_t, n_tiles;
  unsigned long long* tile_counter;
  PartialBuf pb;
};

template <class Net, class DimsT, int ENG>
__global__ void __launch_bounds__(kTile, ENG >= kEngMma ? kMmaMinCtas : 1) energy_kernel(const __grid_constant__ EnergyArgs a) {
  extern __shared__ __align__(1024) float smem[];
  __shared__ double scratch[kWarps];
  __shared__ long long s_tile;
  __shared__ __align__(8) uint64_t tc_mbar;
  __shared__ uint32_t tc_slot;
  using Ctx = typename CtxSelect<Net, ENG>::type;
  Ctx ctx;
  ctx.smem = smem; ctx.gW = a.W; ctx.p = a.plan;
  ctx.bind_partials(nullptr);
  ctx.bind_frags(a.frags);
  ctx_setup(ctx, a.D, a.L, &tc_mbar, &tc_slot);
  const RowTiles<float, Net> tl = make_row_tiles<Net>(smem, a.plan);
  const DimsT dm{a.D, a.L};
  const int D = dm.D();
  double loss[kNumSlots];
#pragma unroll
  for (int s = 0; s < kNumSlots; ++s) loss[s] = 0.0;
  while (true) {
    __syncthreads();
    if (threadIdx.x == 0) s_tile = (long long)atomicAdd(a.tile_counter, 1ULL);
    __syncthreads();
    const long long tile = s_tile;
    if (tile >= a.n_tiles) break;
    const int ti = (int)(tile / a.tiles_per_t);
    const int64_t r = (tile - (long long)ti * a.tiles_per_t) * kTile + ctx.row_in_tile();
    const bool live = r < a.batch;
    const float* src = a.latent + ((int64_t)(ti % a.latent_blocks) * a.batch + r) * D;
    float row[kMaxDim];
    for (int i = 0; i < D; ++i) row[i] = live ? src[i] : 0.f;
    const float v2 = row_kinetic_value<float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), a.t_dev[ti], row, a.dt, a.with_score != 0,
                                                               a.kappa, a.dx, tl, ctx);
    if (live) loss[kSlotKinetic] += (double)v2 * a.weight;
  }
  flush_partials(a.pb, nullptr, 0, loss, scratch);
  ctx_teardown(ctx);
}

// ---- densities on a grid / at Monte-Carlo samples (SURVEY.md section 8f row 3) --------------------------
// The consumers of `log_prob_fn` / `sample_and_log_prob` after training:
//   grid mode  exp(log_prob(params, XY, cond = t)) on an nx x ny grid of [x_min, x_max] x [y_min, y_max] for n_t
//              times in ONE launch -- utils.plot_density_snapshot / plot_density_and_trajectory
//              (cnf_ot/utils.py:572-642: 100 x 100, ten times), solvers.py:184-222 (double-well density at T) and
//              rmse_grid_loss_fn (solvers.py:282-301: 500 x 500).  The grid points are generated in the kernel
//              (XY = hstack(meshgrid(linspace, linspace)) in float64, rounded to float32): no XY array in HBM.
//   MC mode    samples, log_prob = sample_and_log_prob(cond, seed) with the latent drawn on chip --
//              rmse_mc_loss_fn (solvers.py:254-278: 10^6 samples).
// Optional epilogue of both: the squared error against the reference density
// (1 - mix) N(0, var0 I) + mix N(0, var1 I) (solvers.py:238-252,270-276), summed in double.
struct DensityArgs {
  const float* W;
  const float* frags;
  int D, L;
  SmemPlan plan;
  int mode;                 // 0 grid, 1 Monte-Carlo
  int nx, ny, n_t;          // grid
  double x_min, x_step, y_min, y_step;
  const float* t_dev;       // (n_t) times
  unsigned long long key_n; // MC: Philox key of the (n, D) normal draw
  uint32_t step;
  float cond;               // MC: the time
  int64_t n;                // points in total (nx * ny * n_t, or samples)
  float* density;           // (n) exp(log_prob), or nullptr
  float* samples;           // MC: (n, D) samples, or nullptr
  int with_ref;
  float mix, var0, var1;
  PartialBuf pb;            // loss slot kSlotKinetic of each CTA receives its sum of squared errors
};

template <class Net, class DimsT, int ENG>
__global__ void __launch_bounds__(kTile, ENG >= kEngMma ? kMmaMinCtas : 1) density_kernel(const __grid_constant__ DensityArgs a) {
  extern __shared__ __align__(1024) float smem[];
  __shared__ double scratch[kWarps];
  __shared__ __align__(8) uint64_t tc_mbar;
  __shared__ uint32_t tc_slot;
  using Ctx = typename CtxSelect<Net, ENG>::type;
  Ctx ctx;
  ctx.smem = smem; ctx.gW = a.W; ctx.p = a.plan;
  ctx.bind_partials(nullptr);
  ctx.bind_frags(a.frags);
  ctx_setup(ctx, a.D, a.L, &tc_mbar, &tc_slot);
  const RowTiles<float, Net> tl = make_row_tiles<Net>(smem, a.plan);
  const DimsT dm{a.D, a.L};
  const int D = dm.D(), L = dm.L();
  const FixedSplineConsts<float, Net::kK> sc;
  double loss[kNumSlots];
#pragma unroll
  for (int s = 0; s < kNumSlots; ++s) loss[s] = 0.0;
  for (int64_t tile = blockIdx.x; tile * kTile < a.n; tile += gridDim.x) {   // uniform cost per point: static tiles
    const int64_t r = tile * kTile + ctx.row_in_tile();
    const bool live = r < a.n;   // every thread runs the pass: the contexts have CTA / warp barriers
    float st[kMaxStateFloats];
    for (int i = 0; i < D; ++i) st[i] = 0.f;
    float t = a.cond, lp;
    const float* y;
    if (a.mode == 0) {
      const int64_t per_t = (int64_t)a.nx * a.ny;
      const int ti = live ? (int)(r / per_t) : 0;
      const int64_t q = live ? r - (int64_t)ti * per_t : 0;
      const int iy = (int)(q / a.nx), ix = (int)(q - (int64_t)iy * a.nx);
      st[0] = (float)(a.x_min + (double)ix * a.x_step);
      st[1] = (float)(a.y_min + (double)iy * a.y_step);
      t = a.t_dev[ti];
      const float ld = flow_pass<1, float, Net, DimsT, Ctx>(dm, sc, t, st, tl, ctx);
      lp = base_log_prob<float>(st + L * D, D) + ld;
      y = st;
    } else {
      if (live) philox_row(a.key_n, a.key_n, a.step, kRowsNormal, (uint64_t)r, D, st);
      const float fldj = flow_pass<0, float, Net, DimsT, Ctx>(dm, sc, t, st, tl, ctx);
      lp = base_log_prob<float>(st, D) - fldj;
      y = st + L * D;
      if (live && a.samples)
        for (int i = 0; i < D; ++i) a.samples[r * D + i] = y[i];
    }
    if (!live) continue;
    const float p = m_exp(lp);
    if (a.density) a.density[r] = p;
    if (a.with_ref) {
      const float e = ref_mixture_error(p, y, D, a.mix, a.var0, a.var1);
      loss[kSlotKinetic] += (double)e * (double)e;
    }
  }
  flush_partials(a.pb, nullptr, 0, loss, scratch);
  ctx_teardown(ctx);
}

// ---- the fused train step ---------------------------------------------------------------
// One persistent kernel does the WHOLE step (SURVEY.md section 8a, a1): every term of the configured loss and
// its backward pass, the reduction of the CTAs' partial results, (multi-GPU) the all-reduce of
// [gradient | loss slots] over peer-mapped memory, and (device-resident update) Adam.
//   * work = a list of segments (one per loss term and time) cut into 128-row tiles handed out by an atomic
//     counter, most expensive segments first.
//   * rows come from the caller's arrays or are generated on chip (philox.cuh) -- the reference makes
//     every draw inside the jitted step from one key (applications.py:81-82,392).
//   * weight gradients are added (red.global) into one of `n_rows` partial rows (row = CTA index mod
//     n_rows), loss sums into one row of doubles; both are zero on entry (memset by the stateless entry,
//     self-cleaned by the previous launch in the device-resident one).
//   * tail: the last `n_tail` CTAs to finish stay, wait until every CTA has arrived, and each reduces
//     8-column slices of the partial rows in double; with peers the slice is pushed into every peer's
//     exchange buffer (NVLink / NVSwitch stores), flagged, and summed in rank order once every peer's
//     slice has arrived (bit-identical on all ranks); the owner of a column then writes the output and
//     applies the Adam update of that parameter.
enum SegmentKind { kSegNll = 0, kSegSample = 1, kSegKinetic = 2, kSegKineticSplit = 3 /* step_math.cuh: row_kinetic_split */ };

struct Segment {
  int kind;
  int slot;          // loss slot of the fit term (kSegNll / kSegSample)
  int do_fit, do_pot;
  int source;        // RowSource: kRowsMemory reads `rows`, the others draw the rows on chip
  int t_index;       // >= 0: t = horizon * U[0,1) drawn from (key, step, t_index); < 0: use `t`
  float t;
  const float* rows; // (n, D) data or latent rows (kRowsMemory)
  int64_t row0;      // global index of this shard's first row (on-chip draws)
  int64_t n;
  int64_t first_tile;  // in 128-row tiles
  int group;         // kSegKineticSplit: lanes per row (a tile holds 128 / group rows); 1 otherwise
};

constexpr int kMaxSegments = 36;

// header words (uint32) of the step workspace / train state
// Counters are MONOTONIC across launches: kSyncTile (tile claims) and kSyncDone (arrived CTAs) are never reset; their
// values at the start of a launch are kept in kSyncTileBase / kSyncDoneBase, and kSyncSeq counts launches (its parity
// selects which half of the loss row a launch adds into).  All three are advanced by ONE thread of the tail (the first
// tail CTA) once every CTA has arrived -- every CTA read them when it started -- so a launch ends when its last column
// is written, with no "who is last" election.  A zeroed header (memset, cnfot_workspace_register) is a valid state.
enum SyncWord { kSyncTile = 0 /* 64-bit: words 0, 1 */, kSyncDone = 2, kSyncStatus = 4, kSyncDoneBase = 5, kSyncSeq = 6,
                kSyncTileBase = 8 /* 64-bit: words 8, 9 */ };
constexpr int kStateWordOffset = 16;   // 64-bit words [key, step, epoch] start at byte 128 of the header
constexpr int kLossRowOffset = 24;     // 8 doubles at byte 192 of the header
constexpr int kStepRows = 32;          // partial gradient rows of the step kernel (CTA b adds into row b mod 32)

struct PeerArgs {
  int rank, world;     // world <= 1: no exchange
  uint32_t epoch;      // device-resident update: read from the train state instead
  int stride;          // 64-bit slots per (parity, source rank) in an exchange buffer (>= total + kNumSlots)
  unsigned long long timeout_ns;
  unsigned long long* xbuf[8];   // rank k's exchange buffer: [2 parities][world sources][stride] slots of {float bits, epoch}
  uint32_t* flags[8];            // rank k's flag words: [0] = abort
};

struct TailArgs {
  int n_rows;          // partial gradient rows
  int n_tail;          // CTAs that stay for the reduction
  int total;           // gradient floats
  int accumulate;      // out += result (chunked host entry)
  int self_clean;      // zero what was read (device-resident update: the next launch needs no memset)
  long long n_tiles;   // tiles of this launch (the tile counter advances by n_tiles + gridDim.x)
  uint32_t* sync;      // header words
  double* loss_row;    // [kNumSlots], atomically accumulated
  float* grad_rows;    // [n_rows][total]
  float* out;          // [total + kNumSlots] or nullptr
  float* weights;      // Adam (nullptr: none): parameters, first and second moments
  float* adam_m;
  float* adam_v;
  float lr, b1, b2, eps;
  unsigned long long* state;   // device train state [key, step, epoch] or nullptr
  float* loss_hist;    // loss_hist[step] = total loss (device-resident update), or nullptr
  long long loss_hist_len;
  PeerArgs pa;
};

struct StepArgs {
  const float* W;
  const float* frags;
  int D, L;
  SmemPlan plan;
  StepConsts<float> pc;
  int n_seg;
  int64_t n_tiles;     // 128-row tiles
  int stash_cols;      // TMEM columns of the activation stash per CTA (warp-level engines), or 0
  unsigned long long key;       // on-chip draws (philox.cuh): key and step, or read from the train state
  unsigned long long salt_B, salt_Bc, salt_b, salt_t;   // key modifiers: normal (B, D), categorical (B,), normal (b, D), uniform (n_t,)
  uint32_t step;
  unsigned long long* timeline;   // diagnostics (cnfot_debug_step_timeline): globaltimer stamps, or nullptr
  Segment seg[kMaxSegments];
  TailArgs tail;
};

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long v;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(v));
  return v;
}

// optax.adam (scale_by_adam + scale(-lr); cnf_ot/mfc/solvers.py:55,95-96) of one parameter
// (m0, v0, w0: the old moments and parameter, loaded by the caller together with the partial rows: one L2 round trip)
__device__ __forceinline__ void adam_one(const TailArgs& t, int i, float g, float c1, float c2, float m0, float v0, float w0) {
  const float mi = t.b1 * m0 + (1.f - t.b1) * g;
  const float vi = t.b2 * v0 + (1.f - t.b2) * g * g;
  t.adam_m[i] = mi;
  t.adam_v[i] = vi;
  t.weights[i] = w0 - t.lr * (mi / c1) / (sqrtf(vi / c2) + t.eps);
}

__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// The kernel's tail (see above).  Called by every thread of every CTA after its partial results are written.
//
// Reduction: one THREAD per output column sums the (<= 32) partial rows of its column -- up to 16 coalesced loads in
// flight, no shared memory, no barrier -- so the whole buffer is one pass of ceil(columns / 128) CTAs.  The CTAs that
// stay are the FIRST n_tail to finish their tiles: everything that does not depend on the other CTAs (the state words,
// Adam's bias corrections) is done while they wait, and what remains after the last CTA
// has arrived is one L2 round trip, the update and the stores.  (The round-2 start had the last n_tail arrivals run a
// slice-per-CTA reduction over shared memory: 8 us at 592 CTAs, 20 us of a 50 us step at 32 CTAs.)
// Exchange (world > 1): the column's sum is written into every peer's buffer as ONE 64-bit {value, epoch} word (an
// aligned 8-byte store arrives whole, so the data carries its own arrival flag: no fence, no flag round trip -- the
// latency of one NVLink write), and the same thread spins on the epoch of each peer's word for that column.
// Buffers are double-buffered by the epoch's parity: a rank can be at most one step ahead of a peer, because
// finishing a step needs every peer's words of that step.
struct LaunchHeader {   // the header words of the previous launch's end, read once per CTA (thread 0 -> shared memory)
  uint32_t done_base, seq, stepno, epoch;
  unsigned long long tile_base;
};

static __device__ __noinline__ void step_tail(const TailArgs& t, const LaunchHeader& h) {
  __shared__ unsigned s_ticket;
  __shared__ int s_bad;
  const int tid = threadIdx.x;
  __threadfence();
  __syncthreads();
  if (tid == 0) s_ticket = atomicAdd(t.sync + kSyncDone, 1u) - h.done_base;
  __syncthreads();
  const unsigned grid = gridDim.x, S = (unsigned)t.n_tail, ticket = s_ticket;
  if (ticket >= S) return;
  const int k = (int)ticket;
  const int total = t.total, n_out = total + kNumSlots;
  const bool dp = t.pa.world > 1;
  const uint32_t stepno = h.stepno, epoch = h.epoch;   // the state words as every CTA saw them when it started
  double* const loss_row = t.loss_row + 4 * (h.seq & 1u);   // this launch's half of the loss row
  float c1 = 1.f, c2 = 1.f;
  if (t.weights) {
    // 1 - b^(step + 1) without the cancellation: -expm1((step + 1) log b); float32 is accurate to ~2e-7 relative here
    // (optax itself evaluates 1 - b ** count in float32), and two double-precision pow() were 2 us of a small step's tail
    const float n1 = (float)stepno + 1.f;
    c1 = -expm1f(n1 * logf(t.b1));
    c2 = -expm1f(n1 * logf(t.b2));
  }
  const size_t par_off = (size_t)(epoch & 1u) * t.pa.world * t.pa.stride;
  if (tid == 0) {
    while (ld_acquire_gpu(t.sync + kSyncDone) - h.done_base < grid) __nanosleep(20);
    s_bad = (dp && ld_acquire_sys(t.pa.flags[t.pa.rank]) != 0u) ? 1 : 0;   // a peer gave up earlier: stay poisoned
    if (k == 0) {
      // every CTA has arrived, i.e. has read the header: advance it for the next launch (nothing below reads it)
      t.sync[kSyncDoneBase] = h.done_base + grid;
      t.sync[kSyncSeq] = h.seq + 1u;
      *reinterpret_cast<unsigned long long*>(t.sync + kSyncTileBase) = h.tile_base + (unsigned long long)t.n_tiles + grid;
      double* other = t.loss_row + 4 * ((h.seq & 1u) ^ 1u);   // the next launch's half: last read one launch ago
      other[0] = 0.0; other[1] = 0.0; other[2] = 0.0; other[3] = 0.0;
      if (t.state) {
        t.state[1] = (unsigned long long)h.stepno + 1ULL;
        t.state[2] = (unsigned long long)h.epoch + 1ULL;
      }
    }
  }
  __syncthreads();

  auto finish = [&](int col, float v, float m0, float v0, float w0) {   // the owner of an output column
    if (col < total) {
      if (t.out) t.out[col] = t.accumulate ? t.out[col] + v : v;
      if (t.weights && v == v) adam_one(t, col, v, c1, c2, m0, v0, w0);   // a poisoned (NaN) gradient leaves the parameters alone
    } else {
      const int sl = col - total;
      if (t.out) t.out[col] = sl <= 4 ? (t.accumulate ? t.out[col] + v : v) : 0.f;
      if (sl == 0 && t.loss_hist && (long long)stepno < t.loss_hist_len) t.loss_hist[stepno] = v;
    }
  };

  // four adjacent lanes share a column: lane j of the quad sums rows j, j + 4, ... (8 loads in flight for the 32 rows
  // of a persistent workspace), two shuffles fold the quad, its first lane owns the column from there on
  const int stride_cols = (int)S * (int)(blockDim.x >> 2);
  const int rg = tid & 3;
  const bool owner = rg == 0;
  const unsigned long long* mybuf = dp ? t.pa.xbuf[t.pa.rank] + par_off : nullptr;
  const uint32_t* abort_word = dp ? t.pa.flags[t.pa.rank] : nullptr;
  const int n_cols = (n_out + 7) & ~7;   // whole warps take part in the shuffles
  for (int col = k * (int)(blockDim.x >> 2) + (tid >> 2); col < n_cols; col += stride_cols) {
    // phase A: this quad's column of the partial rows -> one float (sent to the peers, or final)
    double acc = 0.0;
    float m0 = 0.f, v0 = 0.f, w0 = 0.f;
    if (t.weights && owner && col < total) {   // in flight together with the partial rows
      m0 = __ldcg(t.adam_m + col); v0 = __ldcg(t.adam_v + col); w0 = __ldcg(t.weights + col);
    }
    if (col < total) {
      float* p = t.grad_rows + col;
      for (int r0 = rg; r0 < t.n_rows; r0 += 32) {
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = r0 + 4 * q < t.n_rows ? __ldcg(p + (size_t)(r0 + 4 * q) * total) : 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) acc += (double)v[q];
        if (t.self_clean) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (r0 + 4 * q < t.n_rows) __stcg(p + (size_t)(r0 + 4 * q) * total, 0.f);
        }
      }
    } else if (col < n_out && owner) {
      // loss slots: out slot 0 = total of the 4 internal slots, 1..4 = internal 0..3, 5..7 = 0
      const int sl = col - total;
      if (sl == 0) acc = __ldcg(loss_row) + __ldcg(loss_row + 1) + __ldcg(loss_row + 2) + __ldcg(loss_row + 3);
      else if (sl <= 4) acc = __ldcg(loss_row + sl - 1);
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (!owner || col >= n_out) continue;
    const float mine = (float)acc;
    if (!dp) {
      finish(col, mine, m0, v0, w0);
      continue;
    }
    const unsigned long long word = ((unsigned long long)epoch << 32) | (unsigned long long)__float_as_uint(mine);
    for (int p = 0; p < t.pa.world; ++p)
      st_relaxed_sys_u64(t.pa.xbuf[p] + par_off + (size_t)t.pa.rank * t.pa.stride + col, word);
    // phase B: every peer's word of this column, summed in rank order.  All (<= 8) words are requested before the first
    // one is looked at: a sys-scope load is an L2 round trip, and eight of them one after the other were 5 us of the
    // 8-GPU step even when every word had long arrived.
    bool bad = *(volatile int*)&s_bad != 0;
    float sum = 0.f;
    if (!bad) {
      const unsigned long long* w0 = mybuf + col;
      unsigned long long v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) v[q] = q < t.pa.world ? ld_relaxed_sys_u64(w0 + (size_t)q * t.pa.stride) : 0ULL;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (q >= t.pa.world || bad) continue;
        if ((uint32_t)(v[q] >> 32) != epoch) {
          const unsigned long long* w = w0 + (size_t)q * t.pa.stride;
          const unsigned long long t0 = global_timer_ns();
          unsigned spins = 0;
          while ((uint32_t)((v[q] = ld_relaxed_sys_u64(w)) >> 32) != epoch) {
            if ((++spins & 255u) == 0u &&
                (ld_acquire_sys(abort_word) != 0u || global_timer_ns() - t0 > t.pa.timeout_ns)) {
              bad = true;
              break;
            }
          }
        }
        sum += __uint_as_float((uint32_t)v[q]);
      }
    }
    if (bad) {
      // a peer never arrived (or gave up): poison this rank's result AND tell every peer, so no rank
      // continues with a sum the others do not have; the status word is read by the host
      for (int p = 0; p < t.pa.world; ++p) st_release_sys(t.pa.flags[p], 1u);
      s_bad = 1;
      t.sync[kSyncStatus] = 1u;
      sum = __int_as_float(0x7fc00000);
    }
    finish(col, sum, m0, v0, w0);
  }
}

// SPLIT: the kinetic segments are of kind kSegKineticSplit (row_kinetic_split: the passes of a row spread over a lane
// group; the host picks this instantiation for steps too small to fill the GPU), else kSegKinetic (row_kinetic).  Two
// kernels rather than one branch: either routine inlined next to the other costs the common path registers.
template <class Net, class DimsT, int ENG, bool SPLIT = false, bool LAT = false>
__global__ void __launch_bounds__(kTile, ENG == kEngMmaStream ? (LAT || SPLIT ? kStepMinCtasStreamLatency : kStepMinCtasStream)
                                                              : (ENG >= kEngMma ? kStepMinCtas : 1))
mfc_step_kernel(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(1024) float smem[];
  __shared__ double scratch4[kWarps][4];
  __shared__ long long s_tile;
  __shared__ LaunchHeader s_hdr;
  __shared__ __align__(8) uint64_t tc_mbar;
  __shared__ uint32_t tc_slot;
  using Ctx = typename CtxSelect<Net, ENG, DimsT::kD, DimsT::kL>::type;
  // Programmatic dependent launch (api.cu: launch_step_kernel): this grid may have been scheduled while the previous
  // kernel of the stream was still in its tail; nothing is read or written before that kernel has completed.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (threadIdx.x == 0) {   // the header as the previous launch left it (visible to the CTA after the set-up's barriers)
    s_hdr.done_base = __ldcg(a.tail.sync + kSyncDoneBase);
    s_hdr.seq = __ldcg(a.tail.sync + kSyncSeq);
    s_hdr.tile_base = __ldcg(reinterpret_cast<const unsigned long long*>(a.tail.sync + kSyncTileBase));
    s_hdr.stepno = a.tail.state ? (uint32_t)__ldcg(a.tail.state + 1) : 0u;
    s_hdr.epoch = a.tail.state && a.tail.pa.world > 1 ? (uint32_t)__ldcg(a.tail.state + 2) : a.tail.pa.epoch;
  }
  unsigned long long t_start = 0;
  if (a.timeline && threadIdx.x == 0) { t_start = global_timer_ns(); atomicMin(a.timeline + 0, t_start); atomicMax(a.timeline + 7, t_start); }   // first / last CTA starts
  float* sAcc = Ctx::kAccInGlobal ? nullptr : smem + a.plan.off_acc;
  float* my_row = a.tail.grad_rows + (int64_t)(blockIdx.x % a.tail.n_rows) * a.plan.total;
  Ctx ctx;
  ctx.smem = smem; ctx.gW = a.W; ctx.p = a.plan;
  ctx.bind_partials(my_row, false);   // shared, pre-zeroed partial rows: the context must not clear them
  ctx.bind_frags(a.frags);
  ctx.stash_acquire(a.stash_cols, DimsT{a.D, a.L}.L() * (DimsT{a.D, a.L}.D() - 1), &tc_slot);
  ctx_setup(ctx, DimsT{a.D, a.L}.D(), DimsT{a.D, a.L}.L(), &tc_mbar, &tc_slot);   // compile-time shape where the kernel has one
  if (a.timeline && threadIdx.x == 0) { const unsigned long long now = global_timer_ns(); atomicMax(a.timeline + 1, now); atomicMax(a.timeline + 6, now - t_start); }   // last CTA is set up; longest setup
  const RowTiles<float, Net> tl = make_row_tiles<Net>(smem, a.plan);
  const DimsT dm{a.D, a.L};
  const int D = dm.D();
  unsigned long long key = a.key;
  uint32_t step = a.step;
  if (a.tail.state) {
    key = __ldcg(a.tail.state);
    step = (uint32_t)__ldcg(a.tail.state + 1);
  }
  unsigned long long* tile_counter = reinterpret_cast<unsigned long long*>(a.tail.sync + kSyncTile);
  FirstGrad<float, Net::kK> gfirst;   // knot adjoints of the shared `first` spline (pulled back once, below)
#pragma unroll
  for (int j = 0; j <= Net::kK; ++j) { gfirst.gx[j] = 0.f; gfirst.gy[j] = 0.f; gfirst.gd[j] = 0.f; }
  double loss[kNumSlots];
#pragma unroll
  for (int s = 0; s < kNumSlots; ++s) loss[s] = 0.0;

  // Work distribution: 128-row tiles handed out by an atomic counter, most expensive segments first.  (Measured and
  // rejected on B200, cfg 2: warps claiming 32-row units on their own, no CTA barrier: 0.196 vs 0.184 ms; tiles
  // pre-assigned round-robin with the next tile's rows prefetched by cp.async: 0.184 vs 0.180 ms -- CTAs that share
  // an SM run at different speeds, and only the counter evens that out.)
  while (true) {
    __syncthreads();
    if (threadIdx.x == 0) s_tile = (long long)(atomicAdd(tile_counter, 1ULL) - s_hdr.tile_base);
    __syncthreads();
    const long long tile = s_tile;
    if (tile >= a.n_tiles) break;
    int si = 0;
    while (si + 1 < a.n_seg && tile >= a.seg[si + 1].first_tile) ++si;
    const Segment& sg = a.seg[si];
    const bool split = SPLIT && sg.kind == kSegKineticSplit;   // the lanes of a group share a row
    const int64_t r = split ? (tile - sg.first_tile) * (kTile / sg.group) + (int)threadIdx.x / sg.group
                            : (tile - sg.first_tile) * kTile + ctx.row_in_tile();
    const bool live = r < sg.n;
    float row[kMaxDim];
    if (sg.source == kRowsMemory) {
      for (int i = 0; i < D; ++i) row[i] = live ? sg.rows[r * D + i] : 0.f;
    } else {
      for (int i = 0; i < D; ++i) row[i] = 0.f;
      if (live)
        philox_row(key ^ (sg.kind >= kSegKinetic ? a.salt_b : a.salt_B), key ^ a.salt_Bc, step, sg.source,
                   (uint64_t)(sg.row0 + r), D, row);
    }
    const float tval = sg.t_index >= 0 ? philox_time(key ^ a.salt_t, step, sg.t_index, a.pc.horizon) : sg.t;
    if (sg.kind == kSegNll) {
      float v = row_nll<float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), tval, row,
                                                           live ? a.pc.w_fit : 0.f, gfirst, tl, ctx);
      loss[sg.slot] += (double)v;
    } else if (sg.kind == kSegSample) {
      StepConsts<float> pc = a.pc;
      if (!live) { pc.w_fit = 0.f; pc.w_pot = 0.f; }
      float lf = 0.f, lp = 0.f;
      row_sample_terms<float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), tval, row, sg.do_fit != 0,
                                                          sg.do_pot != 0, pc, &lf, &lp, gfirst, tl, ctx);
      loss[sg.slot] += (double)lf;
      loss[kSlotPotential] += (double)lp;
    } else {
      StepConsts<float> pc = a.pc;
      if (!live) { pc.w_kin = 0.f; pc.w_pot = 0.f; }
      float lk = 0.f, lp = 0.f;
      if constexpr (SPLIT)
        row_kinetic_split<Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), tval, row, pc, sg.group, &lk, &lp,
                                           gfirst, tl, ctx);
      else
        row_kinetic<float, Net, DimsT, Ctx>(dm, FixedSplineConsts<float, Net::kK>(), tval, row, pc, &lk, &lp, gfirst,
                                            tl, ctx);
      loss[kSlotKinetic] += (double)lk;
      loss[kSlotPotential] += (double)lp;
    }
  }
  // Out of tiles: the next kernel of the stream may take the SM slots this grid frees from here on (every CTA of this
  // grid is resident or done by the time the last one gets here, so the newcomers cannot keep any of them out).  The
  // stash's TMEM columns are freed first, so a newcomer never finds them held.
  ctx.stash_release();
  asm volatile("griddepcontrol.launch_dependents;");
  if (a.timeline && threadIdx.x == 0) {   // this CTA ran out of tiles
    const unsigned long long now = global_timer_ns();
    atomicMin(a.timeline + 2, now);
    atomicMax(a.timeline + 3, now);
  }
  {
    float graw[Net::kPp];
#pragma unroll
    for (int j = 0; j < Net::kPp; ++j) graw[j] = 0.f;
    first_grad_to_raw<float, Net::kK>(gfirst, ctx.first_knots(), FixedSplineConsts<float, Net::kK>(), graw);
    ctx.flush_first(graw, tl);
  }
  // partial results -> the shared rows
  __syncthreads();
  if (sAcc)
    for (int i = threadIdx.x; i < a.plan.total; i += blockDim.x) {
      const float v = sAcc[i];
      if (v != 0.f) atomicAdd(my_row + i, v);
    }
  {   // the four live slots (fit0, fitT, potential, kinetic): warp sums, then one thread per slot
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      double v = loss[s];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0) scratch4[threadIdx.x >> 5][s] = v;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) v += scratch4[w][threadIdx.x];
      if (v != 0.0) atomicAdd(a.tail.loss_row + 4 * (s_hdr.seq & 1u) + threadIdx.x, v);
    }
  }
  ctx_teardown(ctx);
  if (a.timeline && threadIdx.x == 0) atomicMax(a.timeline + 4, global_timer_ns());   // last CTA enters the tail
  step_tail(a.tail, s_hdr);
  if (a.timeline && threadIdx.x == 0) atomicMax(a.timeline + 5, global_timer_ns());   // last CTA leaves
}

}  // namespace cnfot
