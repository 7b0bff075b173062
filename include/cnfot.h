/* cnfot.h -- C ABI of libcnfot.so: B200 (sm_100a) kernels for the cnf_ot flow
 * train step.
 *
 * This is the drop-in boundary for the reference's hot path.  The reference
 * (pure Python/JAX) has no FFI of its own; the seams this library plugs into
 * are the ones SURVEY.md section 8(b) lists:
 *   seam 2  Autoregressive(bijector=...)          cnf_ot/models/flows.py:124-132
 *           -> cnfot_rqs_*                         (one scalar spline per row)
 *   seam 1  Flow namedtuple of RQSFlow(...)        cnf_ot/models/flows.py:213-226
 *           -> cnfot_flow_*                        (whole conditional flow)
 *   seam 3  loss_fn consumed by value_and_grad     cnf_ot/mfc/solvers.py:90-97
 *           -> cnfot_mfc_step*                     (loss + parameter gradient)
 * Every entry point is shaped so an XLA FFI handler can forward to it 1:1
 * (stream + device buffers + scalar attributes); INTEGRATION.md shows the
 * binding.
 *
 * Conventions
 *   - All array pointers are DEVICE pointers to dense row-major float32 unless
 *     the name ends in _host.  Sizes are int64_t, the stream is a cudaStream_t
 *     passed as void*.
 *   - Calls are stream-ordered and never synchronise the stream (the _host
 *     variants synchronise once, to hand results back).
 *   - No persistent allocation behind the caller's back: scratch memory is a
 *     caller-owned workspace sized by the matching *_workspace_bytes().
 *   - Return value 0 = ok; non-zero = error, message via cnfot_last_error()
 *     (thread-local).  Nothing throws.
 *   - There is no CPU fallback: without a CUDA device every compute entry
 *     point fails with CNFOT_ERR_CUDA.
 */
#ifndef CNFOT_H_
#define CNFOT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CNFOT_API __attribute__((visibility("default")))
#else
#define CNFOT_API
#endif

#define CNFOT_ABI_VERSION 2

enum {
  CNFOT_OK = 0,
  CNFOT_ERR_ARG = 1,         /* bad argument / unsupported shape */
  CNFOT_ERR_CUDA = 2,        /* CUDA runtime error (incl. no device) */
  CNFOT_ERR_WORKSPACE = 3    /* workspace too small */
};

/* general.type of config/mfc.yaml (cnf_ot/mfc/solvers.py:58-88) */
enum { CNFOT_OT = 0, CNFOT_RWPO = 1, CNFOT_FP = 2 };
/* ot.subtype, rwpo.pot_type, fp.velocity_field_type */
enum { CNFOT_OT_FREE = 0, CNFOT_OT_OBSTACLE = 1 };
enum { CNFOT_POT_QUADRATIC = 0, CNFOT_POT_DOUBLE_WELL = 1 };
enum { CNFOT_FP_GRADIENT = 0, CNFOT_FP_NONGRADIENT = 1, CNFOT_FP_LORENZ = 2 };

/* Static shape of RQSFlow(event_shape=(dim,), num_layers, hidden_sizes=[hidden]*mlp_layers,
 * num_bins) -- cnf_ot/models/flows.py:178-199 -- plus the spline constants the
 * reference hard-codes at flows.py:124-132 (-10, 10, min_knot_slope 1e-4; min_bin_size
 * 1e-4 is the distrax default). */
typedef struct cnfot_flow_desc {
  int32_t dim;          /* general.dim            */
  int32_t num_layers;   /* cnf.flow_num_layers    */
  int32_t mlp_layers;   /* cnf.mlp_num_layers     */
  int32_t hidden;       /* cnf.hidden_size        */
  int32_t num_bins;     /* cnf.num_bins           */
  float range_min, range_max, min_bin_size, min_knot_slope;
} cnfot_flow_desc;

/* The loss selected by general.type and its hyper-parameters (config/mfc.yaml:6-27). */
typedef struct cnfot_problem_desc {
  int32_t type;     /* CNFOT_OT / CNFOT_RWPO / CNFOT_FP */
  int32_t subtype;  /* see enums above */
  float T;          /* rwpo.T / fp.T (ot uses 1) */
  float beta;       /* rwpo.beta (fp hard-codes 4, applications.py:432) */
  float a;          /* rwpo.a / fp.a */
  float sigma;      /* fp.sigma */
  float dt, dx;     /* general.dt, general.dx (fp hard-codes 0.01, applications.py:286,301) */
} cnfot_problem_desc;

CNFOT_API int cnfot_abi_version(void);
CNFOT_API const char* cnfot_last_error(void);
/* Launch configuration of the calling thread's most recent fused-kernel launch (diagnostics for
 * bench.py / profiles): persistent grid size, dynamic shared memory per CTA in bytes, resident
 * CTAs per SM the grid was sized for, and the conditioner engine that ran (0 CUDA cores,
 * 1 tcgen05 engine, 2 warp-level tensor-core engine, 4 wide-conditioner engine: batched tcgen05
 * GEMMs, the other three fields are 0). */
CNFOT_API void cnfot_last_launch_info(int32_t* grid, int32_t* smem_bytes, int32_t* ctas_per_sm,
                                      int32_t* tensor_cores);
/* Kernel instantiation of the calling thread's most recent fused call, when that call was a step or a VJP that
 * launched its kernel (diagnostics, tests).  plan: 0 CUDA cores, 1 tcgen05 engine, 2 warp-level tensor-core engine with
 * weights resident in shared memory, 3 the same streaming weights from the workspace, 4 wide-conditioner engine; -1 the
 * most recent call was another fused call (evaluation, energies, densities, on either engine), or a step or VJP that
 * launched no kernel (no rows, an argument error).  stash_tmem_cols: TMEM columns per CTA of the activation stash,
 * 0 = the backward pass recomputes.  kinetic_group: lanes per kinetic row of a step (1 = one thread per row), 0 for
 * anything but a step.  latency: 1 = the two-CTAs-per-SM instantiation of the streamed plan. */
CNFOT_API void cnfot_last_launch_variant(int32_t* plan, int32_t* stash_tmem_cols, int32_t* kinetic_group,
                                         int32_t* latency);
/* Diagnostics (tools/step_timeline.py): while `device_words` is non-NULL (8 uint64 in device memory, initialised by the
 * caller to {~0, 0, ~0, 0, 0, 0, 0, 0}) every fused train step records %globaltimer stamps there: [0] first CTA starts,
 * [1] last CTA finished its setup, [2] / [3] first / last CTA ran out of row tiles, [4] last CTA enters the
 * reduction tail, [5] last CTA leaves the kernel, [6] the longest per-CTA setup (a duration), [7] last CTA starts.  NULL switches it off (the default; process-wide, not thread-safe). */
CNFOT_API void cnfot_debug_step_timeline(void* device_words);

/* ---- parameter blob ---------------------------------------------------------------
 * The haiku pytree of SURVEY.md A.3 flattened into one fp32 buffer (layout documented in
 * DESIGN.md and cnf_ot_b200/csrc/flow_math.cuh).  Offsets are in floats. */
CNFOT_API int64_t cnfot_param_count(const cnfot_flow_desc* flow);               /* blob length */
CNFOT_API int64_t cnfot_spline_param_stride(const cnfot_flow_desc* flow);       /* Pp = roundup(3K+1, 4) */
CNFOT_API int64_t cnfot_offset_first(const cnfot_flow_desc* flow);              /* "~/first" */
/* linear m of "mlp_layer{l}_d{d}/~/linear_{m}" (0 <= m < mlp_layers) or, with
 * m == mlp_layers, "linear_out_layer{l}_d{d}"; bias != 0 selects "b" instead of "w". */
CNFOT_API int64_t cnfot_offset_linear(const cnfot_flow_desc* flow, int32_t layer, int32_t d, int32_t m,
                            int32_t bias);
/* 0 if the fused per-row kernels or the wide-conditioner engine support this shape, else
 * CNFOT_ERR_ARG (message says why). */
CNFOT_API int cnfot_flow_supported(const cnfot_flow_desc* flow);

/* ---- seam 2: one scalar spline per row (distrax.RationalQuadraticSpline) ------------
 * params: (rows, 3K+1) raw [K widths | K heights | K+1 slopes], replaces
 * bijector_fn(params).forward_and_log_det / inverse_and_log_det
 * (cnf_ot/models/flows.py:124-132, cnf_ot/models/autoregressive.py:100,130).
 * bin_idx (int32, may be NULL) receives the selected bin (0 in either tail). */
CNFOT_API int cnfot_rqs_forward(void* stream, const float* x, const float* params, int64_t rows,
                      int32_t num_bins, float range_min, float range_max, float min_bin_size,
                      float min_knot_slope, float* y, float* logdet, int32_t* bin_idx);
CNFOT_API int cnfot_rqs_inverse(void* stream, const float* y, const float* params, int64_t rows,
                      int32_t num_bins, float range_min, float range_max, float min_bin_size,
                      float min_knot_slope, float* x, float* logdet, int32_t* bin_idx);
/* Vector-Jacobian products of the two calls above: given the adjoints of (out, logdet)
 * returns the adjoint of the input (rows) and of params (rows, 3K+1). */
CNFOT_API int cnfot_rqs_forward_vjp(void* stream, const float* x, const float* params, const float* g_y,
                          const float* g_logdet, int64_t rows, int32_t num_bins, float range_min,
                          float range_max, float min_bin_size, float min_knot_slope, float* g_x,
                          float* g_params);
CNFOT_API int cnfot_rqs_inverse_vjp(void* stream, const float* y, const float* params, const float* g_x,
                          const float* g_logdet, int64_t rows, int32_t num_bins, float range_min,
                          float range_max, float min_bin_size, float min_knot_slope, float* g_y,
                          float* g_params);

/* ---- seam 1: the conditional flow (Flow namedtuple, cnf_ot/models/flows.py:213-226) --
 * cond is one time per row (cond_stride = 1, like the (N,1) `cond` of sample()) or a single
 * broadcast time (cond_stride = 0, like the (1,) `cond` of log_prob()).
 *   forward : flow.bijector.forward(_and_log_det)   latent -> physical  ("sample direction")
 *   inverse : flow.bijector.inverse(_and_log_det)   physical -> latent  ("log-prob direction")
 * logdet may be NULL.  With add_base != 0, `logdet` instead receives the log-density the
 * reference's ConditionalTransformed returns (cnf_ot/models/conditional.py:316-321,382-402):
 *   forward: log N(in) - fldj  (sample_and_log_prob)   inverse: log N(out) + ildj  (log_prob) */
CNFOT_API int cnfot_flow_forward(void* stream, const cnfot_flow_desc* flow, const float* weights,
                       const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                       float* out, float* logdet, int32_t add_base);
CNFOT_API int cnfot_flow_inverse(void* stream, const cnfot_flow_desc* flow, const float* weights,
                       const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                       float* out, float* logdet, int32_t add_base);
/* The same two calls with a caller-owned workspace of cnfot_flow_workspace_bytes(flow, rows) bytes
 * (0 for flows the fused per-row kernels cover).  Flows with wide conditioners (hidden a multiple of
 * 64, e.g. BASELINE config 5: dim 32, 16 layers, hidden 512) run on the wide-conditioner engine --
 * batched tcgen05 GEMMs over row chunks -- which needs scratch memory; for those the two calls
 * above fail with CNFOT_ERR_WORKSPACE and these must be used. */
CNFOT_API int64_t cnfot_flow_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows);
CNFOT_API int cnfot_flow_forward_ws(void* stream, const cnfot_flow_desc* flow, const float* weights,
                          const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                          float* out, float* logdet, int32_t add_base, void* workspace,
                          int64_t workspace_bytes);
CNFOT_API int cnfot_flow_inverse_ws(void* stream, const cnfot_flow_desc* flow, const float* weights,
                          const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                          float* out, float* logdet, int32_t add_base, void* workspace,
                          int64_t workspace_bytes);
/* VJPs of the two calls above (what a jax.custom_vjp backward rule calls): given g_out (rows,D)
 * and g_logdet (rows, may be NULL = zeros; it is the adjoint of the `logdet` OUTPUT, so it
 * honours add_base) writes g_in (rows,D, may be NULL) and writes the parameter gradient,
 * summed over rows, to g_weights (blob layout, overwritten). */
CNFOT_API int64_t cnfot_flow_vjp_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows);
CNFOT_API int cnfot_flow_forward_vjp(void* stream, const cnfot_flow_desc* flow, const float* weights,
                           const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                           const float* g_out, const float* g_logdet, int32_t add_base,
                           float* g_in, float* g_weights, void* workspace,
                           int64_t workspace_bytes);
CNFOT_API int cnfot_flow_inverse_vjp(void* stream, const cnfot_flow_desc* flow, const float* weights,
                           const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                           const float* g_out, const float* g_logdet, int32_t add_base,
                           float* g_in, float* g_weights, void* workspace,
                           int64_t workspace_bytes);

/* ---- seam 3: the train step's value_and_grad (cnf_ot/mfc/solvers.py:94) --------------
 * Evaluates loss_fn = ot_loss_fn / rwpo_loss_fn / fp_loss_fn
 * (cnf_ot/mfc/applications.py:377-441) and its gradient w.r.t. the parameter blob on this
 * GPU's shard of the batch.  Inputs replace the reference's PRNG draws:
 *   latent  (rows_B, D)  N(0,I) draws; the B//32 sub-batch terms use `latent_sub`
 *   latent_sub (rows_b, D)  this shard's rows of the b = B//32 sub-batch
 *   src, tgt (rows_B, D) data batches of kl_loss_fn (ot only; NULL otherwise)
 *   t_batch (n_t) on the HOST: the uniform times of applications.py:392,416,435
 * rows_B / rows_b are LOCAL row counts, global_B / global_b the whole-job counts used for
 * the means, so out buffers from different GPUs sum to the reference's result.
 * out: [ gradient (param_count) | loss slots (8) ] fp32, overwritten:
 *   slot 0 total loss, 1 fit term at t=0 (lambda-weighted), 2 fit term at t=T, 3 potential,
 *   4 kinetic; 5-7 reserved (zero). */
#define CNFOT_NUM_LOSS_SLOTS 8
CNFOT_API int64_t cnfot_mfc_step_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows_B,
                                       int64_t rows_b, int32_t n_t);
CNFOT_API int cnfot_mfc_step(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                   const float* weights, const float* latent, const float* latent_sub,
                   const float* src, const float* tgt, const float* t_batch_host, int32_t n_t,
                   int64_t rows_B, int64_t rows_b, int64_t global_B, int64_t global_b,
                   float lambda, float* out, void* workspace, int64_t workspace_bytes);
/* Persistent step workspace (optional): cnfot_workspace_register zero-initialises `workspace` (stream-ordered) and
 * records the pointer; from then on cnfot_mfc_step / _dp / _rng calls that are given this workspace skip their
 * per-call memset, because every step's reduction tail leaves the buffers clean for the next one -- two consecutive
 * steps are then two back-to-back kernel launches, and the second is scheduled (programmatic dependent launch) while
 * the first is still in its tail.  Contract: between cnfot_workspace_register and cnfot_workspace_release the memory
 * is only used by those calls, one stream at a time; a step that reported a peer time-out leaves it dirty (register
 * it again).  Not for the wide-conditioner engine.  cnfot_train_state (below) has the same property built in. */
CNFOT_API int cnfot_workspace_register(void* stream, const cnfot_flow_desc* flow, void* workspace, int64_t workspace_bytes);
CNFOT_API int cnfot_workspace_release(void* workspace);
/* ---- data-parallel step: the train step fused with its all-reduce (SURVEY.md section 8e) -------
 * Same as cnfot_mfc_step on this rank's shard, but the step kernel's tail also exchanges the
 * [gradient | loss slots] buffer with the peer GPUs of the node through peer-mapped memory
 * (NVLink / NVSwitch, no NCCL call, no second launch): on return (stream-ordered) `out` holds the SUM
 * over all ranks, bit-identical on every rank.  The caller owns the exchange memory and maps it across
 * processes (e.g. torch.distributed._symmetric_memory, CUDA IPC or VMM handles):
 *   xbuf[k]   rank k's exchange buffer, cnfot_dp_exchange_floats() floats (8-byte aligned), as addressable
 *             from THIS process (k == rank: the local allocation), zero-initialised once.  Every value travels
 *             as ONE 64-bit word {float bits, epoch}: an aligned 8-byte store arrives whole, so the data is its
 *             own arrival flag (no fence, no flag round trip: the latency of one NVLink write)
 *   flags[k]  rank k's flag words, cnfot_dp_flag_count() uint32, zero-initialised once (word 0: abort)
 *   epoch     1, 2, 3, ... : must increase by one per call, identically on all ranks
 * Every rank must make the call (an empty shard passes rows_B = rows_b = 0).  A peer that does not
 * arrive within CNFOT_DP_TIMEOUT_MS (environment, default 20000) makes the waiting rank fill `out` with
 * NaN, raise the abort word of EVERY rank's flag array (the late rank then reports NaN as well, and so
 * does every later call on these buffers: no rank continues with a sum the others do not have) and set
 * word CNFOT_STATUS_WORD of its workspace / train state to 1. */
typedef struct cnfot_peer_desc {
  int32_t rank, world;   /* world <= 8 (one node) */
  uint32_t epoch;        /* ignored by cnfot_mfc_update (the train state carries it) */
  float* xbuf[8];
  uint32_t* flags[8];
} cnfot_peer_desc;
#define CNFOT_STATUS_WORD 4   /* uint32 index into the workspace / train state: 0 ok, 1 a peer never arrived */
CNFOT_API int64_t cnfot_dp_exchange_stride(const cnfot_flow_desc* flow);
CNFOT_API int64_t cnfot_dp_exchange_floats(const cnfot_flow_desc* flow, int32_t world);
CNFOT_API int64_t cnfot_dp_flag_count(const cnfot_flow_desc* flow, int32_t world);
CNFOT_API int cnfot_mfc_step_dp(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                      const float* weights, const float* latent, const float* latent_sub,
                      const float* src, const float* tgt, const float* t_batch_host, int32_t n_t,
                      int64_t rows_B, int64_t rows_b, int64_t global_B, int64_t global_b,
                      float lambda, float* out, void* workspace, int64_t workspace_bytes,
                      const cnfot_peer_desc* peers);

/* ---- the step's random draws, made on chip -----------------------------------------------------------
 * The reference makes every draw of an `update` inside the jitted step from ONE key
 * (cnf_ot/mfc/applications.py:81-82,233-239,392,416,435; solvers.py:104-105).  Here a draw is a pure
 * function of (key, step, kind and leading size n of the drawn array, GLOBAL row, column) -- Philox4x32-10 keyed
 * with key ^ salt(kind, n), Box-Muller; cnf_ot_b200/csrc/philox.cuh -- so, like jax.random, arrays of different
 * shapes drawn from one key are unrelated and equal (key, shape) gives equal numbers; the step kernel
 * generates its rows itself (nothing crosses PCIe or HBM) and any shard is generated independently of how
 * the batch is split over GPUs.  jax.random's threefry streams are not reproduced.
 *   cnfot_philox_rows        rows [row0, row0 + rows) of the (global_rows, dim) array of that draw, as an array:
 *                            feed the explicit-input entries or a CPU check; 1 <= dim <= 255 (the widest flow
 *                            the wide-conditioner engine runs)
 *   cnfot_philox_times_host  the n_t uniform times horizon * U[0,1) of a step, computed on the host
 *   cnfot_mfc_step_rng       cnfot_mfc_step[_dp] (peers may be NULL) with the draws made inside the kernel:
 *                            latent / target rows = NORMAL (global_B, dim), source rows = OT_SOURCE (global_B, dim),
 *                            sub-batch latent = NORMAL (global_b, dim), times = n_t uniforms; this rank's shard is
 *                            rows [row0_B, row0_B + rows_B) of the B-row terms and [row0_b, row0_b + rows_b) of
 *                            the b-row terms
 *                            (both engines; the wide-conditioner engine draws straight into its chunk states and
 *                            refuses `peers`: its workspace is cnfot_mfc_step_workspace_bytes())
 *   cnfot_mfc_step_rng_host  the same with HOST weights in and HOST [gradient | loss] out (transfers inside,
 *                            synchronises): the key is the only other input (fused per-row kernels only) */
enum { CNFOT_ROWS_NORMAL = 1,     /* N(0, I) rows: latent draws and the target of kl_loss_fn (applications.py:73-82) */
       CNFOT_ROWS_OT_SOURCE = 3   /* kl_loss_fn source: z + 8-mode mixture centre (dim 2, applications.py:34-71), z - 3
                                     otherwise; z = the NORMAL draw of the same shape (the reference reuses the key) */ };
CNFOT_API int cnfot_philox_rows(void* stream, uint64_t key, uint32_t step, int32_t source, int64_t global_rows,
                      int64_t row0, int64_t rows, int32_t dim, float* out);
CNFOT_API int cnfot_philox_times_host(uint64_t key, uint32_t step, int32_t n_t, float horizon, float* t_host);
CNFOT_API int cnfot_mfc_step_rng(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                       const float* weights, uint64_t key, uint32_t step, int32_t n_t, int64_t row0_B,
                       int64_t rows_B, int64_t row0_b, int64_t rows_b, int64_t global_B, int64_t global_b,
                       float lambda, float* out, void* workspace, int64_t workspace_bytes,
                       const cnfot_peer_desc* peers);
CNFOT_API int64_t cnfot_mfc_step_rng_host_workspace_bytes(const cnfot_flow_desc* flow);
CNFOT_API int cnfot_mfc_step_rng_host(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                            const float* weights_host, uint64_t key, uint32_t step, int32_t n_t, int64_t row0_B,
                            int64_t rows_B, int64_t row0_b, int64_t rows_b, int64_t global_B, int64_t global_b,
                            float lambda, float* out_host, void* workspace, int64_t workspace_bytes);

/* ---- device-resident update: `update` of cnf_ot/mfc/solvers.py:90-97 as ONE kernel launch -----------------
 * value_and_grad with on-chip draws + (peers) the all-reduce + optax.adam, all inside the step kernel; no host
 * data enters the call after cnfot_train_state_init, so a sequence of calls can be captured in a CUDA graph
 * and replayed (the 30 000-step loop of solvers.py:99-106).  The train state (device memory owned by the caller,
 * cnfot_train_state_bytes()) carries the key, the step count (starts at `step`, +1 per call: it selects the
 * draws, Adam's bias correction and the slot of loss_hist) and the all-reduce epoch, plus the kernel's
 * self-cleaning reduction buffers.  out (may be NULL): [gradient | loss slots] of the step; loss_hist (may be
 * NULL): loss_hist[step] = total loss when step < loss_hist_len.  weights, adam_m, adam_v are updated in place.
 * Flows on the wide-conditioner engine take the same calls: the update is then a sequence of stream-ordered launches
 * (draws made by the chunk-state initialisation, the engine's step, an Adam kernel, a one-thread step advance) with no
 * host synchronisation and no host-memory read, so it is captured like the fused one -- provided one update has run
 * on the device OUTSIDE a capture first (it sets the kernels' shared-memory limits, which a capture must not be the
 * first to do).  Their train state holds the step's gradient and workspace as well, so its size depends on the row
 * counts: cnfot_train_state_bytes_rows(flow, rows_B, rows_b) (this shard's rows; equal to cnfot_train_state_bytes() for
 * the fused kernels, which returns -1 for wide flows); no `peers` (all-reduce the gradient of cnfot_mfc_step with NCCL). */
typedef struct cnfot_adam_desc { float lr, b1, b2, eps; } cnfot_adam_desc;   /* optax.adam defaults: b1 .9 b2 .999 eps 1e-8 */
CNFOT_API int64_t cnfot_train_state_bytes(const cnfot_flow_desc* flow);
CNFOT_API int64_t cnfot_train_state_bytes_rows(const cnfot_flow_desc* flow, int64_t rows_B, int64_t rows_b);
CNFOT_API int cnfot_train_state_init(void* stream, const cnfot_flow_desc* flow, void* state, int64_t state_bytes,
                           uint64_t key, uint64_t step, uint32_t epoch);
CNFOT_API int cnfot_mfc_update(void* stream, const cnfot_flow_desc* flow, const cnfot_problem_desc* problem,
                     void* state, int64_t state_bytes, float* weights, float* adam_m, float* adam_v,
                     const cnfot_adam_desc* adam, int32_t n_t, int64_t row0_B, int64_t rows_B, int64_t row0_b,
                     int64_t rows_b, int64_t global_B, int64_t global_b, float lambda, float* out,
                     float* loss_hist, int64_t loss_hist_len, const cnfot_peer_desc* peers);

/* Same step with HOST buffers in and out (weights, latent, latent_sub, src, tgt, out are host
 * pointers): copies inputs to the device workspace, runs the step, copies `out` back and
 * synchronises the stream.  The workspace must be
 * cnfot_mfc_step_host_workspace_bytes() of DEVICE memory. */
CNFOT_API int64_t cnfot_mfc_step_host_workspace_bytes(const cnfot_flow_desc* flow, int64_t rows_B,
                                            int64_t rows_b, int32_t n_t);
CNFOT_API int cnfot_mfc_step_host(void* stream, const cnfot_flow_desc* flow,
                        const cnfot_problem_desc* problem, const float* weights_host,
                        const float* latent_host, const float* latent_sub_host,
                        const float* src_host, const float* tgt_host, const float* t_batch_host,
                        int32_t n_t, int64_t rows_B, int64_t rows_b, int64_t global_B,
                        int64_t global_b, float lambda, float* out_host, void* workspace,
                        int64_t workspace_bytes);

/* ---- evaluation energies (the callers after the step: cnf_ot/mfc/solvers.py:141-164) ------
 * utils.calc_kinetic_energy (cnf_ot/utils.py:311-340; with_score = 0) and
 * utils.calc_score_kinetic_energy (cnf_ot/utils.py:343-389; with_score != 0, kappa = 1/beta) as ONE
 * forward-only kernel over the whole time grid:
 *   out[0] = (1/n_t) sum_t mean_{rows,dims}(v_t^2) / 2 * dim,
 *   v_t = (r(t+dt/2) - r(t-dt/2)) / dt  [+ kappa * score_t, score by central differences of
 *   log_prob with step dx], r(.) = the flow's samples of the SAME latent rows.
 * latent: (latent_blocks * batch, D); time index i uses block i % latent_blocks (the reference
 * draws a fresh batch per time: latent_blocks = n_t; 1 reuses one batch).  t_host: n_t times on
 * the host.  out: ONE double on the device.  The multiplication by T the rwpo caller applies
 * (solvers.py:154) is left to the caller. */
CNFOT_API int64_t cnfot_kinetic_energy_workspace_bytes(const cnfot_flow_desc* flow, int32_t n_t);
CNFOT_API int cnfot_kinetic_energy(void* stream, const cnfot_flow_desc* flow, const float* weights,
                         const float* latent, int64_t batch, int32_t latent_blocks, const float* t_host,
                         int32_t n_t, float dt, int32_t with_score, float kappa, float dx, double* out,
                         void* workspace, int64_t workspace_bytes);

/* ---- densities on a grid / at Monte-Carlo samples (SURVEY.md 8f row 3): the consumers of log_prob_fn and
 * sample_and_log_prob after training -------------------------------------------------------------------------
 *   cnfot_density_grid  density[(ti, iy, ix)] = exp(log_prob(params, (x_ix, y_iy), cond = t_ti)) on the grid
 *                       XY = hstack(meshgrid(linspace(x_min, x_max, nx), linspace(y_min, y_max, ny))) for n_t times in ONE
 *                       launch, the grid generated in the kernel: utils.plot_density_snapshot / plot_density_and_trajectory
 *                       (cnf_ot/utils.py:572-642), the double-well density at T (cnf_ot/mfc/solvers.py:184-222) and
 *                       rmse_grid_loss_fn (solvers.py:282-301).  dim must be 2.  density: (n_t, ny, nx) floats or NULL.
 *   cnfot_density_mc    samples, log_prob = sample_and_log_prob(cond, seed) for n rows whose latent is the NORMAL (n, dim)
 *                       draw of (key, step) made on chip (cnfot_philox_rows gives the same rows): rmse_mc_loss_fn
 *                       (solvers.py:254-278).  samples: (n, dim) or NULL; density: (n) exp(log_prob) or NULL.
 * with_ref != 0: *sq_err (ONE double on the device) = sum over the points of
 *   (density - ((1 - mix) N(y; 0, var0 I) + mix N(y; 0, var1 I)))^2       (solvers.py:238-252,270-276,296-299);
 * the caller takes sqrt(sq_err / points).
 * Both engines run these calls: the fused kernels in one launch, flows with wide conditioners chunk by chunk on the
 * wide-conditioner engine (cnfot_last_launch_info reports engine 4).  Workspace: for the fused kernels the per-CTA
 * partial sums and the n_t times; for wide flows the chunk buffers of one flow pass and the n_t times -- independent of
 * the number of points (n_t = 0 for cnfot_density_mc). */
CNFOT_API int64_t cnfot_density_workspace_bytes(const cnfot_flow_desc* flow, int32_t n_t);
CNFOT_API int cnfot_density_grid(void* stream, const cnfot_flow_desc* flow, const float* weights, const float* t_host,
                       int32_t n_t, double x_min, double x_max, double y_min, double y_max, int32_t nx, int32_t ny,
                       float* density, int32_t with_ref, float mix, float var0, float var1, double* sq_err,
                       void* workspace, int64_t workspace_bytes);
CNFOT_API int cnfot_density_mc(void* stream, const cnfot_flow_desc* flow, const float* weights, float cond, uint64_t key,
                     uint32_t step, int64_t n, float* samples, float* density, int32_t with_ref, float mix, float var0,
                     float var1, double* sq_err, void* workspace, int64_t workspace_bytes);

/* ---- wide conditioner layers on tcgen05 (BASELINE config 5: hidden = 512) -----------------------
 * Y (rows x N) = epilogue(X (rows x K) * W (K x N) [+ bias]), fp32 in / out with fp32 fidelity (3xTF32):
 * the dense layers of the conditioner MLP (cnf_ot/models/flows.py:65-81) and, with transpose != 0 at
 * prepare time, their data gradients (G * W^T).  tcgen05.mma.kind::tf32 with the accumulator in TMEM,
 * weights staged by 1-D bulk TMA copies from a buffer prepared once per weight update:
 *   cnfot_dense_prepare      W (row stride ldw) -> `prepared` (cnfot_dense_prepared_floats(K, N) floats);
 *                            transpose != 0 prepares W^T, i.e. W is then (N x K) and the call computes X * W^T
 *   cnfot_dense_forward      epilogue 0: + bias, 1: + bias then ReLU, 2: ReLU mask (Y = mask_src > 0 ? acc : 0,
 *                            mask_src (rows x N, row stride ldm)), 3: none, 4: accumulate (Y += X * W)
 * K and N must be multiples of 16; ldx, ldy, ldm multiples of 4. */
CNFOT_API int64_t cnfot_dense_prepared_floats(int32_t K, int32_t N);
CNFOT_API int cnfot_dense_prepare(void* stream, const float* W, int32_t K, int32_t N, int32_t ldw,
                        int32_t transpose, float* prepared);
CNFOT_API int cnfot_dense_forward(void* stream, const float* X, int64_t rows, int32_t K, int32_t ldx,
                        const float* prepared, int32_t N, const float* bias, const float* mask_src,
                        int32_t ldm, int32_t epilogue, float* Y, int32_t ldy);
/* Weight gradient of the same layer, ACCUMULATED: dW (Ka x Nb, row stride ldw) += A^T G over `rows` rows
 * (A (rows x Ka, stride lda) the layer input, G (rows x Nb, stride ldg) the adjoint of its
 * pre-activation), db (Nb, may be NULL) += column sums of G.  tcgen05 with both operands gathered
 * K-major (sample rows contiguous) by the CTA, 3xTF32, split over row ranges, red.global adds. */
CNFOT_API int cnfot_dense_wgrad(void* stream, const float* A, int32_t lda, const float* G, int32_t ldg,
                      int64_t rows, int32_t Ka, int32_t Nb, float* dW, int32_t ldw, float* db);

/* ---- dimension-reduction loss (SURVEY.md 8f row 4; cnf_ot/dr/trainers.py:91-111) -------------------------
 * loss_fn(params, x) = mean_rows sum_dims (x - decoder.forward(mask(encoder.forward(x))))^2 with UNCONDITIONAL
 * flows (cond_shape = (0,), trainers.py:41-68).  The flows are the cnfot_flow_* calls above on a blob whose
 * t-rows (row 0 of every input matrix) are zero, with cond = 0; these two calls are the glue between them:
 *   cnfot_mask_tail    y[:, sub_dim:] = 0                                   (trainers.py:95,108)
 *   cnfot_recon_head   *loss += weight * sum (x - xr)^2, g_xr = -2 weight (x - xr)    (trainers.py:97,110;
 *                      weight = 1 / global rows; loss: one double on the device, zeroed by the caller) */
CNFOT_API int cnfot_mask_tail(void* stream, float* y, int64_t rows, int32_t dim, int32_t sub_dim);
CNFOT_API int cnfot_recon_head(void* stream, const float* x, const float* xr, int64_t rows, int32_t dim,
                     float weight, float* g_xr, double* loss);

/* optax.adam(lr) defaults b1=0.9 b2=0.999 eps=1e-8 (cnf_ot/mfc/solvers.py:55,95-96), fused
 * element-wise update; step is the 1-based update count. */
CNFOT_API int cnfot_adam_update(void* stream, float* params, const float* grads, float* m, float* v,
                      int64_t count, float lr, float b1, float b2, float eps, int64_t step);

#ifdef __cplusplus
}
#endif
#endif /* CNFOT_H_ */
