// Host-side interface of the wide-conditioner engine (wide.cu): flows whose conditioner MLPs do not fit
// the fused per-row kernels (hidden a multiple of 64, e.g. BASELINE config 5: D = 32, L = 16, H = 512).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "flow_math.cuh"
#include "philox.cuh"
#include "step_math.cuh"

namespace cnfot {

// Largest dim the engine takes: a state row [x | t | 0 ..] is then at most 256 columns, one N = 256 tile of the
// input-adjoint GEMM.  cnfot_philox_rows draws rows of every dim up to this bound.
constexpr int kWideMaxDim = 255;

bool wide_supported(const FlowLayout& lay, const char** why);
// workspace: prepared weights (2 x 2 x every matrix) + the chunk buffers
int64_t wide_step_workspace_bytes(const FlowLayout& lay, int64_t rows_B, int64_t rows_b);
int64_t wide_flow_workspace_bytes(const FlowLayout& lay, int64_t rows, bool with_grad);

// The step's draws made on chip, the numbers of the fused step kernel (philox.cuh): key and step by value, or, with
// `state` != NULL, read by the kernels from the train state's words [key, step] (a captured launch then draws the rows of
// whichever update it runs as); salts = step_salts(global_B, global_b, n_t); row0_*: global index of the shard's first row
struct WideDraws {
  uint64_t key;
  uint32_t step;
  const unsigned long long* state;
  StepSalts salts;
  int64_t row0_B, row0_b;
};
// The device-resident update's tail: optax.adam with the step's gradient on weights / m / v in place, for update number
// state[1]; loss_hist[state[1]] = total loss when state[1] < loss_hist_len; then state[1] and the epoch state[2] advance
struct WideAdam {
  unsigned long long* state;
  float* weights;
  float* m;
  float* v;
  float lr, b1, b2, eps;
  float* loss_hist;
  int64_t loss_hist_len;
};

// value_and_grad of ot_loss_fn / rwpo_loss_fn / fp_loss_fn on this shard: out = [gradient (blob) | 8 loss slots], overwritten.
// Rows and times: the explicit arrays, or (draws != NULL) drawn on chip; adam != NULL: the update's tail follows
cudaError_t wide_mfc_step(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const StepConsts<float>& pc,
                          const float* weights, const float* latent, const float* latent_sub, const float* src,
                          const float* tgt, const float* t_batch_host, const WideDraws* draws, int n_t, int64_t rows_B,
                          int64_t rows_b, float* out, const WideAdam* adam, void* workspace, const char** what);
// flow.bijector.forward / inverse (dir 0 / 1) with log-det (or the density with add_base)
cudaError_t wide_flow_eval(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                           int dir, const float* in, const float* cond, int64_t cond_stride, int64_t rows, float* out,
                           float* logdet, int add_base, void* workspace, const char** what);
cudaError_t wide_flow_vjp(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                          int dir, const float* in, const float* cond, int64_t cond_stride, int64_t rows,
                          const float* g_out, const float* g_logdet, int add_base, float* g_in, float* g_weights,
                          void* workspace, const char** what);

// utils.calc_kinetic_energy / calc_score_kinetic_energy over a time grid (forward only); out: one double on the device
int64_t wide_energy_workspace_bytes(const FlowLayout& lay);
cudaError_t wide_kinetic_energy(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                                const float* latent, int64_t batch, int latent_blocks, const float* t_host, int n_t, float dt,
                                int with_score, float kappa, float dx, double* out, void* workspace, const char** what);

// cnfot_density_grid / cnfot_density_mc (density_kernel of flow_kernels.cuh), chunk by chunk: density = exp(log_prob) of
// every point (may be NULL) and, with_ref, the summed squared error against (1 - mix) N(0, var0 I) + mix N(0, var1 I)
// into sq_err (one double on the device).  Workspace: the chunk buffers (independent of the number of points) and the
// n_t grid times.
int64_t wide_density_workspace_bytes(const FlowLayout& lay, int n_t);
// grid: the nx x ny points (x_min + ix x_step, y_min + iy y_step) at each of the n_t times, density[(ti, iy, ix)]
cudaError_t wide_density_grid(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                              const float* t_host, int n_t, double x_min, double x_step, double y_min, double y_step, int nx,
                              int ny, float* density, int with_ref, float mix, float var0, float var1, double* sq_err,
                              void* workspace, const char** what);
// Monte-Carlo: samples (n x D, may be NULL) and densities of sample_and_log_prob at time `cond` for rows [0, n) of the
// NORMAL (n, D) draw of (key_n = key ^ philox_salt(kDrawNormal, n), step)
cudaError_t wide_density_mc(cudaStream_t s, const FlowLayout& lay, const SplineConsts<float>& sc, const float* weights,
                            float cond, uint64_t key_n, uint32_t step, int64_t n, float* samples, float* density,
                            int with_ref, float mix, float var0, float var1, double* sq_err, void* workspace,
                            const char** what);

}  // namespace cnfot
