// Kernel lookup: (hidden, bins, mlp layers, dim, layers) -> compiled kernel.
#pragma once

#include "flow_math.cuh"

namespace cnfot {

// Each returns the __global__ function to pass to cudaLaunchKernel, or nullptr
// when no instantiation exists for the network shape.  Shapes with a
// compile-time (dim, layers) specialisation keep the per-row state in registers;
// all others use the runtime-shape kernel (state in local memory).
// engine: 0 CUDA cores, 1 tcgen05 (tc_engine.cuh), 2 warp-level MMA with weights + fragments resident in
// shared memory (warp_mlp.cuh), 3 warp-level MMA streaming them from global memory; engines 1-3 exist
// for hidden == 16 and num_bins == 5 only (tc_available()).
const void* find_flow_eval_kernel(const FlowLayout& f, int engine = 0);
// stash (engine 2 only): the instantiation that keeps the activation stash in tensor memory (warp_mlp.cuh)
const void* find_flow_vjp_kernel(const FlowLayout& f, int engine = 0, bool stash = false);
// split: flow_kernels.cuh SPLIT; latency: the two-CTAs-per-SM instantiation of the streamed plan (LAT)
const void* find_mfc_step_kernel(const FlowLayout& f, int engine = 0, bool split = false, bool latency = false,
                                 bool stash = false);
const void* find_energy_kernel(const FlowLayout& f, int engine = 0);
const void* find_density_kernel(const FlowLayout& f, int engine = 0);
inline bool tc_available(const FlowLayout& f) { return f.H == 16 && f.K == 5 && f.D >= 2 && f.M <= 3; }

// (hidden, bins, mlp layers) combinations compiled into the fused kernels.
#define CNFOT_NET_LIST(X) \
  X(16, 5, 2)             \
  X(16, 5, 1)             \
  X(16, 5, 3)             \
  X(32, 8, 2)             \
  X(32, 5, 2)             \
  X(64, 5, 2)             \
  X(8, 3, 1)

}  // namespace cnfot
