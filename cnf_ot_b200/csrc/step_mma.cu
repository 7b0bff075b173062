// Instantiations of the fused train-step kernel: the warp-level tensor-core engine, weights + fragments resident in shared memory (warp_mlp.cuh).
// CNFOT_STEP_SPLIT (step_mma_split.cu): the instantiations whose kinetic rows are spread over lane groups.
#ifndef CNFOT_STEP_SPLIT
#define CNFOT_STEP_SPLIT 0
#endif
#include "dispatch.h"
#include "flow_kernels.cuh"

namespace cnfot {

#define STEP_ENG_CASE(M_, E_) \
  if (f.M == M_) return (const void*)&mfc_step_kernel<NetCfg<16, 5, M_>, Dims<0, 0>, E_, CNFOT_STEP_SPLIT != 0>;

// stash: the instantiation with the activation stash in tensor memory (kEngMmaStash)
#if CNFOT_STEP_SPLIT
const void* find_mfc_step_kernel_mma_split(const FlowLayout& f, bool stash) {
#else
const void* find_mfc_step_kernel_mma(const FlowLayout& f, bool stash) {
#endif
  if (stash) {
    if (f.M == 2 && f.D == 2 && f.L == 2)
      return (const void*)&mfc_step_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMmaStash, CNFOT_STEP_SPLIT != 0>;
    STEP_ENG_CASE(1, kEngMmaStash) STEP_ENG_CASE(2, kEngMmaStash) STEP_ENG_CASE(3, kEngMmaStash)
    return nullptr;
  }
  if (f.M == 2 && f.D == 2 && f.L == 2)
    return (const void*)&mfc_step_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMma, CNFOT_STEP_SPLIT != 0>;
  STEP_ENG_CASE(1, kEngMma) STEP_ENG_CASE(2, kEngMma) STEP_ENG_CASE(3, kEngMma)
  return nullptr;
}

}  // namespace cnfot
