// Lookup of the fused train-step kernel; the instantiations live in step_<engine>.cu (one translation unit per
// conditioner engine, so they compile in parallel).
#include "dispatch.h"
#include "flow_kernels.cuh"

namespace cnfot {

const void* find_mfc_step_kernel_tc(const FlowLayout& f);
const void* find_mfc_step_kernel_mma(const FlowLayout& f, bool stash);
const void* find_mfc_step_kernel_mma_stream(const FlowLayout& f);
const void* find_mfc_step_kernel_cuda(const FlowLayout& f);
const void* find_mfc_step_kernel_tc_split(const FlowLayout& f);
const void* find_mfc_step_kernel_mma_split(const FlowLayout& f, bool stash);
const void* find_mfc_step_kernel_mma_stream_split(const FlowLayout& f);
const void* find_mfc_step_kernel_mma_stream_lat(const FlowLayout& f);
const void* find_mfc_step_kernel_cuda_split(const FlowLayout& f);

const void* find_mfc_step_kernel(const FlowLayout& f, int engine, bool split, bool latency, bool stash) {
  if (engine == kEngTc && tc_available(f)) return split ? find_mfc_step_kernel_tc_split(f) : find_mfc_step_kernel_tc(f);
  if (engine == kEngMma && tc_available(f))
    return split ? find_mfc_step_kernel_mma_split(f, stash) : find_mfc_step_kernel_mma(f, stash);
  if (engine == kEngMmaStream && tc_available(f))
    return split ? find_mfc_step_kernel_mma_stream_split(f)
                 : (latency ? find_mfc_step_kernel_mma_stream_lat(f) : find_mfc_step_kernel_mma_stream(f));
  return split ? find_mfc_step_kernel_cuda_split(f) : find_mfc_step_kernel_cuda(f);
}

}  // namespace cnfot
