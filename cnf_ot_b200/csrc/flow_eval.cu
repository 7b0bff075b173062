// Instantiations of the forward-only and VJP flow kernels.
#include "dispatch.h"
#include "flow_kernels.cuh"

namespace cnfot {

#define EVAL_CASE(H_, K_, M_)                                                            \
  if (f.H == H_ && f.K == K_ && f.M == M_)                                               \
    return (const void*)&flow_eval_kernel<NetCfg<H_, K_, M_>, Dims<0, 0>, kEngCuda>;
#define VJP_CASE(H_, K_, M_)                                                             \
  if (f.H == H_ && f.K == K_ && f.M == M_)                                               \
    return (const void*)&flow_vjp_kernel<NetCfg<H_, K_, M_>, Dims<0, 0>, kEngCuda>;
#define EVAL_ENG_CASE(M_, E_)                                                            \
  if (f.M == M_) return (const void*)&flow_eval_kernel<NetCfg<16, 5, M_>, Dims<0, 0>, E_>;
#define VJP_ENG_CASE(M_, E_)                                                             \
  if (f.M == M_) return (const void*)&flow_vjp_kernel<NetCfg<16, 5, M_>, Dims<0, 0>, E_>;

const void* find_flow_eval_kernel(const FlowLayout& f, int engine) {
  if (engine == kEngTc && tc_available(f)) {
    EVAL_ENG_CASE(1, kEngTc) EVAL_ENG_CASE(2, kEngTc) EVAL_ENG_CASE(3, kEngTc)
    return nullptr;
  }
  if (engine == kEngMma && tc_available(f)) {
    if (f.M == 2 && f.D == 2 && f.L == 2)
      return (const void*)&flow_eval_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMma>;
    EVAL_ENG_CASE(1, kEngMma) EVAL_ENG_CASE(2, kEngMma) EVAL_ENG_CASE(3, kEngMma)
    return nullptr;
  }
  if (engine == kEngMmaStream && tc_available(f)) {
    EVAL_ENG_CASE(1, kEngMmaStream) EVAL_ENG_CASE(2, kEngMmaStream) EVAL_ENG_CASE(3, kEngMmaStream)
    return nullptr;
  }
  if (f.H == 16 && f.K == 5 && f.M == 2 && f.D == 2 && f.L == 2)
    return (const void*)&flow_eval_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngCuda>;
  CNFOT_NET_LIST(EVAL_CASE)
  return nullptr;
}

const void* find_flow_vjp_kernel(const FlowLayout& f, int engine, bool stash) {
  if (engine == kEngTc && tc_available(f)) {
    VJP_ENG_CASE(1, kEngTc) VJP_ENG_CASE(2, kEngTc) VJP_ENG_CASE(3, kEngTc)
    return nullptr;
  }
  if (engine == kEngMma && tc_available(f) && stash) {
    if (f.M == 2 && f.D == 2 && f.L == 2)
      return (const void*)&flow_vjp_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMmaStash>;
    VJP_ENG_CASE(1, kEngMmaStash) VJP_ENG_CASE(2, kEngMmaStash) VJP_ENG_CASE(3, kEngMmaStash)
    return nullptr;
  }
  if (engine == kEngMma && tc_available(f)) {
    if (f.M == 2 && f.D == 2 && f.L == 2)
      return (const void*)&flow_vjp_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMma>;
    VJP_ENG_CASE(1, kEngMma) VJP_ENG_CASE(2, kEngMma) VJP_ENG_CASE(3, kEngMma)
    return nullptr;
  }
  if (engine == kEngMmaStream && tc_available(f)) {
    VJP_ENG_CASE(1, kEngMmaStream) VJP_ENG_CASE(2, kEngMmaStream) VJP_ENG_CASE(3, kEngMmaStream)
    return nullptr;
  }
  if (f.H == 16 && f.K == 5 && f.M == 2 && f.D == 2 && f.L == 2)
    return (const void*)&flow_vjp_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngCuda>;
  CNFOT_NET_LIST(VJP_CASE)
  return nullptr;
}

#define ENERGY_CASE(H_, K_, M_)                                                          \
  if (f.H == H_ && f.K == K_ && f.M == M_)                                               \
    return (const void*)&energy_kernel<NetCfg<H_, K_, M_>, Dims<0, 0>, kEngCuda>;
#define ENERGY_ENG_CASE(M_, E_)                                                          \
  if (f.M == M_) return (const void*)&energy_kernel<NetCfg<16, 5, M_>, Dims<0, 0>, E_>;

const void* find_energy_kernel(const FlowLayout& f, int engine) {
  if (engine == kEngMma && tc_available(f)) {
    if (f.M == 2 && f.D == 2 && f.L == 2)
      return (const void*)&energy_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMma>;
    ENERGY_ENG_CASE(1, kEngMma) ENERGY_ENG_CASE(2, kEngMma) ENERGY_ENG_CASE(3, kEngMma)
    return nullptr;
  }
  if (engine == kEngMmaStream && tc_available(f)) {
    ENERGY_ENG_CASE(1, kEngMmaStream) ENERGY_ENG_CASE(2, kEngMmaStream) ENERGY_ENG_CASE(3, kEngMmaStream)
    return nullptr;
  }
  CNFOT_NET_LIST(ENERGY_CASE)
  return nullptr;
}

#define DENSITY_CASE(H_, K_, M_)                                                         \
  if (f.H == H_ && f.K == K_ && f.M == M_)                                               \
    return (const void*)&density_kernel<NetCfg<H_, K_, M_>, Dims<0, 0>, kEngCuda>;
#define DENSITY_ENG_CASE(M_, E_)                                                         \
  if (f.M == M_) return (const void*)&density_kernel<NetCfg<16, 5, M_>, Dims<0, 0>, E_>;

const void* find_density_kernel(const FlowLayout& f, int engine) {
  if (engine == kEngMma && tc_available(f)) {
    if (f.M == 2 && f.D == 2 && f.L == 2)
      return (const void*)&density_kernel<NetCfg<16, 5, 2>, Dims<2, 2>, kEngMma>;
    DENSITY_ENG_CASE(1, kEngMma) DENSITY_ENG_CASE(2, kEngMma) DENSITY_ENG_CASE(3, kEngMma)
    return nullptr;
  }
  if (engine == kEngMmaStream && tc_available(f)) {
    DENSITY_ENG_CASE(1, kEngMmaStream) DENSITY_ENG_CASE(2, kEngMmaStream) DENSITY_ENG_CASE(3, kEngMmaStream)
    return nullptr;
  }
  CNFOT_NET_LIST(DENSITY_CASE)
  return nullptr;
}

}  // namespace cnfot
