// Shared helpers for the fdm_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include "fdm_b200.h"

namespace fdm {

void set_last_error(cudaError_t e);

inline int check_launch() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_last_error(e);
    return FDM_ERR_CUDA;
  }
  return FDM_OK;
}

#define FDM_REQUIRE(cond, code) \
  do {                          \
    if (!(cond)) return (code); \
  } while (0)

__device__ __forceinline__ float silu_f(float v) { return __fdividef(v, 1.0f + __expf(-v)); }

// exact-ish sigmoid for the fp32 parity mode (expf, not __expf): used where 1e-4 end-to-end matters
__device__ __forceinline__ float silu_precise(float v) { return v / (1.0f + expf(-v)); }

template <typename T>
struct OpType;
template <>
struct OpType<float> {
  static __device__ __forceinline__ float load(const float* p) { return *p; }
  static __device__ __forceinline__ void store(float* p, float v) { *p = v; }
  static __device__ __forceinline__ float4 load4(const float* p) { return *reinterpret_cast<const float4*>(p); }
  static __device__ __forceinline__ void store4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
};
template <>
struct OpType<__nv_bfloat16> {
  static __device__ __forceinline__ float load(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float4 load4(const __nv_bfloat16* p) {
    uint2 u = *reinterpret_cast<const uint2*>(p);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&u.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&u.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
  }
  static __device__ __forceinline__ void store4(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&a);
    u.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = u;
  }
};

// ---- programmatic dependent launch (PDL).  Every kernel of the library is launched with the programmatic-stream-
// serialization attribute and calls pdl_wait() before it touches global memory: it blocks until the PREVIOUS kernel of the
// stream has completed and its writes are visible, then releases the NEXT kernel.  The release comes after the wait, not at
// kernel start, so a kernel that is itself still waiting never releases its successor: the next kernel becomes resident
// (TMEM allocation, barrier init, tensor-map prefetch) during this grid's last wave, at most one kernel deep.  DESIGN.md has
// the measurements.  FDM_PDL=0 disables the attribute.
__device__ __forceinline__ void pdl_wait_only() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() {
  pdl_wait_only();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

bool pdl_enabled();  // api.cu

template <typename... KArgs, typename... Args>
inline void launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// the same with thread-block clusters of `cluster` CTAs along x (CTA pairs of the cta_group::2 kernels)
template <typename... KArgs, typename... Args>
inline void launch_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace fdm
