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

// Philox4x32-10 (Salmon et al. 2011; the counter-based generator cuRAND / PyTorch use): 4 x 32 random bits per (counter, key).
// Shared by the sampler's in-kernel noise (fdm_ddpm_step) and the ResBlock dropout mask (fdm_gn_apply / fdm_gn_bwd).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// ResBlock dropout (the nn.Dropout between SiLU and the second conv): the keep mask of the four channels c..c+3 of one
// [N][HW][C] element quad, first element index `o`, regenerated bit for bit by the GroupNorm backward (include/fdm_b200.h).
struct DropMask {
  uint2 key;             // seed = philox[0]
  uint32_t salt, nonce;  // per-launch salt, step nonce = low word of philox[1]
  uint32_t thr;          // keep iff the 32-bit draw >= thr = min(ceil(p * 2^32), 2^32 - 1)
  float scale;           // 1 / (1 - p); 0 for p = 1
  __device__ __forceinline__ void apply(size_t o, float* v) const {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)o, (uint32_t)((unsigned long long)o >> 32), salt, nonce), key);
    v[0] = r.x >= thr ? v[0] * scale : 0.f;
    v[1] = r.y >= thr ? v[1] * scale : 0.f;
    v[2] = r.z >= thr ? v[2] * scale : 0.f;
    v[3] = r.w >= thr ? v[3] * scale : 0.f;
  }
};

// host: the mask parameters of (philox, p, salt); the seed / nonce words are read on the device at run time
struct DropArgs {
  const unsigned long long* philox;
  uint32_t salt, thr;
  float scale;
};

inline DropArgs drop_args(const uint64_t* philox, float p, int32_t salt) {
  DropArgs d{reinterpret_cast<const unsigned long long*>(philox), (uint32_t)salt, 0u, 1.f};
  if (p < 1.f) {
    d.thr = (uint32_t)fmin(ceil((double)p * 4294967296.0), 4294967295.0);
    d.scale = (float)(1.0 / (1.0 - (double)p));
  } else {
    d.thr = 0xffffffffu;
    d.scale = 0.f;
  }
  return d;
}

__device__ __forceinline__ DropMask load_drop_mask(const DropArgs& d) {
  const unsigned long long seed = d.philox[0], nonce = d.philox[1];
  return DropMask{make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), d.salt, (uint32_t)nonce, d.thr, d.scale};
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace fdm
