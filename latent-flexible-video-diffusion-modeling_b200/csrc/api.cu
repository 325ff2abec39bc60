// C-ABI housekeeping: version, status strings, struct sizes (so the ctypes mirror can be verified on CPU); the tensor-map encoder.
#include "tc_common.cuh"
#include <cudaTypedefs.h>
#include <string.h>
#include <stdlib.h>

namespace fdm {
static thread_local char g_last_err[256] = "";
void set_last_error(cudaError_t e) {
  const char* s = cudaGetErrorString(e);
  strncpy(g_last_err, s ? s : "unknown", sizeof(g_last_err) - 1);
  g_last_err[sizeof(g_last_err) - 1] = 0;
}
bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("FDM_PDL");
    return !(e != nullptr && e[0] == '0');
  }();
  return on;
}

bool encode_bf16_map(CUtensorMap* map, const void* ptr, int rank, const cuuint64_t* dims, const cuuint32_t* box,
                     CUtensorMapL2promotion l2, CUtensorMapSwizzle swz, const cuuint64_t* strides, const cuuint32_t* elem_strides) {
  static const PFN_cuTensorMapEncodeTiled encode = [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool found = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
                       q == cudaDriverEntryPointSuccess;
    return found ? reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn) : nullptr;
  }();
  if (encode == nullptr || rank > 5) return false;  // 5: the largest rank of a tiled tensor map
  cuuint64_t dense[4];
  if (strides == nullptr) {
    cuuint64_t s = sizeof(__nv_bfloat16);
    for (int i = 0; i + 1 < rank; ++i) dense[i] = s *= dims[i];
    strides = dense;
  }
  const cuuint32_t ones[5] = {1, 1, 1, 1, 1};
  return encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides, box,
                elem_strides != nullptr ? elem_strides : ones, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, l2,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace fdm

extern "C" int fdm_abi_version(void) { return FDM_ABI_VERSION; }

extern "C" const char* fdm_status_string(int s) {
  switch (s) {
    case FDM_OK: return "ok";
    case FDM_ERR_BAD_ARG: return "bad argument (null pointer or inconsistent sizes)";
    case FDM_ERR_UNSUPPORTED: return "unsupported shape/dtype for the sm_100a kernels";
    case FDM_ERR_CUDA: return "CUDA error (see fdm_last_cuda_error)";
    case FDM_ERR_NO_DEVICE: return "no sm_100 device";
    default: return "unknown status";
  }
}

extern "C" const char* fdm_last_cuda_error(void) { return fdm::g_last_err; }

extern "C" size_t fdm_struct_size(int which) {
  switch (which) {
    case 0: return sizeof(fdm_input_prep_args);
    case 1: return sizeof(fdm_conv_args);
    case 2: return sizeof(fdm_gn_apply_args);
    case 3: return sizeof(fdm_temporal_gn_args);
    case 4: return sizeof(fdm_timestep_embedding_args);
    case 5: return sizeof(fdm_grouped_linear_args);
    case 6: return sizeof(fdm_rpe_hidden_args);
    case 7: return sizeof(fdm_attn_temporal_args);
    case 8: return sizeof(fdm_attn_spatial_args);
    case 9: return sizeof(fdm_cast_args);
    case 10: return sizeof(fdm_ddpm_step_args);
    case 11: return sizeof(fdm_q_sample_args);
    case 12: return sizeof(fdm_masked_mse_args);
    case 13: return sizeof(fdm_linear_problem);
    case 14: return sizeof(fdm_rpe_hidden_problem);
    case 15: return sizeof(fdm_pack_problem);
    case 16: return sizeof(fdm_pack_weights_args);
    case 17: return sizeof(fdm_conv_wgrad_args);
    case 18: return sizeof(fdm_gn_bwd_args);
    case 19: return sizeof(fdm_temporal_gn_bwd_args);
    case 20: return sizeof(fdm_attn_spatial_bwd_args);
    case 21: return sizeof(fdm_attn_temporal_bwd_args);
    case 22: return sizeof(fdm_rpe_hidden_bwd_problem);
    case 23: return sizeof(fdm_rpe_hidden_bwd_args);
    case 24: return sizeof(fdm_linear_bwd_problem);
    case 25: return sizeof(fdm_grouped_linear_bwd_args);
    case 26: return sizeof(fdm_sum_parts_args);
    case 27: return sizeof(fdm_accum_args);
    case 28: return sizeof(fdm_nchw_to_nhwc_args);
    case 29: return sizeof(fdm_adamw_args);
    case 30: return sizeof(fdm_masked_mse_bwd_args);
    case 31: return sizeof(fdm_rpe_table_problem);
    case 32: return sizeof(fdm_rpe_tables_args);
    case 33: return sizeof(fdm_norm_linear_args);
    default: return 0;
  }
}
