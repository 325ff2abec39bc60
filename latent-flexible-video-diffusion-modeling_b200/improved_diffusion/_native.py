"""
ctypes binding of libfdm_sm100.so (the C-ABI declared in include/fdm_b200.h).

There is no CPU fallback: if the library is missing or a call fails, this module raises.  The
structures below mirror the header field by field; `verify_struct_sizes()` cross-checks every
ctypes mirror against `fdm_struct_size()` exported by the library (runs on CPU, no GPU needed).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libfdm_sm100.so")

F32, BF16 = 0, 1
CONV_SIMT, CONV_TC, CONV_TC_TAP = 0, 1, 2

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


def _S(name, fields):
    return type(name, (C.Structure,), {"_fields_": fields})


InputPrepArgs = _S("InputPrepArgs", [("x", vp), ("x0", vp), ("obs_mask", vp), ("xin", vp), ("xin_bf16", vp),
                                     ("N", i32), ("C", i32), ("H", i32), ("W", i32), ("Cpad", i32)])
ConvArgs = _S("ConvArgs", [("a0", vp), ("w0", vp), ("a1", vp), ("w1", vp), ("bias", vp), ("resid", vp),
                           ("y_f32", vp), ("y_op", vp), ("stats", vp),
                           ("N", i32), ("Hin", i32), ("Win", i32), ("C0", i32), ("C1", i32), ("Cout", i32),
                           ("ksize", i32), ("stride", i32), ("upsample", i32),
                           ("a_dtype", i32), ("op_dtype", i32), ("out_nchw", i32), ("engine", i32),
                           ("resid_norm", i32), ("rn_T", i32), ("rn_eps", f32), ("rn_tstats", vp), ("rn_stats", vp),
                           ("rn_gamma", vp), ("rn_beta", vp)])
GnApplyArgs = _S("GnApplyArgs", [("xa", vp), ("xb", vp), ("stats_a", vp), ("stats_b", vp), ("gamma", vp), ("beta", vp),
                                 ("film", vp), ("out_op", vp), ("out_f32", vp), ("raw_op", vp),
                                 ("N", i32), ("HW", i32), ("Ca", i32), ("Cb", i32), ("T", i32),
                                 ("film_stride", i32), ("film_off", i32), ("silu", i32), ("op_dtype", i32), ("eps", f32),
                                 ("xa_bf16", i32), ("film_add", i32), ("drop_philox", vp), ("drop_p", f32), ("drop_salt", i32)])
TemporalGnArgs = _S("TemporalGnArgs", [("x", vp), ("gamma", vp), ("beta", vp), ("out_f32", vp), ("out_op", vp),
                                       ("B", i32), ("T", i32), ("HW", i32), ("C", i32), ("op_dtype", i32), ("eps", f32)])
TimestepEmbeddingArgs = _S("TimestepEmbeddingArgs", [("t", vp), ("t_index", vp), ("t_table", vp), ("freqs", vp), ("out", vp),
                                                     ("B", i32), ("dim", i32)])
LinearProblem = _S("LinearProblem", [("x", vp), ("w", vp), ("b", vp), ("y", vp),
                                     ("M", i32), ("K", i32), ("Nout", i32), ("ldx", i32), ("ldy", i32), ("silu_in", i32)])
GroupedLinearArgs = _S("GroupedLinearArgs", [("problems", vp), ("count", i32), ("max_M", i32), ("max_Nout", i32), ("max_K", i32)])
RpeHiddenProblem = _S("RpeHiddenProblem", [("wd", vp), ("bd", vp), ("hidden", vp), ("C", i32), ("te_off", i32)])
RpeHiddenArgs = _S("RpeHiddenArgs", [("te", vp), ("frame_indices", vp), ("problems", vp),
                                     ("B", i32), ("T", i32), ("te_stride", i32), ("count", i32), ("max_C", i32),
                                     ("hidden_dtype", i32)])
AttnTemporalArgs = _S("AttnTemporalArgs", [("qkv", vp), ("Rq", vp), ("Rk", vp), ("Rv", vp), ("mask", vp), ("out", vp),
                                           ("B", i32), ("T", i32), ("HW", i32), ("C", i32), ("heads", i32),
                                           ("qkv_dtype", i32), ("out_dtype", i32), ("Rq_op", vp), ("Rk_op", vp), ("Rv_op", vp),
                                           ("workspace", vp), ("workspace_bytes", i64), ("attn_mean", vp)])
AttnSpatialArgs = _S("AttnSpatialArgs", [("qkv", vp), ("out", vp), ("N", i32), ("L", i32), ("C", i32), ("heads", i32),
                                         ("qkv_dtype", i32), ("out_dtype", i32), ("engine", i32), ("lse", vp), ("attn_mean", vp)])
CastArgs = _S("CastArgs", [("x", vp), ("out", vp), ("N", i32), ("H", i32), ("W", i32), ("C", i32),
                           ("upsample", i32), ("op_dtype", i32), ("colsum", vp), ("colsum2", vp)])
DdpmStepArgs = _S("DdpmStepArgs", [("x", vp), ("eps", vp), ("noise", vp), ("coef", vp), ("t", vp), ("sample", vp),
                                   ("pred_xstart", vp), ("per_video", i64), ("B", i32), ("clip", i32), ("philox", vp)])
QSampleArgs = _S("QSampleArgs", [("x0", vp), ("noise", vp), ("coef2", vp), ("t", vp), ("x_t", vp),
                                 ("per_video", i64), ("B", i32)])
MaskedMseArgs = _S("MaskedMseArgs", [("eps", vp), ("noise", vp), ("m1", vp), ("m2", vp), ("mse", vp), ("eval", vp),
                                     ("per_frame", i64), ("B", i32), ("T", i32)])

# ---- backward (training) structures
sz = C.c_size_t
PackProblem = _S("PackProblem", [("src", vp), ("src2", vp), ("dst", vp), ("co", i32), ("ci", i32), ("k", i32), ("mode", i32)])
PackWeightsArgs = _S("PackWeightsArgs", [("problems", vp), ("count", i32), ("max_elems", i32)])
ConvWgradArgs = _S("ConvWgradArgs", [("a", vp), ("dy", vp), ("dw", vp), ("dbias", vp), ("dbias2", vp), ("workspace", vp),
                                     ("workspace_bytes", sz),
                                     ("N", i32), ("Hin", i32), ("Win", i32), ("C", i32), ("Cw", i32), ("Cout", i32),
                                     ("ksize", i32), ("stride", i32), ("a_dtype", i32), ("dy_dtype", i32), ("engine", i32)])
GnBwdArgs = _S("GnBwdArgs", [("xa", vp), ("xb", vp), ("stats_a", vp), ("stats_b", vp), ("gamma", vp), ("beta", vp), ("film", vp),
                             ("dy_op", vp), ("dy_f32", vp), ("draw_op", vp), ("gxa", vp), ("gxb", vp), ("ab", vp),
                             ("dgamma", vp), ("dbeta", vp), ("dfilm", vp),
                             ("N", i32), ("HW", i32), ("Ca", i32), ("Cb", i32), ("T", i32), ("film_stride", i32),
                             ("film_off", i32), ("silu", i32), ("op_dtype", i32), ("acc_a", i32), ("acc_b", i32), ("eps", f32),
                             ("dpass_a", vp), ("gop_a", vp), ("cs_a", vp), ("cs2_a", vp), ("phases", i32),
                             ("drop_philox", vp), ("drop_p", f32), ("drop_salt", i32)])
TemporalGnBwdArgs = _S("TemporalGnBwdArgs", [("x", vp), ("gamma", vp), ("dy_op", vp), ("dy_f32", vp), ("gx", vp),
                                             ("dgamma", vp), ("dbeta", vp),
                                             ("B", i32), ("T", i32), ("HW", i32), ("C", i32), ("op_dtype", i32),
                                             ("accumulate", i32), ("eps", f32)])
AttnSpatialBwdArgs = _S("AttnSpatialBwdArgs", [("qkv", vp), ("out", vp), ("dout", vp), ("dqkv", vp), ("lse", vp), ("dsum", vp),
                                               ("N", i32), ("L", i32), ("C", i32), ("heads", i32), ("dtype", i32),
                                               ("lse_from_forward", i32)])
AttnTemporalBwdArgs = _S("AttnTemporalBwdArgs", [("qkv", vp), ("out", vp), ("Rq", vp), ("Rk", vp), ("Rv", vp), ("mask", vp),
                                                 ("dout", vp), ("dqkv", vp), ("dRq", vp), ("dRk", vp), ("dRv", vp),
                                                 ("lse", vp), ("dsum", vp),
                                                 ("B", i32), ("T", i32), ("HW", i32), ("C", i32), ("heads", i32), ("dtype", i32)])
RpeHiddenBwdProblem = _S("RpeHiddenBwdProblem", [("wd", vp), ("bd", vp), ("dhidden", vp), ("dwd", vp), ("dbd", vp),
                                                 ("C", i32), ("te_off", i32)])
RpeHiddenBwdArgs = _S("RpeHiddenBwdArgs", [("te", vp), ("frame_indices", vp), ("problems", vp), ("dte", vp),
                                           ("B", i32), ("T", i32), ("te_stride", i32), ("count", i32), ("max_C", i32),
                                           ("dhidden_dtype", i32)])
LinearBwdProblem = _S("LinearBwdProblem", [("x", vp), ("w", vp), ("dy", vp), ("dw", vp), ("db", vp), ("dx_part", vp),
                                           ("M", i32), ("K", i32), ("Nout", i32), ("ldx", i32), ("ldy", i32), ("silu_in", i32)])
GroupedLinearBwdArgs = _S("GroupedLinearBwdArgs", [("problems", vp), ("count", i32), ("max_M", i32), ("max_Nout", i32),
                                                   ("max_K", i32)])
SumPartsArgs = _S("SumPartsArgs", [("parts", vp), ("out", vp), ("part_stride", i64), ("n", i64), ("count", i32),
                                   ("accumulate", i32)])
AccumArgs = _S("AccumArgs", [("src", vp), ("dst", vp), ("N", i32), ("H", i32), ("W", i32), ("C", i32), ("pool", i32),
                             ("src_dtype", i32), ("accumulate", i32)])
NchwToNhwcArgs = _S("NchwToNhwcArgs", [("src", vp), ("dst", vp), ("N", i32), ("C", i32), ("H", i32), ("W", i32), ("Cpad", i32),
                                       ("op_dtype", i32)])
AdamwArgs = _S("AdamwArgs", [("p", vp), ("g", vp), ("m", vp), ("v", vp), ("ema0", vp), ("ema1", vp), ("n", i64),
                             ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32), ("weight_decay", f32),
                             ("bias_correction1", f32), ("bias_correction2_sqrt", f32), ("ema_rate0", f32), ("ema_rate1", f32)])
MaskedMseBwdArgs = _S("MaskedMseBwdArgs", [("out", vp), ("target", vp), ("m1", vp), ("m2", vp), ("g_mse", vp), ("g_eval", vp),
                                           ("d_out", vp), ("per_frame", i64), ("B", i32), ("T", i32)])
RpeTableProblem = _S("RpeTableProblem", [("wd", vp), ("bd", vp), ("bo", vp), ("w_packed", vp), ("out_op", vp), ("out_f32", vp),
                                         ("C", i32), ("te_off", i32)])
RpeTablesArgs = _S("RpeTablesArgs", [("te", vp), ("frame_indices", vp), ("blob", vp), ("count", i32), ("B", i32), ("T", i32),
                                     ("te_stride", i32), ("max_C", i32)])
NormLinearArgs = _S("NormLinearArgs", [("x", vp), ("stats", vp), ("tstats", vp), ("gamma", vp), ("beta", vp), ("w", vp), ("bias", vp),
                                       ("y_op", vp), ("B", i32), ("T", i32), ("HW", i32), ("K", i32), ("Cout", i32),
                                       ("a_mode", i32), ("eps", f32)])
PACK_TC_FWD, PACK_TC_DGRAD, PACK_SIMT_FWD, PACK_SIMT_DGRAD, PACK_SUM2 = 0, 1, 2, 3, 4

# index = `which` of fdm_struct_size (include/fdm_b200.h)
STRUCTS = [InputPrepArgs, ConvArgs, GnApplyArgs, TemporalGnArgs, TimestepEmbeddingArgs, GroupedLinearArgs,
           RpeHiddenArgs, AttnTemporalArgs, AttnSpatialArgs, CastArgs, DdpmStepArgs, QSampleArgs, MaskedMseArgs,
           LinearProblem, RpeHiddenProblem,
           PackProblem, PackWeightsArgs, ConvWgradArgs, GnBwdArgs, TemporalGnBwdArgs, AttnSpatialBwdArgs, AttnTemporalBwdArgs,
           RpeHiddenBwdProblem, RpeHiddenBwdArgs, LinearBwdProblem, GroupedLinearBwdArgs, SumPartsArgs, AccumArgs,
           NchwToNhwcArgs, AdamwArgs, MaskedMseBwdArgs, RpeTableProblem, RpeTablesArgs, NormLinearArgs]

ENTRY_POINTS = ["fdm_input_prep", "fdm_conv", "fdm_gn_apply", "fdm_temporal_gn", "fdm_timestep_embedding",
                "fdm_grouped_linear", "fdm_rpe_hidden", "fdm_attn_temporal", "fdm_attn_spatial", "fdm_cast",
                "fdm_ddpm_step", "fdm_q_sample", "fdm_masked_mse",
                "fdm_pack_weights", "fdm_conv_wgrad", "fdm_gn_bwd", "fdm_temporal_gn_bwd", "fdm_attn_spatial_bwd",
                "fdm_attn_temporal_bwd", "fdm_rpe_hidden_bwd", "fdm_grouped_linear_bwd", "fdm_sum_parts", "fdm_accum",
                "fdm_nchw_to_nhwc", "fdm_adamw", "fdm_masked_mse_bwd", "fdm_rpe_tables", "fdm_norm_linear"]

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Load libfdm_sm100.so (built in-tree by `make -C csrc` / __graft_entry__.build()).  No fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(f"{LIB_PATH} is missing: build it with `make -C {os.path.join(os.path.dirname(_HERE), 'csrc')}`; "
                              "there is no CPU / PyTorch fallback for the FDM hot path")
        L = C.CDLL(LIB_PATH)
        L.fdm_abi_version.restype = C.c_int
        L.fdm_status_string.restype = C.c_char_p
        L.fdm_status_string.argtypes = [C.c_int]
        L.fdm_last_cuda_error.restype = C.c_char_p
        L.fdm_struct_size.restype = C.c_size_t
        L.fdm_struct_size.argtypes = [C.c_int]
        for name in ENTRY_POINTS:
            fn = getattr(L, name)
            fn.restype = C.c_int
            fn.argtypes = [vp, vp]
        L.fdm_conv_wgrad_workspace.restype = C.c_size_t
        L.fdm_conv_wgrad_workspace.argtypes = [vp]
        L.fdm_rpe_tables_blob_bytes.restype = C.c_size_t
        L.fdm_rpe_tables_blob_bytes.argtypes = [C.c_int32]
        L.fdm_rpe_tables_prepare.restype = C.c_int
        L.fdm_rpe_tables_prepare.argtypes = [vp, C.c_int32, vp, C.c_size_t]
        for name in ("fdm_attn_temporal_workspace", "fdm_attn_temporal_attn_offset"):
            getattr(L, name).restype = C.c_size_t
            getattr(L, name).argtypes = [vp]
        L.fdm_norm_linear_supported.restype = C.c_int
        L.fdm_norm_linear_supported.argtypes = [vp]
        if L.fdm_abi_version() != 2:
            raise NativeError(f"libfdm_sm100.so ABI {L.fdm_abi_version()} != 2")
        _lib = L
    return _lib


def verify_struct_sizes():
    L = lib()
    for which, st in enumerate(STRUCTS):
        n = L.fdm_struct_size(which)
        if n != C.sizeof(st):
            raise NativeError(f"struct #{which} {st.__name__}: library says {n} bytes, ctypes mirror {C.sizeof(st)}")
    return True


def check(rc, what):
    if rc != 0:
        L = lib()
        msg = L.fdm_status_string(rc).decode()
        if rc == -3:
            msg += ": " + L.fdm_last_cuda_error().decode()
        raise NativeError(f"{what} failed: {msg}")


def call(name, args, stream):
    """Launch one entry point on the raw handle `stream`.  The handle must belong to torch's CURRENT device (kernels are launched
    on the calling thread's current CUDA device): callers with tensors on another GPU wrap the call in
    `with torch.cuda.device(tensor.device)` — see `device_guard`."""
    check(getattr(lib(), name)(C.byref(args), C.c_void_p(stream)), name)


def device_guard(device):
    """Context manager making `device` torch's current CUDA device for native launches / graph capture (no-op for CPU)."""
    import contextlib
    import torch as th
    d = th.device(device)
    return th.cuda.device(d) if d.type == "cuda" else contextlib.nullcontext()
