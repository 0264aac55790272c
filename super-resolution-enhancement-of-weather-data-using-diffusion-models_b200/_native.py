"""ctypes binding of libwsr.so (the C ABI declared in include/wsr.h).

There is NO fallback: if the shared library cannot be found/built, or a call returns a non-zero status, a
``WsrError`` is raised.  Device pointers are passed as plain integers (``tensor.data_ptr()``), the stream as the raw
``cudaStream_t`` of torch's current stream.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libwsr.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_LRELU02, ACT_RELU, ACT_SWISH, ACT_MISH = 0, 1, 2, 3, 4


class WsrError(RuntimeError):
    pass


class PackJob(C.Structure):
    """WsrPackJob (include/wsr.h): one entry of the batched weight re-pack."""
    _fields_ = [("src", C.c_void_p), ("src2", C.c_void_p), ("dst", C.c_void_p), ("first_unit", C.c_int64),
                ("kind", C.c_int32), ("transposed", C.c_int32), ("dst_dtype", C.c_int32), ("Cout", C.c_int32), ("Cin", C.c_int32),
                ("taps", C.c_int32), ("Cout_pad", C.c_int32), ("Cin_pad", C.c_int32)]


PACK_CONV, PACK_VMERGE, PACK_UPSAMPLE, PACK_UPSAMPLE_DGRAD, PACK_COPY = 0, 1, 2, 3, 4


class ConvDesc(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("x_dtype", C.c_int), ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Cin", C.c_int), ("x_ld", C.c_int),
        ("w", C.c_void_p), ("w_rows", C.c_int),
        ("ksize", C.c_int), ("stride", C.c_int), ("upsample", C.c_int),
        ("Cout", C.c_int),
        ("x2", C.c_void_p), ("Cin2", C.c_int), ("x2_ld", C.c_int),
        ("w2", C.c_void_p),
        ("bias", C.c_void_p),
        ("rowvec", C.c_void_p), ("rowvec_ld", C.c_int),
        ("act", C.c_int),
        ("out_scale", C.c_float),
        ("res", C.c_void_p), ("res_dtype", C.c_int), ("res_ld", C.c_int), ("res_scale", C.c_float),
        ("res2", C.c_void_p), ("res2_dtype", C.c_int), ("res2_ld", C.c_int), ("res2_scale", C.c_float),
        ("y", C.c_void_p), ("y_dtype", C.c_int), ("y_ld", C.c_int),
        ("gn_stats", C.c_void_p), ("gn_stats_ld", C.c_int),
        ("gn_table", C.c_void_p), ("gn_table_ld", C.c_int), ("gn_act", C.c_int),
        ("w_vmerge", C.c_void_p),
    ]


class GemmDesc(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("a_dtype", C.c_int), ("a_sb", C.c_int64), ("a_sm", C.c_int64), ("a_sk", C.c_int64),
        ("b", C.c_void_p), ("b_dtype", C.c_int), ("b_sb", C.c_int64), ("b_sn", C.c_int64), ("b_sk", C.c_int64),
        ("d", C.c_void_p), ("d_dtype", C.c_int), ("d_sb", C.c_int64), ("d_sm", C.c_int64), ("d_sn", C.c_int64),
        ("res", C.c_void_p), ("res_dtype", C.c_int), ("res_sb", C.c_int64), ("res_sm", C.c_int64), ("res_sn", C.c_int64),
        ("bias", C.c_void_p),
        ("batch", C.c_int), ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("alpha", C.c_float),
    ]


MAX_TAPS = 16


class TapTable(C.Structure):
    """WsrTapTable (include/wsr.h): explicit tap list of a convolution."""
    _fields_ = [
        ("GH", C.c_int), ("GW", C.c_int), ("in_sub", C.c_int),
        ("out_mul", C.c_int), ("out_py", C.c_int), ("out_px", C.c_int),
        ("OH", C.c_int), ("OW", C.c_int), ("ntaps", C.c_int),
        ("py", C.c_int * MAX_TAPS), ("px", C.c_int * MAX_TAPS),
        ("dy", C.c_int * MAX_TAPS), ("dx", C.c_int * MAX_TAPS),
        ("wtap", C.c_int * MAX_TAPS),
    ]


class WgradDesc(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("x_dtype", C.c_int), ("N", C.c_int), ("H", C.c_int), ("W", C.c_int), ("Cin", C.c_int), ("x_ld", C.c_int),
        ("dy", C.c_void_p), ("dy_dtype", C.c_int), ("Cout", C.c_int), ("dy_ld", C.c_int),
        ("dw", C.c_void_p), ("dw_stap", C.c_int64), ("dw_sco", C.c_int64), ("dw_sci", C.c_int64),
        ("dbias", C.c_void_p),
        ("up", C.c_int),
    ]


_P, _I, _L, _F, _U64, _U32 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_uint32

# name -> argument ctypes (every one returns int unless listed in _RESTYPE)
SIGNATURES = {
    "wsr_version": [],
    "wsr_device_is_sm100": [],
    "wsr_conv_simt": [C.POINTER(ConvDesc), _P],
    "wsr_conv_tc": [C.POINTER(ConvDesc), _P],
    "wsr_conv_tc_can_fuse_gn": [C.POINTER(ConvDesc)],
    "wsr_debug_last_tc_config": [],
    "wsr_debug_set_pair": [_I],
    "wsr_set_pdl": [_I],
    "wsr_gn_finalize": [_P, _I, _I, _I, _I, _I, _F, _P, _P, _P, _I, _P],
    "wsr_gemm_simt": [C.POINTER(GemmDesc), _P],
    "wsr_gemm_tc": [C.POINTER(GemmDesc), _P],
    "wsr_attention_tc": [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "wsr_attention_small_tc": [_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "wsr_attention_small_nhwc_tc": [_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _F, _P],
    "wsr_attention_small_tc_supported": [_I, _I, _I],
    "wsr_conv_transpose_k8s4": [_P, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P, _I, _I, _P],
    "wsr_gn_stats": [_P, _I, _I, _I, _I, _I, _P, _I, _P],
    "wsr_gn_apply": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _I, _P, _I, _I, _P],
    "wsr_fill_zero": [_P, _L, _P],
    "wsr_softmax_rows": [_P, _I, _L, _I, _L, _F, _P, _I, _L, _P],
    "wsr_nchw_to_nhwc": [_P, _I, _I, _I, _I, _P, _I, _I, _P],
    "wsr_nhwc_to_nchw": [_P, _I, _I, _I, _I, _I, _I, _P, _P],
    "wsr_pack_conv_weight": [_P, _I, _I, _I, _I, _P, _I, _I, _I, _P],
    "wsr_pack_upsample_weight": [_P, _I, _I, _P, _I, _I, _I, _P],
    "wsr_pack_conv_weight_vmerge": [_P, _I, _I, _P, _I, _I, _P],
    "wsr_pack_convT_weight": [_P, _I, _I, _I, _I, _P, _I, _P],
    "wsr_cast": [_P, _I, _P, _I, _L, _P],
    "wsr_repack_batch": [_P, _I, _L, _P],
    "wsr_upsample2x": [_P, _I, _I, _I, _I, _I, _I, _P, _I, _P],
    "wsr_axpby": [_P, _I, _I, _F, _P, _I, _I, _F, _P, _I, _I, _L, _I, _P],
    "wsr_noise_embed": [_P, _I, _I, _P, _P, _P, _P, _I, _P, _P],
    "wsr_linear_rows": [_P, _I, _I, _P, _P, _I, _P, _P],
    "wsr_fd_precompute_workspace_bytes": [_I, _I, _I, _I],
    "wsr_fd_precompute": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P],
    "wsr_fd_gate": [_P, _I, _P, _I, _I, _I, _P, _P, _I, _P, _P],
    "wsr_stem_assemble": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _I, _I, _P],
    "wsr_haar_detail_sums": [_P, _I, _I, _I, _I, _I, _P, _P, _P],
    "wsr_haar_detail_bands": [_P, _I, _I, _I, _I, _I, _P, _P, _P],
    "wsr_phy_stencils": [_P, _I, _I, _I, _I, _P, _P],
    "wsr_bicubic_upsample": [_P, _I, _I, _I, _I, _P, _P],
    "wsr_standard_scale": [_P, _I, _L, _P, _P, _I, _P, _P],
    "wsr_error_sums": [_P, _P, _I, _L, _P, _P, _P],
    "wsr_ensemble_stats": [_P, _I, _L, _P, _I, _L, _P, _P, _P, _P, _P, _P],
    "wsr_zonal_spectra": [_P, _P, _I, _I, _I, _P, _P, _P, _P],
    "wsr_image_compare_loss": [_P, _P, _I, _I, _I, _F, _F, _P, _P, _P],
    "wsr_relu_mask": [_P, _P, _L, _P],
    "wsr_lrelu_mask": [_P, _I, _I, _P, _I, _I, _L, _I, _F, _P],
    "wsr_sampler_step": [_P, _P, _I, _P, _L, _U64, _P, _I, _P, _I, _P, _L, _P],
    "wsr_final_conv_sampler_step": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _P, _P, _I, _P, _P, _P, _L, _U64, _P, _I, _P, _I, _P],
    "wsr_sampler_step_members": [_P, _P, _I, _P, _L, _P, _L, _P, _I, _P, _I, _P, _L, _P],
    "wsr_final_conv_sampler_step_members": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _P, _P, _I, _P, _P, _P, _L, _P, _L, _P, _I, _P,
                                            _I, _P],
    "wsr_sampler_step_multistep": [_P, _P, _I, _P, _P, _I, _P, _I, _P, _L, _P],
    "wsr_final_conv_sampler_step_multistep": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _P, _P, _I, _P, _P, _P, _P, _I, _P, _I, _P],
    "wsr_head_sampler_supported": [_I, _I, _I],
    "wsr_pack_head_weight": [_P, _I, _I, _P, _P],
    "wsr_broadcast_row": [_P, _I, _P, _I, _P, _P],
    "wsr_step_counter_add": [_P, _I, _P],
    "wsr_randn": [_P, _L, _U64, _U32, _P],
    "wsr_randn_members": [_P, _L, _P, _L, _U32, _P],
    "wsr_q_sample": [_P, _P, _P, _P, _I, _L, _P, _P],
    "wsr_noise_loss": [_P, _P, _L, _I, _P, _P, _F, _P],
    # training step (backward.cu, fd.cu)
    "wsr_conv_taps_simt": [C.POINTER(ConvDesc), C.POINTER(TapTable), _P],
    "wsr_conv_taps_tc": [C.POINTER(ConvDesc), C.POINTER(TapTable), _P],
    "wsr_conv_wgrad_simt": [C.POINTER(WgradDesc), C.POINTER(TapTable), _P],
    "wsr_conv_wgrad_tc": [C.POINTER(WgradDesc), C.POINTER(TapTable), _P],
    "wsr_col_sums": [_P, _I, _L, _I, _I, _P, _P],
    "wsr_gn_apply_dropout": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _I, _P, _I, _I, _F, _U64, _U32, _P],
    "wsr_dropout_mask": [_P, _I, _I, _I, _F, _U64, _U32, _P],
    "wsr_gn_bwd_reduce": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _I, _P, _I, _I, _F, _U64, _U32, _P, _I, _P],
    "wsr_gn_bwd_apply": [_P, _I, _I, _I, _I, _I, _P, _I, _P, _P, _I, _F, _I, _P, _I, _I, _F, _U64, _U32, _P, _I, _P, _I, _I,
                         _I, _P, _P, _P, _I, _P],
    "wsr_softmax_bwd_rows": [_P, _I, _P, _I, _L, _I, _L, _F, _P, _I, _P],
    "wsr_noise_embed_bwd": [_P, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P],
    "wsr_linear_rows_bwd": [_P, _I, _I, _P, _P, _I, _P, _P, _P, _P],
    "wsr_fd_gate_bwd": [_P, _I, _I, _I, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _I, _P, _P, _P],
    "wsr_fd_backward_workspace_bytes": [_I, _I, _I, _I],
    "wsr_fd_backward": [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "wsr_adam_step": [_P, _P, _P, _P, _L, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _I, _P],
    "wsr_adam_step_ema": [_P, _P, _P, _P, _P, _L, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _I, C.c_double, _P],
}
_RESTYPE = {"wsr_fd_precompute_workspace_bytes": C.c_int64, "wsr_fd_backward_workspace_bytes": C.c_int64}
# functions whose return value is data, not a status
_NO_STATUS = {"wsr_version", "wsr_device_is_sm100", "wsr_conv_tc_can_fuse_gn", "wsr_debug_last_tc_config", "wsr_debug_set_pair", "wsr_set_pdl", "wsr_attention_small_tc_supported", "wsr_head_sampler_supported", "wsr_fd_precompute_workspace_bytes", "wsr_fd_backward_workspace_bytes"}

_lib = None
launches = 0          # number of status-returning calls made (bench.py's gpu_launches bookkeeping is done there)


def _load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        # build in-tree (needs nvcc); never silently continue without the native library
        try:
            from .csrc import build as _b
        except Exception:
            import importlib.util
            spec = importlib.util.spec_from_file_location("wsr_build", os.path.join(_HERE, "csrc", "build.py"))
            _b = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(_b)
        _b.build(verbose=False)
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise WsrError("cannot load %s: %s" % (LIB_PATH, e))
    lib.wsr_last_error.restype = C.c_char_p
    lib.wsr_last_error.argtypes = []
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _RESTYPE.get(name, C.c_int)
    _lib = lib
    return lib


def lib():
    return _load()


def last_error():
    return _load().wsr_last_error().decode()


def fn(name):
    """The raw ctypes entry point (argtypes set), for recorded launch lists."""
    return getattr(_load(), name)


def call(name, *args):
    """Call a status-returning entry point; raise WsrError on failure."""
    global launches
    fn = getattr(_load(), name)
    rc = fn(*args)
    if name in _NO_STATUS:
        return rc
    launches += 1
    if rc != 0:
        raise WsrError("%s failed (%d): %s" % (name, rc, last_error()))
    return rc
