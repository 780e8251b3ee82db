"""ctypes binding of libflowk.so (the C ABI declared in include/flowk.h).

There is NO fallback: if the shared library is missing the import fails, and every op
below refuses non-CUDA tensors.  Build it with `python __graft_entry__.py build`
(or `make -C <package>/csrc`)."""
import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libflowk.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "flowk.h")

FLOWK_OK = 0
FLOWK_ERR_SHAPE = 1
FLOWK_ERR_ALIGN = 2
FLOWK_ERR_ARG = 3
FLOWK_ERR_CUDA_BASE = 1000

_fp = ctypes.c_void_p     # device pointers travel as integers
_i = ctypes.c_int
_f = ctypes.c_float
_st = ctypes.c_void_p     # cudaStream_t

SIGNATURES = {
    "flowk_abi_version": ([], _i),
    "flowk_error_string": ([_i], ctypes.c_char_p),
    "flowk_ldj_workspace_bytes": ([_i], ctypes.c_size_t),
    "flowk_squeeze2d": ([_fp, _fp, _i, _i, _i, _i, _i, _st], _i),
    "flowk_unsqueeze2d": ([_fp, _fp, _i, _i, _i, _i, _i, _st], _i),
    "flowk_actnorm_init": ([_fp, _fp, _fp, _i, _i, _i, _f, _f, _st], _i),
    "flowk_channel_scale": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_channel_mix": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _st], _i),
    "flowk_affine_coupling_fwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_affine_coupling_inv": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_affine_coupling_bwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_mixlogcdf_fwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _st], _i),
    "flowk_mixlogcdf_inv": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _st], _i),
    "flowk_mixlogcdf_bwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _st], _i),
    "flowk_mixture_log_cdf": ([_fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_mixture_log_pdf": ([_fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_mixture_inv_cdf": ([_fp, _fp, _fp, _fp, _fp, _i, _i, _i, _st], _i),
    "flowk_conv_gemm": ([ctypes.c_void_p, _st], _i),
    "flowk_nchw_to_nhwc_hilo": ([_fp, ctypes.c_longlong, _i, _i, _i, _i, _fp, _fp, _st], _i),
    "flowk_split_hilo": ([_fp, _fp, _fp, ctypes.c_longlong, _st], _i),
    "flowk_nchw_to_nhwc_hilo_f16": ([_fp, ctypes.c_longlong, _i, _i, _i, _i, _fp, _fp, _st], _i),
    "flowk_split_hilo_f16": ([_fp, _fp, _fp, ctypes.c_longlong, ctypes.c_float, _st], _i),
    "flowk_attention_f16": ([_fp, _fp, _fp, _i, _i, _i, _i, _st], _i),
    "flowk_std_normal_logp": ([_fp, ctypes.c_longlong, _fp, _fp, _i, ctypes.c_longlong, _st], _i),
    "flowk_pack_weight_f16": ([_fp, _fp, _i, ctypes.c_float, _fp, _fp, _i, _i, _i, _i, _fp, _fp, _fp, _st], _i),
    "flowk_fold_actnorm_invconv": ([_fp] * 7 + [_i, _i, _i, _i, _fp, _fp, _fp, _st], _i),
    "flowk_patch_attention": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _st], _i),
    "flowk_patch_attention_train_fwd": ([_fp] * 7 + [_i] * 5 + [_st], _i),
    "flowk_patch_attention_bwd": ([_fp] * 8 + [_i] * 5 + [_st], _i),
    "flowk_attention_tc": ([_fp, _fp, _fp, _i, _i, _i, _i, _i, _fp, _fp, _st], _i),
    "flowk_attention_tc_v2": ([_fp, _fp, _fp, _i, _i, _i, _i, _i, _fp, _fp, _st], _i),
    "flowk_attention_tc_v2_occupancy": ([_i, _i, _i, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)], _i),
    "flowk_attention_inproj_tc": ([_fp, _fp, _fp, _fp, _f, _fp, _fp, _i, _i, _i, _i, _fp, _fp, _st], _i),
    "flowk_attention_inproj_tc_occupancy": ([_i, _i, _i, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)], _i),
    "flowk_attention": ([_fp, _fp, _fp, _i, _i, _i, _i, _st], _i),
    "flowk_concat_elu_fwd": ([_fp, _fp, _fp, ctypes.c_longlong, _i, ctypes.c_longlong, _st], _i),
    "flowk_concat_elu_bwd": ([_fp, _fp, _fp, _fp, ctypes.c_longlong, _i, ctypes.c_longlong, _st], _i),
    "flowk_glu_fwd": ([_fp, _fp, ctypes.c_longlong, _i, ctypes.c_longlong, _st], _i),
    "flowk_weight_norm_operands": ([_fp, _fp, _i, _i, _i, _i, _i, _fp, _fp, _fp, _fp, _fp, _fp, _st], _i),
    "flowk_weight_norm_operands_batched": ([_fp, _i, _i, _st], _i),
    "flowk_weight_norm_bwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _st], _i),
    "flowk_add_layernorm_workspace_bytes": ([ctypes.c_longlong, _i], ctypes.c_longlong),
    "flowk_add_layernorm_fwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, ctypes.c_longlong, _i, _i, _i, _i,
                                 ctypes.c_float, _st], _i),
    "flowk_add_layernorm_bwd": ([_fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, ctypes.c_longlong, _i, _i, _i, _i, _st], _i),
    "flowk_channel_sum_workspace_bytes": ([_i], ctypes.c_longlong),
    "flowk_channel_sum": ([_fp, _fp, _fp, ctypes.c_longlong, _i, ctypes.c_longlong, _st], _i),
    "flowk_conv_wgrad_splits": ([_i, _i, _i, _i, _i, _i, ctypes.POINTER(ctypes.c_int)], _i),
    "flowk_conv_wgrad": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _st], _i),
    "flowk_linear_wgrad_splits": ([ctypes.c_longlong, _i, _i, ctypes.POINTER(ctypes.c_int)], _i),
    "flowk_linear_wgrad": ([_fp, _fp, _fp, _fp, ctypes.c_longlong, _i, _i, _st], _i),
    "flowk_shift_columns": ([_fp, _fp, _fp, ctypes.c_longlong, _i, _st], _i),
    "flowk_weight_norm_bwd_partials": ([_fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _st], _i),
    "flowk_conv_gemm_splitk_slices": ([_fp], _i),
    "flowk_attention_train_fwd": ([_fp, _fp, _fp, _fp, ctypes.c_uint, ctypes.c_float, _i, _i, _i, _i, _st], _i),
    "flowk_attention_train_bwd": ([_i, _fp, _fp, _fp, _fp, _fp, _fp, ctypes.c_uint, ctypes.c_float, _i, _i, _i, _i, _st], _i),
    "flowk_attention_dropout_mask": ([_fp, ctypes.c_uint, ctypes.c_float, _i, _i, _fp, _st], _i),
    "flowk_adamax_step": ([_fp, _i, _fp, ctypes.c_float, ctypes.c_float, ctypes.c_float, _st], _i),
    "flowk_glu_bwd": ([_fp, _fp, _fp, ctypes.c_longlong, _i, ctypes.c_longlong, _st], _i),
    "flowk_mar_step": ([ctypes.c_void_p, _st], _i),
}


class ConvGemmArgs(ctypes.Structure):
    """Mirror of `flowk_conv_gemm_args` (include/flowk.h)."""
    _fields_ = [(n, ctypes.c_void_p) for n in
                ("a_hi", "a_lo", "w_hi", "w_lo", "bias", "res", "gamma", "beta", "pos",
                 "out_f32", "out_hi", "out_lo", "out_nchw", "status", "trace")] + \
               [(n, ctypes.c_int) for n in ("B", "H", "W", "Cin", "N", "taps", "pre", "out_mask")] + \
               [(n, ctypes.c_void_p) for n in ("w2_hi", "w2_lo", "out2_f32")] + [("N2", ctypes.c_int)] + \
               [("splitk_ws", ctypes.c_void_p), ("operand_format", ctypes.c_int), ("acc_scale", ctypes.c_float),
                ("dilation", ctypes.c_int), ("acc_scale2", ctypes.c_float), ("acc_scale_ptr", ctypes.c_void_p)]


class MarStepArgs(ctypes.Structure):
    """Mirror of `flowk_mar_step_args` (include/flowk.h)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("a_hi", "a_lo", "w_hi", "w_lo", "bias", "dst0_hi", "dst0_lo", "dst1_hi",
                                                "dst1_lo", "c", "noise", "z")] + \
               [("z_stride", ctypes.c_longlong), ("status", ctypes.c_void_p)] + \
               [(n, ctypes.c_int) for n in ("mode", "B", "H", "W", "Cin", "taps", "dilation", "hid", "dst0_pitch",
                                            "dst0_col", "dst1_pitch", "dst1_col")] + [("acc_scale", ctypes.c_float)]


class WnJob(ctypes.Structure):
    """Mirror of `flowk_wn_job` (include/flowk.h)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("v", "g", "norm", "w", "fwd_hi", "fwd_lo", "dg_hi", "dg_lo")] + \
               [(n, ctypes.c_int) for n in ("N", "cin", "taps", "cin_pad", "n_pad", "fwd_f16")]


class AdamaxChunk(ctypes.Structure):
    """Mirror of `flowk_adamax_chunk` (include/flowk.h)."""
    _fields_ = [(n, ctypes.c_void_p) for n in ("p", "g", "m", "u")] + [("n", ctypes.c_longlong)]


OPERAND_TF32, OPERAND_F16 = 0, 1
PRE_BIAS, PRE_GLU_RES_LN, PRE_LSTM = 0, 1, 2
MAR_EMBED, MAR_LSTM, MAR_SAMPLE = 0, 1, 2
PACK_PLAIN, PACK_WEIGHT_NORM, PACK_EXP_GAIN = 0, 1, 2
OUT_F32, OUT_HILO, OUT_HILO_POS, OUT_HILO_CELU, OUT_NCHW, OUT_HILO_RELU = 1, 2, 4, 8, 16, 32


# where the integer problem dimensions sit in each entry point's argument list (for per-launch accounting)
DIMS = {
    "flowk_squeeze2d": slice(2, 6), "flowk_unsqueeze2d": slice(2, 6), "flowk_actnorm_init": slice(3, 6),
    "flowk_channel_scale": slice(8, 11), "flowk_channel_mix": slice(7, 11),
    "flowk_affine_coupling_fwd": slice(6, 9), "flowk_affine_coupling_inv": slice(6, 9),
    "flowk_affine_coupling_bwd": slice(6, 9),
    "flowk_mixlogcdf_fwd": slice(7, 10), "flowk_mixlogcdf_inv": slice(7, 10), "flowk_mixlogcdf_bwd": slice(8, 11),
    "flowk_mixture_log_cdf": slice(5, 8), "flowk_mixture_log_pdf": slice(5, 8), "flowk_mixture_inv_cdf": slice(5, 8),
    "flowk_nchw_to_nhwc_hilo": slice(2, 6), "flowk_split_hilo": slice(3, 4), "flowk_attention": slice(3, 7),
    "flowk_nchw_to_nhwc_hilo_f16": slice(2, 6), "flowk_split_hilo_f16": slice(3, 4), "flowk_attention_f16": slice(3, 7),
    "flowk_attention_tc": slice(4, 8), "flowk_attention_tc_v2": slice(4, 8), "flowk_attention_inproj_tc": slice(7, 11),
    "flowk_patch_attention": slice(6, 10),
    "flowk_patch_attention_train_fwd": slice(7, 11), "flowk_patch_attention_bwd": slice(8, 12),
    "flowk_pack_weight_f16": slice(6, 10), "flowk_fold_actnorm_invconv": slice(7, 11),
}


def declared_symbols(header_path=HEADER_PATH):
    """Names of every function include/flowk.h declares (used by the ABI test)."""
    with open(header_path) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(flowk_[a-z0-9_]+)\s*\(", text)))


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libflowk.so not found at %s - the CUDA extension is the product and there is no fallback; "
            "build it with `python __graft_entry__.py build`" % LIB_PATH)
    import torch  # noqa: F401  (makes sure libcudart is resolvable / already mapped)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (argtypes, restype) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    return lib


lib = _load()

# Weights generation: raw-pointer writers (the fused Adamax kernel, CUDA-graph replays of an update, `.data` copies in
# broadcasts and the ActNorm init) change parameters WITHOUT touching torch's per-tensor version counter, so every
# derived-weight cache in the package keys on (GENERATION, data_ptr, _version) and those writers bump GENERATION.
GENERATION = 0


def bump_generation():
    global GENERATION
    GENERATION += 1


def check_device(t, what="flowk"):
    """Kernels are enqueued on the CURRENT device's current stream: a tensor that lives on another GPU would be
    touched from the wrong context.  Fail loudly instead (use torch.cuda.set_device / `with torch.cuda.device(...)`)."""
    import torch
    if t.is_cuda and t.device.index != torch.cuda.current_device():
        raise RuntimeError("%s: tensor lives on %s but the current CUDA device is cuda:%d; select the tensor's device "
                           "first (torch.cuda.set_device or `with torch.cuda.device(t.device)`)"
                           % (what, t.device, torch.cuda.current_device()))


ALLOW_LIBRARY = os.environ.get("FLOWK_ALLOW_LIBRARY", "0") == "1"
LIBRARY_FALLBACKS = 0      # how many times a CUDA tensor was routed to cuDNN / cuBLAS / ATen instead of a flowk kernel


def library_fallback(what, t=None):
    """Called right before a conditioner layer would run a CUDA tensor through a library kernel (F.conv2d, F.linear,
    bmm + softmax attention, ATen LayerNorm) because no flowk kernel takes its shape.  There is no silent multi-backend
    dispatch: this raises unless FLOWK_ALLOW_LIBRARY=1 (or `flowk._lib.ALLOW_LIBRARY = True`) opts in.  CPU tensors pass
    (host-side logic tests; the flow ops themselves are CUDA-only)."""
    global LIBRARY_FALLBACKS
    if t is not None and (not t.is_cuda or t.dtype != torch_float32()):
        return                       # CPU tensors: host-side tests; float64: reference computations of the tests
    if not ALLOW_LIBRARY:
        raise RuntimeError("flowk: %s has no flowk kernel for this shape/mode and would fall back to a library kernel; "
                           "set FLOWK_ALLOW_LIBRARY=1 to allow it" % what)
    LIBRARY_FALLBACKS += 1


def torch_float32():
    import torch
    return torch.float32


def param_key(params):
    return (GENERATION,) + tuple((p.data_ptr(), p._version) for p in params)

LAUNCHES = 0          # number of kernel-launching C-ABI calls made by this process
TIMING = None         # set to a dict to record a CUDA-event pair around every call: name -> [(start, end, int args)]


def check(status, what=""):
    """0 -> ok; shape errors surface as AssertionError like the reference's asserts
    (common_modules.py:21,38), everything else as RuntimeError."""
    if status == FLOWK_OK:
        return
    msg = "%s: %s (flowk status %d)" % (what, lib.flowk_error_string(status).decode(), status)
    if status == FLOWK_ERR_SHAPE:
        raise AssertionError(msg)
    raise RuntimeError(msg)


def call(name, *args, meta=None):
    """Enqueue one C-ABI entry point on the stream passed as its last argument.  `meta` (problem dimensions) is only
    used by the optional per-launch timing table when the dimensions travel inside a struct."""
    global LAUNCHES
    LAUNCHES += 1
    if TIMING is None:
        check(getattr(lib, name)(*args), name)
        return
    import torch
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()                       # torch's current stream == the stream handed to the kernel (ops._stream)
    status = getattr(lib, name)(*args)
    end.record()
    check(status, name)
    TIMING.setdefault(name, []).append((start, end, meta if meta is not None else tuple(args[DIMS.get(name, slice(0, 0))])))
