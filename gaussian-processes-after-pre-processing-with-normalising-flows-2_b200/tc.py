"""Host side of the tensor-core conditioner layers: operand preparation (3xTF32 hi/lo split, NHWC
weight layout) and the ctypes call into `flowk_conv_gemm` (include/flowk.h)."""
import ctypes

import torch

from . import _lib
from ._lib import (OUT_F32, OUT_HILO, OUT_HILO_CELU, OUT_HILO_POS, OUT_HILO_RELU, OUT_NCHW, PRE_BIAS,  # noqa: F401
                   PRE_GLU_RES_LN, PRE_LSTM)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def split_hilo(t):
    """t = hi + lo with both parts rounded to nearest TF32 (13 low mantissa bits zero), like the device-side split."""
    t = t.contiguous().float()
    if t.is_cuda and t.numel():
        return split_rows(t)                      # one kernel (the training path re-splits weights every step)

    def rna(v):
        return ((v.view(torch.int32) + 0x1000) & -8192).view(torch.float32)
    hi = rna(t)
    return hi, rna(t - hi)


def conv_weight_operand(w, cin_pad=None):
    """[N, Cin, kh, kw] conv weight (or [N, Cin] linear weight) -> K-major [N, taps*Cin_pad] in (tap, c) order, hi/lo."""
    if w.dim() == 2:
        w = w[:, :, None, None]
    n, cin, kh, kw = w.shape
    cin_pad = cin_pad or ((cin + 31) // 32 * 32)
    wk = w.permute(0, 2, 3, 1)                                   # [N, kh, kw, Cin]
    if cin_pad != cin:
        wk = torch.nn.functional.pad(wk, (0, cin_pad - cin))
    return split_hilo(wk.reshape(n, kh * kw * cin_pad))


def conv_weight_operand_f16(w, gain=None, mode=_lib.PACK_PLAIN, factor=1.0, bias=None):
    """[N, Cin, kh, kw] conv weight (or [N, Cin] linear weight) -> fp16 (hi, lo) pair [N, taps * ceil64(Cin)] in (tap, c)
    order for FLOWK_OPERAND_F16, pre-scaled by a power of two s so that max|w s| lies in [2^14, 2^15): the lo part then
    keeps its 11 bits clear of fp16's subnormal range.  `gain` / `mode` fuse a per-output-channel factor (weight norm, or an
    ActNorm's exp(factor * logs) with `bias` scaled alike) - see flowk_pack_weight_f16.  Two launches per weight.
    Returns (hi, lo, 1 / s[, bias * gain]); 1 / s goes to conv_gemm(acc_scale=)."""
    if w.dim() == 2:
        w = w[:, :, None, None]
    n, cin, kh, kw = w.shape
    cin_pad = (cin + 63) // 64 * 64
    taps = kh * kw
    w = w.detach().contiguous().float()
    _lib.check_device(w, "conv_weight_operand_f16")
    hi = torch.empty(n, taps * cin_pad, device=w.device, dtype=torch.float16)
    lo = torch.empty_like(hi)
    ws = torch.empty(n + 2, device=w.device, dtype=torch.float32)
    g = None if gain is None else gain.detach().reshape(-1).contiguous().float()
    b_in = None if bias is None else bias.detach().reshape(-1).contiguous().float()
    b_out = None if bias is None else torch.empty_like(b_in)
    assert g is None or g.numel() == n
    _lib.call("flowk_pack_weight_f16", w.data_ptr(), _p(g), int(mode), float(factor), _p(b_in), _p(b_out), n, cin, taps,
              cin_pad, hi.data_ptr(), lo.data_ptr(), ws.data_ptr(), _stream())
    acc_scale = float(ws[n + 1])                       # (host sync: cached per weight version)
    return (hi, lo, acc_scale) if bias is None else (hi, lo, acc_scale, b_out)


def split_rows_f16(x, scale=1.0):
    hi = torch.empty(x.shape, device=x.device, dtype=torch.float16)
    lo = torch.empty_like(hi)
    _lib.call("flowk_split_hilo_f16", x.data_ptr(), hi.data_ptr(), lo.data_ptr(), x.numel(), float(scale), _stream())
    return hi, lo


def _p(t):
    return None if t is None else t.data_ptr()


def conv_gemm(a_hi, a_lo, w_hi, w_lo, B, H, W, Cin, N, taps, pre, out_mask, bias=None, res=None, gamma=None,
              beta=None, pos=None, out_f32=None, out_hi=None, out_lo=None, out_nchw=None, status=None, trace=None,
              w2_hi=None, w2_lo=None, out2_f32=None, n2=0, split_k=False, acc_scale=None, dilation=1, acc_scale2=None,
              acc_scale_ptr=None):
    """The operand format follows the tensors: fp32 tensors = TF32 pairs (FLOWK_OPERAND_TF32), fp16 tensors = fp16 pairs
    (FLOWK_OPERAND_F16, inference; `acc_scale` undoes the weights' power-of-two pre-scaling).
    `split_k=True` (training path: one stream, kernel latency matters) lends the kernel a workspace so that layers
    with few 128-row tiles and a long K loop are shared by several CTAs per output tile."""
    _lib.check_device(a_hi, "conv_gemm")
    args = _lib.ConvGemmArgs(_p(a_hi), _p(a_lo), _p(w_hi), _p(w_lo), _p(bias), _p(res), _p(gamma), _p(beta), _p(pos),
                             _p(out_f32), _p(out_hi), _p(out_lo), _p(out_nchw), _p(status), _p(trace),
                             B, H, W, Cin, N, taps, pre, out_mask, _p(w2_hi), _p(w2_lo), _p(out2_f32), n2, None,
                             _lib.OPERAND_F16 if a_hi.dtype == torch.float16 else _lib.OPERAND_TF32,
                             1.0 if acc_scale is None else float(acc_scale), int(dilation),
                             1.0 if acc_scale2 is None else float(acc_scale2), _p(acc_scale_ptr))
    assert a_hi.dtype == a_lo.dtype == w_hi.dtype == w_lo.dtype, "operand pair formats must agree"
    assert out_hi is None or out_hi.dtype == a_hi.dtype, "out_hi/out_lo are written in the input operand format"
    if split_k:
        slices = _lib.lib.flowk_conv_gemm_splitk_slices(ctypes.addressof(args))
        if slices > 1:
            ws = torch.empty(slices * B * H * W * N, device=a_hi.device, dtype=torch.float32)
            args.splitk_ws = ws.data_ptr()
    _lib.call("flowk_conv_gemm", ctypes.addressof(args), _stream(), meta=(B, H, W, Cin, N, taps, pre))


def nchw_to_nhwc_hilo(x, c_pad, f16=False, out=None):
    """x: NCHW view whose (C,H,W) block is contiguous (e.g. a channel slice) -> ([B*HW, c_pad] hi, lo), written into
    `out` = (hi, lo) when given."""
    b, c, h, w = x.shape
    assert x.stride(3) == 1 and x.stride(2) == w and x.stride(1) == h * w, "channel slice of a contiguous NCHW tensor"
    if out is None:
        hi = torch.empty(b * h * w, c_pad, device=x.device, dtype=torch.float16 if f16 else torch.float32)
        lo = torch.empty_like(hi)
    else:
        hi, lo = out
        assert hi.shape == lo.shape == (b * h * w, c_pad) and hi.is_contiguous() and lo.is_contiguous()
        assert hi.dtype == lo.dtype == (torch.float16 if f16 else torch.float32)
    _lib.call("flowk_nchw_to_nhwc_hilo_f16" if f16 else "flowk_nchw_to_nhwc_hilo", x.data_ptr(), x.stride(0), b, c, h * w,
              c_pad, hi.data_ptr(), lo.data_ptr(), _stream())
    return hi, lo


def mar_step_args(mode, a, w, bias, B, H, W, taps, hid, dst0, dilation=1, dst1=None, c=None, noise=None, z=None,
                  z_stride=0, status=None):
    """flowk_mar_step_args for one step of mAR ancestral sampling (include/flowk.h).  a = (hi, lo) fp16 rows [B*H*W, Cin];
    w = (w_hi, w_lo, acc_scale) from conv_weight_operand_f16; dst0 / dst1 = (hi, lo, pitch, column) with hi / lo the fp16
    row arrays; noise / z are fp32 tensors whose data pointers are the first element the step reads / writes.  The
    struct holds raw pointers: the tensors must outlive every launch made with it."""
    assert a[0].dtype == a[1].dtype == w[0].dtype == w[1].dtype == torch.float16
    _lib.check_device(a[0], "mar_step")
    d1 = dst1 or (None, None, 0, 0)
    return _lib.MarStepArgs(_p(a[0]), _p(a[1]), _p(w[0]), _p(w[1]), _p(bias), _p(dst0[0]), _p(dst0[1]), _p(d1[0]),
                            _p(d1[1]), _p(c), _p(noise), _p(z), int(z_stride), _p(status), int(mode), B, H, W,
                            a[0].shape[1], taps, int(dilation), hid, dst0[2], dst0[3], d1[2], d1[3], float(w[2]))


def mar_step(args):
    """Enqueue flowk_mar_step(args) on the current stream."""
    _lib.call("flowk_mar_step", ctypes.addressof(args), _stream(), meta=(args.mode, args.B, args.H, args.W, args.hid))


def split_rows(x):
    hi = torch.empty_like(x)
    lo = torch.empty_like(x)
    _lib.call("flowk_split_hilo", x.data_ptr(), hi.data_ptr(), lo.data_ptr(), x.numel(), _stream())
    return hi, lo


ATTENTION_TC = __import__("os").environ.get("FLOWK_ATTENTION_TC", "1") != "0"


def attention_tc_supported(HW, C, heads):
    """Shapes the tcgen05 attention kernel (csrc/attention_tc.cu) takes; everything else runs on the mma.sync kernel."""
    d = C // max(heads, 1)
    if not (ATTENTION_TC and C % heads == 0 and HW in (128, 256) and d % 8 == 0 and d <= 64 and C % 4 == 0):
        return False
    dk = (d + 15) // 16 * 16                     # shared memory: P (over Q, K) + V^T + epilogue staging + static
    smem = max(4 * (HW // 64) * 128 * 64, 4 * HW * 128) + 2 * (HW // 64) * dk * 128 + 2 * 128 * (d // 8) * 16 + 9 * 1024
    return smem <= 227 * 1024


# The one-wave tcgen05 kernel (two CTAs per SM) for the shapes it takes; FLOWK_ATTENTION_TC_V2=0 keeps them on the
# one-CTA-per-SM kernel (A/B runs).
ATTENTION_TC_V2 = __import__("os").environ.get("FLOWK_ATTENTION_TC_V2", "1") != "0"


def attention_tc_v2_supported(HW, C, heads):
    """Shapes the one-wave tcgen05 attention kernel (csrc/attention_tc.cu, attention_tc_v2_kernel) takes: seq 128 / 256 with
    head dim 24 or 32 (one 64-byte swizzle row per Q / K row).  Other head dims (cfg4's 40 needs 96-byte rows, which
    would not fit two CTAs per SM) stay on attention_tc_kernel."""
    if not (ATTENTION_TC and ATTENTION_TC_V2 and heads >= 1 and C % heads == 0):
        return False
    return HW in (128, 256) and C // heads in (24, 32)


def attention(qkv, B, HW, C, heads, f16=False, status=None, trace=None):
    """qkv [B*HW, 3C] (k | v | q) -> (hi, lo) [B*HW, C] of softmax(q k^T / sqrt(d)) v."""
    hi = torch.empty(B * HW, C, device=qkv.device, dtype=torch.float16 if f16 else torch.float32)
    lo = torch.empty_like(hi)
    if attention_tc_v2_supported(HW, C, heads):
        _lib.call("flowk_attention_tc_v2", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), int(f16), B, HW, C, heads,
                  _p(status), _p(trace), _stream())
        return hi, lo
    if attention_tc_supported(HW, C, heads):
        _lib.call("flowk_attention_tc", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), int(f16), B, HW, C, heads,
                  _p(status), _p(trace), _stream())
        return hi, lo
    _lib.call("flowk_attention_f16" if f16 else "flowk_attention", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), B, HW, C,
              heads, _stream())
    return hi, lo


# q, k, v computed inside the one-wave kernel from the gate GEMM's normalised rows (flowk_attention_inproj_tc) instead of
# a chained in_proj GEMM writing them as fp32 rows; FLOWK_ATTENTION_INPROJ=0 keeps the in_proj GEMM (A/B runs).
ATTENTION_INPROJ = __import__("os").environ.get("FLOWK_ATTENTION_INPROJ", "1") != "0"


def attention_inproj_supported(HW, C, heads):
    """Shapes the fused in_proj + attention kernel takes: those of the one-wave kernel it extends."""
    return ATTENTION_INPROJ and attention_tc_v2_supported(HW, C, heads)


def attention_inproj(p_hi, p_lo, w_hi, w_lo, acc_scale, B, HW, C, heads, status=None, trace=None):
    """p_hi / p_lo [B*HW, C] fp16 rows in_proj multiplies, (w_hi, w_lo, acc_scale) its fp16 weight operand [3C, ceil64(C)]
    (conv_weight_operand_f16) -> fp16 (hi, lo) [B*HW, C] of softmax(q k^T / sqrt(d)) v with (k | v | q) = rows W^T."""
    assert p_hi.dtype == p_lo.dtype == w_hi.dtype == w_lo.dtype == torch.float16
    # the kernel's tensor maps are built from B, HW and C: the tensors must have exactly these layouts
    assert p_hi.shape == p_lo.shape == (B * HW, C) and p_hi.is_contiguous() and p_lo.is_contiguous(), \
        "p_hi / p_lo must be contiguous [B*HW, C]"
    assert w_hi.shape == w_lo.shape == (3 * C, (C + 63) // 64 * 64) and w_hi.is_contiguous() and w_lo.is_contiguous(), \
        "w_hi / w_lo must be the contiguous in_proj operand [3C, ceil64(C)]"
    _lib.check_device(p_hi, "attention_inproj")
    hi = torch.empty(B * HW, C, device=p_hi.device, dtype=torch.float16)
    lo = torch.empty_like(hi)
    _lib.call("flowk_attention_inproj_tc", p_hi.data_ptr(), p_lo.data_ptr(), w_hi.data_ptr(), w_lo.data_ptr(),
              float(acc_scale), hi.data_ptr(), lo.data_ptr(), B, HW, C, heads, _p(status), _p(trace), _stream())
    return hi, lo


def attention_supported(HW, C, heads):
    if attention_tc_supported(HW, C, heads):
        return True
    return C % heads == 0 and (C // heads) in (8, 16, 24, 32, 40, 64) and (HW <= 256 or HW % 256 == 0) and HW % 4 == 0 \
        and 2 * min(HW, 1 << 30) * (C // heads) * 4 * max(1, 256 // max(HW, 1)) <= 220 * 1024


def chain_supported(C, n2, f16=False):
    """gate -> in_proj fusion: both accumulators in TMEM (2C + n2 <= 512 columns) and the operand tiles in smem."""
    if C % (8 if f16 else 32) or n2 % 16 or 2 * C > 256 or 2 * C + n2 > 512:
        return False
    slab = ((4 * 32 * (C + 4) * 4 + 1023) // 1024) * 1024
    kblocks = (C + 63) // 64 if f16 else C // 32
    return slab + kblocks * 32768 + 2 * n2 * 128 + 2048 <= 227 * 1024
