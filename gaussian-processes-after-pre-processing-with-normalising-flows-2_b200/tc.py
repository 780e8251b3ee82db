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


def conv_weight_operand_f16(w, gain=None, mode=_lib.PACK_PLAIN, factor=1.0, bias=None, device_scale=False):
    """[N, Cin, kh, kw] conv weight (or [N, Cin] linear weight) -> fp16 (hi, lo) pair [N, taps * ceil64(Cin)] in (tap, c)
    order for FLOWK_OPERAND_F16, pre-scaled by a power of two s so that max|w s| lies in [2^14, 2^15): the lo part then
    keeps its 11 bits clear of fp16's subnormal range.  `gain` / `mode` fuse a per-output-channel factor (weight norm, or an
    ActNorm's exp(factor * logs) with `bias` scaled alike) - see flowk_pack_weight_f16.  Two launches per weight.
    Returns (hi, lo, 1 / s[, bias * gain]); 1 / s goes to conv_gemm(acc_scale=).  With `device_scale` 1 / s stays on the
    device as a 1-element tensor for conv_gemm(acc_scale=1, acc_scale_ptr=): no host read, so the packing can be captured
    in a CUDA graph and re-run at every replay."""
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
    if device_scale:
        assert bias is None
        return hi, lo, ws[n + 1:]
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
    if not _attention_mma_supported(HW, C, heads) and attention_long_tc_supported(HW, C, heads):
        _lib.call("flowk_attention_long_tc", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), int(f16), B, HW, C, heads,
                  _p(status), _p(trace), _stream())
        return hi, lo
    _lib.call("flowk_attention_f16" if f16 else "flowk_attention", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), B, HW, C,
              heads, _stream())
    return hi, lo


def attention_long_tc_supported(HW, C, heads):
    """Shapes the long-sequence tcgen05 attention kernel (csrc/attention_long_tc.cu) takes: seq a multiple of 128 and at least
    512, head dim 24, 32, 40 or 64.  `attention` sends it only the shapes no other kernel takes (d > 24 at 1024 tokens: the
    level-1 maps of 64x64 images at widths 128, 160 and 256); the shapes the mma.sync kernel runs keep it."""
    if not (heads >= 1 and C % heads == 0):
        return False
    return HW >= 512 and HW % 128 == 0 and C // heads in (24, 32, 40, 64)


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


def _attention_mma_supported(HW, C, heads):
    """Shapes the mma.sync attention kernel (csrc/attention.cu) takes within its shared-memory budget."""
    return C % heads == 0 and (C // heads) in (8, 16, 24, 32, 40, 64) and (HW <= 256 or HW % 256 == 0) and HW % 4 == 0 \
        and 2 * min(HW, 1 << 30) * (C // heads) * 4 * max(1, 256 // max(HW, 1)) <= 220 * 1024


def attention_supported(HW, C, heads):
    return (attention_tc_supported(HW, C, heads) or _attention_mma_supported(HW, C, heads)
            or attention_long_tc_supported(HW, C, heads))


def chain_supported(C, n2, f16=False):
    """gate -> in_proj fusion: both accumulators in TMEM (2C + n2 <= 512 columns) and the operand tiles in smem."""
    if C % (8 if f16 else 32) or n2 % 16 or 2 * C > 256 or 2 * C + n2 > 512:
        return False
    slab = ((4 * 32 * (C + 4) * 4 + 1023) // 1024) * 1024
    kblocks = (C + 63) // 64 if f16 else C // 32
    return slab + kblocks * 32768 + 2 * n2 * 128 + 2048 <= 227 * 1024


# The attention half of a ConvAttnBlock (gate, LayerNorm, in_proj, attention, attention gate) as one launch where a 128-row
# tile holds whole images (flowk_block_tail_tc); FLOWK_BLOCK_TAIL=0 keeps the chained gate, attention and gate launches
# (A/B runs).
BLOCK_TAIL = __import__("os").environ.get("FLOWK_BLOCK_TAIL", "1") != "0"


def block_tail_supported(HW, C, heads, M):
    """Shapes the conditioner routes to flowk_block_tail_tc: whole images per 128-row tile, head dims 24 / 32, the gate and
    in_proj accumulators side by side in the 512 TMEM columns (5C <= 512), and at least two tiles.  A single-tile batch
    (B = 2 at 8x8) keeps the three-launch route, as the conditioner's route test (tests/test_attention_inproj_fused.py)
    specifies; the kernel takes that shape too and is not slower there (profiles/r8_block_tail_probe.txt)."""
    if not (BLOCK_TAIL and heads >= 1 and C % heads == 0):
        return False
    return (HW <= 128 and 128 % HW == 0 and M % 128 == 0 and M >= 256 and C % 32 == 0 and 5 * C <= 512
            and C // heads in (24, 32))


# The same block tail at 16x16 (an image spans two 128-row tiles) as one launch of two-CTA clusters, one per image
# (flowk_block_tail_pair_tc); FLOWK_BLOCK_TAIL_PAIR=0 keeps the gate GEMM + fused in_proj attention + gate launches (A/B runs).
BLOCK_TAIL_PAIR = __import__("os").environ.get("FLOWK_BLOCK_TAIL_PAIR", "1") != "0"


def block_tail_pair_supported(HW, C, heads, B):
    """Shapes the conditioner routes to flowk_block_tail_pair_tc: 16x16 maps (HW = 256, two tiles per image), head dims 24 /
    32, 5C <= 512 TMEM columns, and B >= 8.  The batch rule is a routing contract: smaller batches (B = 2 and 4 at level 1)
    keep flowk_attention_inproj_tc, as the conditioner's route tests (tests/test_attention_inproj_fused.py,
    tests/test_block_tail_tc.py) specify; the kernel itself takes any B >= 1."""
    if not (BLOCK_TAIL_PAIR and heads >= 1 and C % heads == 0):
        return False
    return HW == 256 and B >= 8 and C % 32 == 0 and 5 * C <= 512 and C // heads in (24, 32)


def block_tail(c1_hi, c1_lo, gate, bias_g, x, ln1, pos, in_proj, attn_gate, bias_a, ln2, B, HW, C, heads, celu,
               status=None, trace=None, pair=False):
    """c1_hi / c1_lo [B*HW, 2C] fp16 rows the block's gate multiplies, x [B*HW, C] the block input; gate / in_proj /
    attn_gate = (w_hi, w_lo, acc_scale) fp16 weight operands (conv_weight_operand_f16), ln1 / ln2 = (gamma, beta), pos
    [HW, C] -> (x2 [B*HW, C] fp32, out_hi, out_lo): concat_elu(x2) as an fp16 pair [B*HW, 2C] when `celu`, else x2 as a
    pair [B*HW, C].  `pair` launches flowk_block_tail_pair_tc (HW = 256) instead of flowk_block_tail_tc."""
    M = B * HW
    # the kernel's tensor maps are built from B, HW and C: the tensors must have exactly these layouts
    assert c1_hi.dtype == c1_lo.dtype == torch.float16 and c1_hi.shape == c1_lo.shape == (M, 2 * C)
    assert c1_hi.is_contiguous() and c1_lo.is_contiguous()
    for (w_hi, w_lo, _), rows, k in ((gate, 2 * C, 2 * C), (in_proj, 3 * C, C), (attn_gate, 2 * C, C)):
        assert w_hi.dtype == w_lo.dtype == torch.float16 and w_hi.shape == w_lo.shape == (rows, (k + 63) // 64 * 64)
        assert w_hi.is_contiguous() and w_lo.is_contiguous()
    for t, shape in ((x, (M, C)), (pos, (HW, C)), (bias_g, (2 * C,)), (bias_a, (2 * C,)), (ln1[0], (C,)), (ln1[1], (C,)),
                     (ln2[0], (C,)), (ln2[1], (C,))):
        assert t.dtype == torch.float32 and tuple(t.shape) == shape and t.is_contiguous()
    _lib.check_device(c1_hi, "block_tail")
    x2 = torch.empty(M, C, device=x.device, dtype=torch.float32)
    width = 2 * C if celu else C
    hi = torch.empty(M, width, device=x.device, dtype=torch.float16)
    lo = torch.empty_like(hi)
    _lib.call("flowk_block_tail_pair_tc" if pair else "flowk_block_tail_tc", c1_hi.data_ptr(), c1_lo.data_ptr(), gate[0].data_ptr(), gate[1].data_ptr(),
              float(gate[2]), bias_g.data_ptr(), x.data_ptr(), ln1[0].data_ptr(), ln1[1].data_ptr(), pos.data_ptr(),
              in_proj[0].data_ptr(), in_proj[1].data_ptr(), float(in_proj[2]), attn_gate[0].data_ptr(),
              attn_gate[1].data_ptr(), float(attn_gate[2]), bias_a.data_ptr(), ln2[0].data_ptr(), ln2[1].data_ptr(),
              x2.data_ptr(), hi.data_ptr(), lo.data_ptr(), int(bool(celu)), B, HW, C, heads, _p(status), _p(trace),
              _stream())
    return x2, hi, lo


def block_tail_pair(c1_hi, c1_lo, gate, bias_g, x, ln1, pos, in_proj, attn_gate, bias_a, ln2, B, HW, C, heads, celu,
                    status=None, trace=None):
    """block_tail for 16x16 maps (HW = 256): one cluster of two CTAs per image (flowk_block_tail_pair_tc)."""
    return block_tail(c1_hi, c1_lo, gate, bias_g, x, ln1, pos, in_proj, attn_gate, bias_a, ln2, B, HW, C, heads, celu,
                      status=status, trace=trace, pair=True)
