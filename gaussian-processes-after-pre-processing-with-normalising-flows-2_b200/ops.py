"""torch.library custom ops over the C ABI of libflowk.so (include/flowk.h).

Each op allocates its outputs with torch, hands raw device pointers + the current CUDA
stream to one `extern "C"` entry point, and owns the autograd / fake-tensor rules.  The ops
are CUDA-only by construction (`device_types="cuda"`): a CPU tensor raises NotImplementedError
from the dispatcher instead of silently running somewhere else.
"""
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import _lib

_WS = {}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _workspace(dev: torch.device, batch: int) -> Tensor:
    """Zero-initialised log-det reduction workspace, one per (device, stream); the kernels leave it
    re-armed (include/flowk.h), so it is allocated and cleared once."""
    key = (dev.index, _stream())
    need = _lib.lib.flowk_ldj_workspace_bytes(int(batch))
    ws = _WS.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.zeros(max(need, 1 << 16), dtype=torch.uint8, device=dev)
        _WS[key] = ws
    return ws


def _f32c(t: Tensor, what: str) -> Tensor:
    if t.dtype != torch.float32:
        raise TypeError("%s: flowk kernels are float32 (got %s)" % (what, t.dtype))
    _lib.check_device(t, what)
    return t.contiguous()


def _hw(x: Tensor) -> int:
    n = 1
    for d in x.shape[2:]:
        n *= int(d)
    return n


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------------------------------------
# squeeze / unsqueeze
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowk::squeeze2d", mutates_args=(), device_types="cuda")
def squeeze2d(x: Tensor, factor: int) -> Tensor:
    x = _f32c(x, "squeeze2d")
    b, c, h, w = x.shape
    assert h % factor == 0 and w % factor == 0, "{}".format((h, w))
    y = x.new_empty(b, c * factor * factor, h // factor, w // factor)
    _lib.call("flowk_squeeze2d", x.data_ptr(), y.data_ptr(), b, c, h, w, factor, _stream())
    return y


@squeeze2d.register_fake
def _(x, factor):
    b, c, h, w = x.shape
    return x.new_empty(b, c * factor * factor, h // factor, w // factor)


@torch.library.custom_op("flowk::unsqueeze2d", mutates_args=(), device_types="cuda")
def unsqueeze2d(x: Tensor, factor: int) -> Tensor:
    x = _f32c(x, "unsqueeze2d")
    b, c, h, w = x.shape
    assert c % (factor * factor) == 0, "{}".format(c)
    y = x.new_empty(b, c // (factor * factor), h * factor, w * factor)
    _lib.call("flowk_unsqueeze2d", x.data_ptr(), y.data_ptr(), b, c, h, w, factor, _stream())
    return y


@unsqueeze2d.register_fake
def _(x, factor):
    b, c, h, w = x.shape
    return x.new_empty(b, c // (factor * factor), h * factor, w * factor)


def _squeeze_setup(ctx, inputs, output):
    ctx.factor = inputs[1]


squeeze2d.register_autograd(lambda ctx, g: (unsqueeze2d(g, ctx.factor), None), setup_context=_squeeze_setup)
unsqueeze2d.register_autograd(lambda ctx, g: (squeeze2d(g, ctx.factor), None), setup_context=_squeeze_setup)


# ------------------------------------------------------------------------------------------------
# ActNorm
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowk::actnorm_init", mutates_args=(), device_types="cuda")
def actnorm_init(x: Tensor, scale: float, eps: float) -> Tuple[Tensor, Tensor]:
    x = _f32c(x, "actnorm_init")
    b, c = x.shape[0], x.shape[1]
    hw = _hw(x)
    bias = x.new_empty(c)
    logs = x.new_empty(c)
    _lib.call("flowk_actnorm_init", x.data_ptr(), bias.data_ptr(), logs.data_ptr(), b, c, hw,
              float(scale), float(eps), _stream())
    return bias, logs


@actnorm_init.register_fake
def _(x, scale, eps):
    return x.new_empty(x.shape[1]), x.new_empty(x.shape[1])


@torch.library.custom_op("flowk::channel_scale", mutates_args=(), device_types="cuda")
def channel_scale(x: Tensor, pre: Tensor, mul: Tensor, post: Tensor, ldj: Tensor, ldj_add: Tensor
                  ) -> Tuple[Tensor, Tensor]:
    """y = (x + pre[c]) * mul[c] + post[c];  ldj_out = ldj + ldj_add."""
    x = _f32c(x, "channel_scale")
    b, c = x.shape[0], x.shape[1]
    hw = _hw(x)
    y = torch.empty_like(x)
    out = torch.empty_like(ldj)
    _lib.call("flowk_channel_scale", x.data_ptr(), _f32c(pre, "pre").data_ptr(), _f32c(mul, "mul").data_ptr(),
              _f32c(post, "post").data_ptr(), y.data_ptr(), _f32c(ldj, "ldj").data_ptr(),
              _f32c(ldj_add, "ldj_add").data_ptr(), out.data_ptr(), b, c, hw, _stream())
    return y, out


@channel_scale.register_fake
def _(x, pre, mul, post, ldj, ldj_add):
    return torch.empty_like(x), torch.empty_like(ldj)


def _cs_setup(ctx, inputs, output):
    x, pre, mul, post, ldj, ldj_add = inputs
    ctx.save_for_backward(x, pre, mul)


def _cs_backward(ctx, gy, gldj):
    x, pre, mul = ctx.saved_tensors
    shape = (1, -1) + (1,) * (x.dim() - 2)
    red = [0] + list(range(2, x.dim()))
    gx = gy * mul.view(shape)
    g_post = gy.sum(red)
    g_pre = g_post * mul
    g_mul = (gy * (x + pre.view(shape))).sum(red)
    return gx, g_pre, g_mul, g_post, gldj, gldj.sum().reshape(1)


channel_scale.register_autograd(_cs_backward, setup_context=_cs_setup)


# ------------------------------------------------------------------------------------------------
# channel mixing (1x1 conv, optionally with squeeze/unsqueeze folded in)
# ------------------------------------------------------------------------------------------------
def _mix_out_shape(x: Tensor, in_squeeze: bool, out_unsqueeze: bool) -> List[int]:
    b, c, h, w = x.shape
    if in_squeeze:
        return [b, c * 4, h // 2, w // 2]
    if out_unsqueeze:
        return [b, c // 4, h * 2, w * 2]
    return [b, c, h, w]


MIX_TC_MIN_ELEMENTS = int(__import__("os").environ.get("FLOWK_MIX_TC_MIN", str(1 << 23)))   # below: one launch of the
#                                          CUDA-core kernel is latency-bound either way (10-20 us at the named batch sizes)
MIX_TC_MIN_CHANNELS = 96
_MIX_W = {}


def _mix_on_tensor_cores(x: Tensor, c: int, h: int, w: int, in_squeeze: bool, out_unsqueeze: bool) -> bool:
    # measured (B200, working set >> L2): C = 96: 604 us on tcgen05 vs 704 us on CUDA cores; C = 48: 438 vs 194 us (the
    # NCHW <-> NHWC conversion and the NCHW epilogue on 4x4 maps cost more than the FMA bound) - so from C = 96 up only
    if in_squeeze or out_unsqueeze or c < MIX_TC_MIN_CHANNELS or c % 8 or x.numel() < MIX_TC_MIN_ELEMENTS:
        return False
    hw = h * w
    return w <= 128 and 128 % w == 0 and ((hw % 128 == 0) if hw >= 128 else (128 % hw == 0))


def _mix_weight_operand(weight: Tensor):
    """fp16 (hi, lo) operand of the [C, C] mixing matrix, cached per weight version (its scale needs one host read)."""
    key = (weight.data_ptr(), weight._version, _lib.GENERATION, tuple(weight.shape))
    hit = _MIX_W.get(weight.device)
    if hit is None or hit[0] != key:
        from . import tc
        hit = (key, tc.conv_weight_operand_f16(weight))
        _MIX_W[weight.device] = hit
    return hit[1]


@torch.library.custom_op("flowk::channel_mix", mutates_args=(), device_types="cuda")
def channel_mix(x: Tensor, weight: Tensor, bias: Optional[Tensor], ldj: Tensor, ldj_add: Tensor,
                in_squeeze: bool, out_unsqueeze: bool) -> Tuple[Tensor, Tensor]:
    """y[b,o,p] = sum_i weight[o,i] x[b,i,p] + bias[o];  ldj_out = ldj + ldj_add."""
    x = _f32c(x, "channel_mix")
    b, cx, hx, wx = x.shape
    if in_squeeze:
        assert hx % 2 == 0 and wx % 2 == 0, "{}".format((hx, wx))
        c, h, w = cx * 4, hx // 2, wx // 2
    else:
        c, h, w = cx, hx, wx
    if out_unsqueeze:
        assert c % 4 == 0, "{}".format(c)
    assert weight.shape[0] == c and weight.shape[1] == c, "weight must be [%d,%d]" % (c, c)
    y = x.new_empty(_mix_out_shape(x, in_squeeze, out_unsqueeze))
    if _mix_on_tensor_cores(x, c, h, w, in_squeeze, out_unsqueeze):
        # Wide 1x1 convs over large batches: the CUDA-core kernel is FP32-FMA-bound from C = 48 up (2 C^2 flop per 8 C bytes),
        # so the channel GEMM runs on tcgen05: NCHW -> NHWC fp16 (hi, lo) rows, implicit GEMM with taps = 1, NCHW epilogue.
        from . import tc
        a_hi, a_lo = tc.nchw_to_nhwc_hilo(x, c, True)
        w_hi, w_lo, sc = _mix_weight_operand(_f32c(weight, "weight"))
        tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, b, h, w, c, c, 1, tc.PRE_BIAS, tc.OUT_NCHW,
                     bias=None if bias is None else _f32c(bias, "bias"), out_nchw=y, acc_scale=sc)
        return y, ldj + ldj_add
    out = torch.empty_like(ldj)
    _lib.call("flowk_channel_mix", x.data_ptr(), _f32c(weight, "weight").data_ptr(),
              _ptr(None if bias is None else _f32c(bias, "bias")), y.data_ptr(), _f32c(ldj, "ldj").data_ptr(),
              _f32c(ldj_add, "ldj_add").data_ptr(), out.data_ptr(), b, c, h, w, int(in_squeeze),
              int(out_unsqueeze), _stream())
    return y, out


@channel_mix.register_fake
def _(x, weight, bias, ldj, ldj_add, in_squeeze, out_unsqueeze):
    return x.new_empty(_mix_out_shape(x, in_squeeze, out_unsqueeze)), torch.empty_like(ldj)


def _mix_setup(ctx, inputs, output):
    x, weight, bias, ldj, ldj_add, in_squeeze, out_unsqueeze = inputs
    ctx.save_for_backward(x, weight)
    ctx.flags = (in_squeeze, out_unsqueeze, bias is not None)


def _mix_backward(ctx, gy, gldj):
    x, weight = ctx.saved_tensors
    in_squeeze, out_unsqueeze, has_bias = ctx.flags
    gy = gy.contiguous()
    zero = gldj.new_zeros(1)
    # dL/dx = W^T gy, routed back through whichever index map the forward applied
    gx, _ = channel_mix(gy, weight.t().contiguous(), None, gldj, zero, out_unsqueeze, in_squeeze)
    xs = squeeze2d(x, 2) if in_squeeze else x
    gs = squeeze2d(gy, 2) if out_unsqueeze else gy
    g_w = torch.einsum("bop,bip->oi", gs.flatten(2), xs.flatten(2))
    g_b = gs.sum((0, 2, 3)) if has_bias else None
    return gx, g_w, g_b, gldj, gldj.sum().reshape(1), None, None


channel_mix.register_autograd(_mix_backward, setup_context=_mix_setup)


# ------------------------------------------------------------------------------------------------
# affine coupling arithmetic
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowk::affine_coupling", mutates_args=(), device_types="cuda")
def affine_coupling(x: Tensor, h: Tensor, ldj: Tensor, reverse: bool) -> Tuple[Tensor, Tensor]:
    x = _f32c(x, "affine_coupling")
    h = _f32c(h, "affine_coupling h")
    assert h.shape == x.shape, "conditioner output %s must match input %s" % (tuple(h.shape), tuple(x.shape))
    b, c = x.shape[0], x.shape[1]
    hw = _hw(x)
    y = torch.empty_like(x)
    out = torch.empty_like(ldj)
    fn = "flowk_affine_coupling_inv" if reverse else "flowk_affine_coupling_fwd"
    _lib.call(fn, x.data_ptr(), h.data_ptr(), y.data_ptr(), _f32c(ldj, "ldj").data_ptr(), out.data_ptr(),
              _workspace(x.device, b).data_ptr(), b, c, hw, _stream())
    return y, out


@affine_coupling.register_fake
def _(x, h, ldj, reverse):
    return torch.empty_like(x), torch.empty_like(ldj)


@torch.library.custom_op("flowk::affine_coupling_bwd", mutates_args=(), device_types="cuda")
def affine_coupling_bwd(x: Tensor, h: Tensor, gy: Tensor, gldj: Tensor) -> Tuple[Tensor, Tensor]:
    b, c = x.shape[0], x.shape[1]
    hw = _hw(x)
    gx = torch.empty_like(x)
    gh = torch.empty_like(h)
    _lib.call("flowk_affine_coupling_bwd", x.data_ptr(), h.data_ptr(), _f32c(gy, "gy").data_ptr(),
              _f32c(gldj, "gldj").data_ptr(), gx.data_ptr(), gh.data_ptr(), b, c, hw, _stream())
    return gx, gh


@affine_coupling_bwd.register_fake
def _(x, h, gy, gldj):
    return torch.empty_like(x), torch.empty_like(h)


def _aff_setup(ctx, inputs, output):
    x, h, ldj, reverse = inputs
    if reverse:
        ctx.reverse = True
        return
    ctx.reverse = False
    ctx.save_for_backward(x.contiguous(), h.contiguous())


def _aff_backward(ctx, gy, gldj):
    if ctx.reverse:
        raise RuntimeError("flowk::affine_coupling: the reverse (sampling) direction is inference-only")
    x, h = ctx.saved_tensors
    gx, gh = affine_coupling_bwd(x, h, gy, gldj)
    return gx, gh, gldj, None


affine_coupling.register_autograd(_aff_backward, setup_context=_aff_setup)


# ------------------------------------------------------------------------------------------------
# MixLogCDF coupling arithmetic
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowk::mixlogcdf_coupling", mutates_args=(), device_types="cuda")
def mixlogcdf_coupling(x: Tensor, raw: Tensor, rescale: Tensor, ldj: Tensor, reverse: bool, flip: bool,
                       num_components: int) -> Tuple[Tensor, Tensor]:
    x = _f32c(x, "mixlogcdf_coupling")
    raw = _f32c(raw, "mixlogcdf_coupling raw")
    b, c = x.shape[0], x.shape[1]
    hw = _hw(x)
    planes = 2 + 3 * num_components
    assert raw.shape[0] == b and raw.shape[1] == planes * (c // 2) and raw.numel() == b * planes * (c // 2) * hw, \
        "raw conditioner output %s does not match input %s" % (tuple(raw.shape), tuple(x.shape))
    y = torch.empty_like(x)
    out = torch.empty_like(ldj)
    fn = "flowk_mixlogcdf_inv" if reverse else "flowk_mixlogcdf_fwd"
    _lib.call(fn, x.data_ptr(), raw.data_ptr(), _f32c(rescale, "rescale").data_ptr(), y.data_ptr(),
              _f32c(ldj, "ldj").data_ptr(), out.data_ptr(), _workspace(x.device, b).data_ptr(),
              b, c, hw, num_components, int(flip), _stream())
    return y, out


@mixlogcdf_coupling.register_fake
def _(x, raw, rescale, ldj, reverse, flip, num_components):
    return torch.empty_like(x), torch.empty_like(ldj)


@torch.library.custom_op("flowk::mixlogcdf_coupling_bwd", mutates_args=(), device_types="cuda")
def mixlogcdf_coupling_bwd(x: Tensor, raw: Tensor, rescale: Tensor, gy: Tensor, gldj: Tensor, flip: bool,
                           num_components: int) -> Tuple[Tensor, Tensor, Tensor]:
    b, c = x.shape[0], x.shape[1]
    hw = _hw(x)
    gx = torch.empty_like(x)
    graw = torch.empty_like(raw)
    ga_tanh = x.new_empty(b, c // 2, hw)
    _lib.call("flowk_mixlogcdf_bwd", x.data_ptr(), raw.data_ptr(), rescale.data_ptr(), _f32c(gy, "gy").data_ptr(),
              _f32c(gldj, "gldj").data_ptr(), gx.data_ptr(), graw.data_ptr(), ga_tanh.data_ptr(),
              b, c, hw, num_components, int(flip), _stream())
    return gx, graw, ga_tanh.sum((0, 2))


@mixlogcdf_coupling_bwd.register_fake
def _(x, raw, rescale, gy, gldj, flip, num_components):
    return torch.empty_like(x), torch.empty_like(raw), x.new_empty(x.shape[1] // 2)


def _mix_c_setup(ctx, inputs, output):
    x, raw, rescale, ldj, reverse, flip, k = inputs
    ctx.reverse, ctx.flip, ctx.k = reverse, flip, k
    if not reverse:
        ctx.save_for_backward(x.contiguous(), raw.contiguous(), rescale.contiguous())


def _mix_c_backward(ctx, gy, gldj):
    if ctx.reverse:
        raise RuntimeError("flowk::mixlogcdf_coupling: the reverse (sampling) direction is inference-only")
    x, raw, rescale = ctx.saved_tensors
    gx, graw, gres = mixlogcdf_coupling_bwd(x, raw, rescale, gy, gldj, ctx.flip, ctx.k)
    return gx, graw, gres.view_as(rescale), gldj, None, None, None


mixlogcdf_coupling.register_autograd(_mix_c_backward, setup_context=_mix_c_setup)


# ------------------------------------------------------------------------------------------------
# Transformer_attn (patch attention), forward direction for training
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("flowk::patch_attention", mutates_args=(), device_types="cuda")
def patch_attention(x: Tensor, g: Tensor, prm: Tensor, ldj: Tensor, permute: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """y, ldj_out = Transformer_attn(x) with G = g [C, C], prm = {offset, offset2, offset3, scale}; `scores` [B, 8] are
    kept for the backward pass."""
    x = _f32c(x, "patch_attention")
    b, c, h, w = x.shape
    y = torch.empty_like(x)
    out = torch.empty_like(ldj)
    scores = x.new_empty(b, 8)
    _lib.call("flowk_patch_attention_train_fwd", x.data_ptr(), _f32c(g, "patch_attention G").data_ptr(),
              _f32c(prm, "patch_attention prm").data_ptr(), y.data_ptr(), _f32c(ldj, "ldj").data_ptr(), out.data_ptr(),
              scores.data_ptr(), b, c, h, w, int(permute), _stream())
    return y, out, scores


@patch_attention.register_fake
def _(x, g, prm, ldj, permute):
    return torch.empty_like(x), torch.empty_like(ldj), x.new_empty(x.shape[0], 8)


@torch.library.custom_op("flowk::patch_attention_bwd", mutates_args=(), device_types="cuda")
def patch_attention_bwd(x: Tensor, g: Tensor, prm: Tensor, scores: Tensor, gy: Tensor, gldj: Tensor,
                        permute: bool) -> Tuple[Tensor, Tensor]:
    """gx [B, C, H, W] and partials [B, C*C + 4]: per sample the gradient of G, then of offset, offset2, offset3, scale."""
    b, c, h, w = x.shape
    gx = torch.empty_like(x)
    partials = x.new_empty(b, c * c + 4)
    _lib.call("flowk_patch_attention_bwd", x.data_ptr(), g.data_ptr(), prm.data_ptr(), scores.data_ptr(),
              _f32c(gy, "gy").data_ptr(), _f32c(gldj, "gldj").data_ptr(), gx.data_ptr(), partials.data_ptr(),
              b, c, h, w, int(permute), _stream())
    return gx, partials


@patch_attention_bwd.register_fake
def _(x, g, prm, scores, gy, gldj, permute):
    return torch.empty_like(x), x.new_empty(x.shape[0], x.shape[1] * x.shape[1] + 4)


def _pa_setup(ctx, inputs, output):
    x, g, prm, ldj, permute = inputs
    ctx.permute = permute
    ctx.mark_non_differentiable(output[2])
    ctx.save_for_backward(x.contiguous(), g.contiguous(), prm.contiguous(), output[2])


def _pa_backward(ctx, gy, gldj, gscores):
    from .tc_autograd import channel_sum
    x, g, prm, scores = ctx.saved_tensors
    c = x.shape[1]
    gx, partials = patch_attention_bwd(x, g, prm, scores, gy, gldj, ctx.permute)
    red = channel_sum(partials, False)                     # deterministic fixed-order sum over the batch
    return gx, red[:c * c].view(c, c), red[c * c:], gldj, None


patch_attention.register_autograd(_pa_backward, setup_context=_pa_setup)


# ------------------------------------------------------------------------------------------------
# log_dist functions on explicit [B,K,...] parameter tensors
# ------------------------------------------------------------------------------------------------
def _mixture_call(fn: str, x: Tensor, pi: Tensor, mu: Tensor, s: Tensor) -> Tensor:
    x = _f32c(x, fn)
    b, k = pi.shape[0], pi.shape[1]
    n = 1
    for d in x.shape[1:]:
        n *= int(d)
    assert pi.shape == mu.shape == s.shape and pi.numel() == b * k * n, "parameter tensors must be [B,K,*x.shape[1:]]"
    out = torch.empty_like(x)
    _lib.call(fn, x.data_ptr(), _f32c(pi, "pi").data_ptr(), _f32c(mu, "mu").data_ptr(), _f32c(s, "s").data_ptr(),
              out.data_ptr(), b, k, n, _stream())
    return out


@torch.library.custom_op("flowk::mixture_log_cdf", mutates_args=(), device_types="cuda")
def mixture_log_cdf(x: Tensor, pi: Tensor, mu: Tensor, s: Tensor) -> Tensor:
    return _mixture_call("flowk_mixture_log_cdf", x, pi, mu, s)


@torch.library.custom_op("flowk::mixture_log_pdf", mutates_args=(), device_types="cuda")
def mixture_log_pdf(x: Tensor, pi: Tensor, mu: Tensor, s: Tensor) -> Tensor:
    return _mixture_call("flowk_mixture_log_pdf", x, pi, mu, s)


@torch.library.custom_op("flowk::mixture_inv_cdf", mutates_args=(), device_types="cuda")
def mixture_inv_cdf(y: Tensor, pi: Tensor, mu: Tensor, s: Tensor) -> Tensor:
    return _mixture_call("flowk_mixture_inv_cdf", y, pi, mu, s)


for _op in (mixture_log_cdf, mixture_log_pdf, mixture_inv_cdf):
    _op.register_fake(lambda x, pi, mu, s: torch.empty_like(x))
