"""Training path of the MixLogCDF conditioner on libflowk: `autograd.Function`s whose forward AND backward are C-ABI calls.

The training forward keeps torch's module graph (so dropout semantics, autograd and the reference's module tree stay), but
every kernel between the flow-level ops is ours:

    wn_conv2d / wn_linear    weight norm + operand construction (batched over the model: `WeightNormBatch`), forward GEMM,
                             input-gradient GEMM (taps flipped, weight transposed), weight-gradient GEMM (tcgen05 split-K:
                             `flowk_conv_wgrad` on NCHW operands, `flowk_linear_wgrad` on row-major MN-major operands),
                             weight-norm backward fused with the split-K reduction, bias gradient
    concat_elu / glu         one pass each way
    add_layernorm            residual + LayerNorm + the block's NCHW<->NHWC permutes, forward / backward
    attention_core           softmax(q k^T / sqrt d) with weight dropout times v: flash-style forward + two backward kernels,
                             dropout mask regenerated from a counter-based hash (`advance_dropout_seed` once per step)

All of them are fp32-accurate (3xTF32 split on the tensor cores) and deterministic (no atomics).  `conv2d` / `linear`
(without weight norm) are the plain building blocks, used by tests.  Unsupported shapes fall back to the torch layers in
`flow_modules/` - never to a CPU path.
"""
import ctypes

import torch

from . import _lib, tc

ENABLED = True
FWD_F16 = __import__("os").environ.get("FLOWK_TRAIN_FWD_F16", "1") != "0"
# Forward GEMMs of the batched weight-norm path on fp16 (hi, lo) operand pairs (FLOWK_OPERAND_F16: half the operand bytes and
# MMA instructions, the same 22 significant bits; activations are O(1) in magnitude and the weights are scaled on the device).
# Gradient GEMMs stay on TF32 pairs: gradients need fp32's exponent range.


def conv_supported(x, w):
    if not (ENABLED and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4):
        return False
    n, cin, kh, kw = w.shape
    if (kh, kw) not in ((1, 1), (3, 3)) or n < 1 or cin < 1:          # both serve as the GEMM N (forward / dgrad)
        return False
    b, _, h, ww = x.shape
    if ww > 128 or 128 % ww:
        return False
    hw = h * ww
    return (hw % 128 == 0) if hw >= 128 else (128 % hw == 0)


def _nchw_operand(x, c_pad):
    x = x.contiguous()
    return tc.nchw_to_nhwc_hilo(x, c_pad)


def _pad32(c):
    return (c + 31) // 32 * 32


class _Conv2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, bias):
        b, cin, h, ww = x.shape
        n, _, kh, kw = w.shape
        taps = kh * kw
        cp = _pad32(cin)
        a_hi, a_lo = _nchw_operand(x, cp)
        w_hi, w_lo = tc.conv_weight_operand(w.detach(), cp)
        y = torch.empty(b, n, h, ww, device=x.device, dtype=torch.float32)
        tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, b, h, ww, cp, n, taps, tc.PRE_BIAS, tc.OUT_NCHW,
                     bias=None if bias is None else bias.detach().contiguous(), out_nchw=y, split_k=True)
        ctx.save_for_backward(x, w)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        b, cin, h, ww = x.shape
        n, _, kh, kw = w.shape
        taps = kh * kw
        gy = gy.contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            # dL/dx = conv(dL/dy, w^T with the taps flipped): weight [cin, n, kh, kw] from w[n, cin, ::-1, ::-1]
            np_ = _pad32(n)
            g_hi, g_lo = _nchw_operand(gy, np_)
            wt = w.detach().flip(2, 3).permute(1, 0, 2, 3).contiguous()
            wt_hi, wt_lo = tc.conv_weight_operand(wt, np_)
            gx = torch.empty(x.shape, device=x.device, dtype=torch.float32)      # contiguous NCHW whatever x's strides
            tc.conv_gemm(g_hi, g_lo, wt_hi, wt_lo, b, h, ww, np_, cin, taps, tc.PRE_BIAS, tc.OUT_NCHW, out_nchw=gx, split_k=True)
        if ctx.needs_input_grad[1]:
            partial = wgrad_partials(x.contiguous(), gy, taps)
            if partial is not None:                      # tcgen05 split-K slices [S, taps, N, Cin] (or [S, taps, Cin, N])
                p, transposed = partial
                gw = p.sum(0)
                gw = (gw.permute(2, 1, 0) if transposed else gw.permute(1, 2, 0)).reshape(n, cin, kh, kw).contiguous()
            else:
                _lib.library_fallback("conv weight gradient %s" % (tuple(w.shape),), x)
                gw = torch.nn.grad.conv2d_weight(x, w.shape, gy, padding=kh // 2)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = channel_sum(gy, True)
        return gx, gw, gb


def conv2d(x, w, bias, padding):
    """F.conv2d(x, w, bias, padding='same') for 1x1 / 3x3 kernels, stride 1."""
    assert padding == w.shape[2] // 2
    return _Conv2d.apply(x, w, bias)


def linear_supported(x, w):
    if not (ENABLED and x.is_cuda and x.dtype == torch.float32):
        return False
    m = x.numel() // x.shape[-1]
    return m % 16 == 0 and w.shape[0] % 4 == 0 and w.shape[1] % 32 == 0 and x.shape[-1] == w.shape[1]


def _rows_as_images(m):
    """[m, K] rows as the (B, H, W) "image" grid flowk_conv_gemm tiles over (taps = 1: positions are independent): whole
    128-row tiles when m % 128 == 0, else images of gcd(m, 128) rows (the TMA unit zero-fills the tile's missing images)."""
    if m % 128 == 0:
        return m // 128, 8, 16
    hw = 128
    while m % hw:
        hw //= 2
    w = min(hw, 16)
    return m // hw, hw // w, w


def _rows_gemm(a, wmat, bias, n):
    """[M, K] rows (K % 32 == 0, M % 128 == 0) times wmat[n, K]^T -> [M, n] fp32."""
    m, k = a.shape
    a_hi, a_lo = tc.split_rows(a.contiguous())
    w_hi, w_lo = tc.split_hilo(wmat)
    y = torch.empty(m, n, device=a.device, dtype=torch.float32)
    tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, *_rows_as_images(m), k, n, 1, tc.PRE_BIAS, tc.OUT_F32, bias=bias, out_f32=y, split_k=True)
    return y


class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, bias):
        shape = x.shape
        x2 = x.reshape(-1, shape[-1])
        y = _rows_gemm(x2, w.detach(), None if bias is None else bias.detach().contiguous(), w.shape[0])
        ctx.save_for_backward(x2, w)
        ctx.has_bias = bias is not None
        ctx.shape = shape
        return y.view(*shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, gy):
        x2, w = ctx.saved_tensors
        n, k = w.shape
        g2 = gy.reshape(-1, n).contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            if n % 32 == 0:
                gx = _rows_gemm(g2, w.detach().t().contiguous(), None, k).view(ctx.shape)
            else:
                _lib.library_fallback("linear input gradient, N=%d" % n, g2)
                gx = (g2 @ w).view(ctx.shape)
        if ctx.needs_input_grad[1]:
            partial = linear_wgrad_partials(x2, g2)
            if partial is not None:
                p, transposed = partial
                gw = p.sum(0)[0]
                gw = gw.t().contiguous() if transposed else gw
            else:
                _lib.library_fallback("linear weight gradient [%d, %d]" % (n, k), g2)
                gw = g2.t() @ x2
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = channel_sum(g2, False)
        return gx, gw, gb


def linear(x, w, bias):
    return _Linear.apply(x, w, bias)


def channel_sum(x, nchw):
    """Bias gradient: x [B, C, H, W] summed over (0, 2, 3) when nchw, else rows [M, C] summed over 0; contiguous fp32."""
    if nchw:
        outer, c, inner = x.shape[0], x.shape[1], x.shape[2] * x.shape[3]
    else:
        outer, c, inner = x.shape[0], x.shape[1], 1
    out = torch.empty(c, device=x.device, dtype=torch.float32)
    ws = torch.empty(_lib.lib.flowk_channel_sum_workspace_bytes(c) // 4, device=x.device, dtype=torch.float32)
    _lib.call("flowk_channel_sum", x.data_ptr(), out.data_ptr(), ws.data_ptr(), outer, c, inner, tc._stream())
    return out


def _wn_operands(v, g, cin_pad, n_pad, want_w=False, want_dg=True):
    """Fused weight norm + GEMM operands (two launches): returns norm, w (or None), (fwd_hi, fwd_lo), (dg_hi, dg_lo)."""
    n, cin = v.shape[0], v.shape[1]
    taps = v.numel() // (n * cin)
    dev = v.device
    norm = torch.empty(n, device=dev, dtype=torch.float32)
    w = torch.empty(v.shape, device=dev, dtype=torch.float32) if want_w else None
    fwd = torch.empty(2, n, taps * cin_pad, device=dev, dtype=torch.float32)
    dg = torch.empty(2, cin, taps * n_pad, device=dev, dtype=torch.float32) if want_dg else None
    _lib.call("flowk_weight_norm_operands", v.data_ptr(), g.data_ptr(), n, cin, taps, cin_pad, n_pad, norm.data_ptr(),
              tc._p(w), fwd[0].data_ptr(), fwd[1].data_ptr(), None if dg is None else dg[0].data_ptr(),
              None if dg is None else dg[1].data_ptr(), tc._stream())
    return norm, w, fwd, dg


WGRAD_LINEAR_TC = True    # Linear weight gradients on the tcgen05 kernel, row-major operands as MN-major tiles
WGRAD_TC = True      # weight gradients on the tcgen05 split-K kernels (False: torch.nn.grad.conv2d_weight / matmul, for A/B tests)


def wgrad_partials(x_cm, gy_cm, taps):
    """Split-K partial weight gradients from channel-major fp32 x [B,Cin,H,W], gy [B,N,H,W]: (partial, transposed) with
    partial [S, taps, N, Cin] (or [S, taps, Cin, N] when transposed); None when the tcgen05 kernel does not take the shape."""
    b, cin, h, w = x_cm.shape
    n = gy_cm.shape[1]
    if not WGRAD_TC:
        return None
    transposed = ctypes.c_int(0)
    splits = _lib.lib.flowk_conv_wgrad_splits(b, h, w, cin, n, taps, ctypes.byref(transposed))
    if splits <= 0:
        return None
    transposed = bool(transposed.value)
    partial = torch.empty((splits, taps, cin, n) if transposed else (splits, taps, n, cin), device=x_cm.device,
                          dtype=torch.float32)
    xl = xr = None
    if taps == 9:
        shifted = torch.empty((2,) + tuple(x_cm.shape), device=x_cm.device, dtype=torch.float32)
        xl, xr = shifted[0], shifted[1]
        _lib.call("flowk_shift_columns", x_cm.data_ptr(), xl.data_ptr(), xr.data_ptr(), x_cm.numel(), w, tc._stream())
    _lib.call("flowk_conv_wgrad", x_cm.data_ptr(), tc._p(xl), tc._p(xr), gy_cm.data_ptr(), partial.data_ptr(), None,
              b, h, w, cin, n, taps, tc._stream())
    return partial, transposed


def linear_wgrad_partials(x2, g2):
    """Split-K partial weight gradients of y = x2 @ w^T from row-major x2 [M, K], g2 [M, N]: (partial, transposed) with
    partial [S, 1, N, K] (or [S, 1, K, N]); None when the tcgen05 kernel does not take the shape."""
    m, k = x2.shape
    n = g2.shape[1]
    if not (WGRAD_TC and WGRAD_LINEAR_TC):
        return None
    transposed = ctypes.c_int(0)
    splits = _lib.lib.flowk_linear_wgrad_splits(m, k, n, ctypes.byref(transposed))
    if splits <= 0:
        return None
    transposed = bool(transposed.value)
    partial = torch.empty((splits, 1, k, n) if transposed else (splits, 1, n, k), device=x2.device, dtype=torch.float32)
    _lib.call("flowk_linear_wgrad", x2.data_ptr(), g2.data_ptr(), partial.data_ptr(), None, m, k, n, tc._stream())
    return partial, transposed


def _wn_backward_partials(v, g, norm, partial_t):
    partial, transposed = partial_t
    n, cin = v.shape[0], v.shape[1]
    taps = v.numel() // (n * cin)
    gv = torch.empty(v.shape, device=v.device, dtype=torch.float32)
    gg = torch.empty(g.shape, device=v.device, dtype=torch.float32)
    _lib.call("flowk_weight_norm_bwd_partials", v.data_ptr(), g.data_ptr(), norm.data_ptr(), partial.data_ptr(),
              gv.data_ptr(), gg.data_ptr(), n, cin, taps, partial.shape[0], int(transposed), tc._stream())
    return gv, gg


def _wn_backward(v, g, norm, gw):
    gv = torch.empty(v.shape, device=v.device, dtype=torch.float32)
    gg = torch.empty(g.shape, device=v.device, dtype=torch.float32)
    _lib.call("flowk_weight_norm_bwd", v.data_ptr(), g.data_ptr(), norm.data_ptr(), gw.contiguous().data_ptr(),
              gv.data_ptr(), gg.data_ptr(), v.shape[0], v.numel() // v.shape[0], tc._stream())
    return gv, gg


OVERLAP_WGRAD = True      # backward: weight/bias-gradient kernels on a side stream, concurrent with the input-gradient GEMM
_SIDE = {}


class _fork_wgrad:
    """`with _fork_wgrad(device): ...` runs the body on a side stream that has waited for the current one; `join()` makes
    the current stream wait for it.  The two gradient chains of a layer are independent, and below level 1 neither fills
    the GPU.  (Capturable: inside a CUDA graph the fork becomes a parallel branch.)"""

    def __init__(self, device):
        self.on = OVERLAP_WGRAD
        if self.on:
            self.main = torch.cuda.current_stream(device)
            side = _SIDE.get(device)
            if side is None:
                side = _SIDE[device] = torch.cuda.Stream(device)
            self.side = side
            self.ctx = torch.cuda.stream(side)

    def __enter__(self):
        if self.on:
            self.side.wait_stream(self.main)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.on:
            self.ctx.__exit__(*exc)
        return False

    def join(self):
        if self.on:
            self.main.wait_stream(self.side)


class WeightNormBatch:
    """All weight-normalised conv / Linear layers of a model, normalised and turned into GEMM operands in TWO launches
    per training step (instead of two per layer).  `refresh()` fills the preallocated outputs and hands each module its
    (norm, w, fwd, dg) tuple through `module._prepared`; the module's next forward consumes it (one use per refresh, so
    a forward that was not preceded by a refresh falls back to the per-layer path and can never see stale weights)."""

    def __init__(self, modules):
        self.modules = [m for m in modules if self._eligible(m)]
        self._key = None
        self._build()

    @staticmethod
    def _eligible(m):
        v = m.weight_v
        if not (ENABLED and v.is_cuda and v.dtype == torch.float32 and v.dim() in (2, 4)):
            return False
        n, cin = v.shape[0], v.shape[1]
        if v.dim() == 4:
            return (v.shape[2], v.shape[3]) in ((1, 1), (3, 3)) and n >= 1 and cin >= 1
        return n % 4 == 0 and cin % 32 == 0

    def _pointers(self):
        return tuple((m.weight_v.data_ptr(), m.weight_g.data_ptr()) for m in self.modules)

    def _build(self):
        self._key = self._pointers()
        self.slots = []
        if not self.modules:
            return
        dev = self.modules[0].weight_v.device
        jobs = (_lib.WnJob * len(self.modules))()
        self.max_rows = 1
        # one buffer for every layer's [row norms | max |w| scratch | acc_scale]: a single fill resets all the scratch words
        offs = [0]
        for m in self.modules:
            offs.append(offs[-1] + (m.weight_v.shape[0] + 2 + 3) // 4 * 4)
        self.norms = torch.zeros(offs[-1], device=dev, dtype=torch.float32)
        for i, m in enumerate(self.modules):
            v, g = m.weight_v, m.weight_g
            n, cin = v.shape[0], v.shape[1]
            taps = v.numel() // (n * cin)
            linear = v.dim() == 2
            f16 = FWD_F16 and cin % 8 == 0
            cin_pad = (cin + 63) // 64 * 64 if f16 else (cin if linear else _pad32(cin))
            n_pad = n if linear else _pad32(n)
            want_w = linear and n % 32 != 0                      # the Linear dgrad falls back to g2 @ w
            norm = self.norms[offs[i]:offs[i] + n + 2]
            w = torch.empty(v.shape, device=dev, dtype=torch.float32) if want_w else None
            fwd = torch.empty(2, n, taps * cin_pad, device=dev, dtype=torch.float16 if f16 else torch.float32)
            dg = None if want_w else torch.empty(2, cin, taps * n_pad, device=dev, dtype=torch.float32)
            jobs[i] = _lib.WnJob(v.data_ptr(), g.data_ptr(), norm.data_ptr(), tc._p(w), fwd[0].data_ptr(), fwd[1].data_ptr(),
                                 None if dg is None else dg[0].data_ptr(), None if dg is None else dg[1].data_ptr(),
                                 n, cin, taps, cin_pad, n_pad, int(f16))
            self.max_rows = max(self.max_rows, n)
            self.slots.append((norm, w, fwd, dg))
        raw = bytes(jobs)
        self.table = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)

    def refresh(self):
        if not self.modules:
            return
        if self._pointers() != self._key:          # parameters were re-allocated (.to(), load with assign=True, ...)
            self._build()
        self.norms.zero_()                          # the per-layer max |w| words accumulate by atomicMax
        _lib.call("flowk_weight_norm_operands_batched", self.table.data_ptr(), len(self.modules), self.max_rows,
                  tc._stream())
        for m, slot in zip(self.modules, self.slots):
            m._prepared = slot


def take_prepared(module):
    """The (norm, w, fwd, dg) tuple the last WeightNormBatch.refresh() left for this module, at most once."""
    slot = getattr(module, "_prepared", None)
    if slot is not None:
        module._prepared = None
    return slot


class _WNConv2d(torch.autograd.Function):
    """conv2d(x, v * g / ||v||, bias) with weight norm, operand construction, forward and dgrad on libflowk."""

    @staticmethod
    def forward(ctx, x, v, g, bias, prepared=None):
        b, cin, h, ww = x.shape
        n, _, kh, kw = v.shape
        cp, np_ = _pad32(cin), _pad32(n)
        vd, gd = v.detach().contiguous(), g.detach().contiguous()
        if prepared is not None:
            norm, _, fwd, dg = prepared
        else:
            norm, _, fwd, dg = _wn_operands(vd, gd, cp, np_, want_dg=ctx.needs_input_grad[0])
        y = torch.empty(b, n, h, ww, device=x.device, dtype=torch.float32)
        bias_d = None if bias is None else bias.detach().contiguous()
        if fwd.dtype == torch.float16:              # batched operands in fp16 pairs; norm = [row norms | scratch | acc_scale]
            c8 = (cin + 7) // 8 * 8
            a_hi, a_lo = tc.nchw_to_nhwc_hilo(x.contiguous(), c8, True)
            tc.conv_gemm(a_hi, a_lo, fwd[0], fwd[1], b, h, ww, c8, n, kh * kw, tc.PRE_BIAS, tc.OUT_NCHW, bias=bias_d,
                         out_nchw=y, acc_scale=1.0, acc_scale_ptr=norm[n + 1:])
            norm = norm[:n]
        else:
            a_hi, a_lo = _nchw_operand(x, cp)
            tc.conv_gemm(a_hi, a_lo, fwd[0], fwd[1], b, h, ww, cp, n, kh * kw, tc.PRE_BIAS, tc.OUT_NCHW, bias=bias_d,
                         out_nchw=y, split_k=True)
        ctx.save_for_backward(x, vd, gd, norm, dg)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, v, g, norm, dg = ctx.saved_tensors
        b, cin, h, ww = x.shape
        n, _, kh, kw = v.shape
        gy = gy.contiguous()
        gx = gv = gg = gb = None
        fork = _fork_wgrad(x.device)
        with fork:                                  # side stream: weight and bias gradients
            if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
                partial = wgrad_partials(x.contiguous(), gy, kh * kw)
                if partial is not None:
                    gv, gg = _wn_backward_partials(v, g, norm, partial)
                else:
                    _lib.library_fallback("conv weight gradient %s" % (tuple(v.shape),), x)
                    gv, gg = _wn_backward(v, g, norm, torch.nn.grad.conv2d_weight(x, v.shape, gy, padding=kh // 2))
            if ctx.has_bias and ctx.needs_input_grad[3]:
                gb = channel_sum(gy, True)
        if ctx.needs_input_grad[0]:                 # main stream: input gradient
            np_ = _pad32(n)
            g_hi, g_lo = _nchw_operand(gy, np_)
            gx = torch.empty(x.shape, device=x.device, dtype=torch.float32)
            tc.conv_gemm(g_hi, g_lo, dg[0], dg[1], b, h, ww, np_, cin, kh * kw, tc.PRE_BIAS, tc.OUT_NCHW, out_nchw=gx, split_k=True)
        fork.join()
        return gx, gv, gg, gb, None


class _WNLinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, v, g, bias, prepared=None):
        shape = x.shape
        n, k = v.shape
        x2 = x.reshape(-1, k).contiguous()
        vd, gd = v.detach().contiguous(), g.detach().contiguous()
        tc_dgrad = n % 32 == 0
        if prepared is not None:
            norm, w, fwd, dg = prepared
        else:
            norm, w, fwd, dg = _wn_operands(vd, gd, k, n, want_w=not tc_dgrad, want_dg=tc_dgrad)
        y = torch.empty(x2.shape[0], n, device=x.device, dtype=torch.float32)
        bias_d = None if bias is None else bias.detach().contiguous()
        if fwd.dtype == torch.float16:
            a_hi, a_lo = tc.split_rows_f16(x2)
            tc.conv_gemm(a_hi, a_lo, fwd[0], fwd[1], *_rows_as_images(x2.shape[0]), k, n, 1, tc.PRE_BIAS, tc.OUT_F32,
                         bias=bias_d, out_f32=y, acc_scale=1.0, acc_scale_ptr=norm[n + 1:])
            norm = norm[:n]
        else:
            a_hi, a_lo = tc.split_rows(x2)
            tc.conv_gemm(a_hi, a_lo, fwd[0], fwd[1], *_rows_as_images(x2.shape[0]), k, n, 1, tc.PRE_BIAS, tc.OUT_F32,
                         bias=bias_d, out_f32=y, split_k=True)
        ctx.save_for_backward(x2, vd, gd, norm, dg if tc_dgrad else w)
        ctx.tc_dgrad, ctx.has_bias, ctx.shape = tc_dgrad, bias is not None, shape
        return y.view(*shape[:-1], n)

    @staticmethod
    def backward(ctx, gy):
        x2, v, g, norm, wd = ctx.saved_tensors
        n, k = v.shape
        g2 = gy.reshape(-1, n).contiguous()
        gx = gv = gg = gb = None
        fork = _fork_wgrad(g2.device)
        with fork:                                  # side stream: weight and bias gradients
            if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
                partial = linear_wgrad_partials(x2, g2)
                if partial is not None:
                    gv, gg = _wn_backward_partials(v, g, norm, partial)
                else:
                    _lib.library_fallback("linear weight gradient [%d, %d]" % (n, k), g2)
                    gv, gg = _wn_backward(v, g, norm, g2.t() @ x2)
            if ctx.has_bias and ctx.needs_input_grad[3]:
                gb = channel_sum(g2, False)
        if ctx.needs_input_grad[0]:                 # main stream: input gradient
            if ctx.tc_dgrad:
                g_hi, g_lo = tc.split_rows(g2)
                gx = torch.empty(g2.shape[0], k, device=g2.device, dtype=torch.float32)
                tc.conv_gemm(g_hi, g_lo, wd[0], wd[1], *_rows_as_images(g2.shape[0]), n, k, 1, tc.PRE_BIAS, tc.OUT_F32,
                             out_f32=gx, split_k=True)
                gx = gx.view(ctx.shape)
            else:
                _lib.library_fallback("linear input gradient, N=%d" % n, g2)
                gx = (g2 @ wd).view(ctx.shape)
        fork.join()
        return gx, gv, gg, gb, None


def wn_conv2d(x, v, g, bias, prepared=None):
    """F.conv2d(x, weight_norm(v, g), bias, padding='same'), 1x1 / 3x3, stride 1 (mixlogcdf_nn.py:12-29)."""
    return _WNConv2d.apply(x, v, g, bias, prepared)


def wn_linear(x, v, g, bias, prepared=None):
    return _WNLinearFn.apply(x, v, g, bias, prepared)


def _oci(x, dim):
    """(outer, channels, inner) view of splitting / concatenating along `dim`."""
    dim = dim % x.dim()
    outer = 1
    for d in x.shape[:dim]:
        outer *= int(d)
    inner = 1
    for d in x.shape[dim + 1:]:
        inner *= int(d)
    return outer, int(x.shape[dim]), inner


class _ConcatElu(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, dim, mask):
        x = x.contiguous()
        outer, c, inner = _oci(x, dim)
        shape = list(x.shape)
        shape[dim] = 2 * c
        y = torch.empty(shape, device=x.device, dtype=torch.float32)
        _lib.call("flowk_concat_elu_fwd", x.data_ptr(), y.data_ptr(), tc._p(mask), outer, c, inner, tc._stream())
        ctx.save_for_backward(x, mask)
        ctx.dim = dim
        return y

    @staticmethod
    def backward(ctx, gy):
        x, mask = ctx.saved_tensors
        outer, c, inner = _oci(x, ctx.dim)
        gx = torch.empty_like(x)
        _lib.call("flowk_concat_elu_bwd", x.data_ptr(), gy.contiguous().data_ptr(), gx.data_ptr(), tc._p(mask), outer, c, inner,
                  tc._stream())
        return gx, None, None


class _Glu(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, dim):
        x = x.contiguous()
        outer, c2, inner = _oci(x, dim)
        shape = list(x.shape)
        shape[dim] = c2 // 2
        y = torch.empty(shape, device=x.device, dtype=torch.float32)
        _lib.call("flowk_glu_fwd", x.data_ptr(), y.data_ptr(), outer, c2 // 2, inner, tc._stream())
        ctx.save_for_backward(x)
        ctx.dim = dim
        return y

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        outer, c2, inner = _oci(x, ctx.dim)
        gx = torch.empty_like(x)
        _lib.call("flowk_glu_bwd", x.data_ptr(), gy.contiguous().data_ptr(), gx.data_ptr(), outer, c2 // 2, inner,
                  tc._stream())
        return gx, None


class _AddLayerNorm(torch.autograd.Function):
    """y = LayerNorm_C(a + b); a, b NCHW [B,C,H,W] (in_nchw) or NHWC [B,H,W,C]; y NCHW or NHWC by out_nchw."""

    @staticmethod
    def forward(ctx, a, b, gamma, beta, eps, in_nchw, out_nchw):
        a, b = a.contiguous(), b.contiguous()
        if in_nchw:
            bsz, c, h, w = a.shape
        else:
            bsz, h, w, c = a.shape
        m, hw = bsz * h * w, h * w
        dev = a.device
        y = torch.empty((bsz, c, h, w) if out_nchw else (bsz, h, w, c), device=dev, dtype=torch.float32)
        s = torch.empty(m, c, device=dev, dtype=torch.float32)
        stats = torch.empty(2, m, device=dev, dtype=torch.float32)
        gd, bd = gamma.detach().contiguous(), beta.detach().contiguous()
        _lib.call("flowk_add_layernorm_fwd", a.data_ptr(), b.data_ptr(), gd.data_ptr(), bd.data_ptr(), y.data_ptr(),
                  s.data_ptr(), stats[0].data_ptr(), stats[1].data_ptr(), m, c, hw, int(in_nchw), int(out_nchw),
                  float(eps), tc._stream())
        ctx.save_for_backward(s, stats, gd)
        ctx.cfg = (tuple(a.shape), m, c, hw, in_nchw, out_nchw)
        return y

    @staticmethod
    def backward(ctx, gy):
        s, stats, gamma = ctx.saved_tensors
        shape, m, c, hw, in_nchw, out_nchw = ctx.cfg
        dev = gy.device
        gs = torch.empty(shape, device=dev, dtype=torch.float32)
        dgb = torch.empty(2, c, device=dev, dtype=torch.float32)
        ws = torch.empty(_lib.lib.flowk_add_layernorm_workspace_bytes(m, c) // 4, device=dev, dtype=torch.float32)
        _lib.call("flowk_add_layernorm_bwd", gy.contiguous().data_ptr(), s.data_ptr(), stats[0].data_ptr(),
                  stats[1].data_ptr(), gamma.data_ptr(), gs.data_ptr(), dgb[0].data_ptr(), dgb[1].data_ptr(),
                  ws.data_ptr(), m, c, hw, int(in_nchw), int(out_nchw), tc._stream())
        return gs, gs, dgb[0], dgb[1], None, None, None


def add_layernorm(a, b, norm, in_nchw, out_nchw):
    """`norm(a + b)` for an nn.LayerNorm over the channel dim, with the NCHW<->NHWC permutes of ConvAttnBlock folded in."""
    return _AddLayerNorm.apply(a, b, norm.weight, norm.bias, norm.eps, in_nchw, out_nchw)


_DROPOUT_SEED = {}


def dropout_seed(device):
    """Per-device scalar the attention-dropout masks are keyed on; `advance_dropout_seed` bumps it once per training
    step ON THE DEVICE, so a captured CUDA graph draws fresh masks at every replay.  (The backward pass re-reads it: run
    backward before the next training forward.)"""
    t = _DROPOUT_SEED.get(device)
    if t is None:
        t = torch.randint(0, 2 ** 31 - 1, (1,), dtype=torch.int32).to(device)
        _DROPOUT_SEED[device] = t
    return t


def advance_dropout_seed(device):
    dropout_seed(device).add_(1)


def attention_train_supported(qkv, heads):
    if not (ENABLED and ATTENTION_TC and qkv.is_cuda and qkv.dtype == torch.float32 and qkv.dim() == 3):
        return False
    b, s, c3 = qkv.shape
    c = c3 // 3
    return c3 % 3 == 0 and c % heads == 0 and c // heads in (8, 16, 24, 32, 40, 64) and s % 8 == 0 and \
        b * heads * s * s < 2 ** 32 - 1


# the two attention backward kernels are independent and may run on two streams; measured: no gain (62.2 vs 61-63 ms/step,
# both already fill the GPU at level 1), so they stay on one stream unless FLOWK_ATTN_FORK=1
ATTENTION_BWD_FORK = __import__("os").environ.get("FLOWK_ATTN_FORK", "0") == "1"
FOLD_DROPOUT = __import__("os").environ.get("FLOWK_FOLD_DROPOUT", "1") != "0"   # Dropout2d folded into concat_elu
ATTENTION_TC = True      # training attention core (softmax(q k^T) v with dropout, forward + backward) on the flowk kernels


def _attention_train_entry(seq, head_dim):
    """Head dim 64 at 128 / 256 tokens runs on the tcgen05 kernels (csrc/attention_train_tc.cu); every other admitted shape,
    head dim 64 at the shorter sequences of the deep levels included, on the mma.sync kernels (csrc/attention_train.cu)."""
    return "flowk_attention_train_tc" if head_dim == 64 and seq in (128, 256) else "flowk_attention_train"


class _AttentionCore(torch.autograd.Function):
    """att = dropout(softmax(q k^T / sqrt(d))) v per (image, head); qkv [B, S, 3C] rows in (k | v | q) order -> [B, S, C]."""

    @staticmethod
    def forward(ctx, qkv, heads, p_drop, salt):
        qkv = qkv.contiguous()
        b, s, c3 = qkv.shape
        c = c3 // 3
        out = torch.empty(b, s, c, device=qkv.device, dtype=torch.float32)
        lse = torch.empty(b * heads, s, device=qkv.device, dtype=torch.float32)
        seed = dropout_seed(qkv.device)
        _lib.call(_attention_train_entry(s, c // heads) + "_fwd", qkv.data_ptr(), out.data_ptr(), lse.data_ptr(),
                  seed.data_ptr(), salt, float(p_drop), b, s, c, heads, tc._stream())
        ctx.save_for_backward(qkv, out, lse)
        ctx.cfg = (heads, float(p_drop), salt)
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, out, lse = ctx.saved_tensors
        heads, p_drop, salt = ctx.cfg
        b, s, c3 = qkv.shape
        dqkv = torch.empty_like(qkv)
        dout = dout.contiguous()
        seed = dropout_seed(qkv.device)
        args = (qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), dqkv.data_ptr(), seed.data_ptr(), salt, p_drop,
                b, s, c3 // 3, heads)
        bwd = _attention_train_entry(s, c3 // 3 // heads) + "_bwd"
        fork = _fork_wgrad(qkv.device)
        fork.on = fork.on and ATTENTION_BWD_FORK
        with fork:                                  # side stream: key side (dk, dv columns)
            _lib.call(bwd, 2, *args, tc._stream())
        _lib.call(bwd, 1, *args, tc._stream())       # main stream: query side (dq columns)
        fork.join()
        return dqkv, None, None, None


def attention_core(qkv, heads, p_drop, salt):
    return _AttentionCore.apply(qkv, heads, p_drop, salt)


def attention_dropout_mask(device, salt, p_drop, pairs, seq):
    """The multipliers (0 or 1/(1-p)) the kernels apply, [pairs, seq, seq] - test helper."""
    mask = torch.empty(pairs, seq, seq, device=device, dtype=torch.float32)
    _lib.call("flowk_attention_dropout_mask", dropout_seed(device).data_ptr(), salt, float(p_drop), pairs, seq,
              mask.data_ptr(), tc._stream())
    return mask


def pointwise_ok(x):
    return ENABLED and x.is_cuda and x.dtype == torch.float32


def concat_elu(x, dim=1, mask=None):
    """elu(cat(x, -x)) along `dim`; `mask` [outer, 2C] (fp32, 0 or 1/(1-p)) folds the following feature dropout in."""
    return _ConcatElu.apply(x, dim, mask)


def feature_dropout_mask(x, channels, p):
    """nn.Dropout2d's mask for a [B, channels, H, W] tensor as a [B, channels] multiplier (0 or 1/(1-p))."""
    return torch.empty(x.shape[0], channels, device=x.device, dtype=torch.float32).bernoulli_(1.0 - p).div_(1.0 - p)


def glu(x, dim):
    return _Glu.apply(x, dim)
