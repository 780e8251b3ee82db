"""The mAR channel prior's networks on the flowk tensor-core kernels: inference / sampling (autograd off) and, at the end
of this file, training (autograd over one prior level, backward through time on flowk kernels).

Reference: mar_prior/corr_prior.py:58-139 (likelihood / ancestral sampling over the channel sequence),
mar_prior/lstm.py:7-43 (conv_embed -> Conv2dLSTM -> conv_out1), mar_prior/convolutional_rnn/functional.py:30-52 (the
LSTM cell) and :248-275 ("same" padding of dilated kernels).

Everything is a `flowk_conv_gemm` launch over NHWC rows in TIME-MAJOR order (row = (t, b, pixel)), fp16 (hi, lo) operand
pairs (fp32-accurate two-term split, csrc/tc_gemm.cu):

    conv_embed              k x k conv of all T steps at once                     -> operand pair [T*B*HW, E]
    per LSTM layer          input-to-hidden gates of all T steps in ONE GEMM      -> fp32 [T*B*HW, 4E]
                            T recurrent launches: hidden-to-hidden k x k (dilated) conv with the cell update in the
                            epilogue (FLOWK_PRE_LSTM): gates = W_hh * h_{t-1} + b_hh + gi_t, c_t, h_t; h_t is written
                            as the operand pair the next step AND the next layer read, c_t as fp32 rows
    conv_out1               3 x 3 conv -> (mean, log-std)
    z1_cond_network         5 x 5 conv, ReLU (epilogue), 5 x 5 conv

so one likelihood evaluation of a level is 3 + L (T + 1) launches and nothing but the T-step recurrence is sequential.

Ancestral sampling (`AncestralSampler`) runs the same networks one channel at a time with `flowk_mar_step`: conv_embed,
one launch per LSTM layer (input-to-hidden and hidden-to-hidden convolutions as ONE GEMM over the rows [x_t | h_{t-1}]),
and conv_out1 with the Gaussian sample drawn in its epilogue - 2 + L launches per channel and no host work in between.
"""
import ctypes

import torch

from .. import _lib, tc

ENABLED = True


def usable(module, x):
    """CUDA tensors, autograd off, feature maps the GEMM tiles over (W | 128, H*W | 128 or 128 | H*W)."""
    if not (ENABLED and x.is_cuda and x.dtype == torch.float32 and not torch.is_grad_enabled()):
        return False
    h, w = x.shape[-2], x.shape[-1]
    if w > 128 or 128 % w:
        return False
    hw = h * w
    return (hw % 128 == 0) if hw >= 128 else (128 % hw == 0)


def _pad8(c):
    return (c + 7) // 8 * 8


class _Cache:
    def __init__(self):
        self.key, self.value = None, None

    def get(self, params, build):
        key = _lib.param_key(params)
        if key != self.key:
            with torch.no_grad():
                self.value = build()
            self.key = key
        return self.value


def _prep(weight, bias, pad_out=None):
    """conv weight [N, Cin, k, k] (+ bias [N]) -> ((w_hi, w_lo, acc_scale), bias, taps); N zero-padded to `pad_out`."""
    w, b = weight.detach(), bias.detach()
    if pad_out is not None and pad_out > w.shape[0]:
        w = torch.cat([w, w.new_zeros(pad_out - w.shape[0], *w.shape[1:])], 0)
        b = torch.cat([b, b.new_zeros(pad_out - b.shape[0])], 0)
    return tc.conv_weight_operand_f16(w), b.contiguous(), w.shape[2] * w.shape[3]


def _encoder_operands(enc):
    lstm = enc.lstm
    ops = {"embed": _prep(enc.conv_embed.weight, enc.conv_embed.bias),
           "out": _prep(enc.conv_out1.weight, enc.conv_out1.bias, pad_out=4), "layers": []}
    for layer in range(lstm.num_layers):
        ops["layers"].append((
            _prep(getattr(lstm, "weight_ih_l%d" % layer), getattr(lstm, "bias_ih_l%d" % layer)),
            _prep(getattr(lstm, "weight_hh_l%d" % layer), getattr(lstm, "bias_hh_l%d" % layer))))
    return ops


def _conv(a_hi, a_lo, prepared, images, h, w, cin, n, pre, mask, dilation=1, **kw):
    (w_hi, w_lo, sc), bias, taps = prepared
    tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, images, h, w, cin, n, taps, pre, mask, bias=bias, acc_scale=sc, dilation=dilation,
                 **kw)


def run_sequence(enc, x):
    """ConvSeqEncoder.forward on the flowk kernels from a zero state: x [B, T, Cin, H, W] -> out [B, T, 2, H, W]."""
    B, T, cin, H, W = x.shape
    HW, E = H * W, enc.embed_ch
    rows, step_rows = T * B * HW, B * HW
    dev = x.device
    lstm = enc.lstm
    cache = enc.__dict__.setdefault("_flowk_cache", _Cache())
    ops = cache.get(list(enc.parameters()), lambda: _encoder_operands(enc))

    def f16(*shape):
        return torch.empty(*shape, device=dev, dtype=torch.float16)

    def f32(*shape):
        return torch.empty(*shape, device=dev, dtype=torch.float32)

    cpad = _pad8(cin)
    x_tb = x.transpose(0, 1).reshape(T * B, cin, H, W).contiguous()                # time-major images
    a_hi, a_lo = tc.nchw_to_nhwc_hilo(x_tb, cpad, True)
    x_hi, x_lo = f16(rows, E), f16(rows, E)
    _conv(a_hi, a_lo, ops["embed"], T * B, H, W, cpad, E, tc.PRE_BIAS, tc.OUT_HILO, out_hi=x_hi, out_lo=x_lo)
    for layer, (ih, hh) in enumerate(ops["layers"]):
        gi = f32(T, step_rows, 4 * E)                                                # input-to-hidden gates, all steps
        _conv(x_hi, x_lo, ih, T * B, H, W, E, 4 * E, tc.PRE_BIAS, tc.OUT_F32, dilation=lstm.dilation, out_f32=gi)
        h_hi, h_lo = f16(T, step_rows, E), f16(T, step_rows, E)
        hp_hi = hp_lo = torch.zeros(step_rows, E, device=dev, dtype=torch.float16)
        c_prev = torch.zeros(step_rows, E, device=dev, dtype=torch.float32)
        for t in range(T):                                                           # the recurrence: one launch per step
            c_next = f32(step_rows, E)
            _conv(hp_hi, hp_lo, hh, B, H, W, E, 4 * E, tc.PRE_LSTM, 0, dilation=lstm.dilation, res=gi[t], gamma=c_prev,
                  out_f32=c_next, out_hi=h_hi[t], out_lo=h_lo[t])
            hp_hi, hp_lo, c_prev = h_hi[t], h_lo[t], c_next
        x_hi, x_lo = h_hi.view(rows, E), h_lo.view(rows, E)
    out = f32(rows, 4)
    _conv(x_hi, x_lo, ops["out"], T * B, H, W, E, 4, tc.PRE_BIAS, tc.OUT_F32, out_f32=out)
    return out.view(T, B, H, W, 4)[..., :enc.out_ch].permute(1, 0, 4, 2, 3).contiguous()


def z1_embedding(net, z1):
    """z1_cond_network (corr_prior.py:26-28): conv5x5 -> ReLU -> conv5x5 on the half that continues through the flow.
    z1 [B, nc, H, W] (a channel slice of a contiguous NCHW tensor) -> [B, 4, H, W]."""
    B, nc, H, W = z1.shape
    dev = z1.device
    cache = net.__dict__.setdefault("_flowk_cache", _Cache())
    ops = cache.get(list(net.parameters()), lambda: (_prep(net[0].weight, net[0].bias), _prep(net[2].weight, net[2].bias)))
    cpad = _pad8(nc)
    if not (z1.stride(3) == 1 and z1.stride(2) == W and z1.stride(1) == H * W):
        z1 = z1.contiguous()
    a_hi, a_lo = tc.nchw_to_nhwc_hilo(z1, cpad, True)
    mid = ops[0][0][0].shape[0]
    h_hi = torch.empty(B * H * W, mid, device=dev, dtype=torch.float16)
    h_lo = torch.empty_like(h_hi)
    _conv(a_hi, a_lo, ops[0], B, H, W, cpad, mid, tc.PRE_BIAS, tc.OUT_HILO_RELU, out_hi=h_hi, out_lo=h_lo)
    n_out = ops[1][0][0].shape[0]
    out = torch.empty(B * H * W, n_out, device=dev, dtype=torch.float32)
    _conv(h_hi, h_lo, ops[1], B, H, W, mid, n_out, tc.PRE_BIAS, tc.OUT_F32, out_f32=out)
    return out.view(B, H, W, n_out).permute(0, 3, 1, 2).contiguous()


def _sampling_operands(enc):
    """Weights of one sampling step: conv_embed; per layer [W_ih | W_hh] (one GEMM over the [x | h] rows) with b_ih + b_hh;
    conv_out1 as [0 | W_out], so that it reads the same rows (under fp16's 64-channel k-blocks that costs no extra MMA)."""
    lstm = enc.lstm
    w_out = enc.conv_out1.weight.detach()
    ops = {"embed": _prep(enc.conv_embed.weight, enc.conv_embed.bias),
           "out": _prep(torch.cat([torch.zeros_like(w_out), w_out], 1), enc.conv_out1.bias, pad_out=4), "layers": []}
    for layer in range(lstm.num_layers):
        w_ih, w_hh = getattr(lstm, "weight_ih_l%d" % layer), getattr(lstm, "weight_hh_l%d" % layer)
        b_ih, b_hh = getattr(lstm, "bias_ih_l%d" % layer), getattr(lstm, "bias_hh_l%d" % layer)
        ops["layers"].append(_prep(torch.cat([w_ih.detach(), w_hh.detach()], 1), b_ih.detach() + b_hh.detach()))
    return ops


class AncestralSampler:
    """Ancestral sampling of one level of the channel prior (ChannelPriorUniScale.get_sample, corr_prior.py:66-101) for a
    fixed batch size and device.  All buffers are allocated and zeroed here, once:

        S      fp16 pair [B*HW, 8]            step input [previous channel's sample | z1 embedding | 0]
        A      fp16 pairs [L][2][B*HW, 2 hid]  per layer and step parity, rows [x_t | h_{t-1}]
        c      fp32 [L][B*HW, hid]             cell states
        noise  fp32 [nc, B*HW]                 the standard-normal draw of every channel

    Channel t (parity p = t % 2) is 2 + L flowk_mar_step launches, none of which writes a buffer it reads (the 3x3 / 5x5
    taps read rows of other CTAs): EMBED S -> x of A_0[p]; LSTM l reads A_l[p], writes h to A_l[1-p] and to x of A_{l+1}[p];
    SAMPLE reads A_{L-1}[1-p] and writes z[:, t] and column 0 of S.  SAMPLE multiplies the stale x half of its rows by zero
    weights, which is why the buffers start zeroed (uninitialised fp16 can hold NaN, and 0 * NaN = NaN).  The per-channel
    loop makes no allocation, no host synchronisation and no ATen call, so `sample` can be captured in a CUDA graph."""

    def __init__(self, prior, batch, device):
        enc = prior.prior_lstm
        self.prior, self.enc = prior, enc
        self.B, self.H, self.W, self.nc = batch, prior.height, prior.width, prior.nc
        self.hid, self.layers = enc.embed_ch, enc.lstm.num_layers
        self.M = batch * self.H * self.W
        f16 = dict(device=device, dtype=torch.float16)
        self.S = torch.zeros(2, self.M, 8, **f16)
        self.A = torch.zeros(self.layers, 2, 2, self.M, 2 * self.hid, **f16)
        self.c = torch.zeros(self.layers, self.M, self.hid, device=device)
        self.noise = torch.zeros(self.nc, self.M, device=device)
        self._cache = enc.__dict__.setdefault("_flowk_sample_cache", _Cache())

    def _steps(self, ops, z):
        """The launch arguments of an even and an odd channel (SAMPLE's noise / z pointers are set per channel)."""
        B, H, W, hid, L = self.B, self.H, self.W, self.hid, self.layers
        S = (self.S[0], self.S[1])

        def rows(layer, parity, col):
            return (self.A[layer, parity, 0], self.A[layer, parity, 1], 2 * hid, col)

        steps = []
        for p in (0, 1):
            (ew, eb, etaps), (ow, ob, otaps) = ops["embed"], ops["out"]
            seq = [tc.mar_step_args(_lib.MAR_EMBED, S, ew, eb, B, H, W, etaps, hid, rows(0, p, 0))]
            for layer, (lw, lb, ltaps) in enumerate(ops["layers"]):
                seq.append(tc.mar_step_args(_lib.MAR_LSTM, rows(layer, p, 0)[:2], lw, lb, B, H, W, ltaps, hid,
                                            rows(layer, 1 - p, hid), dilation=self.enc.lstm.dilation,
                                            dst1=rows(layer + 1, p, 0) if layer + 1 < L else None, c=self.c[layer]))
            seq.append(tc.mar_step_args(_lib.MAR_SAMPLE, rows(L - 1, 1 - p, 0)[:2], ow, ob, B, H, W, otaps, hid,
                                        S + (8, 0), noise=self.noise, z=z, z_stride=self.nc * H * W))
            steps.append(seq)
        return steps

    def sample(self, z1=None, noise=None):
        """z2 [B, nc, H, W] given z1 (the half that continues through the flow; None at the last level).  `noise`
        [nc, B, ..., H, W] (any device) is copied into the noise buffer first; None samples with what it holds."""
        B, H, W = self.B, self.H, self.W
        ops = self._cache.get(list(self.enc.parameters()), lambda: _sampling_operands(self.enc))
        if noise is not None:
            self.noise.copy_(noise.reshape(self.nc, self.M))
        if z1 is None:
            self.S.zero_()
        else:
            emb = z1_embedding(self.prior.z1_cond_network, z1)
            tc.nchw_to_nhwc_hilo(torch.cat([emb.new_zeros(B, 1, H, W), emb], 1), 8, True, out=(self.S[0], self.S[1]))
        self.A.zero_()                                   # h_{-1} = 0, c_{-1} = 0
        self.c.zero_()
        z2 = torch.empty(B, self.nc, H, W, device=self.noise.device)
        steps = self._steps(ops, z2)
        noise0, z0 = self.noise.data_ptr(), z2.data_ptr()
        for t in range(self.nc):
            seq = steps[t % 2]
            seq[-1].noise = noise0 + 4 * t * self.M
            seq[-1].z = z0 + 4 * t * H * W
            for args in seq:
                tc.mar_step(args)
        return z2


def sampler_for(prior, batch, device):
    """The AncestralSampler eager sampling uses for (prior, batch size, device)."""
    samplers = prior.__dict__.setdefault("_flowk_samplers", {})
    key = (batch, str(torch.device(device)))
    if key not in samplers:
        samplers[key] = AncestralSampler(prior, batch, device)
    return samplers[key]


# ----------------------------------------------------------------------------------------------------------- training
# Autograd over one level of the prior.  The forward makes the launches of run_sequence / z1_embedding and keeps what the
# backward needs: every layer's input rows, gi, h for all T in a [T + 1] buffer whose slot 0 is the zero state (so that
# h_prev = h[0:T]) and every c_t.  The backward per layer, from the top:
#   one batched GEMM recomputes W_hh * h_prev + b_hh for all T steps (the forward's fp16 operands, the same packed weights)
#   for t = T-1 .. 0: flowk_lstm_cell_bwd, then (t > 0) the dgrad GEMM of dgates_t against W_hh (taps flipped, weight
#   transposed, same dilation) -> the recurrent dh of step t-1: the only sequential part
#   one batched dgrad GEMM against W_ih -> the gradient of the layer's input
#   weight gradients of W_ih over the inputs and of W_hh over h_prev (flowk_conv_wgrad_nhwc), one channel sum for both biases
# Gradient GEMMs use TF32 pairs (fp32's exponent range).  Weight operands are packed by launches made in every call (no
# cache, no host read), so a captured training step sees the weights the optimizer wrote.  Channel counts the GEMMs read
# are zero-padded (inputs to 8 or 32, conv_out1's N to 4 / 32) in both operands and gradients.

def trainable(module, x):
    """CUDA fp32 with autograd on, the feature maps `usable` takes, a hidden width the training kernels take (whole
    32-channel blocks, 4 hid <= 256 gate columns per CTA) and B*H*W pixels that tile 32-pixel weight-gradient k-blocks.
    `module`: the ChannelPriorUniScale, `x`: its z2 [B, nc, H, W]."""
    if not (ENABLED and x.is_cuda and x.dtype == torch.float32 and torch.is_grad_enabled()):
        return False
    h, w = x.shape[-2], x.shape[-1]
    if w > 128 or 128 % w:
        return False
    hw = h * w
    if not ((hw % 128 == 0) if hw >= 128 else (128 % hw == 0)):
        return False
    hid = module.prior_lstm.embed_ch
    if hid % 32 or 4 * hid > 256:
        return False
    return _lib.lib.flowk_conv_wgrad_nhwc_splits(x.shape[0], h, w, 32, 32, 9, 1, None) > 0


def _pad32(c):
    return (c + 31) // 32 * 32


def _pack(weight, bias, pad_out=None):
    """Forward operand of a conv: fp16 pair with its scale on the device (tc.conv_weight_operand_f16(device_scale=True))."""
    w, b = weight.detach(), bias.detach()
    if pad_out is not None and pad_out > w.shape[0]:
        w = torch.cat([w, w.new_zeros(pad_out - w.shape[0], *w.shape[1:])], 0)
        b = torch.cat([b, b.new_zeros(pad_out - b.shape[0])], 0)
    return tc.conv_weight_operand_f16(w, device_scale=True), b.contiguous(), w.shape[2] * w.shape[3]


def _conv_t(a_hi, a_lo, packed, images, h, w, cin, n, pre, mask, dilation=1, **kw):
    (w_hi, w_lo, sc), bias, taps = packed
    tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, images, h, w, cin, n, taps, pre, mask, bias=bias, acc_scale=1.0, acc_scale_ptr=sc,
                 dilation=dilation, **kw)


def _dgrad_operand(weight, n_out, n_in):
    """dL/dx = conv(dL/dy, W^T with the taps flipped): [N, Cin, k, k] -> TF32 pair [n_out, taps * n_in] (rows Cin padded
    to n_out, channels N to n_in, with zeros)."""
    wt = weight.detach().flip(2, 3).transpose(0, 1)
    if n_out > wt.shape[0]:
        wt = torch.cat([wt, wt.new_zeros(n_out - wt.shape[0], *wt.shape[1:])], 0)
    return tc.conv_weight_operand(wt, n_in)


def _dgrad(g_rows, wt, images, h, w, n_out, taps, dilation=1):
    """[images*h*w, n_in] fp32 gradient rows -> [images*h*w, n_out] fp32 input-gradient rows."""
    g_hi, g_lo = g_rows if isinstance(g_rows, tuple) else tc.split_rows(g_rows)
    out = torch.empty(g_hi.shape[0], n_out, device=g_hi.device, dtype=torch.float32)
    tc.conv_gemm(g_hi, g_lo, wt[0], wt[1], images, h, w, g_hi.shape[1], n_out, taps, tc.PRE_BIAS, tc.OUT_F32, out_f32=out,
                 dilation=dilation, split_k=True)
    return out


def wgrad(x_rows, gy_rows, images, h, w, taps, dilation=1):
    """Weight gradient of a "same" conv over NHWC rows x [images*h*w, Cin], gy [images*h*w, N] (both % 32 channels):
    [N, Cin, k, k], the split-K slices of flowk_conv_wgrad_nhwc summed in index order."""
    cin, n = x_rows.shape[1], gy_rows.shape[1]
    transposed = ctypes.c_int(0)
    splits = _lib.lib.flowk_conv_wgrad_nhwc_splits(images, h, w, cin, n, taps, dilation, ctypes.byref(transposed))
    assert splits > 0, "flowk_conv_wgrad_nhwc does not take %s" % ((images, h, w, cin, n, taps, dilation),)
    transposed = bool(transposed.value)
    partial = torch.empty((splits, taps, cin, n) if transposed else (splits, taps, n, cin), device=x_rows.device,
                          dtype=torch.float32)
    _lib.call("flowk_conv_wgrad_nhwc", x_rows.data_ptr(), gy_rows.data_ptr(), partial.data_ptr(), None, images, h, w, cin,
              n, taps, dilation, tc._stream())
    g = partial.sum(0)
    g = g.permute(2, 1, 0) if transposed else g.permute(1, 2, 0)
    k = 5 if taps == 25 else 3 if taps == 9 else 1
    return g.reshape(n, cin, k, k)


def pair_to_f32(hi, lo, c_out=None):
    """fp16 (hi, lo) rows [M, C] -> fp32 rows [M, c_out] (extra columns zero)."""
    m, c = hi.shape[0], hi.shape[-1]
    out = torch.empty(m, c_out or c, device=hi.device, dtype=torch.float32)
    _lib.call("flowk_f16_pair_to_f32", hi.data_ptr(), lo.data_ptr(), out.data_ptr(), m, c, c_out or c, tc._stream())
    return out


def cell_backward(gi, hh, c_prev, c, dh, dh_rec, dc, dgates, dg_hi, dg_lo):
    """flowk_lstm_cell_bwd over rows [M, 4 hid]; `dc` holds dL/dc_t from step t+1 (None at the last step) on entry and
    receives dL/dc_{t-1}."""
    m, hid = c.shape
    _lib.call("flowk_lstm_cell_bwd", gi.data_ptr(), hh.data_ptr(), c_prev.data_ptr(), c.data_ptr(), dh.data_ptr(),
              tc._p(dh_rec), None if dh_rec is None else dc.data_ptr(), dgates.data_ptr(), dg_hi.data_ptr(),
              dg_lo.data_ptr(), dc.data_ptr(), m, hid, tc._stream())


def _channel_sum(rows):
    from ..tc_autograd import channel_sum
    return channel_sum(rows, False)


def _encoder_params(enc):
    lstm = enc.lstm
    ps = [enc.conv_embed.weight, enc.conv_embed.bias]
    for layer in range(lstm.num_layers):
        ps += [getattr(lstm, n % layer) for n in ("weight_ih_l%d", "weight_hh_l%d", "bias_ih_l%d", "bias_hh_l%d")]
    return ps + [enc.conv_out1.weight, enc.conv_out1.bias]


class _Encoder(torch.autograd.Function):
    """ConvSeqEncoder.forward from a zero state (dropout 0): x [B, T, Cin, H, W] -> [B, T, out_ch, H, W]."""

    @staticmethod
    def forward(ctx, enc, x, *params):
        B, T, cin, H, W = x.shape
        E, L, d = enc.embed_ch, enc.lstm.num_layers, enc.lstm.dilation
        rows, srows = T * B * H * W, B * H * W
        dev = x.device

        def f16(*shape):
            return torch.empty(*shape, device=dev, dtype=torch.float16)

        cpad = _pad8(cin)
        x_tb = x.detach().transpose(0, 1).reshape(T * B, cin, H, W).contiguous()
        a_hi, a_lo = tc.nchw_to_nhwc_hilo(x_tb, cpad, True)
        embed = _pack(enc.conv_embed.weight, enc.conv_embed.bias)
        x_hi, x_lo = f16(rows, E), f16(rows, E)
        _conv_t(a_hi, a_lo, embed, T * B, H, W, cpad, E, tc.PRE_BIAS, tc.OUT_HILO, out_hi=x_hi, out_lo=x_lo)
        layers = []
        for layer in range(L):
            lw = [getattr(enc.lstm, n % layer) for n in ("weight_ih_l%d", "weight_hh_l%d", "bias_ih_l%d", "bias_hh_l%d")]
            ih, hh = _pack(lw[0], lw[2]), _pack(lw[1], lw[3])
            gi = torch.empty(T, srows, 4 * E, device=dev, dtype=torch.float32)
            _conv_t(x_hi, x_lo, ih, T * B, H, W, E, 4 * E, tc.PRE_BIAS, tc.OUT_F32, dilation=d, out_f32=gi)
            h_hi, h_lo = f16(T + 1, srows, E), f16(T + 1, srows, E)
            c = torch.empty(T + 1, srows, E, device=dev, dtype=torch.float32)
            h_hi[0].zero_()
            h_lo[0].zero_()
            c[0].zero_()
            for t in range(T):
                _conv_t(h_hi[t], h_lo[t], hh, B, H, W, E, 4 * E, tc.PRE_LSTM, 0, dilation=d, res=gi[t], gamma=c[t],
                        out_f32=c[t + 1], out_hi=h_hi[t + 1], out_lo=h_lo[t + 1])
            layers.append((x_hi, x_lo, gi, h_hi, h_lo, c, hh))
            x_hi, x_lo = h_hi[1:].reshape(rows, E), h_lo[1:].reshape(rows, E)
        out = torch.empty(rows, 4, device=dev, dtype=torch.float32)
        _conv_t(x_hi, x_lo, _pack(enc.conv_out1.weight, enc.conv_out1.bias, pad_out=4), T * B, H, W, E, 4, tc.PRE_BIAS,
                tc.OUT_F32, out_f32=out)
        ctx.enc, ctx.shape = enc, (B, T, cin, H, W)
        ctx.state = (a_hi, a_lo, layers)
        return out.view(T, B, H, W, 4)[..., :enc.out_ch].permute(1, 0, 4, 2, 3).contiguous()

    @staticmethod
    def backward(ctx, gy):
        enc = ctx.enc
        B, T, cin, H, W = ctx.shape
        a_hi, a_lo, layers = ctx.state
        ctx.state = None
        E, L, d, k = enc.embed_ch, enc.lstm.num_layers, enc.lstm.dilation, enc.lstm.kernel_size
        taps, TB = k * k, T * B
        rows, srows = TB * H * W, B * H * W
        dev = gy.device
        f32 = dict(device=dev, dtype=torch.float32)
        # conv_out1: gradient rows zero-padded to one 32-channel block
        dy = torch.zeros(T, B, H, W, 32, **f32)
        dy[..., :enc.out_ch] = gy.permute(1, 0, 3, 4, 2)
        dy = dy.view(rows, 32)
        w_out = enc.conv_out1.weight
        top = layers[-1]
        g_out_w = wgrad(pair_to_f32(top[3][1:].reshape(rows, E), top[4][1:].reshape(rows, E)), dy, TB, H, W, 9)
        g_out_b = _channel_sum(dy)[:enc.out_ch]
        dh = _dgrad(dy, _dgrad_operand(w_out, E, 32), TB, H, W, E, 9)
        grads = []
        for layer in reversed(range(L)):
            x_hi, x_lo, gi, h_hi, h_lo, c, hh_op = layers[layer]
            w_ih, w_hh = getattr(enc.lstm, "weight_ih_l%d" % layer), getattr(enc.lstm, "weight_hh_l%d" % layer)
            hf = pair_to_f32(h_hi.view(-1, E), h_lo.view(-1, E)).view(T + 1, srows, E)
            hh = torch.empty(T, srows, 4 * E, **f32)
            _conv_t(h_hi[:T].reshape(rows, E), h_lo[:T].reshape(rows, E), hh_op, TB, H, W, E, 4 * E, tc.PRE_BIAS, tc.OUT_F32,
                    dilation=d, out_f32=hh)
            dgates = torch.empty(T, srows, 4 * E, **f32)
            dg_hi, dg_lo = torch.empty_like(dgates), torch.empty_like(dgates)
            dc = torch.empty(srows, E, **f32)
            dh_rec = torch.empty(srows, E, **f32)
            w_hh_t = _dgrad_operand(w_hh, E, 4 * E)
            dh_t = dh.view(T, srows, E)
            for t in reversed(range(T)):
                last = t == T - 1
                cell_backward(gi[t], hh[t], c[t], c[t + 1], dh_t[t], None if last else dh_rec, dc, dgates[t], dg_hi[t],
                              dg_lo[t])
                if t > 0:
                    tc.conv_gemm(dg_hi[t], dg_lo[t], w_hh_t[0], w_hh_t[1], B, H, W, 4 * E, E, taps, tc.PRE_BIAS, tc.OUT_F32,
                                 out_f32=dh_rec, dilation=d, split_k=True)
            dg_rows = dgates.view(rows, 4 * E)
            dh = _dgrad((dg_hi.view(rows, 4 * E), dg_lo.view(rows, 4 * E)), _dgrad_operand(w_ih, E, 4 * E), TB, H, W, E,
                        taps, d)
            g_ih = wgrad(pair_to_f32(x_hi, x_lo), dg_rows, TB, H, W, taps, d)
            g_hh = wgrad(hf[:T].reshape(rows, E), dg_rows, TB, H, W, taps, d)
            g_b = _channel_sum(dg_rows)
            grads = [g_ih, g_hh, g_b, g_b.clone()] + grads
        # conv_embed: input rows padded to 32 channels for the weight gradient, its dgrad's N to 8
        ke = enc.conv_embed.kernel_size[0]
        cpad = a_hi.shape[1]
        g_emb_w = wgrad(pair_to_f32(a_hi, a_lo, 32), dh, TB, H, W, ke * ke)[:, :cin]
        g_emb_b = _channel_sum(dh)
        gx = _dgrad(dh, _dgrad_operand(enc.conv_embed.weight, cpad, E), TB, H, W, cpad, ke * ke)
        gx = gx.view(T, B, H, W, cpad)[..., :cin].permute(1, 0, 4, 2, 3)
        return (None, gx, g_emb_w, g_emb_b, *grads, g_out_w[:enc.out_ch], g_out_b)


def run_sequence_train(enc, x):
    """ConvSeqEncoder.forward with autograd on the flowk kernels: x [B, T, Cin, H, W] -> out [B, T, 2, H, W]."""
    return _Encoder.apply(enc, x, *_encoder_params(enc))


class _Z1Embedding(torch.autograd.Function):
    """z1_cond_network (conv5x5 -> ReLU -> conv5x5, corr_prior.py:26-28) with autograd: z1 [B, nc, H, W] -> [B, 4, H, W]."""

    @staticmethod
    def forward(ctx, net, z1, w1, b1, w2, b2):
        B, nc, H, W = z1.shape
        dev = z1.device
        cpad = _pad8(nc)
        a_hi, a_lo = tc.nchw_to_nhwc_hilo(z1.detach().contiguous(), cpad, True)
        mid, n_out = w1.shape[0], w2.shape[0]
        h_hi = torch.empty(B * H * W, mid, device=dev, dtype=torch.float16)
        h_lo = torch.empty_like(h_hi)
        _conv_t(a_hi, a_lo, _pack(w1, b1), B, H, W, cpad, mid, tc.PRE_BIAS, tc.OUT_HILO_RELU, out_hi=h_hi, out_lo=h_lo)
        out = torch.empty(B * H * W, n_out, device=dev, dtype=torch.float32)
        _conv_t(h_hi, h_lo, _pack(w2, b2), B, H, W, mid, n_out, tc.PRE_BIAS, tc.OUT_F32, out_f32=out)
        ctx.net, ctx.shape, ctx.state = net, (B, nc, H, W), (a_hi, a_lo, h_hi, h_lo)
        return out.view(B, H, W, n_out).permute(0, 3, 1, 2).contiguous()

    @staticmethod
    def backward(ctx, ge):
        net = ctx.net
        B, nc, H, W = ctx.shape
        a_hi, a_lo, h_hi, h_lo = ctx.state
        ctx.state = None
        w1, w2 = net[0].weight, net[2].weight
        mid, n_out, k1, k2 = w1.shape[0], w2.shape[0], w1.shape[2], w2.shape[2]
        cpad = a_hi.shape[1]
        g = torch.zeros(B * H * W, 32, device=ge.device, dtype=torch.float32)
        g[:, :n_out] = ge.permute(0, 2, 3, 1).reshape(-1, n_out)
        mid_f = pair_to_f32(h_hi, h_lo, _pad32(mid))
        g_w2 = wgrad(mid_f, g, B, H, W, k2 * k2)[:n_out, :mid]
        g_b2 = _channel_sum(g)[:n_out]
        dmid = _dgrad(g, _dgrad_operand(w2, _pad32(mid), 32), B, H, W, _pad32(mid), k2 * k2)
        dmid.mul_(mid_f > 0)                                       # ReLU
        g_w1 = wgrad(pair_to_f32(a_hi, a_lo, 32), dmid, B, H, W, k1 * k1)[:mid, :nc]
        g_b1 = _channel_sum(dmid)[:mid]
        gz = _dgrad(dmid, _dgrad_operand(w1, cpad, _pad32(mid)), B, H, W, cpad, k1 * k1)
        return None, gz.view(B, H, W, cpad)[..., :nc].permute(0, 3, 1, 2), g_w1, g_b1, g_w2, g_b2


def z1_embedding_train(net, z1):
    """z1_embedding with autograd on the flowk kernels."""
    return _Z1Embedding.apply(net, z1, net[0].weight, net[0].bias, net[2].weight, net[2].bias)
