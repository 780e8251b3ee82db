"""The mAR channel prior's networks on the flowk tensor-core kernels (inference / sampling, autograd off).

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
