"""Tensor-core (tcgen05) execution of the coupling conditioners, inference / no-grad mode.

`mixlogcdf_nn_raw(nn_module, x_id)` computes what `NN.forward_raw` computes (flow_modules/mixlogcdf_nn.py:64-69:
in_conv -> 10 x ConvAttnBlock -> out_conv) as a chain of `flowk_conv_gemm` launches over NHWC activations:

    per block   G1 conv3x3  concat_elu(x)      -> concat_elu(conv + bias)                         (hi/lo operand)
                G2 gate1x1                      -> LayerNorm(GLU + x)          = x1 (+ pos. enc.)   (fp32 + operand)
                G3 in_proj  x1 + pos            -> (k | v | q)                                      (fp32)
                   attention  softmax(q k^T / sqrt(d)) v   per image and head
                G4 gate     attention output    -> LayerNorm(GLU + x1)         = x2, concat_elu(x2) (fp32 + operand)

Every nonlinearity lives in a GEMM epilogue, so a block is 4 GEMM launches + attention; where a 128-row tile holds whole
images (8x8 and 4x4 maps), G2 to G4 and the attention are one launch (tc.block_tail), and at 16x16 from B = 8 one launch of
two-CTA clusters, one per image (tc.block_tail_pair).  Weight-normalised,
re-laid-out, hi/lo-split weights are cached per parameter version.
"""
import os

import torch

from . import _lib, tc

F16 = os.environ.get("FLOWK_F16", "1") != "0"   # operand format of the inference chain: fp16 (hi, lo) pairs (tcgen05
                    # kind::f16: half the operand bytes, twice the MMA rate, same 22-bit accuracy) or TF32 pairs ("0")
ENABLED = True      # set False to force the torch/cuDNN conditioner (used by tests to A/B the two paths)
CHAIN = os.environ.get("FLOWK_CHAIN", "1") != "0"   # gate -> LayerNorm -> (+pos) -> in_proj as ONE launch: the epilogue warps
                    # write the normalised rows as (hi, lo) operand tiles into swizzled shared memory and the MMA warp runs
                    # the second GEMM while its weights stream in behind the GLU / LayerNorm epilogue


def supported(channels, h, w):
    """Shapes the tcgen05 path takes: channel counts that are multiples of 32 (K blocks) and 16 (MMA N), spatial
    tiles that pack into 128-row M tiles."""
    if channels % 32:
        return False
    if w > 128 or 128 % w:
        return False
    hw = h * w
    return (hw % 128 == 0) if hw >= 128 else (128 % hw == 0)


class _Cache:
    """Per-module operand cache keyed on the parameters' (data_ptr, version)."""

    def __init__(self):
        self.key = None
        self.value = None

    def get(self, params, build):
        key = _lib.param_key(params)
        if key != self.key:
            with torch.no_grad():
                self.value = build()
            self.key = key
        return self.value


def _weight_operand(w):
    """(w_hi, w_lo, acc_scale) of a conv / linear weight in the chain's operand format."""
    if F16:
        return tc.conv_weight_operand_f16(w)
    return tc.conv_weight_operand(w) + (None,)


def _act_buf(dev, *shape):
    return torch.empty(*shape, device=dev, dtype=torch.float16 if F16 else torch.float32)


def _cin_pad(c):
    return (c + 7) // 8 * 8 if F16 else (c + 31) // 32 * 32


def _wn_operand(core):
    """(w_hi, w_lo, bias, acc_scale) of a weight-normed conv / linear (`_WeightNormed`)."""
    bias = None if core.bias is None else core.bias.detach().contiguous()
    if F16:                                            # weight norm fused into the operand packing (two launches)
        w_hi, w_lo, sc = tc.conv_weight_operand_f16(core.weight_v, core.weight_g, _lib.PACK_WEIGHT_NORM)
        return w_hi, w_lo, bias, sc
    w_hi, w_lo, sc = _weight_operand(core.normed_weight())
    return w_hi, w_lo, bias, sc


def _nn_operands(nn_module):
    ops = {"in": _wn_operand(nn_module.in_conv.conv), "out": _wn_operand(nn_module.out_conv.conv), "blocks": []}
    for blk in nn_module.mid_convs:
        d = {"conv": _wn_operand(blk.conv.conv.conv), "gate": _wn_operand(blk.conv.gate.conv),
             "ln1": (blk.norm_1.weight.detach().contiguous(), blk.norm_1.bias.detach().contiguous())}
        if blk.attn is not None:
            d["in_proj"] = _wn_operand(blk.attn.in_proj)
            d["attn_gate"] = _wn_operand(blk.attn.gate)
            d["ln2"] = (blk.norm_2.weight.detach().contiguous(), blk.norm_2.bias.detach().contiguous())
            d["heads"] = blk.attn.num_heads
        ops["blocks"].append(d)
    return ops


def mixlogcdf_nn_raw(nn_module, x_id, status=None):
    """x_id: [B,c,H,W] channel slice of a contiguous NCHW tensor.  Returns raw [B,(2+3K)c,H,W] fp32."""
    assert not torch.is_grad_enabled() or not any(p.requires_grad for p in nn_module.parameters()), \
        "tcgen05 conditioner path is inference-only"
    B, c, H, W = x_id.shape
    dev = x_id.device
    M, HW = B * H * W, H * W
    C = nn_module.in_conv.conv.weight_v.shape[0]
    cache = nn_module.__dict__.setdefault("_tc_cache", _Cache())
    ops = cache.get(list(nn_module.parameters()), lambda: _nn_operands(nn_module))

    def buf(*shape):
        return torch.empty(*shape, device=dev, dtype=torch.float32)

    def obuf(*shape):                                  # operand (hi or lo) buffer in the chain's format
        return _act_buf(dev, *shape)

    cin0 = _cin_pad(c)
    a_hi, a_lo = tc.nchw_to_nhwc_hilo(x_id, cin0, F16)
    x = buf(M, C)
    nxt_hi, nxt_lo = obuf(M, 2 * C), obuf(M, 2 * C)
    w_hi, w_lo, bias, sc = ops["in"]
    tc.conv_gemm(a_hi, a_lo, w_hi, w_lo, B, H, W, cin0, C, 9, tc.PRE_BIAS, tc.OUT_F32 | tc.OUT_HILO_CELU, bias=bias,
                 out_f32=x, out_hi=nxt_hi, out_lo=nxt_lo, status=status, acc_scale=sc)
    nblocks = len(ops["blocks"])
    for bi, blk in enumerate(ops["blocks"]):
        last = bi == nblocks - 1
        # G1: conv3x3 on concat_elu(x) -> concat_elu(. + bias)
        c1_hi, c1_lo = obuf(M, 2 * C), obuf(M, 2 * C)
        w_hi, w_lo, bias, sc = blk["conv"]
        tc.conv_gemm(nxt_hi, nxt_lo, w_hi, w_lo, B, H, W, 2 * C, C, 9, tc.PRE_BIAS, tc.OUT_HILO_CELU, bias=bias,
                     out_hi=c1_hi, out_lo=c1_lo, status=status, acc_scale=sc)
        # G2: gate 1x1 -> GLU + x -> LayerNorm
        w_hi, w_lo, bias, sc = blk["gate"]
        has_attn = "in_proj" in blk
        pair = has_attn and F16 and tc.block_tail_pair_supported(HW, C, blk["heads"], B)
        if has_attn and F16 and (pair or tc.block_tail_supported(HW, C, blk["heads"], M)):
            # G2, G3, the attention and G4 in one launch: x1, q, k, v and the attention output stay on chip (at 16x16 in a
            # cluster of two CTAs per image)
            pos = nn_module.mid_convs[bi].attn._pos_enc(HW, C, dev).reshape(HW, C).contiguous()
            w3_hi, w3_lo, _, sc3 = blk["in_proj"]
            w4_hi, w4_lo, bias4, sc4 = blk["attn_gate"]
            x, nxt_hi, nxt_lo = tc.block_tail(c1_hi, c1_lo, (w_hi, w_lo, sc), bias, x, blk["ln1"], pos, (w3_hi, w3_lo, sc3),
                                              (w4_hi, w4_lo, sc4), bias4, blk["ln2"], B, HW, C, blk["heads"], not last,
                                              status=status, pair=pair)
            continue
        x1 = buf(M, C)
        if has_attn:
            pos = nn_module.mid_convs[bi].attn._pos_enc(HW, C, dev).reshape(HW, C).contiguous()
            heads = blk["heads"]
            fused = F16 and tc.attention_inproj_supported(HW, C, heads)
            if fused:
                # G2 writes the normalised rows (+ positional encoding) as an fp16 pair; G3 and the attention run in one
                # launch, q, k and v never leaving the SM
                p_hi, p_lo = obuf(M, C), obuf(M, C)
                tc.conv_gemm(c1_hi, c1_lo, w_hi, w_lo, B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN,
                             tc.OUT_F32 | tc.OUT_HILO_POS, bias=bias, res=x, gamma=blk["ln1"][0], beta=blk["ln1"][1],
                             pos=pos, out_f32=x1, out_hi=p_hi, out_lo=p_lo, status=status, acc_scale=sc)
                w3_hi, w3_lo, _, sc3 = blk["in_proj"]
                t_hi, t_lo = tc.attention_inproj(p_hi, p_lo, w3_hi, w3_lo, sc3, B, HW, C, heads, status=status)
            else:
                qkv = buf(M, 3 * C)
                if CHAIN and tc.chain_supported(C, 3 * C, F16):
                    # G2 + G3 in one launch: the normalised rows (+ positional encoding) go from the epilogue into swizzled
                    # shared-memory operand tiles and are multiplied by in_proj's weight in the same CTA
                    w3_hi, w3_lo, _, sc3 = blk["in_proj"]
                    tc.conv_gemm(c1_hi, c1_lo, w_hi, w_lo, B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN, tc.OUT_F32, bias=bias,
                                 res=x, gamma=blk["ln1"][0], beta=blk["ln1"][1], pos=pos, out_f32=x1, status=status,
                                 w2_hi=w3_hi, w2_lo=w3_lo, out2_f32=qkv, n2=3 * C, acc_scale=sc, acc_scale2=sc3)
                else:
                    p_hi, p_lo = obuf(M, C), obuf(M, C)
                    tc.conv_gemm(c1_hi, c1_lo, w_hi, w_lo, B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN,
                                 tc.OUT_F32 | tc.OUT_HILO_POS, bias=bias, res=x, gamma=blk["ln1"][0], beta=blk["ln1"][1],
                                 pos=pos, out_f32=x1, out_hi=p_hi, out_lo=p_lo, status=status, acc_scale=sc)
                    # G3: in_proj -> (k | v | q)
                    w_hi, w_lo, _, sc = blk["in_proj"]
                    tc.conv_gemm(p_hi, p_lo, w_hi, w_lo, B, H, W, C, 3 * C, 1, tc.PRE_BIAS, tc.OUT_F32, out_f32=qkv,
                                 status=status, acc_scale=sc)
                if tc.attention_supported(HW, C, heads):
                    t_hi, t_lo = tc.attention(qkv, B, HW, C, heads, F16, status=status)
                else:                                                     # odd head sizes: library matmuls
                    _lib.library_fallback("attention core (seq %d, head dim %d)" % (HW, C // heads), qkv)
                    d = C // heads
                    t = qkv.view(B, HW, 3, heads, d)
                    k, v, q = (t[:, :, i].permute(0, 2, 1, 3) for i in range(3))
                    att = torch.softmax((q * (d ** -0.5)) @ k.transpose(-1, -2), dim=-1) @ v      # [B, heads, HW, d]
                    att = att.permute(0, 2, 1, 3).reshape(M, C).contiguous()
                    t_hi, t_lo = tc.split_rows_f16(att) if F16 else tc.split_rows(att)
            # G4: attention gate -> GLU + x1 -> LayerNorm
            w_hi, w_lo, bias, sc = blk["attn_gate"]
            x2 = buf(M, C)
            if last:
                nxt_hi, nxt_lo = obuf(M, C), obuf(M, C)
            else:
                nxt_hi, nxt_lo = obuf(M, 2 * C), obuf(M, 2 * C)
            tc.conv_gemm(t_hi, t_lo, w_hi, w_lo, B, H, W, C, 2 * C, 1, tc.PRE_GLU_RES_LN,
                         tc.OUT_F32 | (tc.OUT_HILO if last else tc.OUT_HILO_CELU), bias=bias, res=x1,
                         gamma=blk["ln2"][0], beta=blk["ln2"][1], out_f32=x2, out_hi=nxt_hi, out_lo=nxt_lo, status=status,
                         acc_scale=sc)
            x = x2
        else:
            if last:
                nxt_hi, nxt_lo = obuf(M, C), obuf(M, C)
            else:
                nxt_hi, nxt_lo = obuf(M, 2 * C), obuf(M, 2 * C)
            tc.conv_gemm(c1_hi, c1_lo, w_hi, w_lo, B, H, W, 2 * C, 2 * C, 1, tc.PRE_GLU_RES_LN,
                         tc.OUT_F32 | (tc.OUT_HILO if last else tc.OUT_HILO_CELU), bias=bias, res=x,
                         gamma=blk["ln1"][0], beta=blk["ln1"][1], out_f32=x1, out_hi=nxt_hi, out_lo=nxt_lo, status=status,
                         acc_scale=sc)
            x = x1
    if nblocks == 0:                                   # out_conv takes the plain activation
        nxt_hi, nxt_lo = tc.split_rows_f16(x) if F16 else tc.split_rows(x)
    w_hi, w_lo, bias, sc = ops["out"]
    n_out = w_hi.shape[0]
    raw = buf(B, n_out, H, W)
    tc.conv_gemm(nxt_hi, nxt_lo, w_hi, w_lo, B, H, W, C, n_out, 9, tc.PRE_BIAS, tc.OUT_NCHW, bias=bias, out_nchw=raw,
                 status=status, acc_scale=sc)
    return raw


def _affine_operands(net):
    """NN_net (flow_modules/affine_coupling.py:68-80) with both ActNorms folded into the conv weights:
    (conv(x) + b) e^{logs} = conv(x; w e^{logs}) + b e^{logs};  Conv2dZeros: (conv + bias) e^{3 logs}."""
    ops = []
    if F16:                                            # gains and biases folded by the packing kernel
        for conv in (net.conv1, net.conv2):
            w_hi, w_lo, sc, b = tc.conv_weight_operand_f16(conv.weight, conv.actnorm.logs, _lib.PACK_EXP_GAIN, 1.0,
                                                           conv.actnorm.bias)
            ops.append((w_hi, w_lo, b, sc))
        w_hi, w_lo, sc, b = tc.conv_weight_operand_f16(net.conv3.weight, net.conv3.logs, _lib.PACK_EXP_GAIN,
                                                       float(net.conv3.logscale_factor), net.conv3.bias)
        ops.append((w_hi, w_lo, b, sc))
        return ops
    for conv in (net.conv1, net.conv2):
        gain = torch.exp(conv.actnorm.logs.detach().reshape(-1))
        w_hi, w_lo, sc = _weight_operand(conv.weight.detach() * gain.view(-1, 1, 1, 1))
        ops.append((w_hi, w_lo, (conv.actnorm.bias.detach().reshape(-1) * gain).contiguous(), sc))
    gain = torch.exp(net.conv3.logs.detach().reshape(-1) * net.conv3.logscale_factor)
    w_hi, w_lo, sc = _weight_operand(net.conv3.weight.detach() * gain.view(-1, 1, 1, 1))
    ops.append((w_hi, w_lo, (net.conv3.bias.detach() * gain).contiguous(), sc))
    return ops


def affine_supported(net, h, w):
    hidden = net.conv1.weight.shape[0]
    return (tuple(net.conv1.weight.shape[2:]) == (3, 3) and tuple(net.conv2.weight.shape[2:]) == (1, 1)
            and net.conv3.weight.shape[0] % 4 == 0 and supported(hidden, h, w))


def affine_nn_net(net, z1, status=None):
    """h = NN_net(z1) as three tcgen05 implicit GEMMs (3x3 -> ReLU -> 1x1 -> ReLU -> 3x3), NCHW output [B,C,H,W]."""
    B, c, H, W = z1.shape
    dev = z1.device
    M = B * H * W
    hidden = net.conv1.weight.shape[0]
    n_out = net.conv3.weight.shape[0]
    cache = net.__dict__.setdefault("_tc_cache", _Cache())
    ops = cache.get(list(net.parameters()), lambda: _affine_operands(net))

    def buf(*shape):
        return torch.empty(*shape, device=dev, dtype=torch.float32)

    cin0 = _cin_pad(c)
    a_hi, a_lo = tc.nchw_to_nhwc_hilo(z1, cin0, F16)
    h1_hi, h1_lo = _act_buf(dev, M, hidden), _act_buf(dev, M, hidden)
    tc.conv_gemm(a_hi, a_lo, ops[0][0], ops[0][1], B, H, W, cin0, hidden, 9, tc.PRE_BIAS, tc.OUT_HILO_RELU, bias=ops[0][2],
                 out_hi=h1_hi, out_lo=h1_lo, status=status, acc_scale=ops[0][3])
    h2_hi, h2_lo = _act_buf(dev, M, hidden), _act_buf(dev, M, hidden)
    tc.conv_gemm(h1_hi, h1_lo, ops[1][0], ops[1][1], B, H, W, hidden, hidden, 1, tc.PRE_BIAS, tc.OUT_HILO_RELU,
                 bias=ops[1][2], out_hi=h2_hi, out_lo=h2_lo, status=status, acc_scale=ops[1][3])
    out = buf(B, n_out, H, W)
    tc.conv_gemm(h2_hi, h2_lo, ops[2][0], ops[2][1], B, H, W, hidden, n_out, 9, tc.PRE_BIAS, tc.OUT_NCHW, bias=ops[2][2],
                 out_nchw=out, status=status, acc_scale=ops[2][3])
    return out
