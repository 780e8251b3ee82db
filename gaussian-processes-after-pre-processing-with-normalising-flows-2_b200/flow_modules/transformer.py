"""`Transformer_attn`: the fork's invertible patch-attention layer (reference flow_modules/transformer.py:31-326, used twice
per FlowStep at marscf_main.py:50-51,69-70).  Same class name, call signature and state-dict keys (`convq1..3`,
`convk1..3` [C,C,1,1], `offset`, `offset2`, `offset3`, `scale` [1,1,1]) so the fork's checkpoints load.

The layer is outside the north-star hot path (SURVEY.md section 8f-2) and is a plug-in (`FlowStep(..., attn=True)`), written
as device-agnostic torch ops - no `.cuda()` calls, no float64 / host round trips - on a restructured form of the
reference's arithmetic:

  * the image is a 2x2 grid of (W/2)-sized patches, each flattened to L = C*p*p values; entries whose (patch + index)
    parity is even (odd with `permute`) condition the attention and pass through unchanged;
  * the six 1x1 convolutions and three Q K^T products collapse to ONE 1x1 convolution: with G = sum_i Wq_i^T Wk_i,
    sum_i Q_i K_i^T = Z (G Z)^T over the masked input Z - G is cached per weight version;
  * attn = sigmoid(score / scale + offset2) + offset3 gives two 2x2 matrices, M1 for patches (0, 2) and M2 for patches
    (1, 3) (`offset` added on the diagonal); the free entries of the two patches are mixed by M (forward) or by its
    closed-form inverse (reverse); logdet +-= (log|det M1| + log|det M2|) * p * (p // 2) * C.

On CUDA fp32 the layer runs on flowk kernels (csrc/patch_attention.cu): inference and sampling in one fused launch, and
training of the forward direction through `flowk::patch_attention` (a forward launch that keeps the scores, a closed-form
backward launch and a fixed-order batch sum of the parameter gradients); G and its weight gradients stay in torch.  The
torch-op form below serves CPU / fp64 tensors, autograd through the reverse direction, and maps too large for the
kernels' shared memory.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib, ops

KERNEL_TRAINING = True     # False: train the forward direction on the torch-op form (A/B measurements, tests)


def _fits(c, h, w, copies):
    """Shared memory of csrc/patch_attention.cu: `copies` [C, H, W] fp32 samples (padded to 4) plus G, at most 200 KB."""
    return (copies * ((c * h * w + 3) & ~3) + c * c) * 4 <= 200 * 1024


def _patches(x, p):
    b, c, h, w = x.shape
    return x.reshape(b, c, h // p, p, w // p, p).permute(0, 2, 4, 1, 3, 5).reshape(b, (h // p) * (w // p), c * p * p)


def _unpatches(t, p, shape):
    b, c, h, w = shape
    return t.reshape(b, h // p, w // p, c, p, p).permute(0, 3, 1, 4, 2, 5).reshape(b, c, h, w)


class Transformer_attn(nn.Module):
    def __init__(self, num_channels):
        super().__init__()
        self.c = num_channels
        for name in ("convq1", "convk1", "convq2", "convk2", "convq3", "convk3"):
            w = torch.empty(num_channels, num_channels, 1, 1)
            nn.init.kaiming_uniform_(w, a=math.sqrt(5))
            setattr(self, name, nn.Parameter(w))
        self.offset = nn.Parameter(torch.ones(1, 1, 1) * 0.99)
        self.offset2 = nn.Parameter(torch.ones(1, 1, 1) * 0.65)
        self.offset3 = nn.Parameter(torch.ones(1, 1, 1) * -0.6)
        self.scale = nn.Parameter(torch.ones(1, 1, 1) * 100)
        self._masks = {}
        self._g = None

    def _mask(self, n, length, permute, like):
        key = (n, length, bool(permute), like.device, like.dtype)
        m = self._masks.get(key)
        if m is None:
            i = torch.arange(n, device=like.device).view(-1, 1)
            j = torch.arange(length, device=like.device).view(1, -1)
            m = (1 - (i + j) % 2).to(like.dtype)
            if permute:
                m = 1 - m
            self._masks[key] = m
        return m

    def _bilinear(self):
        """G = sum_i Wq_i^T Wk_i as a [C, C, 1, 1] conv weight (cached outside autograd)."""
        ws = (self.convq1, self.convk1, self.convq2, self.convk2, self.convq3, self.convk3)
        track = torch.is_grad_enabled() and any(w.requires_grad for w in ws)
        key = _lib.param_key(ws)
        if not track and self._g is not None and self._g[0] == key:
            return self._g[1]
        g = sum(q[:, :, 0, 0].t() @ k[:, :, 0, 0] for q, k in zip(ws[0::2], ws[1::2]))
        g = g[:, :, None, None]
        if not track:
            self._g = (key, g)
        return g

    def _kernel_operands(self):
        """(G [C, C], prm = {offset, offset2, offset3, scale}) for flowk_patch_attention, cached per weight version."""
        ps = (self.convq1, self.convk1, self.convq2, self.convk2, self.convq3, self.convk3, self.offset, self.offset2,
              self.offset3, self.scale)
        key = _lib.param_key(ps)
        hit = getattr(self, "_kop", None)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                g = self._bilinear()[:, :, 0, 0].contiguous().float()
                prm = torch.cat([t.reshape(1) for t in (self.offset, self.offset2, self.offset3, self.scale)]).float().contiguous()
            hit = self._kop = (key, g, prm)
        return hit[1], hit[2]

    def forward(self, input, logdet=0, reverse=False, permute=False):
        z = input
        b, c, h, w = z.shape
        assert h == w and w % 2 == 0, "Transformer_attn expects square maps with an even side"
        tracking = torch.is_grad_enabled() and (z.requires_grad or any(q.requires_grad for q in self.parameters()))
        if (KERNEL_TRAINING and tracking and not reverse and z.is_cuda and z.dtype == torch.float32 and
                _fits(c, h, w, 3)):
            # training: flowk::patch_attention (forward kernel + closed-form backward kernel); G = sum_i Wq_i^T Wk_i and
            # prm are built with autograd, so torch turns the kernel's gradient of G into the six conv-weight gradients
            _lib.check_device(z, "Transformer_attn")
            g = self._bilinear()[:, :, 0, 0]
            prm = torch.cat([t.reshape(1) for t in (self.offset, self.offset2, self.offset3, self.scale)])
            batch_ld = torch.is_tensor(logdet) and logdet.dim() == 1 and logdet.shape[0] == b
            ld_in = logdet.float() if batch_ld else z.new_zeros(b)
            out, ld_out, _ = ops.patch_attention(z, g, prm, ld_in, bool(permute))
            return out, (ld_out if batch_ld else ld_out + logdet)
        if z.is_cuda and z.dtype == torch.float32 and (2 * c * h * w + c * c) * 4 <= 200 * 1024 and not tracking:
            # inference / sampling: one fused flowk kernel (csrc/patch_attention.cu), one read + one write of the activations
            g, prm = self._kernel_operands()
            _lib.check_device(z, "Transformer_attn")
            z = z.contiguous()
            out = torch.empty_like(z)
            ld_in = None
            if torch.is_tensor(logdet) and logdet.dim() == 1 and logdet.shape[0] == b:
                ld_in = logdet.float().contiguous()
            ld_out = torch.empty(b, device=z.device, dtype=torch.float32)
            _lib.call("flowk_patch_attention", z.data_ptr(), g.data_ptr(), prm.data_ptr(), out.data_ptr(),
                      None if ld_in is None else ld_in.data_ptr(), ld_out.data_ptr(), b, c, h, w, int(bool(permute)),
                      int(bool(reverse)), torch.cuda.current_stream().cuda_stream)
            if ld_in is None:
                ld_out = ld_out + logdet                         # scalar / broadcastable start value
            return out, ld_out
        p = w // 2
        full = _patches(z, p)                                   # [B, 4, L]
        mask = self._mask(full.shape[1], full.shape[2], permute, z)
        cond = full * mask
        # score[n, m] = sum_pixels z_n^T G z_m over the conditioning entries
        t = _patches(F.conv2d(_unpatches(cond, p, z.shape), self._bilinear()), p)
        score = torch.matmul(cond, t.transpose(1, 2)) / self.scale
        attn = torch.sigmoid(score + self.offset2) + self.offset3
        off = self.offset.reshape(())
        a1, b1, c1, d1 = attn[:, 0, 0] + off, attn[:, 0, 2], attn[:, 2, 0], attn[:, 2, 2] + off      # M1: patches 0, 2
        a2, b2, c2, d2 = attn[:, 1, 1] + off, attn[:, 1, 3], attn[:, 3, 1], attn[:, 3, 3] + off      # M2: patches 1, 3
        det1, det2 = a1 * d1 - b1 * c1, a2 * d2 - b2 * c2
        ld = (torch.log(det1.abs()) + torch.log(det2.abs())) * (p * (p // 2) * self.c)
        if reverse:                                             # closed-form 2x2 inverses
            a1, b1, c1, d1 = d1 / det1, -b1 / det1, -c1 / det1, a1 / det1
            a2, b2, c2, d2 = d2 / det2, -b2 / det2, -c2 / det2, a2 / det2
        free = full * (1 - mask)
        x0, x1, x2, x3 = free[:, 0], free[:, 1], free[:, 2], free[:, 3]
        col = lambda v: v.view(-1, 1)                           # noqa: E731
        mixed = torch.stack((col(a1) * x0 + col(b1) * x2, col(a2) * x1 + col(b2) * x3,
                             col(c1) * x0 + col(d1) * x2, col(c2) * x1 + col(d2) * x3), dim=1)
        out = _unpatches(mixed * (1 - mask) + cond, p, z.shape)
        return out, (logdet - ld if reverse else logdet + ld)
