"""FlowStep / FlowNet / MarScfFlow with the reference's constructor arguments, module tree
(state-dict keys) and `forward(x, logdet, reverse=...)` contract (marscf_main.py:35-220).

This is variant "A minus attention" of SURVEY.md section 0: ActNorm -> invertible 1x1 conv ->
(affine | MixLogCDF) coupling (-> TupleFlip), the stack BASELINE.json's north_star names.  The
fork's two `Transformer_attn` layers and the ConvLSTM channel prior are outside that path; both are
plug-ins: `attn=True` inserts the patch-attention layers (flow_modules/transformer.py) where the fork
has them, and `prior=` takes anything with the reference's `c_prior(z, level, reverse)` call
signature (`"mar"` = the ConvLSTM channel prior port), defaulting to a standard normal.

Per FlowStep the activations are touched twice: one fused ActNorm∘InvConv (∘Squeeze) channel-mix
kernel and one fused coupling kernel (which also applies the TupleFlip and accumulates the log-det).
"""
import math

import torch
import torch.nn as nn

from . import _lib, ops
from .flow_modules.affine_coupling import AffineCoupling
from .flow_modules.common_modules import (Actnormlayer, GaussianDiag, InvertibleConv1x1, Split2dMsC, SqueezeLayer,
                                          TupleFlip, _batch_ldj, fold_actnorm_invconv, squeeze2d)
from .flow_modules.mixlogcdf_coupling import MixLogCDFCoupling
from .flow_modules.transformer import Transformer_attn


class FlowStep(nn.Module):
    def __init__(self, H, W, C, in_channels, out_channels, hidden_channels, actnorm_scale, coupling_type,
                 num_blocks=10, num_components=32, drop_prob=0.2, attn=False):
        super().__init__()
        self.coupling_type = coupling_type
        # attn=True adds the fork's two invertible patch-attention layers after the 1x1 conv (marscf_main.py:50-51,
        # 69-70); they are outside the north-star path, so the default stack is variant A minus Transformer_attn
        self.attn1 = Transformer_attn(in_channels) if attn else None
        self.attn2 = Transformer_attn(in_channels) if attn else None
        if coupling_type == 'mixlogcdf':
            self.coupling = MixLogCDFCoupling(in_channels, hidden_channels, num_blocks=num_blocks,
                                              num_components=num_components, drop_prob=drop_prob)
            self.tuple_flip = TupleFlip()
        else:
            self.coupling = AffineCoupling(in_channels, out_channels, hidden_channels)
        self.actnormlayer = Actnormlayer(in_channels, actnorm_scale)
        self.invert_1x1_layer = InvertibleConv1x1(in_channels)
        self._fold_cache = {}

    def _folded(self, hw, reverse):
        """(matrix, bias, ldj_add) of ActNorm∘InvConv; cached per parameter version in no-grad mode."""
        an, ic = self.actnormlayer, self.invert_1x1_layer
        params = (an.bias, an.logs) + tuple(ic._params())
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            return fold_actnorm_invconv(an, ic, hw, reverse)
        key = (hw, bool(reverse)) + _lib.param_key(params)
        hit = self._fold_cache.get(bool(reverse))
        if hit is None or hit[0] != key:
            with torch.no_grad():
                hit = (key, tuple(t.contiguous() for t in fold_actnorm_invconv(an, ic, hw, reverse)))
            self._fold_cache[bool(reverse)] = hit
        return hit[1]

    def forward_inference(self, x, logdet=0., reverse=False, squeeze_input=False):
        an = self.actnormlayer
        if an.training and not an._seen_initialized:
            if squeeze_input:
                x, squeeze_input = squeeze2d(x, 2), False
            an.maybe_initialize(x)
        ldj, had = _batch_ldj(logdet, x)
        hw = (x.size(2) // 2, x.size(3) // 2) if squeeze_input else (x.size(2), x.size(3))
        mat, bias, add = self._folded(hw, False)
        x, ldj = ops.channel_mix(x, mat, bias, ldj, add, bool(squeeze_input), False)
        if self.attn1 is not None:
            x, ldj = self.attn1(x, logdet=ldj, reverse=False)
            x, ldj = self.attn2(x, logdet=ldj, reverse=False, permute=True)
        if self.coupling_type == 'mixlogcdf':
            x, ldj = self.coupling(x, ldj, False, flip=True)
        else:
            x, ldj = self.coupling(x, ldj, False)
        return x, (ldj if had else None)

    def reverse_sampling(self, x, logdet=0., reverse=True, unsqueeze_output=False):
        ldj, had = _batch_ldj(logdet, x)
        if self.coupling_type == 'mixlogcdf':
            x, ldj = self.coupling(x, ldj, True, flip=True)
        else:
            x, ldj = self.coupling(x, ldj, True)
        if self.attn1 is not None:
            x, ldj = self.attn2(x, logdet=ldj, reverse=True, permute=True)
            x, ldj = self.attn1(x, logdet=ldj, reverse=True)
        mat, bias, add = self._folded((x.size(2), x.size(3)), True)
        x, ldj = ops.channel_mix(x, mat, bias, ldj, add, False, bool(unsqueeze_output))
        return x, (ldj if had else None)

    def forward(self, input, logdet=0., reverse=False):
        if not reverse:
            return self.forward_inference(input, logdet, reverse)
        return self.reverse_sampling(input, logdet, reverse)


class StandardNormalPrior(nn.Module):
    """Default `c_prior` plug-in: i.i.d. N(0,1) on every latent, with the call signature of the
    reference's ChannelPriorMultiScale (marscf_main.py:159-164,168,172): forward returns the [B]
    log-likelihood of z2 (given z1, ignored here) or of the final z; reverse samples."""

    def __init__(self, image_shape, L):
        super().__init__()
        h, w, c = image_shape
        self.L = L
        self.final_shape = (c * 4 ** L // 2 ** (L - 1), h // 2 ** L, w // 2 ** L)

    def forward(self, z, level, reverse=False, eps_std=None, batch_size=None, device=None):
        if not reverse:
            z2 = z[1] if isinstance(z, (tuple, list)) else z
            # log N(z2; 0, I) per sample = -(sum z^2 + D log 2 pi) / 2: GaussianDiag.logp with zero mean / log-std in two
            # launches instead of ~12 (common_modules.py:223-240; same value up to fp32 summation order)
            return self.accumulate(z, level, None)
        if z is None:
            return torch.randn((batch_size,) + self.final_shape, device=device) * (eps_std or 1.0)
        return torch.randn_like(z) * (eps_std or 1.0)

    def accumulate(self, z, level, logdet):
        """logdet + log N(z2; 0, I) ([B]; `logdet` None, a float or a [B] tensor) - on CUDA without autograd one flowk launch
        (flowk_std_normal_logp) instead of five library kernels."""
        z2 = z[1] if isinstance(z, (tuple, list)) else z
        b, d = z2.shape[0], z2[0].numel()
        vec = torch.is_tensor(logdet) and logdet.dim() == 1 and logdet.shape[0] == b and logdet.dtype == torch.float32
        if (z2.is_cuda and z2.dtype == torch.float32 and b > 0 and not (torch.is_grad_enabled() and (z2.requires_grad or (
                torch.is_tensor(logdet) and logdet.requires_grad))) and (logdet is None or vec)
                and z2[0].is_contiguous() and (b == 1 or z2.stride(0) >= d)):
            _lib.check_device(z2, "StandardNormalPrior")
            out = torch.empty(b, device=z2.device, dtype=torch.float32)
            ld = logdet.contiguous() if vec else None
            _lib.call("flowk_std_normal_logp", z2.data_ptr(), z2.stride(0) if b > 1 else d, None if ld is None else ld.data_ptr(),
                      out.data_ptr(), b, d, torch.cuda.current_stream().cuda_stream)
            return out
        ll = -0.5 * (z2.square().flatten(1).sum(1) + d * GaussianDiag.Log2PI)
        return ll if logdet is None else logdet + ll


class FlowNet(nn.Module):
    def __init__(self, batch_size, image_shape, hidden_channels, K, L, coupling_type, actnorm_scale=1.0,
                 prior=None, num_blocks=10, fuse_squeeze=True, attn=False, drop_prob=0.2):
        super().__init__()
        self.layers = nn.ModuleList()
        self.output_shapes = []
        self.K, self.L = K, L
        self.batch_size = batch_size
        self.fuse_squeeze = fuse_squeeze
        H, W, C = image_shape
        assert C == 1 or C == 3, ("image_shape should be HWC, like (64, 64, 3)"
                                  "C == 1 or C == 3")
        for i in range(L):
            C, H, W = C * 4, H // 2, W // 2
            self.layers.append(SqueezeLayer(factor=2))
            self.output_shapes.append([-1, C, H, W])
            for _ in range(K):
                self.layers.append(FlowStep(H, W, C, in_channels=C, out_channels=C, hidden_channels=hidden_channels,
                                            actnorm_scale=actnorm_scale, coupling_type=coupling_type,
                                            num_blocks=num_blocks, attn=attn, drop_prob=drop_prob))
                self.output_shapes.append([-1, C, H, W])
            if i < L - 1:
                self.layers.append(Split2dMsC(C, i + 1))
                self.output_shapes.append([-1, C // 2, H, W])
                C = C // 2
        if prior == "mar":          # the reference's prior (marscf_main.py:147-148), sized from the image instead of 3x32x32
            from .mar_prior import ChannelPriorMultiScale
            h0, w0, c0 = image_shape
            prior = ChannelPriorMultiScale(batch_size, c0, h0, w0, L, mog=False, dp_rate=0, num_layers=3, hidden_size=32)
        self.c_prior = prior if prior is not None else StandardNormalPrior(image_shape, L)

    def forward(self, input, logdet=0., reverse=False, eps_std=None):
        if not reverse:
            return self.encode(input, logdet)
        return self.decode(input, eps_std)

    # -- forward ---------------------------------------------------------------------------------
    def encode_latents(self, z, logdet=0.0, pairs=None):
        """Layer loop of FlowNet.encode (marscf_main.py:156-165) without the prior terms.
        Returns (z_final, [z2 of every split], flow logdet); `pairs` (a list) receives the (z1, z2) of every split."""
        outs = []
        layers = list(self.layers)
        i = 0
        while i < len(layers):
            layer = layers[i]
            nxt = layers[i + 1] if i + 1 < len(layers) else None
            if (self.fuse_squeeze and isinstance(layer, SqueezeLayer) and layer.factor == 2
                    and isinstance(nxt, FlowStep)):
                assert z.size(2) % 2 == 0 and z.size(3) % 2 == 0, "{}".format((z.size(2), z.size(3)))
                z, logdet = nxt.forward_inference(z, logdet, squeeze_input=True)
                i += 2
                continue
            z, logdet = layer(z, logdet, reverse=False)
            if isinstance(layer, Split2dMsC):
                z, z2 = z
                outs.append(z2)
                if pairs is not None:
                    pairs.append((z, z2))
            i += 1
        return z, outs, logdet

    def encode(self, z, logdet=0.0):
        pairs = []
        z, outs, logdet = self.encode_latents(z, logdet, pairs)
        acc = getattr(self.c_prior, "accumulate", None)        # priors that can add their term to the objective in place
        for level, pair in enumerate(pairs, start=1):          # marscf_main.py:159-163
            logdet = acc(pair, level, logdet) if acc else logdet + self.c_prior(pair, level, reverse=False)
        logdet = acc(z, self.L, logdet) if acc else logdet + self.c_prior(z, self.L, reverse=False)
        return z, logdet

    # -- reverse ---------------------------------------------------------------------------------
    def decode_latents(self, z, z2s, with_logdet=False):
        """Layer loop of FlowNet.decode (marscf_main.py:169-175) with the factored-out halves given."""
        z2s = list(z2s)
        layers = list(self.layers)
        ldj = z.new_zeros(z.shape[0]) if with_logdet else None
        i = len(layers) - 1
        while i >= 0:
            layer = layers[i]
            prev = layers[i - 1] if i > 0 else None
            if isinstance(layer, Split2dMsC):
                z = torch.cat((z, z2s.pop()), dim=1)
            elif (self.fuse_squeeze and isinstance(layer, FlowStep) and isinstance(prev, SqueezeLayer)
                  and prev.factor == 2):
                z, ldj = layer.reverse_sampling(z, ldj, unsqueeze_output=True)
                i -= 1
            else:
                z, ldj = layer(z, ldj, reverse=True)
            i -= 1
        return (z, ldj) if with_logdet else z

    def decode(self, z, eps_std=None, prior=None):
        """Sample (marscf_main.py:167-175): the last level's latent, then at every split z2 given the decoded z1.
        `prior` (default: self.c_prior) takes the same calls as c_prior, e.g. one whose samples come from a CUDA graph's
        device-side noise."""
        prior = self.c_prior if prior is None else prior
        if z is None:
            z = prior(None, self.L, reverse=True, eps_std=eps_std, batch_size=self.batch_size,
                      device=next(self.parameters()).device)
        else:
            z = prior(z, self.L, reverse=True, eps_std=eps_std)
        layers = list(self.layers)
        i = len(layers) - 1
        while i >= 0:
            layer = layers[i]
            prev = layers[i - 1] if i > 0 else None
            if isinstance(layer, Split2dMsC):
                z2 = prior(z, layer.level, reverse=True, eps_std=eps_std)
                z, _ = layer((z, z2), logdet=0, reverse=True)
            elif (self.fuse_squeeze and isinstance(layer, FlowStep) and isinstance(prev, SqueezeLayer)
                  and prev.factor == 2):
                z, _ = layer.reverse_sampling(z, None, unsqueeze_output=True)
                i -= 1
            else:
                z, _ = layer(z, logdet=None, reverse=True)
            i -= 1
        return z


class MarScfFlow(nn.Module):
    def __init__(self, batch_size, image_shape, coupling_type, L, K, C, prior=None, num_blocks=10,
                 fuse_squeeze=True, attn=False, drop_prob=0.2):
        super().__init__()
        self.flow = FlowNet(batch_size, image_shape=image_shape, hidden_channels=C, K=K, L=L,
                            coupling_type=coupling_type, prior=prior, num_blocks=num_blocks,
                            fuse_squeeze=fuse_squeeze, attn=attn, drop_prob=drop_prob)
        self.batch_size = batch_size
        from .flow_modules.mixlogcdf_nn import assign_dropout_salts
        assign_dropout_salts(self)

    def forward(self, x=None, z=None, eps_std=None, reverse=False, noise=None):
        if not reverse:
            return self.normal_flow(x, noise)
        return self.reverse_flow(z, eps_std)

    def normal_flow(self, x, noise=None):
        """Uniform dequantisation, logdet0 = -ln(256) D, encode, bits/dim (marscf_main.py:192-206).
        `noise` (U[0,1), same shape as x) can be injected for reproducible parity runs."""
        d = x.size(1) * x.size(2) * x.size(3)
        if self.training and torch.is_grad_enabled() and x.is_cuda:
            self._weight_norm_batch().refresh()         # every weight-normed layer's GEMM operands in two launches
            from . import tc_autograd
            tc_autograd.advance_dropout_seed(x.device)  # fresh attention-dropout masks (also on every graph replay)
        if noise is None:
            noise = torch.rand_like(x)
        z = x + noise * (1. / 256.)
        logdet = x.new_full((x.size(0),), float(-math.log(256.) * d))
        z, objective = self.flow(z, logdet=logdet, reverse=False)
        nll = (-objective) / float(math.log(2.) * d)
        return z, nll, None

    def _weight_norm_batch(self):
        from . import tc_autograd
        from .flow_modules.mixlogcdf_nn import _WNConvCore, _WNLinear
        if getattr(self, "_wn_batch", None) is None:
            self._wn_batch = tc_autograd.WeightNormBatch([m for m in self.modules() if isinstance(m, (_WNConvCore, _WNLinear))])
        return self._wn_batch

    def reverse_flow(self, z, eps_std):
        with torch.no_grad():
            return self.flow(z, eps_std=eps_std, reverse=True)

    def load_my_state_dict(self, state_dict):
        own_state = self.state_dict()
        for name, param in state_dict.items():
            if isinstance(param, nn.Parameter):
                param = param.data
            own_state[name].copy_(param)
