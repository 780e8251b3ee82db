"""Generate the golden fixtures in this directory from the REFERENCE's own modules.

Run in the build container only (it imports /root/reference read-only):

    python tests/golden/make_golden.py

Nothing here runs on the GPU box: the committed ``*.npz`` files are what travels.
The reference ships no known-answer vectors of its own (SURVEY.md section 4), so
these files - outputs of its live modules on seeded inputs - are the pin for
``oracle/flow_oracle.py`` and, through it, for the CUDA kernels.

What is NOT the reference here, and why (SURVEY.md section 8c):
  * ``marscf_main.py`` cannot be imported (``utils/`` package shadows ``utils.py``), so the
    ~40 lines of FlowStep/FlowNet/MarScfFlow composition are re-stated below from
    marscf_main.py:35-206, WITHOUT the fork's Transformer_attn add-on (not on the north-star
    path) and with a standard-normal prior instead of the ConvLSTM prior (outside the path).
  * ``InvertibleConv1x1`` reverse ends in ``.cuda()`` (common_modules.py:110); ``Tensor.cuda``
    is patched to the identity while generating so that the reference's own lines run on CPU.
Every arithmetic module (Actnormlayer, InvertibleConv1x1, AffineCoupling, MixLogCDFCoupling,
SqueezeLayer, Split2dMsC, TupleFlip, log_dist.*) is the reference's code, unmodified.
"""
import json
import os
import sys
import warnings

import numpy as np
import torch
import torch.nn as nn

REF = os.environ.get("FLOWK_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")

from flow_modules.common_modules import (Actnormlayer, InvertibleConv1x1, SqueezeLayer,  # noqa: E402
                                         Split2dMsC, TupleFlip, GaussianDiag, squeeze2d, unsqueeze2d)
from flow_modules.affine_coupling import AffineCoupling  # noqa: E402
from flow_modules.mixlogcdf_coupling import MixLogCDFCoupling  # noqa: E402
import flow_modules.log_dist as logistic  # noqa: E402

torch.Tensor.cuda = lambda self, *a, **k: self      # see module docstring
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from conftest import rebuild_weight, sha256  # noqa: E402

RECIPE_MIN = 1 << 16      # weights with more elements are stored as generator states (keeps every fixture under 1 MB)


def save(name, meta, **arrays):
    out = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()}
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print("%-28s %7.1f KB  %d arrays" % (name, os.path.getsize(path) / 1024, len(out)))


def sd_arrays(module, prefix="sd/"):
    return {prefix + k: v.clone() for k, v in module.state_dict().items()}


def perturb(module, gen, std=0.05, states=None):
    """Move every parameter off its (partly zero / identity) init so no term is trivially 0.  `states`, if given,
    collects the generator state before each parameter's draw."""
    with torch.no_grad():
        for n, p in module.named_parameters():
            if states is not None:
                states[n] = gen.get_state()
            p.add_(torch.randn(p.shape, generator=gen) * std)


class RefFlowStep(nn.Module):
    """marscf_main.py:35-113 minus attn1/attn2; num_blocks exposed so fixtures stay small."""

    def __init__(self, in_channels, hidden, coupling, num_blocks=10):
        super().__init__()
        self.coupling_type = coupling
        if coupling == "mixlogcdf":
            self.coupling = MixLogCDFCoupling(in_channels, hidden, num_blocks=num_blocks,
                                              num_components=32, drop_prob=0.2)
            self.tuple_flip = TupleFlip()
        else:
            self.coupling = AffineCoupling(in_channels, in_channels, hidden)
        self.actnormlayer = Actnormlayer(in_channels, 1.0)
        self.invert_1x1_layer = InvertibleConv1x1(in_channels)

    def forward(self, x, logdet=0., reverse=False):
        if not reverse:
            x, logdet = self.actnormlayer(x, logdet, reverse)
            x, logdet = self.invert_1x1_layer(x, logdet, reverse)
            x, logdet = self.coupling(x, logdet, reverse)
            if self.coupling_type == "mixlogcdf":
                x, logdet = self.tuple_flip(x, logdet, reverse)
        else:
            if self.coupling_type == "mixlogcdf":
                x, logdet = self.tuple_flip(x, logdet, reverse)
            x, logdet = self.coupling(x, logdet, reverse)
            x, logdet = self.invert_1x1_layer(x, logdet, reverse)
            x, logdet = self.actnormlayer(x, logdet, reverse)
        return x, logdet


class RefFlowNet(nn.Module):
    """marscf_main.py:116-175 with the layer list of :127-145; splits return their z2."""

    def __init__(self, image_shape, hidden, K, L, coupling, num_blocks=10):
        super().__init__()
        self.layers = nn.ModuleList()
        H, W, C = image_shape
        for i in range(L):
            C, H, W = C * 4, H // 2, W // 2
            self.layers.append(SqueezeLayer(factor=2))
            for _ in range(K):
                self.layers.append(RefFlowStep(C, hidden, coupling, num_blocks))
            if i < L - 1:
                self.layers.append(Split2dMsC(C, i + 1))
                C = C // 2

    def encode(self, z, logdet):
        outs = []
        for layer in self.layers:
            z, logdet = layer(z, logdet, reverse=False)
            if isinstance(layer, Split2dMsC):
                z, z2 = z
                outs.append(z2)
        return z, outs, logdet

    def decode(self, z, z2s):
        z2s = list(z2s)
        total = torch.zeros(z.shape[0])
        for layer in reversed(self.layers):
            if isinstance(layer, Split2dMsC):
                z = (z, z2s.pop())
            z, total = layer(z, logdet=total, reverse=True)
        return z, total


class RefModel(nn.Module):
    def __init__(self, *a, **k):
        super().__init__()
        self.flow = RefFlowNet(*a, **k)


def gen_squeeze():
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 3, 8, 12, generator=g)
    y = squeeze2d(x, 2)
    idx = torch.arange(2 * 3 * 8 * 12, dtype=torch.float32).view(2, 3, 8, 12)
    save("squeeze", {"factor": 2}, x=x, y=y, back=unsqueeze2d(y, 2), idx=idx,
         idx_squeezed=squeeze2d(idx, 2))


def gen_actnorm():
    g = torch.Generator().manual_seed(12)
    m = Actnormlayer(6, 1.0)
    x = torch.randn(4, 6, 5, 7, generator=g) * 1.7 + 0.3
    m.train()
    ldj0 = torch.randn(4, generator=g)
    y_init, ldj_init = m(x, ldj0.clone())            # data-dependent init happens here
    init_bias, init_logs = m.bias.detach().clone(), m.logs.detach().clone()
    perturb(m, g, 0.2)
    m.eval()
    with torch.no_grad():
        y, ldj = m(x, ldj0.clone())
        xr, ldjr = m(y, ldj.clone(), reverse=True)
    save("actnorm", {"scale": 1.0}, x=x, ldj0=ldj0, y_init=y_init, ldj_init=ldj_init,
         init_bias=init_bias, init_logs=init_logs, bias=m.bias, logs=m.logs, y=y, ldj=ldj, xr=xr, ldjr=ldjr)


def gen_invconv():
    g = torch.Generator().manual_seed(13)
    np.random.seed(13)
    for c, hw in ((12, (4, 4)), (24, (2, 6))):
        m = InvertibleConv1x1(c)
        perturb(m, g, 0.05)
        x = torch.randn(3, c, *hw, generator=g)
        ldj0 = torch.randn(3, generator=g)
        with torch.no_grad():
            w_fwd, _ = m.get_weight(x, False)
            z, ldj = m(x, ldj0.clone())
            w_rev, _ = m.get_weight(z, True)
            xr, ldjr = m(z, ldj.clone(), reverse=True)
        save("invconv_c%d" % c, {"c": c}, x=x, ldj0=ldj0, z=z, ldj=ldj, xr=xr, ldjr=ldjr,
             w_fwd=w_fwd.view(c, c), w_rev=w_rev.view(c, c), **sd_arrays(m))


def init_then_perturb(m, x_init, g, std):
    m.train()
    with torch.no_grad():
        m(x_init, torch.zeros(x_init.shape[0]))
    perturb(m, g, std)
    m.eval()


def gen_affine():
    g = torch.Generator().manual_seed(14)
    torch.manual_seed(14)
    m = AffineCoupling(12, 12, 16)
    x = torch.randn(3, 12, 6, 6, generator=g)
    init_then_perturb(m, x, g, 0.05)
    ldj0 = torch.randn(3, generator=g)
    with torch.no_grad():
        h = m.NN_net(x[:, :6])
        y, ldj = m(x, ldj0.clone())
        xr, ldjr = m(y, ldj.clone(), reverse=True)
    save("affine", {"in": 12, "hidden": 16}, x=x, ldj0=ldj0, h=h, y=y, ldj=ldj, xr=xr, ldjr=ldjr,
         **sd_arrays(m, "sd/coupling."))


def gen_mixlogcdf_elementwise():
    g = torch.Generator().manual_seed(15)
    torch.manual_seed(15)
    B, c, H, W, K = 3, 4, 4, 6, 32
    m = MixLogCDFCoupling(2 * c, 8, 1, K, 0.0)
    x = torch.randn(B, 2 * c, H, W, generator=g)
    a = 0.3 * torch.randn(B, c, H, W, generator=g)
    b = 0.3 * torch.randn(B, c, H, W, generator=g)
    pi = torch.randn(B, K, c, H, W, generator=g)
    mu = torch.randn(B, K, c, H, W, generator=g)
    s = (0.7 * torch.randn(B, K, c, H, W, generator=g) - 0.5).clamp(min=-7)

    class FixedParams(nn.Module):          # stands in for the conditioner: returns the drawn params
        def forward(self, x_id, aux=None):
            return a, b, pi, mu, s
    m.nn = FixedParams()
    ldj0 = torch.randn(B, generator=g)
    with torch.no_grad():
        y, ldj = m(x, ldj0.clone())
        xr, ldjr = m(y, ldj.clone(), reverse=True)
        xc = x[:, :c]
        log_cdf = logistic.mixture_log_cdf(xc, pi, mu, s)
        log_pdf = logistic.mixture_log_pdf(xc, pi, mu, s)
        u = torch.rand(B, c, H, W, generator=g).clamp(1e-5, 1 - 1e-5)
        xinv = logistic.mixture_inv_cdf(u, pi, mu, s)
    save("mixlogcdf_elementwise", {"K": K}, x=x, a=a, b=b, pi=pi, mu=mu, s=s, ldj0=ldj0, y=y, ldj=ldj,
         xr=xr, ldjr=ldjr, log_cdf=log_cdf, log_pdf=log_pdf, u=u, xinv=xinv)


def gen_mixlogcdf_coupling():
    g = torch.Generator().manual_seed(16)
    torch.manual_seed(16)
    m = MixLogCDFCoupling(12, 16, 2, 32, 0.2)
    perturb(m, g, 0.03)
    m.eval()
    x = torch.randn(2, 12, 4, 4, generator=g)
    ldj0 = torch.randn(2, generator=g)
    with torch.no_grad():
        a, b, pi, mu, s = m.nn(x[:, 6:], None)
        y, ldj = m(x, ldj0.clone())
        xr, ldjr = m(y, ldj.clone(), reverse=True)
    save("mixlogcdf_coupling", {"in": 12, "hidden": 16, "blocks": 2, "K": 32}, x=x, ldj0=ldj0, a=a, b=b, pi=pi,
         mu=mu, s=s, y=y, ldj=ldj, xr=xr, ldjr=ldjr, **sd_arrays(m, "sd/coupling."))


def gaussian_logp(z):
    return GaussianDiag.logp(torch.zeros_like(z), torch.zeros_like(z), z)


def gen_flownet(name, coupling, image, L, K, hidden, blocks, B, seed):
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    np.random.seed(seed)
    init_states = {}                  # data_ptr -> global generator state right before nn.Conv2d's default weight init
    kaiming = nn.init.kaiming_uniform_

    def recording_kaiming(t, *a, **k):
        init_states[t.data_ptr()] = torch.get_rng_state()
        return kaiming(t, *a, **k)
    nn.init.kaiming_uniform_ = recording_kaiming
    try:
        model = RefModel(image, hidden, K, L, coupling, blocks)
    finally:
        nn.init.kaiming_uniform_ = kaiming
    H, W, C = image
    x = torch.rand(B, C, H, W, generator=g) - 0.5
    noise = torch.rand(B, C, H, W, generator=g)
    D = C * H * W
    z0 = x + noise * (1. / 256.)
    ld0 = torch.zeros(B) + float(-np.log(256.) * D)
    model.train()
    with torch.no_grad():
        model.flow.encode(z0, ld0)                       # ActNorm data-dependent init
    perturb_states = {}
    perturb(model, g, 0.02, perturb_states)
    model.eval()
    with torch.no_grad():
        z, outs, logdet = model.flow.encode(z0, ld0)
        objective = logdet + gaussian_logp(z)
        for o in outs:
            objective = objective + gaussian_logp(o)
        nll = (-objective) / float(np.log(2.) * D)
        xr, ldr = model.flow.decode(z, outs)
    arrays = dict(x=x, noise=noise, z=z, logdet=logdet, nll=nll, xr=xr, ldr=ldr)
    for i, o in enumerate(outs):
        arrays["z2_%d" % i] = o
    meta = {"coupling": coupling, "image_hwc": list(image), "L": L, "K": K, "hidden": hidden,
            "blocks": blocks, "B": B}
    sd = sd_arrays(model)
    rebuilt = {}
    for k, v in model.state_dict().items():
        if v.numel() < RECIPE_MIN:
            continue
        init, pert = init_states[v.data_ptr()], perturb_states[k]
        assert torch.equal(rebuild_weight(list(v.shape), init, pert, 0.02), v), k
        rebuilt[k] = {"shape": list(v.shape), "std": 0.02, "sha256": sha256(v)}
        arrays["rng_init/" + k], arrays["rng_perturb/" + k] = init, pert
        del sd["sd/" + k]
    if rebuilt:
        meta["rebuilt"] = rebuilt
    save(name, meta, **arrays, **sd)


def gen_mar_prior():
    """mAR channel prior (mar_prior/corr_prior.py) - outside the hot path, pinned for the plug-in port.
    `collections.Iterable` is aliased first: mar_prior/convolutional_rnn/utils.py:10 predates its removal."""
    import collections
    import collections.abc
    collections.Iterable = collections.abc.Iterable
    from mar_prior.corr_prior import ChannelPriorMultiScale
    g = torch.Generator().manual_seed(31)
    torch.manual_seed(31)
    B, L = 2, 2
    prior = ChannelPriorMultiScale(B, 3, 16, 16, L, mog=False, dp_rate=0, num_layers=2, hidden_size=8)
    prior.eval()
    z1 = torch.randn(B, 6, 8, 8, generator=g)
    z2 = torch.randn(B, 6, 8, 8, generator=g)
    zf = torch.randn(B, 24, 4, 4, generator=g)
    with torch.no_grad():
        ll1 = prior((z1, z2), 1, reverse=False)
        ll2 = prior(zf, 2, reverse=False)
        torch.manual_seed(77)
        s2 = prior(None, 2, reverse=True)
        torch.manual_seed(78)
        s1 = prior(z1, 1, reverse=True)
    save("mar_prior", {"B": B, "L": L, "hidden": 8, "num_layers": 2, "image_hwc": [16, 16, 3]}, z1=z1, z2=z2, zf=zf,
         ll1=ll1, ll2=ll2, s2=s2, s1=s1, **sd_arrays(prior))


def gen_transformer_attn():
    """The fork's invertible patch attention (flow_modules/transformer.py) - SURVEY.md section 8f-2.  Its constructor and
    forward call `.cuda()` throughout; with `Tensor.cuda` patched to the identity its own lines run on CPU."""
    from flow_modules.transformer import Transformer_attn
    g = torch.Generator().manual_seed(41)
    cases = {}
    for tag, (B, C, H) in {"c12": (3, 12, 8), "c24": (2, 24, 4)}.items():
        torch.manual_seed(41 + C)
        m = Transformer_attn(C)
        with torch.no_grad():
            # spread the attention logits: the default scale=100 leaves sigmoid() almost constant
            m.scale.fill_(3.0)
            m.offset.fill_(0.9)
            m.offset2.fill_(0.4)
            m.offset3.fill_(-0.55)
        x = torch.randn(B, C, H, H, generator=g)
        ld0 = torch.randn(B, generator=g)
        arrays = {"x": x, "ld0": ld0}
        with torch.no_grad():
            for permute in (False, True):
                y, ld = m(x.clone(), logdet=ld0.clone(), reverse=False, permute=permute)
                xr, ldr = m(y.clone(), logdet=ld.clone(), reverse=True, permute=permute)
                sfx = "_perm" if permute else ""
                arrays.update({"y" + sfx: y, "ld" + sfx: ld, "xr" + sfx: xr, "ldr" + sfx: ldr})
        arrays.update(sd_arrays(m))
        cases[tag] = arrays
    for tag, arrays in cases.items():
        save("transformer_attn_" + tag, {"case": tag}, **arrays)


if __name__ == "__main__":
    only = set(sys.argv[1:])          # `make_golden.py wide` regenerates only the width-32 nets below

    def want(tag):
        return not only or tag in only
    if want("base"):
        gen_transformer_attn()
        gen_mar_prior()
        gen_squeeze()
        gen_actnorm()
        gen_invconv()
        gen_affine()
        gen_mixlogcdf_elementwise()
        gen_mixlogcdf_coupling()
        gen_flownet("flownet_affine", "affine", (16, 16, 3), 3, 2, 8, 0, 2, 21)
        gen_flownet("flownet_mixlogcdf", "mixlogcdf", (8, 8, 3), 2, 1, 8, 1, 2, 22)
    if want("wide"):
        # hidden width 32: the narrowest nets whose conditioners run ENTIRELY on the tcgen05 / flowk kernels (channel
        # blocks of 32, attention head dim 8), so the tensor-core path is pinned to the reference's own outputs
        gen_flownet("flownet_affine_h32", "affine", (16, 16, 3), 2, 2, 32, 0, 2, 23)
        gen_flownet("flownet_mixlogcdf_h32", "mixlogcdf", (16, 16, 3), 2, 1, 32, 1, 2, 24)
