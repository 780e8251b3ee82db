"""The MixLogCDF model on 64x64 images: the long-sequence tcgen05 attention core (csrc/attention_long_tc.cu) over the
1024-token level-1 maps, its route in tc.attention, the model's eval and sampling paths against the fp64 oracle, and
training attention at 1024 tokens on the existing kernels."""
import math

import numpy as np
import pytest
import torch

from oracle import flow_oracle as O


def _lib():
    import flowk  # noqa: F401
    from flowk import _lib
    return _lib


def dev():
    return torch.device("cuda:0")


def rel_err(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def parity(got, ref, rel, what=""):
    ref = ref.to(torch.float32)
    got = got.detach().float().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    scale = max(1.0, float(ref.abs().max())) if ref.numel() else 1.0
    err = float((got - ref).abs().max()) if ref.numel() else 0.0
    assert err <= rel * scale, "%s: max abs err %.3e > %.1e * %.3g" % (what, err, rel, scale)


# ---------------------------------------------------------------------------------------------------------------------
# C ABI: argument checks before any launch (no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def test_long_attention_validates_arguments():
    L = _lib()
    f, ARG, SHAPE = L.lib.flowk_attention_long_tc, L.FLOWK_ERR_ARG, L.FLOWK_ERR_SHAPE
    one = 16                                        # any non-NULL address: validation fails before a launch
    assert f(None, one, one, 1, 2, 1024, 128, 4, None, None, None) == ARG
    assert f(one, None, one, 1, 2, 1024, 128, 4, None, None, None) == ARG
    assert f(one, one, None, 0, 2, 1024, 128, 4, None, None, None) == ARG
    assert f(one, one, one, 1, 2, 256, 128, 4, None, None, None) == SHAPE          # < 512 tokens
    assert f(one, one, one, 1, 2, 1000, 128, 4, None, None, None) == SHAPE         # not a multiple of 128
    assert f(one, one, one, 1, 2, 1024, 192, 4, None, None, None) == SHAPE         # d = 48
    assert f(one, one, one, 1, 2, 1024, 128, 0, None, None, None) == SHAPE         # heads = 0
    assert f(one, one, one, 1, -1, 1024, 128, 4, None, None, None) == SHAPE
    assert f(None, None, None, 1, 0, 1024, 128, 4, None, None, None) == L.FLOWK_OK  # B = 0: nothing to do


def test_long_attention_routes_by_shape():
    import flowk  # noqa: F401
    from flowk import tc
    for hw, c in ((1024, 128), (1024, 160), (1024, 256), (512, 256), (2048, 128)):
        assert tc.attention_long_tc_supported(hw, c, 4) and tc.attention_supported(hw, c, 4)
        assert not tc._attention_mma_supported(hw, c, 4)
    for hw, c in ((256, 128), (1000, 128), (1024, 192), (1024, 224), (1024, 64)):
        assert not tc.attention_long_tc_supported(hw, c, 4)
    assert tc._attention_mma_supported(1024, 96, 4) and tc._attention_mma_supported(1024, 64, 4)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernel against fp64 and against the mma.sync kernel
# ---------------------------------------------------------------------------------------------------------------------
def _reference(qkv, B, HW, C, heads):
    d = C // heads
    x = qkv.double().view(B, HW, 3 * C)
    k, v, q = x[..., :C], x[..., C:2 * C], x[..., 2 * C:]
    hf = lambda m: m.reshape(B, HW, heads, d).permute(0, 2, 1, 3)          # noqa: E731
    w = torch.softmax((hf(q) * d ** -0.5) @ hf(k).transpose(-1, -2), dim=-1)
    return (w @ hf(v)).permute(0, 2, 1, 3).reshape(B * HW, C)


def _long(qkv, B, HW, C, heads, f16, status=None):
    L = _lib()
    dt = torch.float16 if f16 else torch.float32
    hi = torch.full((B * HW, C), float("nan"), device=qkv.device, dtype=dt)
    lo = torch.full_like(hi, float("nan"))
    L.call("flowk_attention_long_tc", qkv.data_ptr(), hi.data_ptr(), lo.data_ptr(), int(f16), B, HW, C, heads,
           None if status is None else status.data_ptr(), None, torch.cuda.current_stream().cuda_stream)
    return hi, lo


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [True, False])
@pytest.mark.parametrize("B,HW,C,heads,late_max", [(2, 1024, 96, 4, False), (2, 1024, 128, 4, False),
                                                   (2, 1024, 160, 4, False), (2, 1024, 256, 4, False),
                                                   (3, 512, 128, 4, False), (1, 2048, 96, 4, False),
                                                   (2, 1024, 256, 4, True)])
def test_long_attention_matches_fp64(B, HW, C, heads, late_max, f16):
    g = torch.Generator().manual_seed(B * 1000 + HW + C)
    qkv = torch.randn(B * HW, 3 * C, generator=g) * 1.5
    if late_max:
        # one large key in the last 128-key block, aligned with every query: each row's largest logit sits there, so
        # the running output is rescaled after every earlier block has been folded in
        d = C // heads
        q = qkv[:, 2 * C:].view(B, HW, heads, d)
        k = qkv[:, :C].view(B, HW, heads, d)
        key = HW - 1 - 37
        q.abs_()
        k[:, key] = 2.0
    qkv = qkv.to(dev())
    status = torch.zeros(1, dtype=torch.int32, device=dev())
    hi, lo = _long(qkv, B, HW, C, heads, f16, status)
    hi2, lo2 = _long(qkv, B, HW, C, heads, f16, status)
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    ref = _reference(qkv.cpu(), B, HW, C, heads)
    if late_max:
        logits = _reference_logit_argmax(qkv.cpu(), B, HW, C, heads)
        assert bool((logits >= HW - 128).all())
    assert rel_err((hi.float() + lo.float()).cpu(), ref) < 2e-5
    if not f16:
        assert int((hi.view(torch.int32) & 0x1fff).abs().max()) == 0
    assert torch.equal(hi, hi2) and torch.equal(lo, lo2)


def _reference_logit_argmax(qkv, B, HW, C, heads):
    d = C // heads
    x = qkv.double().view(B, HW, 3 * C)
    hf = lambda m: m.reshape(B, HW, heads, d).permute(0, 2, 1, 3)          # noqa: E731
    return (hf(x[..., 2 * C:]) @ hf(x[..., :C]).transpose(-1, -2)).argmax(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [True, False])
@pytest.mark.parametrize("C", [96, 128, 160, 256])
def test_long_attention_agrees_with_mma_sync_kernel(C, f16):
    L = _lib()
    B, HW, heads = 2, 1024, 4
    g = torch.Generator().manual_seed(C)
    qkv = (torch.randn(B * HW, 3 * C, generator=g) * 1.5).to(dev())
    hi, lo = _long(qkv, B, HW, C, heads, f16)
    dt = torch.float16 if f16 else torch.float32
    ohi = torch.empty(B * HW, C, device=dev(), dtype=dt)
    olo = torch.empty_like(ohi)
    L.call("flowk_attention_f16" if f16 else "flowk_attention", qkv.data_ptr(), ohi.data_ptr(), olo.data_ptr(), B, HW, C,
           heads, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    old = (ohi.float() + olo.float()).double()
    assert rel_err(hi.float() + lo.float(), old) < 2e-5


@pytest.mark.gpu
def test_attention_routes_at_long_sequences():
    import flowk  # noqa: F401
    from flowk import tc
    L = _lib()
    for HW, C, route in ((1024, 128, "flowk_attention_long_tc"), (1024, 256, "flowk_attention_long_tc"),
                         (1024, 96, "flowk_attention_f16"), (1024, 64, "flowk_attention_f16"),
                         (256, 96, "flowk_attention_tc_v2")):
        qkv = torch.randn(2 * HW, 3 * C, device=dev())
        L.TIMING = {}
        try:
            tc.attention(qkv, 2, HW, C, 4, f16=True)
            torch.cuda.synchronize()
            names = [n for n in L.TIMING if "attention" in n]
        finally:
            L.TIMING = None
        assert names == [route], (HW, C, names)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the 64x64 MixLogCDF model
# ---------------------------------------------------------------------------------------------------------------------
def _initialised_model(B, L, K, hidden, seed, image=(64, 64, 3), **kw):
    from flowk.marscf import MarScfFlow
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = MarScfFlow(B, image, "mixlogcdf", L, K, hidden, **kw).to(dev())
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(B, image[2], image[0], image[1], generator=gen) - 0.5
    noise = torch.rand(B, image[2], image[0], image[1], generator=gen)
    model.train()
    with torch.no_grad():
        model(x.to(dev()), noise=noise.to(dev()))            # ActNorm data-dependent init (first training batch)
        for p in model.parameters():                         # move the zero-initialised output convs off zero
            p.add_((torch.randn(p.shape, generator=gen) * 0.005).to(p.device))
    return model, x, noise


@pytest.mark.gpu
@pytest.mark.parametrize("hidden", [128, 256])
def test_64x64_model_vs_oracle(no_library, hidden):
    L = _lib()
    Lv, K, B = 4, 2, 2
    model, x, noise = _initialised_model(B, Lv, K, hidden, seed=300 + hidden, num_blocks=2)
    model.eval()
    d = x[0].numel()
    L.TIMING = {}
    try:
        with torch.no_grad():
            z, nll, _ = model(x.to(dev()), noise=noise.to(dev()))
            zf, outs, ld = model.flow.encode_latents((x + noise / 256.0).to(dev()), torch.zeros(B, device=dev()))
            xr, ldr = model.flow.decode_latents(zf, outs, with_logdet=True)
        torch.cuda.synchronize()
        names = set(L.TIMING)
    finally:
        L.TIMING = None
    assert "flowk_attention_long_tc" in names and "flowk_conv_gemm" in names, sorted(names)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    z_ref, outs_ref, ld_ref, nll_ref = O.normal_flow(sd, x, noise, Lv, K, "mixlogcdf")
    parity(z, z_ref, 1e-4, what="z")
    for i, (a, b) in enumerate(zip(outs, outs_ref)):
        parity(a, b, 1e-4, what="z2_%d" % i)
    parity(ld, ld_ref - float(-math.log(256.0) * d), 1e-4, what="logdet")
    assert float((nll.cpu() - nll_ref).abs().max()) < 1e-3
    parity(xr, x + noise / 256.0, 2e-3, what="round trip")
    assert float((ld + ldr).abs().max()) < 2e-3 * max(1.0, float(ld.abs().max()))


@pytest.mark.gpu
def test_64x64_sampling_eager_and_graphed(no_library):
    from flowk.graphs import GraphedSampler
    B, image = 4, (64, 64, 3)
    model, _, _ = _initialised_model(B, 4, 2, 256, seed=41, num_blocks=1)
    model.eval()
    with torch.no_grad():
        x = model(None, None, reverse=True)
    x = x[0] if isinstance(x, tuple) else x
    assert x.shape == (B, 3, 64, 64) and bool(torch.isfinite(x).all())
    lane = GraphedSampler(model, B, image)
    recs = []
    for _ in range(2):
        lane.run()
        with torch.cuda.stream(lane.stream):
            recs.append((lane.z.clone(), [t.clone() for t in lane.z2s], lane.images.clone()))
    torch.cuda.synchronize()
    assert not torch.equal(recs[0][0], recs[1][0])
    with torch.no_grad():
        for i, (z, z2s, images) in enumerate(recs):
            x = model.flow.decode_latents(z, z2s)
            nan = torch.isnan(x)
            assert torch.equal(torch.clamp(torch.where(nan, torch.full_like(x, -0.5), x), -0.5, 0.5), images), i


# ---------------------------------------------------------------------------------------------------------------------
# GPU: training at 1024 tokens on the existing kernels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,S,C,heads,p", [(2, 1024, 128, 4, 0.2), (2, 1024, 256, 4, 0.2)])
def test_training_attention_1024_tokens_matches_fp64(B, S, C, heads, p):
    from flowk import tc_autograd
    g = torch.Generator(device="cpu").manual_seed(29)
    qkv = torch.randn(B, S, 3 * C, generator=g).to(dev()).requires_grad_()
    dout = torch.randn(B, S, C, generator=g).to(dev())
    salt, d = 7, C // heads
    out = tc_autograd.attention_core(qkv, heads, p, salt)
    out.backward(dout)
    mask = tc_autograd.attention_dropout_mask(dev(), salt, p, B * heads, S).double().view(B, heads, S, S)
    keep = float((mask > 0).double().mean())
    assert abs(keep - (1 - p)) < 0.02
    x = qkv.detach().double().requires_grad_()
    k, v, q = x[..., :C], x[..., C:2 * C], x[..., 2 * C:]
    hf = lambda m: m.reshape(B, S, heads, d).permute(0, 2, 1, 3)          # noqa: E731
    w = torch.softmax((hf(q) * d ** -0.5) @ hf(k).transpose(-1, -2), dim=-1) * mask
    ref = (w @ hf(v)).permute(0, 2, 1, 3).reshape(B, S, C)
    ref.backward(dout.double())
    assert rel_err(out.detach(), ref.detach()) < 2e-5
    assert rel_err(qkv.grad, x.grad) < 5e-5


@pytest.mark.gpu
def test_64x64_training_gradients_vs_oracle(no_library):
    L = _lib()
    Lv, K, hidden, B = 4, 1, 128, 2
    model, x, noise = _initialised_model(B, Lv, K, hidden, seed=91, num_blocks=1, drop_prob=0.0)
    sd64 = {k: v.detach().cpu().double().requires_grad_(v.dtype.is_floating_point and "is_initialized" not in k and
                                                         not k.endswith(".p") and not k.endswith("sign_s"))
            for k, v in model.state_dict().items()}
    _, _, _, nll = O.normal_flow(sd64, x.double(), noise.double(), Lv, K, "mixlogcdf")
    nll.mean().backward()
    model.train()
    L.TIMING = {}
    try:
        _, nll_d, _ = model(x.to(dev()), noise=noise.to(dev()))
        nll_d.mean().backward()
        torch.cuda.synchronize()
        names = set(L.TIMING)
    finally:
        L.TIMING = None
    assert {"flowk_attention_train_fwd", "flowk_attention_train_bwd"} <= names, sorted(names)
    assert float((nll_d.detach().cpu() - nll.float()).abs().max()) < 1e-3
    checked = 0
    for name, p in model.named_parameters():
        ref = sd64[name].grad
        if ref is None:
            continue
        if name.endswith(".l") or name.endswith(".u"):
            c = ref.shape[0]
            ref = ref * (torch.tril(torch.ones(c, c), -1) if name.endswith(".l") else torch.triu(torch.ones(c, c), 1))
        parity(p.grad, ref, 1e-3, what="grad " + name)
        checked += 1
    assert checked > 50
