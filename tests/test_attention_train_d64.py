"""Training attention at head dim 64 (the width-256 MixLogCDF model: 4 heads x 64): the tcgen05 kernels of
csrc/attention_train_tc.cu at 128 / 256 tokens, the D = 64 mma.sync instances at the deep levels' 64 / 16 tokens, and the
width-256 model trained end to end on flowk kernels."""
import copy
import math
import os

import numpy as np
import pytest
import torch

from oracle import flow_oracle as O


def _lib():
    import flowk  # noqa: F401
    from flowk import _lib
    return _lib


# ---------------------------------------------------------------------------------------------------------------------
# C ABI: argument checks before any launch (no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def test_tc_entry_points_validate_arguments():
    L = _lib()
    lib, ARG, SHAPE = L.lib, L.FLOWK_ERR_ARG, L.FLOWK_ERR_SHAPE
    assert lib.flowk_abi_version() == 3
    one = 16                                        # any non-NULL address: validation fails before a launch
    fwd, bwd = lib.flowk_attention_train_tc_fwd, lib.flowk_attention_train_tc_bwd
    assert fwd(None, one, one, None, 1, 0.2, 2, 256, 256, 4, None) == ARG
    assert fwd(one, None, one, None, 1, 0.2, 2, 256, 256, 4, None) == ARG
    assert fwd(one, one, None, None, 1, 0.2, 2, 256, 256, 4, None) == ARG
    assert fwd(one, one, one, None, 1, 0.2, 2, 256, 128, 4, None) == SHAPE        # D = 32
    assert fwd(one, one, one, None, 1, 0.2, 2, 256, 192, 4, None) == SHAPE        # D = 48
    for S in (16, 64, 136, 512):
        assert fwd(one, one, one, None, 1, 0.2, 2, S, 256, 4, None) == SHAPE
    for p in (-0.1, 1.0, float("nan")):
        assert fwd(one, one, one, None, 1, p, 2, 256, 256, 4, None) == SHAPE
    assert fwd(one, one, one, None, 1, 0.2, 16384, 256, 256, 4, None) == SHAPE    # B*heads*S^2 = 2^32: mask counter
    for which in (0, 4):
        assert bwd(which, one, one, one, one, one, None, 1, 0.2, 2, 256, 256, 4, None) == ARG
    for i in range(5):
        ptrs = [one] * 5
        ptrs[i] = None
        assert bwd(3, *ptrs, None, 1, 0.2, 2, 256, 256, 4, None) == ARG
    assert bwd(3, one, one, one, one, one, None, 1, 0.2, 2, 256, 160, 4, None) == SHAPE
    assert bwd(3, one, one, one, one, one, None, 1, 0.2, 2, 64, 256, 4, None) == SHAPE
    assert bwd(3, one, one, one, one, one, None, 1, 1.5, 2, 256, 256, 4, None) == SHAPE
    assert bwd(1, one, one, one, one, one, None, 1, 0.2, 16384, 256, 256, 4, None) == SHAPE


def test_head_dim_64_is_admitted_for_training(monkeypatch):
    import flowk  # noqa: F401
    from flowk import tc_autograd
    monkeypatch.setattr(tc_autograd, "ENABLED", True)

    class Q:                                         # the predicate reads only these attributes
        is_cuda, dtype = True, torch.float32

        def __init__(self, *shape):
            self.shape = shape

        def dim(self):
            return len(self.shape)
    for s in (16, 64, 128, 256, 136):
        assert tc_autograd.attention_train_supported(Q(2, s, 768), 4)
    assert not tc_autograd.attention_train_supported(Q(2, 12, 768), 4)              # S % 8
    assert not tc_autograd.attention_train_supported(Q(2, 256, 576), 4)             # D = 48
    assert not tc_autograd.attention_train_supported(Q(16384, 256, 768), 4)         # mask counter
    assert tc_autograd._attention_train_entry(256, 64) == tc_autograd._attention_train_entry(128, 64) == \
        "flowk_attention_train_tc"
    for s, d in ((64, 64), (16, 64), (256, 32), (256, 24), (136, 64)):
        assert tc_autograd._attention_train_entry(s, d) == "flowk_attention_train"


# ---------------------------------------------------------------------------------------------------------------------
# GPU: kernels against fp64 autograd with the kernels' own mask
# ---------------------------------------------------------------------------------------------------------------------
def rel_err(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _run(qkv, dout, heads, p, salt):
    from flowk import tc_autograd
    q = qkv.detach().clone().requires_grad_()
    out = tc_autograd.attention_core(q, heads, p, salt)
    out.backward(dout)
    return out.detach(), q.grad


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,C,heads,p", [(2, 256, 256, 4, 0.2), (3, 128, 256, 4, 0.0), (1, 256, 128, 2, 0.3),
                                           (2, 64, 256, 4, 0.2), (4, 16, 256, 4, 0.5)])
def test_d64_training_attention_matches_fp64(B, S, C, heads, p):
    from flowk import tc_autograd
    L = _lib()
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(31)
    qkv = torch.randn(B, S, 3 * C, generator=g).to(dev)
    dout = torch.randn(B, S, C, generator=g).to(dev)
    salt, d = 5, C // heads
    L.TIMING = {}
    try:
        out, grad = _run(qkv, dout, heads, p, salt)
        torch.cuda.synchronize()
        names = set(L.TIMING)
    finally:
        L.TIMING = None
    tc_route = S in (128, 256)
    want = {"flowk_attention_train_tc_fwd", "flowk_attention_train_tc_bwd"} if tc_route else \
        {"flowk_attention_train_fwd", "flowk_attention_train_bwd"}
    other = {"flowk_attention_train_fwd", "flowk_attention_train_bwd"} if tc_route else \
        {"flowk_attention_train_tc_fwd", "flowk_attention_train_tc_bwd"}
    assert want <= names and not (other & names), sorted(names)
    mask = tc_autograd.attention_dropout_mask(dev, salt, p, B * heads, S).double().view(B, heads, S, S)
    x = qkv.double().requires_grad_()
    k, v, q = x[..., :C], x[..., C:2 * C], x[..., 2 * C:]
    hf = lambda m: m.reshape(B, S, heads, d).permute(0, 2, 1, 3)          # noqa: E731
    w = torch.softmax((hf(q) * d ** -0.5) @ hf(k).transpose(-1, -2), dim=-1) * mask
    ref = (w @ hf(v)).permute(0, 2, 1, 3).reshape(B, S, C)
    ref.backward(dout.double())
    assert rel_err(out, ref.detach()) < 2e-5
    assert rel_err(grad, x.grad) < 5e-5


@pytest.mark.gpu
@pytest.mark.parametrize("S", [128, 256])
def test_d64_tc_route_is_deterministic_and_draws_fresh_masks(S):
    from flowk import tc_autograd
    L = _lib()
    dev = torch.device("cuda:0")
    B, C, heads, p, salt = 3, 256, 4, 0.2, 9
    g = torch.Generator(device="cpu").manual_seed(41)
    qkv = torch.randn(B, S, 3 * C, generator=g).to(dev)
    dout = torch.randn(B, S, C, generator=g).to(dev)
    out, grad = _run(qkv, dout, heads, p, salt)
    out2, grad2 = _run(qkv, dout, heads, p, salt)                          # two forward + two backward calls
    assert torch.equal(out, out2) and torch.equal(grad, grad2)
    # the backward kernels on their own, twice: bit-identical dqkv
    lse = torch.empty(B * heads, S, device=dev)
    o = torch.empty(B, S, C, device=dev)
    seed = tc_autograd.dropout_seed(dev)
    L.call("flowk_attention_train_tc_fwd", qkv.data_ptr(), o.data_ptr(), lse.data_ptr(), seed.data_ptr(), salt, p, B, S,
           C, heads, None)
    assert torch.equal(o, out)
    d1, d2 = torch.full_like(qkv, float("nan")), torch.full_like(qkv, float("nan"))
    for dq in (d1, d2):
        L.call("flowk_attention_train_tc_bwd", 3, qkv.data_ptr(), o.data_ptr(), dout.data_ptr(), lse.data_ptr(),
               dq.data_ptr(), seed.data_ptr(), salt, p, B, S, C, heads, None)
    torch.cuda.synchronize()
    assert torch.isfinite(d1).all() and torch.equal(d1, d2) and torch.equal(d1, grad)
    mask = tc_autograd.attention_dropout_mask(dev, salt, p, B * heads, S)
    keep = float((mask > 0).double().mean())
    assert abs(keep - (1 - p)) < 0.02
    tc_autograd.advance_dropout_seed(dev)
    out3, _ = _run(qkv, dout, heads, p, salt)
    assert not torch.equal(out3, out)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the width-256 MixLogCDF model
# ---------------------------------------------------------------------------------------------------------------------
def _model(B, L, K, hidden, seed, **kw):
    from flowk.marscf import MarScfFlow
    dev = torch.device("cuda:0")
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = MarScfFlow(B, (32, 32, 3), "mixlogcdf", L, K, hidden, **kw).to(dev)
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(B, 3, 32, 32, generator=gen) - 0.5
    noise = torch.rand(B, 3, 32, 32, generator=gen)
    model.train()
    with torch.no_grad():
        model(x.to(dev), noise=noise.to(dev))                 # ActNorm data-dependent init
        for prm in model.parameters():                        # move the zero-initialised output convs off zero
            prm.add_((torch.randn(prm.shape, generator=gen) * 0.005).to(prm.device))
    return model, x, noise


@pytest.mark.gpu
def test_width256_training_gradients_vs_oracle(no_library):
    """A width-256 training step (16x16 / 8x8 / 4x4, 2 ConvAttnBlocks, dropout p = 0) against fp64 autograd through the
    oracle for every parameter; the attention of all three levels runs forward and backward on flowk kernels."""
    L = _lib()
    dev = torch.device("cuda:0")
    Lv, K, hidden, B = 3, 1, 256, 8
    model, x, noise = _model(B, Lv, K, hidden, 83, num_blocks=2, drop_prob=0.0)
    sd64 = {k: v.detach().cpu().double().requires_grad_(v.dtype.is_floating_point and "is_initialized" not in k and
                                                         not k.endswith(".p") and not k.endswith("sign_s"))
            for k, v in model.state_dict().items()}
    _, _, _, nll = O.normal_flow(sd64, x.double(), noise.double(), Lv, K, "mixlogcdf")
    nll.mean().backward()
    model.train()
    L.TIMING = {}
    try:
        _, nll_d, _ = model(x.to(dev), noise=noise.to(dev))
        nll_d.mean().backward()
        torch.cuda.synchronize()
        timing = dict(L.TIMING)
    finally:
        L.TIMING = None
    assert len(timing.get("flowk_attention_train_tc_fwd", [])) > 0      # level 1 (256 tokens)
    assert len(timing.get("flowk_attention_train_tc_bwd", [])) > 0
    assert len(timing.get("flowk_attention_train_fwd", [])) > 0         # levels 2 and 3 (64 and 16 tokens)
    assert len(timing.get("flowk_attention_train_bwd", [])) > 0
    assert float((nll_d.detach().cpu() - nll.detach().float()).abs().max()) < 1e-3
    checked = 0
    for name, prm in model.named_parameters():
        ref = sd64[name].grad
        if ref is None:
            continue
        if name.endswith(".l") or name.endswith(".u"):
            c = ref.shape[0]
            ref = ref * (torch.tril(torch.ones(c, c), -1) if name.endswith(".l") else torch.triu(torch.ones(c, c), 1))
        ref = ref.float()
        got = prm.grad.detach().float().cpu()
        err = float((got - ref).abs().max())
        assert err <= 1e-3 * max(1.0, float(ref.abs().max())), (name, err)
        checked += 1
    assert checked > 100


@pytest.mark.gpu
def test_width256_graphed_step_with_dropout_matches_eager(no_library):
    from flowk import sharding

    class FixedNoise(torch.nn.Module):
        def __init__(self, m, noise):
            super().__init__()
            self.m, self.noise = m, noise

        def forward(self, x):
            return self.m(x, noise=self.noise)

    dev = torch.device("cuda:0")
    B = 8
    base, x, noise = _model(B, 3, 1, 256, 12, num_blocks=1, drop_prob=0.2)
    for m in base.modules():                  # feature dropout draws from torch's RNG: off, the attention dropout stays on
        if isinstance(m, torch.nn.Dropout2d):
            m.p = 0.0
    x, noise = x.to(dev), noise.to(dev)
    results = []
    for use_graph in (False, True):
        from flowk import tc_autograd
        tc_autograd.dropout_seed(dev).fill_(1234)          # both runs draw the same attention masks
        model = FixedNoise(copy.deepcopy(base), noise)
        trainer = sharding.ShardedTrainer(model, lr=1e-4, warm_up=40, global_batch=B, use_graph=use_graph, graph_after=2)
        losses = [float(trainer.step(x)) for _ in range(5)]
        results.append((losses, [prm.detach().clone() for prm in model.parameters()]))
    (l0, p0), (l1, p1) = results
    assert all(math.isfinite(v) for v in l0)
    for a, b in zip(l0, l1):
        assert abs(a - b) < 1e-4 * max(1.0, abs(a)), (l0, l1)
    for a, b in zip(p0, p1):
        assert float((a - b).abs().max()) <= 1e-4 * max(1.0, float(a.abs().max()))


@pytest.mark.gpu
def test_width256_fit_end_to_end(tmp_path, no_library):
    from flowk import driver
    from flowk.marscf import MarScfFlow
    dev = torch.device("cuda:0")
    torch.manual_seed(4)
    np.random.seed(4)
    model = MarScfFlow(8, (32, 32, 3), "mixlogcdf", 3, 1, 256, num_blocks=1, drop_prob=0.2).to(dev)
    g = torch.Generator().manual_seed(6)
    train = [(torch.rand(8, 3, 32, 32, generator=g) - 0.5, None) for _ in range(3)]
    test = [(torch.rand(8, 3, 32, 32, generator=g) - 0.5, None) for _ in range(2)]
    path = os.path.join(tmp_path, "best.pt")
    hist = driver.fit(model, train, test, epochs=2, checkpoint_path=path, lr=1e-4, warm_up=16, device=dev, use_graph=False)
    assert all(math.isfinite(h["train_nll"]) and math.isfinite(h["test_nll"]) for h in hist)
    assert os.path.exists(path)
