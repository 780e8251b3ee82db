"""Training of `Transformer_attn` on the flowk kernels (csrc/patch_attention.cu: flowk_patch_attention_train_fwd +
flowk_patch_attention_bwd, wrapped as `flowk::patch_attention`): argument validation without a GPU, then on the GPU every
gradient against float64 autograd of the torch-op form of the same layer, bit-exact forward and determinism, the whole
attention model against the float64 oracle, and the CUDA-graph training step."""
import copy
import ctypes

import pytest
import torch

import flowk  # noqa: F401  (registers the package alias)
from flowk import _lib
from flowk.flow_modules import transformer
from flowk.flow_modules.transformer import Transformer_attn
from oracle import flow_oracle as O

PARAMS = ("convq1", "convk1", "convq2", "convk2", "convq3", "convk3", "offset", "offset2", "offset3", "scale")


def close(got, ref, rel, what):
    ref = ref.detach().double().cpu()
    got = got.detach().double().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    scale = max(1.0, float(ref.abs().max()))
    err = float((got - ref).abs().max())
    assert err <= rel * scale, "%s: max abs err %.3e > %.1e * %.3g" % (what, err, rel, scale)


def test_train_entry_points_validate_without_gpu():
    L = _lib.lib
    one = ctypes.c_void_p(16)       # never dereferenced: validation fails first
    fwd, bwd = L.flowk_patch_attention_train_fwd, L.flowk_patch_attention_bwd
    assert fwd(one, one, one, one, None, None, None, 2, 12, 16, 16, 0, None) == _lib.FLOWK_ERR_ARG       # scores
    assert fwd(None, one, one, one, None, None, one, 2, 12, 16, 16, 0, None) == _lib.FLOWK_ERR_ARG
    assert fwd(one, one, one, one, None, None, one, 2, 12, 16, 8, 0, None) == _lib.FLOWK_ERR_SHAPE       # H != W
    assert fwd(one, one, one, one, None, None, one, 2, 12, 7, 7, 0, None) == _lib.FLOWK_ERR_SHAPE        # odd side
    assert fwd(one, one, one, one, None, None, one, 2, 64, 32, 32, 0, None) == _lib.FLOWK_ERR_SHAPE      # > 200 KB
    assert fwd(None, None, None, None, None, None, None, 0, 12, 16, 16, 0, None) == _lib.FLOWK_OK
    args = [one] * 8
    for k in range(8):                                                                                # every pointer
        a = list(args)
        a[k] = None
        assert bwd(*a, 2, 12, 16, 16, 1, None) == _lib.FLOWK_ERR_ARG, k
    assert bwd(*args, -1, 12, 16, 16, 0, None) == _lib.FLOWK_ERR_SHAPE
    assert bwd(*args, 2, 0, 16, 16, 0, None) == _lib.FLOWK_ERR_SHAPE
    assert bwd(*args, 2, 12, 5, 5, 0, None) == _lib.FLOWK_ERR_SHAPE
    # (16, 36, 36) fits the forward's two copies of the sample but not the backward's three
    assert bwd(*args, 2, 16, 36, 36, 0, None) == _lib.FLOWK_ERR_SHAPE
    assert transformer._fits(16, 36, 36, 2) and not transformer._fits(16, 36, 36, 3)
    assert transformer._fits(12, 32, 32, 3) and transformer._fits(96, 4, 4, 3)
    assert bwd(None, None, None, None, None, None, None, None, 0, 12, 16, 16, 0, None) == _lib.FLOWK_OK


def test_cpu_training_keeps_torch_ops():
    """CPU tensors never reach the CUDA-only op: the torch-op form trains as before."""
    torch.manual_seed(0)
    m = Transformer_attn(12)
    x = torch.randn(2, 12, 8, 8, requires_grad=True)
    y, ld = m(x, logdet=torch.zeros(2))
    (y.square().sum() + ld.sum()).backward()
    assert x.grad is not None and m.convq1.grad is not None


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def _layer(C, seed, dev):
    torch.manual_seed(seed)
    m = Transformer_attn(C).to(dev)
    with torch.no_grad():
        m.scale.fill_(4.0 + seed % 4)                          # 4..7: the scores move the attention matrices visibly
    return m


def _grads(m, x, ld0, gy, gl, permute):
    """(gradients of x, ldj_in and every parameter) of <y, gy> + <ldj_out, gl>."""
    x = x.clone().requires_grad_()
    ld0 = ld0.clone().requires_grad_()
    m.zero_grad(set_to_none=True)
    y, ld = m(x, logdet=ld0, permute=permute)
    torch.autograd.backward([y, ld], [gy, gl])
    return [x.grad, ld0.grad] + [getattr(m, n).grad for n in PARAMS]


@pytest.mark.gpu
@pytest.mark.parametrize("permute", [False, True])
@pytest.mark.parametrize("C,H,B", [(12, 16, 64), (24, 8, 64), (48, 4, 64), (12, 32, 5), (96, 4, 3)])
def test_layer_gradients_vs_fp64(C, H, B, permute):
    dev = torch.device("cuda:0")
    m = _layer(C, C + H, dev)
    gen = torch.Generator().manual_seed(C * H + B)
    x = torch.randn(B, C, H, H, generator=gen).to(dev)
    ld0 = torch.randn(B, generator=gen).to(dev)
    gy = torch.randn(B, C, H, H, generator=gen).to(dev)
    gl = (0.05 * torch.randn(B, generator=gen)).to(dev)
    _lib.TIMING = {}
    try:
        got = _grads(m, x, ld0, gy, gl, permute)
        torch.cuda.synchronize()
        names = set(_lib.TIMING)
    finally:
        _lib.TIMING = None
    assert {"flowk_patch_attention_train_fwd", "flowk_patch_attention_bwd", "flowk_channel_sum"} <= names, names
    m64 = copy.deepcopy(m).double()                               # fp64 takes the torch-op form
    ref = _grads(m64, x.double(), ld0.double(), gy.double(), gl.double(), permute)
    for what, a, r in zip(("x", "ldj_in") + PARAMS, got, ref):
        close(a, r, 1e-3, "grad %s (C=%d H=%d B=%d permute=%s)" % (what, C, H, B, permute))


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,B", [(12, 16, 64), (48, 4, 64), (12, 32, 5)])
def test_training_forward_is_the_inference_kernel(C, H, B):
    """The training route's forward (flowk_patch_attention_train_fwd) gives the inference kernel's y and ldj bit for bit."""
    dev = torch.device("cuda:0")
    m = _layer(C, C + H + 1, dev)
    x = torch.randn(B, C, H, H, device=dev)
    ld0 = torch.randn(B, device=dev)
    for permute in (False, True):
        with torch.no_grad():
            y0, l0 = m(x, logdet=ld0, permute=permute)
        _lib.TIMING = {}
        try:
            y1, l1 = m(x.clone().requires_grad_(), logdet=ld0, permute=permute)
            torch.cuda.synchronize()
            assert "flowk_patch_attention_train_fwd" in _lib.TIMING
        finally:
            _lib.TIMING = None
        assert torch.equal(y0, y1.detach()) and torch.equal(l0, l1.detach())


@pytest.mark.gpu
def test_backward_is_deterministic():
    dev = torch.device("cuda:0")
    for C, H, B in ((12, 16, 64), (96, 4, 3)):
        m = _layer(C, 5, dev)
        x = torch.randn(B, C, H, H, device=dev)
        ld0 = torch.randn(B, device=dev)
        gy = torch.randn_like(x)
        gl = torch.randn(B, device=dev)
        a = _grads(m, x, ld0, gy, gl, True)
        b = _grads(m, x, ld0, gy, gl, True)
        for t, u in zip(a, b):
            assert torch.equal(t, u)


@pytest.mark.gpu
def test_kernel_training_switch_selects_torch_ops():
    """KERNEL_TRAINING = False trains the fp32 layer on the torch-op form (no flowk launch); both routes agree."""
    dev = torch.device("cuda:0")
    m = _layer(24, 9, dev)
    x = torch.randn(8, 24, 8, 8, device=dev)
    ld0 = torch.randn(8, device=dev)
    gy, gl = torch.randn_like(x), 0.05 * torch.randn(8, device=dev)
    got = _grads(m, x, ld0, gy, gl, False)
    transformer.KERNEL_TRAINING = False
    _lib.TIMING = {}
    try:
        ref = _grads(m, x, ld0, gy, gl, False)
        torch.cuda.synchronize()
        assert not any(k.startswith("flowk_patch_attention") for k in _lib.TIMING)
    finally:
        _lib.TIMING = None
        transformer.KERNEL_TRAINING = True
    for what, a, r in zip(("x", "ldj_in") + PARAMS, got, ref):
        close(a, r, 1e-3, "grad " + what)


def _initialised_model(coupling, hidden, B, seed, dev, **kw):
    """As tests/test_gpu_parity.py builds its models (ActNorm data init, every parameter moved off its init), then the
    attention scales set to 4 so that the scores matter."""
    import numpy as np
    from flowk.marscf import MarScfFlow
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = MarScfFlow(B, (32, 32, 3), coupling, 3, 1, hidden, attn=True, **kw).to(dev)
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(B, 3, 32, 32, generator=gen) - 0.5
    noise = torch.rand(B, 3, 32, 32, generator=gen)
    model.train()
    with torch.no_grad():
        model(x.to(dev), noise=noise.to(dev))
        for name, p in model.named_parameters():
            p.add_((torch.randn(p.shape, generator=gen) * 0.02).to(p.device))
            if name.endswith(".scale"):
                p.fill_(4.0)
    return model, x, noise


@pytest.mark.gpu
@pytest.mark.parametrize("coupling,hidden,kw", [("mixlogcdf", 96, {"num_blocks": 2, "drop_prob": 0.0}), ("affine", 32, {})])
def test_model_with_attn_training_gradients_vs_oracle(no_library, coupling, hidden, kw):
    """cfg2-shaped model with both attention layers in every FlowStep (levels 16x16x12, 8x8x24, 4x4x48): every parameter
    gradient of the training step against float64 autograd through the oracle, with no library layer anywhere."""
    dev = torch.device("cuda:0")
    model, x, noise = _initialised_model(coupling, hidden, 8, 91, dev, **kw)
    sd64 = {k: v.detach().cpu().double().requires_grad_(v.dtype.is_floating_point and "is_initialized" not in k and
                                                         not k.endswith(".p") and not k.endswith("sign_s"))
            for k, v in model.state_dict().items()}
    _, _, _, nll = O.normal_flow(sd64, x.double(), noise.double(), 3, 1, coupling, attn=True)
    nll.mean().backward()
    _lib.TIMING = {}
    try:
        _, nll_d, _ = model(x.to(dev), noise=noise.to(dev))
        nll_d.mean().backward()
        torch.cuda.synchronize()
        calls = len(_lib.TIMING.get("flowk_patch_attention_bwd", ()))
    finally:
        _lib.TIMING = None
    assert calls == 6, calls                                       # 3 FlowSteps x 2 attention layers
    assert float((nll_d.detach().cpu() - nll.float()).abs().max()) < 1e-3
    checked = 0
    for name, p in model.named_parameters():
        ref = sd64[name].grad
        if ref is None:
            continue
        if name.endswith(".l") or name.endswith(".u"):
            c = ref.shape[0]
            ref = ref * (torch.tril(torch.ones(c, c), -1) if name.endswith(".l") else torch.triu(torch.ones(c, c), 1))
        close(p.grad, ref, 1e-3, "grad " + name)
        checked += 1
    assert checked > 60


@pytest.mark.gpu
def test_graphed_training_step_with_attn_matches_eager():
    """ShardedTrainer replaying forward + backward and the update as CUDA graphs == the eager step, attention layers on."""
    import numpy as np
    from flowk import sharding
    from flowk.marscf import MarScfFlow
    dev = torch.device("cuda:0")

    class FixedNoise(torch.nn.Module):
        def __init__(self, m, noise):
            super().__init__()
            self.m, self.noise = m, noise

        def forward(self, x):
            return self.m(x, noise=self.noise)

    torch.manual_seed(11)
    np.random.seed(11)
    B = 8
    base = MarScfFlow(B, (16, 16, 3), "affine", 2, 2, 32, attn=True).to(dev)
    x = torch.rand(B, 3, 16, 16, device=dev) - 0.5
    noise = torch.rand_like(x)
    base.train()
    with torch.no_grad():
        base(x, noise=noise)
        for name, p in base.named_parameters():
            p.add_(torch.randn_like(p) * 0.02)
            if name.endswith(".scale"):
                p.fill_(4.0)
    results = []
    for use_graph in (False, True):
        model = FixedNoise(copy.deepcopy(base), noise)
        trainer = sharding.ShardedTrainer(model, lr=1e-3, warm_up=40, global_batch=B, use_graph=use_graph, graph_after=2)
        losses = [float(trainer.step(x)) for _ in range(5)]
        results.append((losses, [p.detach().clone() for p in model.parameters()]))
    (l0, p0), (l1, p1) = results
    assert l0[-1] < l0[0]
    for a, b in zip(l0, l1):
        assert abs(a - b) < 1e-4 * max(1.0, abs(a)), (l0, l1)
    for a, b in zip(p0, p1):
        close(b, a, 1e-4, "parameters after 5 steps")
