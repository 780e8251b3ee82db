"""Training the mAR channel prior on flowk kernels: the NHWC weight-gradient kernel (5x5 / dilated taps), the ConvLSTM cell
backward, autograd over one prior level against float64 on the CPU, the full model against the torch-layer route, and the
graphed training step against eager execution."""
import copy
import ctypes

import numpy as np
import pytest
import torch

from flowk import _lib
from flowk.mar_prior import ChannelPriorUniScale, cuda_path


def close(got, ref, rel, what):
    ref = ref.detach().double().cpu()
    got = got.detach().double().cpu()
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    scale = max(1.0, float(ref.abs().max()))
    err = float((got - ref).abs().max())
    assert err <= rel * scale, "%s: max abs err %.3e > %.1e * %.3g" % (what, err, rel, scale)
    return err / scale


def test_new_entry_points_validate_without_gpu():
    splits = _lib.lib.flowk_conv_wgrad_nhwc_splits
    t = ctypes.c_int(0)
    for args in ((48, 16, 16, 32, 128, 25, 2), (96, 8, 8, 32, 32, 25, 1), (3072, 4, 4, 32, 128, 9, 1), (8, 16, 16, 32, 32, 1, 1)):
        assert splits(*args, ctypes.byref(t)) > 0, args
    for bad in ((48, 16, 16, 5, 128, 25, 2),          # channels not whole 32-blocks
                (48, 16, 16, 32, 130, 25, 2),
                (3, 4, 4, 32, 128, 9, 1),             # 4x4 maps: a 32-pixel k-block spans two images
                (48, 16, 16, 32, 128, 16, 1),         # taps
                (48, 16, 16, 32, 128, 25, 0),         # dilation
                (48, 12, 12, 32, 128, 9, 1)):         # 12 columns do not tile 32
        assert splits(*bad, None) == 0, bad
    assert _lib.lib.flowk_conv_wgrad_nhwc(None, None, None, None, 48, 16, 16, 32, 128, 25, 2, None) == _lib.FLOWK_ERR_ARG
    assert _lib.lib.flowk_conv_wgrad_nhwc(None, None, None, None, 3, 4, 4, 32, 128, 9, 1, None) == _lib.FLOWK_ERR_SHAPE
    assert _lib.lib.flowk_lstm_cell_bwd(*([None] * 11), 64, 32, None) == _lib.FLOWK_ERR_ARG
    assert _lib.lib.flowk_lstm_cell_bwd(*([None] * 11), 0, 32, None) == _lib.FLOWK_OK
    assert _lib.lib.flowk_f16_pair_to_f32(None, None, None, 64, 8, 4, None) == _lib.FLOWK_ERR_SHAPE
    assert _lib.lib.flowk_f16_pair_to_f32(None, None, None, 64, 8, 32, None) == _lib.FLOWK_ERR_ARG


def test_cpu_and_no_grad_do_not_take_the_training_path():
    prior = ChannelPriorUniScale(2, 3, 32, 32, 1, 3, hidden_size=32, num_layers=1, dp_rate=0)
    z = torch.randn(2, 6, 16, 16)
    assert not cuda_path.trainable(prior, z)                  # CPU tensors: torch layers
    z1 = torch.randn(2, 6, 16, 16, requires_grad=True)
    ll = prior((z1, z)).sum()
    ll.backward()
    assert z1.grad is not None and prior.prior_lstm.lstm.weight_hh_l0.grad is not None


# (taps, dilation, H, Cin, N, T): every weight gradient of the cfg2 prior (3x32x32, hidden 32): conv_embed (input padded to
# 32 channels), W_ih / W_hh, conv_out1 (N padded 2 -> 32) and z1_cond_network (T = 1: its maps are not repeated over time)
WGRAD_SHAPES = [
    (25, 1, 16, 32, 32, 6), (25, 2, 16, 32, 128, 6), (9, 1, 16, 32, 32, 6), (25, 1, 16, 32, 32, 1),
    (25, 1, 8, 32, 32, 12), (25, 1, 8, 32, 128, 12), (9, 1, 8, 32, 32, 12), (25, 1, 8, 32, 32, 1),
    (9, 1, 4, 32, 32, 48), (9, 1, 4, 32, 128, 48),
]


@pytest.mark.gpu
@pytest.mark.parametrize("taps,dil,H,cin,n,T", WGRAD_SHAPES)
def test_conv_wgrad_nhwc_matches_fp64(taps, dil, H, cin, n, T):
    dev = torch.device("cuda:0")
    B = 8
    NB, k = T * B, int(round(taps ** 0.5))
    gen = torch.Generator().manual_seed(taps * 1000 + dil * 100 + H + n + T)
    x = torch.randn(NB, cin, H, H, generator=gen, dtype=torch.float64)
    gy = torch.randn(NB, n, H, H, generator=gen, dtype=torch.float64)
    ref = torch.nn.grad.conv2d_weight(x, (n, cin, k, k), gy, padding=dil * (k - 1) // 2, dilation=dil)
    x_rows = x.permute(0, 2, 3, 1).reshape(-1, cin).float().contiguous().to(dev)
    g_rows = gy.permute(0, 2, 3, 1).reshape(-1, n).float().contiguous().to(dev)
    got = cuda_path.wgrad(x_rows, g_rows, NB, H, H, taps, dil)
    rel = float((got.double().cpu() - ref).abs().max() / ref.abs().max())
    print("taps %d dil %d %dx%d Cin %d N %d images %d: rel err %.2e" % (taps, dil, H, H, cin, n, NB, rel))
    assert rel < 2e-5, rel
    # repeated calls give identical split-K partials (no atomics)
    transposed = ctypes.c_int(0)
    s = _lib.lib.flowk_conv_wgrad_nhwc_splits(NB, H, H, cin, n, taps, dil, ctypes.byref(transposed))
    parts = []
    for _ in range(2):
        p = torch.full((s, taps, n, cin), float("nan"), device=dev)
        _lib.call("flowk_conv_wgrad_nhwc", x_rows.data_ptr(), g_rows.data_ptr(), p.data_ptr(), None, NB, H, H, cin, n,
                  taps, dil, torch.cuda.current_stream().cuda_stream)
        parts.append(p)
    torch.cuda.synchronize()
    assert torch.equal(parts[0], parts[1])


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 20.0])
def test_lstm_cell_backward_matches_fp64(scale):
    """flowk_lstm_cell_bwd against float64 autograd of the cell in mar_prior/lstm.py, with random and saturated gates."""
    dev = torch.device("cuda:0")
    M, hid = 1000, 32
    gen = torch.Generator().manual_seed(int(scale))
    gi = (torch.randn(M, 4 * hid, generator=gen, dtype=torch.float64) * scale).float()
    hh = torch.randn(M, 4 * hid, generator=gen, dtype=torch.float64).float()
    c_prev = (torch.randn(M, hid, generator=gen, dtype=torch.float64) * 2).float()
    dh = torch.randn(M, hid, generator=gen, dtype=torch.float64).float()
    dh_rec = torch.randn(M, hid, generator=gen, dtype=torch.float64).float()
    dc_next = torch.randn(M, hid, generator=gen, dtype=torch.float64).float()
    a = (gi.double() + hh.double()).requires_grad_(True)
    cp = c_prev.double().requires_grad_(True)
    i, f, g, o = a.chunk(4, 1)
    c = torch.sigmoid(f) * cp + torch.sigmoid(i) * torch.tanh(g)
    h = torch.sigmoid(o) * torch.tanh(c)
    ((dh.double() + dh_rec.double()) * h + dc_next.double() * c).sum().backward()
    d = {k: v.to(dev) for k, v in dict(gi=gi, hh=hh, c_prev=c_prev, dh=dh, dh_rec=dh_rec).items()}
    dc = dc_next.to(dev)
    dgates = torch.empty(M, 4 * hid, device=dev)
    dg_hi, dg_lo = torch.empty_like(dgates), torch.empty_like(dgates)
    cuda_path.cell_backward(d["gi"], d["hh"], d["c_prev"], c.detach().float().to(dev), d["dh"], d["dh_rec"], dc, dgates,
                            dg_hi, dg_lo)
    torch.cuda.synchronize()
    close(dgates, a.grad, 1e-5, "dgates")
    close(dc, cp.grad, 1e-5, "dc_prev")
    assert torch.equal(dg_hi.view(torch.int32) & 0x1FFF, torch.zeros_like(dg_hi, dtype=torch.int32))     # TF32 containers
    close(dg_hi.double() + dg_lo.double(), dgates.double(), 1e-6, "hi + lo")


def _level(level, B, dev):
    torch.manual_seed(100 + level)
    prior = ChannelPriorUniScale(B, 3, 32, 32, level, 3, hidden_size=32, num_layers=3, dp_rate=0)
    gen = torch.Generator().manual_seed(level)
    with torch.no_grad():
        for p in prior.parameters():                              # move the zero-mean init to something less symmetric
            p.add_(torch.randn(p.shape, generator=gen) * 0.02)
    z2 = torch.randn(B, prior.nc, prior.height, prior.width, generator=gen)
    z1 = torch.randn(B, prior.nc, prior.height, prior.width, generator=gen) if level < 3 else None
    return prior, z1, z2


def _ll(prior, z1, z2):
    return prior((z1, z2) if z1 is not None else z2)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [8, 64])
@pytest.mark.parametrize("level", [1, 2, 3])
def test_level_gradients_match_fp64(no_library, level, B):
    dev = torch.device("cuda:0")
    prior, z1, z2 = _level(level, B, dev)
    ref = copy.deepcopy(prior).double()
    r1 = None if z1 is None else z1.double().requires_grad_(True)
    r2 = z2.double().requires_grad_(True)
    old = cuda_path.ENABLED
    cuda_path.ENABLED = False
    try:
        ll_ref = _ll(ref, r1, r2)
        ll_ref.sum().backward()
    finally:
        cuda_path.ENABLED = old
    prior = prior.to(dev)
    g1 = None if z1 is None else z1.to(dev).requires_grad_(True)
    g2 = z2.to(dev).requires_grad_(True)
    assert cuda_path.trainable(prior, g2)
    _lib.TIMING = {}
    try:
        ll = _ll(prior, g1, g2)
        ll.sum().backward()
        torch.cuda.synchronize()
        names = set(_lib.TIMING)
    finally:
        _lib.TIMING = None
    assert {"flowk_conv_wgrad_nhwc", "flowk_lstm_cell_bwd", "flowk_f16_pair_to_f32"} <= names, names
    with torch.no_grad():
        ll_eval = _ll(prior, None if g1 is None else g1.detach(), g2.detach())
    scale = max(1.0, float(ll_eval.abs().max()))
    assert float((ll.detach() - ll_eval).abs().max()) <= 1e-4 * scale
    close(ll, ll_ref, 1e-4, "ll")
    worst = close(g2.grad, r2.grad, 1e-3, "z2")
    if g1 is not None:
        worst = max(worst, close(g1.grad, r1.grad, 1e-3, "z1"))
    for (name, p), (_, q) in zip(prior.named_parameters(), ref.named_parameters()):
        if q.grad is None:                                        # the last level has no z1 (z1_cond_network unused)
            assert p.grad is None and level == 3 and name.startswith("z1_cond_network"), name
            continue
        worst = max(worst, close(p.grad, q.grad, 1e-3, name))
    print("level %d B %d: worst gradient error %.2e (of max(1, max|ref|))" % (level, B, worst))


@pytest.mark.gpu
def test_no_library_convolution_in_prior_training():
    dev = torch.device("cuda:0")
    prior, z1, z2 = _level(1, 8, dev)
    prior = prior.to(dev)
    z1, z2 = z1.to(dev).requires_grad_(True), z2.to(dev).requires_grad_(True)
    _ll(prior, z1, z2).sum().backward()                         # warm-up (module loads)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        _ll(prior, z1, z2).sum().backward()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    bad = [n for n in names if "cudnn" in n.lower() or "aten::conv" in n or "aten::_conv" in n or "aten::cudnn" in n
           or "xmma" in n.lower() or "implicit_convolve" in n.lower()]
    assert not bad, sorted(set(bad))[:10]
    assert any("conv_wgrad_kernel" in n for n in names) and any("lstm_cell_bwd_kernel" in n for n in names)


def _model(dev, B=8):
    from flowk.marscf import MarScfFlow
    torch.manual_seed(5)
    np.random.seed(5)
    model = MarScfFlow(B, (32, 32, 3), "mixlogcdf", 3, 1, 96, prior="mar", num_blocks=2, drop_prob=0).to(dev)
    gen = torch.Generator().manual_seed(6)
    x = torch.rand(B, 3, 32, 32, generator=gen) - 0.5
    noise = torch.rand(B, 3, 32, 32, generator=gen)
    model.train()
    with torch.no_grad():
        model(x.to(dev), noise=noise.to(dev))
        for p in model.parameters():
            p.add_((torch.randn(p.shape, generator=gen) * 0.02).to(dev))
    return model, x.to(dev), noise.to(dev)


@pytest.mark.gpu
def test_full_model_gradients_match_torch_layer_route(no_library):
    dev = torch.device("cuda:0")
    model, x, noise = _model(dev)
    ref = copy.deepcopy(model)
    old, old_tf32 = cuda_path.ENABLED, torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    cuda_path.ENABLED = False
    try:
        _, nll_ref, _ = ref(x, noise=noise)
        nll_ref.mean().backward()
    finally:
        cuda_path.ENABLED = old
        torch.backends.cudnn.allow_tf32 = old_tf32
    _lib.TIMING = {}
    try:
        _, nll, _ = model(x, noise=noise)
        nll.mean().backward()
        torch.cuda.synchronize()
        calls = len(_lib.TIMING.get("flowk_lstm_cell_bwd", ()))
    finally:
        _lib.TIMING = None
    assert calls == 3 * (6 + 12 + 48), calls                   # 3 layers x T per level
    close(nll, nll_ref, 1e-4, "nll")
    checked = set()
    for (name, p), (_, q) in zip(model.named_parameters(), ref.named_parameters()):
        if q.grad is None:
            assert p.grad is None, name
            continue
        close(p.grad, q.grad, 1e-3, "grad " + name)
        checked.add(name)
    # per level conv_embed 2 + 3 LSTM layers x 4 + conv_out1 2, and z1_cond_network 4 at the two split levels
    assert len([n for n in checked if "c_prior" in n]) == 3 * (2 + 12 + 2) + 2 * 4


@pytest.mark.gpu
def test_graphed_training_step_matches_eager():
    """ShardedTrainer's graphed step == eager steps, and after two updates the graph's gradients equal an eager backward
    with the updated weights (the prior's weight operands are rebuilt inside the graph, never cached)."""
    from flowk import sharding
    dev = torch.device("cuda:0")
    base, x, noise = _model(dev)

    class FixedNoise(torch.nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m = m

        def forward(self, xx):
            return self.m(xx, noise=noise)

    results = []
    for use_graph in (False, True):
        model = FixedNoise(copy.deepcopy(base))
        trainer = sharding.ShardedTrainer(model, lr=1e-3, warm_up=1, global_batch=8, use_graph=use_graph, graph_after=1)
        losses = [float(trainer.step(x)) for _ in range(4)]
        results.append((losses, [p.detach().clone() for p in model.parameters()], model, trainer))
    (l0, p0, _, _), (l1, p1, gm, gt) = results
    for a, b in zip(l0, l1):
        assert abs(a - b) < 1e-4 * max(1.0, abs(a)), (l0, l1)
    for a, b in zip(p0, p1):
        close(b, a, 1e-4, "parameters after 4 steps")
    # stale-operand check: the last replay's gradients against an eager backward at the weights that replay saw
    fb, up, static_x, _ = gt._graphs
    fb.replay()
    torch.cuda.synchronize()
    graphed = [None if p.grad is None else p.grad.detach().clone() for p in gm.parameters()]
    eager = FixedNoise(copy.deepcopy(base))
    eager.load_state_dict(gm.state_dict())
    _, nll, _ = eager(static_x)
    nll.mean().backward()
    n = 0
    for (name, p), g in zip(eager.named_parameters(), graphed):
        if p.grad is None:
            continue
        close(g, p.grad, 1e-4, "graphed grad " + name)
        n += "prior" in name
    assert n > 0
