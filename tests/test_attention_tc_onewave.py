"""The one-wave tcgen05 attention kernel (csrc/attention_tc.cu, attention_tc_v2_kernel): two CTAs per SM, key blocks of 128
with per-block softmax statistics, P in tensor memory.  Checked against fp64 attention, against the one-CTA-per-SM kernel,
for determinism, occupancy, routing and CUDA-graph capture."""
import ctypes

import pytest
import torch


@pytest.fixture(scope="module")
def tc():
    import flowk  # noqa: F401
    from flowk import tc as mod
    return mod


def rel_err(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def qkv_for(B, HW, C, seed, scale=1.5):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(B * HW, 3 * C, generator=g) * scale).to("cuda:0")


def reference(qkv, B, HW, C, heads):
    d = C // heads
    t = qkv.double().view(B, HW, 3, heads, d)
    k, v, q = (t[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    return (torch.softmax((q * d ** -0.5) @ k.transpose(-1, -2), dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * HW, C)


def run(tc, route, qkv, B, HW, C, heads, f16):
    """route: "v2" (one-wave kernel), "v1" (one CTA per SM) - through tc.attention with the module flags."""
    saved = tc.ATTENTION_TC_V2
    tc.ATTENTION_TC_V2 = route == "v2"
    try:
        status = torch.zeros(1, dtype=torch.int32, device=qkv.device)
        hi, lo = tc.attention(qkv, B, HW, C, heads, f16, status=status)
        torch.cuda.synchronize()
    finally:
        tc.ATTENTION_TC_V2 = saved
    assert int(status) == 0, "barrier wait timed out inside the kernel"
    return hi, lo


def test_support_predicate_needs_no_gpu():
    import flowk  # noqa: F401
    from flowk import tc
    saved = tc.ATTENTION_TC_V2
    try:
        tc.ATTENTION_TC_V2 = True
        assert tc.attention_tc_v2_supported(256, 96, 4)          # cfg2 level 1
        assert tc.attention_tc_v2_supported(128, 128, 4)
        assert not tc.attention_tc_v2_supported(256, 160, 4)     # cfg4 level 1 (d = 40): one-CTA-per-SM kernel
        assert not tc.attention_tc_v2_supported(64, 96, 4)       # levels 2, 3: mma.sync kernel
        assert not tc.attention_tc_v2_supported(256, 32, 4)      # d = 8
        assert not tc.attention_tc_v2_supported(256, 100, 4)
        tc.ATTENTION_TC_V2 = False
        assert not tc.attention_tc_v2_supported(256, 96, 4)
    finally:
        tc.ATTENTION_TC_V2 = saved


def test_entry_points_validate_without_gpu():
    import flowk  # noqa: F401
    from flowk import _lib
    L = _lib.lib
    one = ctypes.c_void_p(16)
    n = ctypes.c_int(-1)
    assert L.flowk_attention_tc_v2(one, one, one, 1, 2, 256, 160, 4, None, None, None) == _lib.FLOWK_ERR_SHAPE
    assert L.flowk_attention_tc_v2(one, one, one, 1, 2, 64, 96, 4, None, None, None) == _lib.FLOWK_ERR_SHAPE
    assert L.flowk_attention_tc_v2(None, one, one, 1, 2, 256, 96, 4, None, None, None) == _lib.FLOWK_ERR_ARG
    assert L.flowk_attention_tc_v2(None, None, None, 1, 0, 256, 96, 4, None, None, None) == _lib.FLOWK_OK
    assert L.flowk_attention_tc_v2_occupancy(256, 160, 4, ctypes.byref(n), None) == _lib.FLOWK_ERR_SHAPE


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["tf32", "f16"])
@pytest.mark.parametrize("B,HW,C,heads", [(64, 256, 96, 4), (3, 128, 96, 4), (5, 256, 128, 4), (7, 128, 32, 1),
                                          (1, 256, 24, 1), (149, 256, 96, 4), (75, 256, 96, 4), (37, 128, 64, 2)])
def test_onewave_matches_fp64_and_one_cta_kernel(tc, fmt, B, HW, C, heads):
    """seq 128 / 256, head dims 24 and 32; B gives fewer (1..37 images) and more (149 images: 596 CTAs) CTAs than the
    2 x 148 slots of one wave, odd B included."""
    assert tc.attention_tc_v2_supported(HW, C, heads)
    qkv = qkv_for(B, HW, C, B * HW + C)
    f16 = fmt == "f16"
    hi, lo = run(tc, "v2", qkv, B, HW, C, heads, f16)
    if f16:
        assert hi.dtype == torch.float16
    else:
        assert int((hi.view(torch.int32) & 8191).abs().max()) == 0     # TF32 pair: hi exactly representable
    got = hi.double() + lo.double()
    ref = reference(qkv, B, HW, C, heads)
    assert rel_err(got, ref) < 2e-5
    h1, l1 = run(tc, "v1", qkv, B, HW, C, heads, f16)
    assert rel_err(got, h1.double() + l1.double()) < 2e-5


@pytest.mark.gpu
def test_onewave_large_scores(tc):
    """Scores far apart between the two key blocks: the exact combination O = sum_b O_b 2^(m_b - m) / sum_b l_b 2^(m_b - m)."""
    B, HW, C, heads = 4, 256, 96, 4
    qkv = qkv_for(B, HW, C, 11, scale=4.0)
    qkv.view(B, HW, 3, C)[:, 128:, 0] *= 3.0      # keys of the second block: much larger logits for some rows
    hi, lo = run(tc, "v2", qkv, B, HW, C, heads, True)
    assert rel_err(hi.double() + lo.double(), reference(qkv, B, HW, C, heads)) < 2e-5


@pytest.mark.gpu
def test_onewave_is_deterministic(tc):
    B, HW, C, heads = 64, 256, 96, 4
    qkv = qkv_for(B, HW, C, 5)
    a = run(tc, "v2", qkv, B, HW, C, heads, True)
    b = run(tc, "v2", qkv, B, HW, C, heads, True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize("HW,C,heads", [(256, 96, 4), (128, 96, 4), (256, 128, 4)])
def test_two_ctas_per_sm(tc, HW, C, heads):
    from flowk import _lib
    n, smem = ctypes.c_int(0), ctypes.c_int(0)
    _lib.check(_lib.lib.flowk_attention_tc_v2_occupancy(HW, C, heads, ctypes.byref(n), ctypes.byref(smem)))
    assert n.value == 2
    assert smem.value <= 110 * 1024


@pytest.mark.gpu
def test_unsupported_shapes_route_to_one_cta_kernel(tc, monkeypatch):
    from flowk import _lib
    calls = []
    real = _lib.call

    def spy(name, *args, **kw):
        calls.append(name)
        return real(name, *args, **kw)

    monkeypatch.setattr(_lib, "call", spy)
    monkeypatch.setattr(tc, "ATTENTION_TC_V2", True)
    for HW, C, route in ((256, 160, "flowk_attention_tc"), (256, 32, "flowk_attention_tc"), (128, 256, "flowk_attention_tc"),
                         (64, 96, "flowk_attention_f16"), (256, 96, "flowk_attention_tc_v2")):
        calls.clear()
        qkv = qkv_for(2, HW, C, HW + C)
        hi, lo = tc.attention(qkv, 2, HW, C, 4, True)
        torch.cuda.synchronize()
        assert calls == [route], (HW, C, calls)
        assert rel_err(hi.double() + lo.double(), reference(qkv, 2, HW, C, 4)) < 2e-5
    monkeypatch.setattr(tc, "ATTENTION_TC_V2", False)
    calls.clear()
    tc.attention(qkv_for(2, 256, 96, 1), 2, 256, 96, 4, True)
    assert calls == ["flowk_attention_tc"]


@pytest.mark.gpu
def test_conditioner_graph_capture_matches_eager(tc):
    """The cfg2 level-1 conditioner (MixLogCDF NN with its ConvAttnBlocks at 16 x 16, width 96) captured in a CUDA graph
    gives the eager output bit for bit, and the eager output agrees with the one-CTA-per-SM kernel's."""
    from flowk import conditioner_tc
    from flowk.flow_modules.mixlogcdf_nn import NN
    torch.manual_seed(3)
    dev = torch.device("cuda:0")
    net = NN(6, 96, 2, 4, 0.0).to(dev).eval()
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * 0.02)
        x = torch.randn(64, 12, 16, 16, device=dev)
        x_id = x[:, 6:]
        eager = conditioner_tc.mixlogcdf_nn_raw(net, x_id).clone()
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            conditioner_tc.mixlogcdf_nn_raw(net, x_id)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            captured = conditioner_tc.mixlogcdf_nn_raw(net, x_id)
        g.replay()
        torch.cuda.synchronize()
        saved = tc.ATTENTION_TC_V2
        tc.ATTENTION_TC_V2 = False
        try:
            old = conditioner_tc.mixlogcdf_nn_raw(net, x_id).clone()
        finally:
            tc.ATTENTION_TC_V2 = saved
    assert torch.equal(eager, captured)
    assert rel_err(eager, old) < 1e-4
