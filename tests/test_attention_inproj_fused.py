"""The one-wave tcgen05 attention kernel with the in_proj GEMM fused in front (flowk_attention_inproj_tc,
attention_tc_v2_kernel<.., true>): q, k, v computed per (image, head) from the gate GEMM's fp16 (hi, lo) rows and the in_proj
weight operand.  Checked against fp64 attention of the projected rows, against the unfused route (in_proj GEMM, then the
one-wave kernel), for determinism, occupancy, routing and, inside the cfg2 conditioner, against the unfused conditioner and
under CUDA-graph capture."""
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


def operands(tc, B, HW, C, seed):
    """Rows P as an fp16 pair and the in_proj weight operand, as the conditioner hands them to the kernel."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    rows = (torch.randn(B * HW, C, generator=g) * 1.5).to("cuda:0")
    w = (torch.randn(3 * C, C, generator=g) / C ** 0.5).to("cuda:0")
    p_hi, p_lo = tc.split_rows_f16(rows)
    w_hi, w_lo, sc = tc.conv_weight_operand_f16(w)
    return p_hi, p_lo, w_hi, w_lo, sc


def qkv_fp64(p_hi, p_lo, w_hi, w_lo, sc, C):
    w = (w_hi.double() + w_lo.double())[:, :C] * sc
    return (p_hi.double() + p_lo.double()) @ w.t()


def reference(qkv, B, HW, C, heads):
    d = C // heads
    t = qkv.double().view(B, HW, 3, heads, d)
    k, v, q = (t[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    return (torch.softmax((q * d ** -0.5) @ k.transpose(-1, -2), dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * HW, C)


def fused(tc, ops, B, HW, C, heads, trace=None):
    status = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    hi, lo = tc.attention_inproj(*ops, B, HW, C, heads, status=status, trace=trace)
    torch.cuda.synchronize()
    assert int(status) == 0, "barrier wait timed out inside the kernel"
    assert hi.dtype == torch.float16
    return hi, lo


def test_support_predicate_needs_no_gpu(monkeypatch):
    import flowk  # noqa: F401
    from flowk import tc
    monkeypatch.setattr(tc, "ATTENTION_TC_V2", True)
    monkeypatch.setattr(tc, "ATTENTION_INPROJ", True)
    assert tc.attention_inproj_supported(256, 96, 4)          # cfg2 level 1
    assert tc.attention_inproj_supported(128, 128, 4)
    assert not tc.attention_inproj_supported(256, 160, 4)     # cfg4 level 1 (d = 40)
    assert not tc.attention_inproj_supported(64, 96, 4)       # levels 2, 3
    assert not tc.attention_inproj_supported(16, 96, 4)
    monkeypatch.setattr(tc, "ATTENTION_INPROJ", False)
    assert not tc.attention_inproj_supported(256, 96, 4)
    monkeypatch.setattr(tc, "ATTENTION_INPROJ", True)
    monkeypatch.setattr(tc, "ATTENTION_TC_V2", False)
    assert not tc.attention_inproj_supported(256, 96, 4)


def test_entry_points_validate_without_gpu():
    import flowk  # noqa: F401
    from flowk import _lib
    L = _lib.lib
    one, odd = ctypes.c_void_p(16), ctypes.c_void_p(17)
    n = ctypes.c_int(-1)
    assert L.flowk_attention_inproj_tc(one, one, one, one, 1.0, one, one, 2, 256, 160, 4, None, None, None) == _lib.FLOWK_ERR_SHAPE
    assert L.flowk_attention_inproj_tc(one, one, one, one, 1.0, one, one, 2, 64, 96, 4, None, None, None) == _lib.FLOWK_ERR_SHAPE
    assert L.flowk_attention_inproj_tc(None, one, one, one, 1.0, one, one, 2, 256, 96, 4, None, None, None) == _lib.FLOWK_ERR_ARG
    assert L.flowk_attention_inproj_tc(one, one, one, one, 0.0, one, one, 2, 256, 96, 4, None, None, None) == _lib.FLOWK_ERR_ARG
    assert L.flowk_attention_inproj_tc(one, odd, one, one, 1.0, one, one, 2, 256, 96, 4, None, None, None) == _lib.FLOWK_ERR_ALIGN
    assert L.flowk_attention_inproj_tc(None, None, None, None, 1.0, None, None, 0, 256, 96, 4, None, None, None) == _lib.FLOWK_OK
    assert L.flowk_attention_inproj_tc_occupancy(256, 160, 4, ctypes.byref(n), None) == _lib.FLOWK_ERR_SHAPE


def test_wrapper_rejects_wrong_layouts_without_gpu():
    """tc.attention_inproj checks the layouts its tensor maps assume before anything reaches the device."""
    import flowk  # noqa: F401
    from flowk import tc
    B, HW, C, heads = 2, 256, 96, 4
    f16 = dict(dtype=torch.float16)
    p, w = torch.zeros(B * HW, C, **f16), torch.zeros(3 * C, 128, **f16)
    bad = [(torch.zeros(B * HW, C + 8, **f16)[:, :C], p, w, w),      # rows not contiguous
           (torch.zeros(B * HW - 1, C, **f16), p, w, w),              # too few rows
           (p, p, torch.zeros(3 * C, C, **f16), w),                   # weight K not padded to 64
           (p, p, w, torch.zeros(3 * C, 128, **f16).t().contiguous().t())]   # weight not row-major
    for p_hi, p_lo, w_hi, w_lo in bad:
        with pytest.raises(AssertionError):
            tc.attention_inproj(p_hi, p_lo, w_hi, w_lo, 1.0, B, HW, C, heads)


SHAPES = [(64, 256, 96, 4), (3, 128, 96, 4), (5, 256, 128, 4), (7, 128, 32, 1), (1, 256, 24, 1), (149, 256, 96, 4),
          (75, 256, 96, 4), (37, 128, 64, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,HW,C,heads", SHAPES)
def test_fused_matches_fp64(tc, B, HW, C, heads):
    """seq 128 / 256, head dims 24 and 32, one to four 32-channel K slices; B gives fewer (1..37 images) and more (149
    images: 596 CTAs) CTAs than the 2 x 148 slots of one wave, odd B included."""
    assert tc.attention_inproj_supported(HW, C, heads)
    ops = operands(tc, B, HW, C, B * HW + C)
    hi, lo = fused(tc, ops, B, HW, C, heads)
    ref = reference(qkv_fp64(*ops, C), B, HW, C, heads)
    assert rel_err(hi.double() + lo.double(), ref) < 2e-5


@pytest.mark.gpu
@pytest.mark.parametrize("B,HW,C,heads", [s for s in SHAPES if s[2] % 32 == 0])
def test_fused_matches_unfused_route(tc, B, HW, C, heads):
    """The in_proj GEMM (flowk_conv_gemm, fp32 rows) followed by the one-wave kernel, on the same operands.  Only widths
    that are multiples of 32: the conditioner's GEMM route takes no others (conditioner_tc.supported), so C = 24 is
    checked against fp64 alone; head dim 24 meets the unfused route here through C = 96 with 4 heads."""
    ops = operands(tc, B, HW, C, 7 * B + HW + C)
    p_hi, p_lo, w_hi, w_lo, sc = ops
    qkv = torch.empty(B * HW, 3 * C, device="cuda:0")
    H = 16 if HW == 256 else 8
    tc.conv_gemm(p_hi, p_lo, w_hi, w_lo, B, H, HW // H, C, 3 * C, 1, tc.PRE_BIAS, tc.OUT_F32, out_f32=qkv, acc_scale=sc)
    assert tc.attention_tc_v2_supported(HW, C, heads)
    o_hi, o_lo = tc.attention(qkv, B, HW, C, heads, True)
    hi, lo = fused(tc, ops, B, HW, C, heads)
    assert rel_err(hi.double() + lo.double(), o_hi.double() + o_lo.double()) < 2e-5


@pytest.mark.gpu
def test_fused_is_deterministic(tc):
    B, HW, C, heads = 64, 256, 96, 4
    ops = operands(tc, B, HW, C, 5)
    a = fused(tc, ops, B, HW, C, heads)
    b = fused(tc, ops, B, HW, C, heads)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize("HW,C,heads", [(256, 96, 4), (128, 96, 4), (256, 128, 4)])
def test_two_ctas_per_sm(tc, HW, C, heads):
    from flowk import _lib
    n, smem = ctypes.c_int(0), ctypes.c_int(0)
    _lib.check(_lib.lib.flowk_attention_inproj_tc_occupancy(HW, C, heads, ctypes.byref(n), ctypes.byref(smem)))
    assert n.value == 2
    assert smem.value <= 110 * 1024


def cfg2_conditioner(seed=3):
    from flowk.flow_modules.mixlogcdf_nn import NN
    torch.manual_seed(seed)
    dev = torch.device("cuda:0")
    net = NN(6, 96, 2, 4, 0.0).to(dev).eval()
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    return net


@pytest.mark.gpu
def test_conditioner_routes(tc, monkeypatch):
    """Level 1 (16 x 16, d = 24) takes the fused kernel and no in_proj GEMM; levels 2 and 3 keep the chained GEMM and the
    mma.sync kernel; FLOWK_ATTENTION_INPROJ=0 (tc.ATTENTION_INPROJ) restores the one-wave kernel at level 1."""
    from flowk import _lib, conditioner_tc
    net = cfg2_conditioner()
    calls = []
    real = _lib.call

    def spy(name, *args, **kw):
        calls.append(name)
        return real(name, *args, **kw)

    monkeypatch.setattr(_lib, "call", spy)
    with torch.no_grad():
        for hw, attn in ((16, ["flowk_attention_inproj_tc"]), (8, ["flowk_attention_f16"]), (4, ["flowk_attention_f16"])):
            calls.clear()
            conditioner_tc.mixlogcdf_nn_raw(net, torch.randn(2, 12, hw, hw, device="cuda:0")[:, 6:])
            assert [c for c in calls if "attention" in c] == attn * 2, (hw, calls)
            per_block = 3 if hw == 16 or conditioner_tc.CHAIN else 4   # conv, gate (+ in_proj unless fused / chained), attn gate
            assert calls.count("flowk_conv_gemm") == 2 + 2 * per_block, (hw, calls)
        monkeypatch.setattr(tc, "ATTENTION_INPROJ", False)
        calls.clear()
        conditioner_tc.mixlogcdf_nn_raw(net, torch.randn(2, 12, 16, 16, device="cuda:0")[:, 6:])
        assert [c for c in calls if "attention" in c] == ["flowk_attention_tc_v2"] * 2


@pytest.mark.gpu
def test_conditioner_fused_vs_unfused_and_graph_capture(tc, monkeypatch):
    """The cfg2 level-1 conditioner (width 96, 4 heads, B = 64): fused and unfused routes agree to 1e-4 of max(1, max|ref|),
    and a CUDA-graph capture of the fused route gives the eager output bit for bit."""
    from flowk import conditioner_tc
    net = cfg2_conditioner()
    dev = torch.device("cuda:0")
    with torch.no_grad():
        x_id = torch.randn(64, 12, 16, 16, device=dev)[:, 6:]
        eager = conditioner_tc.mixlogcdf_nn_raw(net, x_id).clone()
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
        monkeypatch.setattr(tc, "ATTENTION_INPROJ", False)
        ref = conditioner_tc.mixlogcdf_nn_raw(net, x_id).clone()
    assert torch.equal(eager, captured)
    err = float((eager.double() - ref.double()).abs().max())
    assert err <= 1e-4 * max(1.0, float(ref.abs().max())), err
