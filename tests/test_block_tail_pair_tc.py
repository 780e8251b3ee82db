"""The attention half of a ConvAttnBlock at 16x16 in one tcgen05 launch of two-CTA clusters (flowk_block_tail_pair_tc,
csrc/block_tail_tc.cu with PAIR = true): each CTA owns 128 of an image's 256 rows, and the two exchange each head's K and
V so that every row attends over the whole image.  Checked against an fp64 reference of the whole tail (including a grid of
more than one wave), for attention that crosses the pair and stops at the image, for determinism and the trace stamps,
against the gate GEMM + fused in_proj attention + gate route inside the cfg2 conditioner, under CUDA-graph capture, and for
the routes the conditioner takes at level 1."""
import ctypes

import pytest
import torch

HW, C, HEADS = 256, 96, 4


@pytest.fixture(scope="module")
def tc():
    import flowk  # noqa: F401
    from flowk import tc as mod
    return mod


def test_support_predicate_needs_no_gpu(monkeypatch):
    import flowk  # noqa: F401
    from flowk import tc
    monkeypatch.setattr(tc, "BLOCK_TAIL_PAIR", True)
    assert tc.block_tail_pair_supported(256, 96, 4, 64)         # cfg2 level 1 at the benchmark's batch
    assert tc.block_tail_pair_supported(256, 96, 4, 8)
    assert tc.block_tail_pair_supported(256, 64, 2, 149)        # head dim 32
    assert not tc.block_tail_pair_supported(256, 96, 4, 2)      # small batches keep flowk_attention_inproj_tc
    assert not tc.block_tail_pair_supported(256, 96, 4, 4)
    assert not tc.block_tail_pair_supported(256, 160, 4, 64)    # cfg4: 5C > 512 TMEM columns, head dim 40
    assert not tc.block_tail_pair_supported(64, 96, 4, 64)      # deep levels take flowk_block_tail_tc
    assert not tc.block_tail_pair_supported(16, 96, 4, 64)
    assert not tc.block_tail_pair_supported(256, 96, 2, 64)     # head dim 48
    monkeypatch.setattr(tc, "BLOCK_TAIL_PAIR", False)
    assert not tc.block_tail_pair_supported(256, 96, 4, 64)


def test_entry_point_validates_without_gpu():
    import flowk  # noqa: F401
    from flowk import _lib
    one, odd = ctypes.c_void_p(16), ctypes.c_void_p(17)

    def call(*, ptr=one, first=one, sc=1.0, B=2, HW=256, C=96, heads=4):
        return _lib.lib.flowk_block_tail_pair_tc(first, ptr, ptr, ptr, sc, ptr, ptr, ptr, ptr, ptr, ptr, ptr, 1.0, ptr, ptr,
                                                 1.0, ptr, ptr, ptr, ptr, ptr, ptr, 1, B, HW, C, heads, None, None, None)
    assert call(HW=64) == _lib.FLOWK_ERR_SHAPE                  # whole images per tile: flowk_block_tail_tc's shapes
    assert call(HW=128) == _lib.FLOWK_ERR_SHAPE
    assert call(C=160, heads=4) == _lib.FLOWK_ERR_SHAPE         # 5C > 512
    assert call(C=96, heads=2) == _lib.FLOWK_ERR_SHAPE          # head dim 48
    assert call(C=80, heads=4) == _lib.FLOWK_ERR_SHAPE          # C % 32 != 0
    assert call(B=-1) == _lib.FLOWK_ERR_SHAPE
    assert call(first=None) == _lib.FLOWK_ERR_ARG
    assert call(sc=0.0) == _lib.FLOWK_ERR_ARG
    assert call(first=odd) == _lib.FLOWK_ERR_ALIGN
    assert call(ptr=None, first=None, B=0) == _lib.FLOWK_OK


def operands(tc, B, seed):
    """The block's inputs as the conditioner hands them to the kernel: c1 as an fp16 pair, fp16 weight operands."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    M = B * HW

    def rnd(*shape, s=1.0):
        return (torch.randn(*shape, generator=g) * s).to("cuda:0")
    c1_hi, c1_lo = tc.split_rows_f16(rnd(M, 2 * C, s=0.8))
    gate = tc.conv_weight_operand_f16(rnd(2 * C, 2 * C, s=(2 * C) ** -0.5))
    # in_proj scaled so that the scores q k / sqrt(d) spread over several units: the softmax is far from flat
    in_proj = tc.conv_weight_operand_f16(rnd(3 * C, C, s=1.5 * C ** -0.5))
    attn_gate = tc.conv_weight_operand_f16(rnd(2 * C, C, s=C ** -0.5))
    return dict(c1_hi=c1_hi, c1_lo=c1_lo, gate=gate, bias_g=rnd(2 * C, s=0.1), x=rnd(M, C), pos=rnd(HW, C, s=0.5),
                ln1=(1 + rnd(C, s=0.1), rnd(C, s=0.1)), in_proj=in_proj, attn_gate=attn_gate, bias_a=rnd(2 * C, s=0.1),
                ln2=(1 + rnd(C, s=0.1), rnd(C, s=0.1)))


def run(tc, o, B, celu, trace=None):
    status = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    out = tc.block_tail_pair(o["c1_hi"], o["c1_lo"], o["gate"], o["bias_g"], o["x"], o["ln1"], o["pos"], o["in_proj"],
                             o["attn_gate"], o["bias_a"], o["ln2"], B, HW, C, HEADS, celu, status=status, trace=trace)
    torch.cuda.synchronize()
    assert int(status) == 0, "barrier wait timed out inside the kernel"
    return out


def reference(o, B, celu):
    """fp64 gate -> GLU -> +x -> LN -> +pos -> in_proj -> per-image softmax attention over all 256 keys -> gate -> GLU -> +x1
    -> LN (-> concat_elu) from the operand pairs and packed weights as the kernel sees them."""
    def w(op, k):
        return (op[0].double() + op[1].double())[:, :k] * op[2]

    def glu_ln(t, res, bias, ln):
        t = t + bias.double()
        y = t[:, :C] * torch.sigmoid(t[:, C:]) + res
        return torch.nn.functional.layer_norm(y, (C,), ln[0].double(), ln[1].double(), 1e-5)
    c1 = o["c1_hi"].double() + o["c1_lo"].double()
    x1 = glu_ln(c1 @ w(o["gate"], 2 * C).t(), o["x"].double(), o["bias_g"], o["ln1"])
    qkv = (x1 + o["pos"].double().repeat(B, 1)) @ w(o["in_proj"], C).t()
    d = C // HEADS
    t = qkv.view(B, HW, 3, HEADS, d)
    k, v, q = (t[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    a = (torch.softmax((q * d ** -0.5) @ k.transpose(-1, -2), dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * HW, C)
    x2 = glu_ln(a @ w(o["attn_gate"], C).t(), x1, o["bias_a"], o["ln2"])
    out = torch.cat([torch.nn.functional.elu(x2), torch.nn.functional.elu(-x2)], 1) if celu else x2
    return x2, out


def bound(ref):
    return 1e-4 * max(1.0, float(ref.abs().max()))


@pytest.mark.gpu
@pytest.mark.parametrize("celu", [True, False])
@pytest.mark.parametrize("B", [8, 9, 64, 149])
def test_matches_fp64(tc, B, celu):
    """cfg2's level 1 (C = 96, 4 heads); B = 149 is 298 CTAs, more than one wave of 148 SMs."""
    o = operands(tc, B, 7 * B + 1)
    x2, hi, lo = run(tc, o, B, celu)
    ref_x2, ref_out = reference(o, B, celu)
    assert float((x2.double() - ref_x2).abs().max()) <= bound(ref_x2)
    got = hi.double() + lo.double()
    assert got.shape == ref_out.shape
    assert float((got - ref_out).abs().max()) <= bound(ref_out)


@pytest.mark.gpu
def test_attention_crosses_the_pair_and_stops_at_the_image(tc):
    """Perturbing only rank 1's rows of image 1 changes rank 0's outputs of that image (its keys reach the other CTA of the
    cluster) and no other image's outputs, bit for bit."""
    B = 16
    o = operands(tc, B, 5)
    x2, hi, lo = run(tc, o, B, True)
    rows = slice(HW + 128, 2 * HW)              # image 1, rank 1
    o["x"] = o["x"].clone()
    o["x"][rows] += 0.5
    o["c1_hi"] = o["c1_hi"].clone()
    o["c1_hi"][rows] = -o["c1_hi"][rows]
    x2b, hib, lob = run(tc, o, B, True)
    rank0 = slice(HW, HW + 128)
    assert not torch.equal(x2[rank0], x2b[rank0])
    assert not torch.equal(hi[rank0], hib[rank0])
    other = torch.ones(B * HW, dtype=torch.bool, device="cuda:0")
    other[HW:2 * HW] = False
    for a, b in ((x2, x2b), (hi, hib), (lo, lob)):
        assert torch.equal(a[other], b[other])


@pytest.mark.gpu
def test_deterministic_and_traced(tc):
    B = 64
    o = operands(tc, B, 9)
    trace = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    a = run(tc, o, B, True, trace=trace)
    b = run(tc, o, B, True)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    t = trace.cpu().tolist()
    assert all(t[i] < t[i + 1] for i in range(7)), t


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
def test_conditioner_matches_inproj_route(tc, monkeypatch, no_library):
    """A cfg2-width conditioner (96 channels, 4 heads, two blocks: the concat-ELU and the last-block outputs) at level 1,
    B = 64: the cluster route against the gate GEMM + flowk_attention_inproj_tc + gate route, and CUDA-graph replay of the
    cluster route against its eager run bit for bit."""
    from flowk import conditioner_tc
    net = cfg2_conditioner()
    with torch.no_grad():
        x_id = torch.randn(64, 12, 16, 16, device="cuda:0")[:, 6:]
        status = torch.zeros(1, dtype=torch.int32, device="cuda:0")
        eager = conditioner_tc.mixlogcdf_nn_raw(net, x_id, status=status).clone()
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
        monkeypatch.setattr(tc, "BLOCK_TAIL_PAIR", False)
        ref = conditioner_tc.mixlogcdf_nn_raw(net, x_id).clone()
    assert int(status) == 0
    assert torch.equal(eager, captured)
    err = float((eager.double() - ref.double()).abs().max())
    assert err <= 1e-4 * max(1.0, float(ref.abs().max())), err


@pytest.mark.gpu
def test_conditioner_routes_block_tail_pair(tc, monkeypatch):
    """Level 1 takes the cluster launch (one per attention block, no separate gate GEMMs) from B = 8, and
    flowk_attention_inproj_tc below that or with FLOWK_BLOCK_TAIL_PAIR=0 (tc.BLOCK_TAIL_PAIR)."""
    from flowk import _lib, conditioner_tc
    net = cfg2_conditioner()
    calls = []
    real = _lib.call

    def spy(name, *args, **kw):
        calls.append(name)
        return real(name, *args, **kw)

    def route(B, hw):
        calls.clear()
        conditioner_tc.mixlogcdf_nn_raw(net, torch.randn(B, 12, hw, hw, device="cuda:0")[:, 6:])
        return [c for c in calls if "attention" in c or "block_tail" in c], calls.count("flowk_conv_gemm")

    monkeypatch.setattr(_lib, "call", spy)
    with torch.no_grad():
        assert route(64, 16) == (["flowk_block_tail_pair_tc"] * 2, 2 + 2 * 1)
        assert route(8, 16) == (["flowk_block_tail_pair_tc"] * 2, 2 + 2 * 1)
        assert route(4, 16) == (["flowk_attention_inproj_tc"] * 2, 2 + 2 * 3)
        assert route(64, 8) == (["flowk_block_tail_tc"] * 2, 2 + 2 * 1)
        monkeypatch.setattr(tc, "BLOCK_TAIL_PAIR", False)
        assert route(64, 16) == (["flowk_attention_inproj_tc"] * 2, 2 + 2 * 3)
