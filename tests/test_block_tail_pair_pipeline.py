"""The pipelined attention of the level-1 block tail (flowk_block_tail_pair_tc, csrc/block_tail_tc.cu with PAIR = true): per
head four 64-key blocks (the CTA's own keys 0-63 and 64-127, then the peer's), each with its own row maximum, folded into
the output as they retire.  Checked against an fp64 reference of the whole tail at the widths the kernel instantiates
besides cfg2's (C = 32 / 1 head, 64 / 2 heads, 96 / 3 heads), with the row maximum placed in each of the four blocks, with
block maxima so far apart that 2^(m_b - m) underflows to zero, and for determinism at C = 64."""
import pytest
import torch

HW = 256


@pytest.fixture(scope="module")
def tc():
    import flowk  # noqa: F401
    from flowk import tc as mod
    return mod


def operands(tc, B, C, heads, seed, hot=None, p0=0.0, p1=0.0, cold=0.0):
    """The block's inputs as the conditioner hands them to the kernel.  With `hot` (an image position), dim 0 of every head's
    q is (x1 + pos)[:, 0] and dim 0 of its k is (x1 + pos)[:, 1], the rest of in_proj is small, and pos puts p0 in channel
    0 of every row, p1 in channel 1 of row `hot` and `cold` in channel 1 of the others: key `hot` then scores about
    p0 (p1 - cold) / sqrt(d) above the others in every row."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    M, d = B * HW, C // heads

    def rnd(*shape, s=1.0):
        return torch.randn(*shape, generator=g) * s
    w_in = rnd(3 * C, C, s=(1.5 if hot is None else 0.3) * C ** -0.5)
    pos = rnd(HW, C, s=0.5)
    if hot is not None:
        for h in range(heads):
            w_in[h * d] = 0.0
            w_in[h * d, 1] = 1.0
            w_in[2 * C + h * d] = 0.0
            w_in[2 * C + h * d, 0] = 1.0
        pos[:, 0] = p0
        pos[:, 1] = cold
        pos[hot, 1] = p1
    dev = "cuda:0"
    c1_hi, c1_lo = tc.split_rows_f16(rnd(M, 2 * C, s=0.8).to(dev))
    return dict(c1_hi=c1_hi, c1_lo=c1_lo, gate=tc.conv_weight_operand_f16(rnd(2 * C, 2 * C, s=(2 * C) ** -0.5).to(dev)),
                bias_g=rnd(2 * C, s=0.1).to(dev), x=rnd(M, C).to(dev), pos=pos.to(dev),
                ln1=(1 + rnd(C, s=0.1).to(dev), rnd(C, s=0.1).to(dev)), in_proj=tc.conv_weight_operand_f16(w_in.to(dev)),
                attn_gate=tc.conv_weight_operand_f16(rnd(2 * C, C, s=C ** -0.5).to(dev)), bias_a=rnd(2 * C, s=0.1).to(dev),
                ln2=(1 + rnd(C, s=0.1).to(dev), rnd(C, s=0.1).to(dev)))


def run(tc, o, B, C, heads, celu=True):
    status = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    out = tc.block_tail_pair(o["c1_hi"], o["c1_lo"], o["gate"], o["bias_g"], o["x"], o["ln1"], o["pos"], o["in_proj"],
                             o["attn_gate"], o["bias_a"], o["ln2"], B, HW, C, heads, celu, status=status)
    torch.cuda.synchronize()
    assert int(status) == 0, "barrier wait timed out inside the kernel"
    return out


def reference(o, B, C, heads, celu=True):
    """fp64 tail from the operand pairs and packed weights as the kernel sees them -> (x2, output, scores in log2 units
    [B, heads, HW, HW])."""
    def w(op, k):
        return (op[0].double() + op[1].double())[:, :k] * op[2]

    def glu_ln(t, res, bias, ln):
        t = t + bias.double()
        y = t[:, :C] * torch.sigmoid(t[:, C:]) + res
        return torch.nn.functional.layer_norm(y, (C,), ln[0].double(), ln[1].double(), 1e-5)
    c1 = o["c1_hi"].double() + o["c1_lo"].double()
    x1 = glu_ln(c1 @ w(o["gate"], 2 * C).t(), o["x"].double(), o["bias_g"], o["ln1"])
    qkv = (x1 + o["pos"].double().repeat(B, 1)) @ w(o["in_proj"], C).t()
    d = C // heads
    t = qkv.view(B, HW, 3, heads, d)
    k, v, q = (t[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    s = (q * d ** -0.5) @ k.transpose(-1, -2)
    a = (torch.softmax(s, dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * HW, C)
    x2 = glu_ln(a @ w(o["attn_gate"], C).t(), x1, o["bias_a"], o["ln2"])
    out = torch.cat([torch.nn.functional.elu(x2), torch.nn.functional.elu(-x2)], 1) if celu else x2
    return x2, out, s / torch.log(torch.tensor(2.0, dtype=torch.float64))


def check(tc, o, B, C, heads, celu=True):
    x2, hi, lo = run(tc, o, B, C, heads, celu)
    ref_x2, ref_out, s = reference(o, B, C, heads, celu)
    for got, ref in ((x2.double(), ref_x2), (hi.double() + lo.double(), ref_out)):
        assert got.shape == ref.shape
        assert bool(torch.isfinite(got).all())
        err = float((got - ref).abs().max())
        assert err <= 1e-4 * max(1.0, float(ref.abs().max())), err
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("B", [8, 149])
@pytest.mark.parametrize("C,heads", [(32, 1), (64, 2), (96, 3)])
def test_other_widths_match_fp64(tc, C, heads, B):
    """Head dim 32 at every NKB instantiation; C = 32 and 64 place S / P and O after in_proj (s_col = 5C), C = 96 over the
    drained gate accumulator.  B = 149 is more than one wave of clusters."""
    check(tc, operands(tc, B, C, heads, 11 * C + B), B, C, heads, celu=B == 8)


@pytest.mark.gpu
@pytest.mark.parametrize("hot", [10, 70, 138, 200])
def test_row_maximum_in_each_key_block(tc, hot):
    """Key `hot` scores highest in nearly every row.  Rank 0's rows see it in their block hot // 64 (own 0-63, own 64-127,
    the peer's 0-63 or 64-127); rank 1's in (hot // 64 + 2) % 4, so 200 is rank 0's peer-second block and 70 rank 1's."""
    B, C, heads = 8, 96, 4
    o = operands(tc, B, C, heads, 3 + hot, hot=hot, p0=4.0, p1=8.0)
    s = check(tc, o, B, C, heads)
    assert float((s.argmax(-1) == hot).double().mean()) > 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("hot", [10, 200])
def test_block_maxima_far_apart_underflow(tc, hot):
    """Key `hot` scores more than 126 (log2 units) above every other key of its row, so the weight 2^(m_b - m) of every
    other key block underflows to zero: when the hot block comes last (200 for rank 0's rows) the running output is
    dropped entirely, when it comes first (10 for rank 0's rows) the later blocks add nothing."""
    B, C, heads = 8, 96, 4
    o = operands(tc, B, C, heads, 5 + hot, hot=hot, p0=12.0, p1=40.0, cold=-30.0)
    s = check(tc, o, B, C, heads)
    others = s.clone()
    others[..., hot] = -float("inf")
    gap = s[..., hot] - others.max(-1).values
    assert float(gap.min()) > 126.0, float(gap.min())


@pytest.mark.gpu
def test_deterministic_at_c64(tc):
    B, C, heads = 16, 64, 2
    o = operands(tc, B, C, heads, 2)
    a = run(tc, o, B, C, heads)
    b = run(tc, o, B, C, heads)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
