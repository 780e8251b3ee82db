"""Ancestral sampling from the mAR channel prior on flowk_mar_step (one launch per network stage and channel) and its CUDA
graph: argument validation without a GPU; on the GPU every epilogue against the torch layers in float64, the sampler
against the teacher-forced likelihood kernels, eager sampling against the float64 prior, and the graph against eager."""
import copy
import ctypes

import pytest
import torch
import torch.nn.functional as F

import flowk  # noqa: F401
from flowk import _lib

FILL = ctypes.c_void_p(16)        # never dereferenced: validation fails first


def _args(mode, **kw):
    """A flowk_mar_step_args that is valid for `mode` at level 1 of the reference configuration, with `kw` overriding
    fields (the tests below always break at least one)."""
    a = _lib.MarStepArgs()
    for name in ("a_hi", "a_lo", "w_hi", "w_lo", "bias", "dst0_hi", "dst0_lo", "c", "noise", "z"):
        setattr(a, name, FILL.value)
    a.mode, a.B, a.H, a.W, a.taps, a.dilation, a.hid, a.acc_scale = mode, 64, 16, 16, 25, 2, 32, 1.0
    a.Cin = 8 if mode == _lib.MAR_EMBED else 64
    a.dst0_pitch, a.dst0_col = (8, 0) if mode == _lib.MAR_SAMPLE else (64, 32)
    a.z_stride = 6 * 256
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def _step(a):
    return _lib.lib.flowk_mar_step(ctypes.addressof(a), None)


def test_mar_step_validates_without_gpu():
    ARG, SHAPE = _lib.FLOWK_ERR_ARG, _lib.FLOWK_ERR_SHAPE
    assert _lib.lib.flowk_mar_step(None, None) == ARG
    assert _step(_args(3)) == ARG
    needs = {_lib.MAR_EMBED: [], _lib.MAR_LSTM: ["c"], _lib.MAR_SAMPLE: ["noise", "z"]}
    for mode, extra in needs.items():
        for name in ["a_hi", "a_lo", "w_hi", "w_lo", "bias", "dst0_hi", "dst0_lo"] + extra:
            assert _step(_args(mode, **{name: None})) == ARG, (mode, name)
        assert _step(_args(mode, taps=4)) == ARG
        assert _step(_args(mode, acc_scale=0.0)) == ARG
        for hid in (0, 12, 72):                                      # hid % 8, 4 hid <= 256
            assert _step(_args(mode, hid=hid)) == SHAPE, (mode, hid)
        assert _step(_args(mode, Cin=12)) == SHAPE
        assert _step(_args(mode, W=24)) == SHAPE                     # W must divide 128
        assert _step(_args(mode, H=3)) == SHAPE                      # H*W = 48 neither divides nor is a multiple of 128
        assert _step(_args(mode, B=0)) == SHAPE
        pitch = _args(mode).dst0_pitch
        assert _step(_args(mode, dst0_col=pitch)) == SHAPE           # column + width beyond the pitch
        assert _step(_args(mode, dst0_col=-1)) == SHAPE
    assert _step(_args(_lib.MAR_EMBED, dst0_col=2)) == SHAPE         # 8-byte stores: column % 4
    assert _step(_args(_lib.MAR_LSTM, dst0_pitch=66, dst0_col=0)) == SHAPE
    # LSTM's second destination is optional, but complete and in range when given
    assert _step(_args(_lib.MAR_LSTM, dst1_hi=FILL.value)) == ARG
    assert _step(_args(_lib.MAR_LSTM, dst1_hi=FILL.value, dst1_lo=FILL.value, dst1_pitch=64, dst1_col=40)) == SHAPE
    assert _step(_args(_lib.MAR_SAMPLE, z_stride=255)) == SHAPE      # z_stride >= H*W


def test_graphed_sampler_rejects_temperature_with_mar_prior():
    """The reference's channel prior has no temperature (corr_prior.py:96-101): asking for one is an error, not a no-op."""
    from flowk.graphs import GraphedSampler
    from flowk.marscf import MarScfFlow
    model = MarScfFlow(4, (16, 16, 3), "affine", 2, 1, 16, prior="mar")
    with pytest.raises(ValueError):
        GraphedSampler(model, 4, (16, 16, 3), eps_std=2.0)


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
LEVELS = [(16, 16, 5, 2), (8, 8, 5, 1), (4, 4, 3, 1)]               # cfg2's level shapes: H, W, kernel, dilation
B = 64


def dev():
    return torch.device("cuda:0")


def bound(got, ref, what):
    err = float((got.double().cpu() - ref.double().cpu()).abs().max())
    lim = 1e-4 * max(1.0, float(ref.abs().max()))
    assert err <= lim, "%s: max error %.3e > %.3e" % (what, err, lim)
    return err


def pair(hi, lo):
    return hi.float() + lo.float()


def rows_to_nchw(x, H, W):
    return x.view(-1, H, W, x.shape[-1]).permute(0, 3, 1, 2).double().cpu()


def nchw_to_rows(x):
    return x.permute(0, 2, 3, 1).reshape(-1, x.shape[1])


def sentinel(M, C):
    """fp16 pair rows holding finite garbage: columns a launch must not write keep it bit for bit."""
    return torch.randn(M, C, device=dev()).half(), torch.randn(M, C, device=dev()).half()


@pytest.mark.gpu
@pytest.mark.parametrize("hid", [32, 8])
@pytest.mark.parametrize("level", [0, 1, 2])
def test_each_mode_matches_fp64_layers(no_library, level, hid):
    from flowk import tc
    from flowk.mar_prior import cuda_path
    from flowk.mar_prior.lstm import ConvSeqEncoder
    H, W, k, dil = LEVELS[level]
    M = B * H * W
    torch.manual_seed(10 + level + hid)
    enc = ConvSeqEncoder(input_ch=5, out_ch=2, embed_ch=hid, kernel_size=k, dilation=dil, num_layers=3).to(dev()).eval()
    ops = cuda_path._sampling_operands(enc)
    sd = {n: p.detach().double().cpu() for n, p in enc.named_parameters()}
    lstm = enc.lstm
    worst = {}
    with torch.no_grad():
        # EMBED: S [prev sample | z1 embedding | 0] -> x half of [x | h] rows
        s = torch.zeros(M, 8, device=dev())
        s[:, :5] = torch.randn(M, 5, device=dev())
        s_pair = tc.split_rows_f16(s)
        dst = sentinel(M, 2 * hid)
        keep = [t.clone() for t in dst]
        (w, b, taps) = ops["embed"]
        tc.mar_step(tc.mar_step_args(_lib.MAR_EMBED, s_pair, w, b, B, H, W, taps, hid, dst + (2 * hid, 0)))
        ref = F.conv2d(rows_to_nchw(s[:, :5], H, W), sd["conv_embed.weight"], sd["conv_embed.bias"], padding=k // 2)
        worst["embed"] = bound(pair(dst[0][:, :hid], dst[1][:, :hid]), nchw_to_rows(ref), "EMBED x")
        assert torch.equal(dst[0][:, hid:], keep[0][:, hid:]) and torch.equal(dst[1][:, hid:], keep[1][:, hid:])

        # LSTM (layer 1): [x | h_{t-1}], c_{t-1} -> c_t in place, h_t to the h half of one buffer and the x half of another
        x, h, c = (torch.randn(M, hid, device=dev()) for _ in range(3))
        c_prev = c.clone()
        a_pair = tc.split_rows_f16(torch.cat([x, h], 1))
        d0, d1 = sentinel(M, 2 * hid), sentinel(M, 2 * hid)
        keep0, keep1 = [t.clone() for t in d0], [t.clone() for t in d1]
        (w, b, taps) = ops["layers"][1]
        tc.mar_step(tc.mar_step_args(_lib.MAR_LSTM, a_pair, w, b, B, H, W, taps, hid, d0 + (2 * hid, hid), dilation=dil,
                                     dst1=d1 + (2 * hid, 0), c=c))
        pad = dil * (k - 1) // 2
        gates = (F.conv2d(rows_to_nchw(x, H, W), sd["lstm.weight_ih_l1"], sd["lstm.bias_ih_l1"], padding=pad, dilation=dil)
                 + F.conv2d(rows_to_nchw(h, H, W), sd["lstm.weight_hh_l1"], sd["lstm.bias_hh_l1"], padding=pad,
                            dilation=dil))
        i, f, g, o = gates.chunk(4, 1)
        c_ref = torch.sigmoid(f) * rows_to_nchw(c_prev, H, W) + torch.sigmoid(i) * torch.tanh(g)
        h_ref = torch.sigmoid(o) * torch.tanh(c_ref)
        worst["c"] = bound(c, nchw_to_rows(c_ref), "LSTM c_t")
        worst["h"] = bound(pair(d0[0][:, hid:], d0[1][:, hid:]), nchw_to_rows(h_ref), "LSTM h_t")
        assert torch.equal(d0[0][:, hid:], d1[0][:, :hid]) and torch.equal(d0[1][:, hid:], d1[1][:, :hid]), \
            "the two h destinations differ"
        assert torch.equal(d0[0][:, :hid], keep0[0][:, :hid]) and torch.equal(d0[1][:, :hid], keep0[1][:, :hid])
        assert torch.equal(d1[0][:, hid:], keep1[0][:, hid:]) and torch.equal(d1[1][:, hid:], keep1[1][:, hid:])
        assert lstm.dilation == dil

        # SAMPLE: conv_out1 on the h half ([0 | W_out] ignores the stale x half) -> z[:, t] and column 0 of S
        x, h = torch.randn(M, hid, device=dev()), torch.randn(M, hid, device=dev())
        a_pair = tc.split_rows_f16(torch.cat([x, h], 1))
        noise = torch.randn(M, device=dev())
        nc, t = 3, 1
        z = torch.randn(B, nc, H, W, device=dev())
        z_keep = z.clone()
        s_dst = sentinel(M, 8)
        s_keep = [u.clone() for u in s_dst]
        (w, b, taps) = ops["out"]
        tc.mar_step(tc.mar_step_args(_lib.MAR_SAMPLE, a_pair, w, b, B, H, W, taps, hid, s_dst + (8, 0), noise=noise,
                                     z=z[:, t], z_stride=nc * H * W))
        out = F.conv2d(rows_to_nchw(h, H, W), sd["conv_out1.weight"], sd["conv_out1.bias"], padding=1)
        ref = noise.double().cpu().view(B, H, W) * torch.exp(out[:, 1]) + out[:, 0]
        worst["z"] = bound(z[:, t], ref, "SAMPLE z")
        assert torch.equal(z[:, :t], z_keep[:, :t]) and torch.equal(z[:, t + 1:], z_keep[:, t + 1:])
        s0 = pair(s_dst[0][:, 0], s_dst[1][:, 0])
        zr = z[:, t].reshape(-1)
        assert bool(((s0 - zr).abs() <= 2 ** -20 * zr.abs() + 2 ** -24).all()), "S column 0 is not the fp16 pair of z"
        assert torch.equal(s_dst[0][:, 1:], s_keep[0][:, 1:]) and torch.equal(s_dst[1][:, 1:], s_keep[1][:, 1:])
    print("level %d hid %d: worst %s" % (level + 1, hid, {k_: "%.2e" % v for k_, v in worst.items()}))


def _prior(batch, seed=3):
    from flowk.mar_prior import ChannelPriorMultiScale
    torch.manual_seed(seed)
    return ChannelPriorMultiScale(batch, 3, 32, 32, 3, mog=False, dp_rate=0, num_layers=3, hidden_size=32).to(dev()).eval()


def _z1(prior, level, batch, gen=None):
    if level == 3:
        return None
    p = prior.prior_list[level - 1]
    return torch.randn(batch, p.nc, p.height, p.width, generator=gen).to(dev())


def recovered_noise(p, z1, z2):
    """eps = (z2 - mean) / exp(logs) with (mean, logs) from the teacher-forced likelihood kernels (run_sequence over the
    sampled channels, the input get_likelihood builds)."""
    from flowk.mar_prior import cuda_path
    x = z2.unsqueeze(2)
    inp = torch.cat([torch.zeros_like(x[:, :1]), x[:, :-1]], 1)
    if z1 is not None:
        emb = cuda_path.z1_embedding(p.z1_cond_network, z1).unsqueeze(1).repeat(1, x.size(1), 1, 1, 1)
        inp = torch.cat([inp, emb], 2)
    out = cuda_path.run_sequence(p.prior_lstm, inp)
    return ((z2 - out[:, :, 0]) / torch.exp(out[:, :, 1]))


@pytest.mark.gpu
def test_ancestral_sampler_inverts_the_likelihood_path(no_library):
    """Sample each cfg2 level with injected noise; the likelihood kernels recover that noise from the samples."""
    from flowk.mar_prior import cuda_path
    prior = _prior(B)
    gen = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for level in (1, 2, 3):
            p = prior.prior_list[level - 1]
            z1 = _z1(prior, level, B, gen)
            noise = torch.randn(p.nc, B, p.height, p.width, generator=gen).to(dev())
            s = cuda_path.AncestralSampler(p, B, dev())
            z2 = s.sample(z1, noise)
            eps = recovered_noise(p, z1, z2)
            err = float((eps - noise.permute(1, 0, 2, 3)).abs().max())
            print("level %d: max |eps - noise| %.2e" % (level, err))
            assert err <= 1e-3, "level %d: %.3e" % (level, err)


def fp64_sample(p, z1, b):
    """corr_prior.py:66-101 in float64 on the CPU: one float32 host draw [b, 1, 1, H, W] per channel, in order."""
    p = copy.deepcopy(p).cpu().double()
    emb = None if z1 is None else p.z1_cond_network(z1.cpu().double()).unsqueeze(1)
    inp = torch.zeros(b, 1, 1, p.height, p.width, dtype=torch.float64)
    if emb is not None:
        inp = torch.cat([inp, emb], 2)
    hidden, chans = None, []
    for _ in range(p.nc):
        out, hidden = p.prior_lstm(inp, None, hidden)
        sample = torch.randn(out[:, :, 0:1].size()).double() * torch.exp(out[:, :, 1:2]) + out[:, :, 0:1]
        chans.append(sample)
        inp = sample if emb is None else torch.cat([sample, emb], 2)
    return torch.cat(chans, 1).squeeze(2)


@pytest.mark.gpu
def test_eager_sampling_matches_fp64_prior(no_library):
    """prior(z1, level, reverse=True) on CUDA (the sampler, host noise in the reference's order) against the same prior in
    float64 on the CPU under the same seed: hidden 32, 3 layers, B = 8, all three levels."""
    Bs = 8
    prior = _prior(Bs)
    gen = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for level in (1, 2, 3):
            z1 = _z1(prior, level, Bs, gen)
            torch.manual_seed(100 + level)
            got = prior(z1, level, reverse=True, batch_size=Bs, device=dev())
            torch.manual_seed(100 + level)
            ref = fp64_sample(prior.prior_list[level - 1], z1, Bs)
            err = bound(got, ref, "level %d sample" % level)
            print("level %d: worst |sample - fp64| %.2e (max |ref| %.2f)" % (level, err, float(ref.abs().max())))


def _mar_model():
    from flowk.marscf import MarScfFlow
    torch.manual_seed(0)
    model = MarScfFlow(B, (32, 32, 3), "mixlogcdf", 3, 4, 96, prior="mar").to(dev())
    x = torch.rand(B, 3, 32, 32, generator=torch.Generator().manual_seed(1)) - 0.5
    model.train()
    with torch.no_grad():
        model(x.to(dev()))                                          # ActNorm data-dependent init
    return model.eval()


def _postprocess(x):
    return torch.clamp(torch.where(torch.isnan(x), torch.full_like(x, -0.5), x), -0.5, 0.5)


def _replay(gs):
    """Replay on the lane's stream and copy the images there (run() does not order the caller's stream after it)."""
    gs.run()
    with torch.cuda.stream(gs.stream):
        images = gs.images.clone()
    torch.cuda.current_stream().wait_stream(gs.stream)
    return images


def _fill_eager_order(gs, prior, seed):
    """Host draws exactly as eager sampling takes them: last level first, then the splits from the top, one
    [B, 1, 1, H, W] draw per channel."""
    torch.manual_seed(seed)
    for level in (3, 2, 1):
        p = prior.prior_list[level - 1]
        draws = torch.stack([torch.randn(B, 1, 1, p.height, p.width) for _ in range(p.nc)])
        gs.noise[level - 1].copy_(draws.reshape(p.nc, -1))


@pytest.fixture(scope="module")
def mar_model():
    return _mar_model()


@pytest.mark.gpu
def test_graphed_mar_sampler_equals_eager(no_library, mar_model):
    from flowk.graphs import GraphedSampler
    model = mar_model
    prior = model.flow.c_prior
    gs = GraphedSampler(model, B, (32, 32, 3), draw_noise=False)
    _fill_eager_order(gs, prior, 123)
    images = _replay(gs)
    torch.cuda.synchronize()
    torch.manual_seed(123)
    eager = _postprocess(model(None, None, reverse=True))
    assert torch.equal(images, eager), "graph replay differs from eager sampling"
    # launches: (2 + num_layers) per channel, 4 per split level (z1 embedding: 3, step input: 1), then the flow decode
    zs = [prior.prior_list[2].nc] + [p.nc for p in prior.prior_list[:2]]
    assert sum(zs) == 66
    with torch.no_grad():
        before = _lib.LAUNCHES
        model.flow.decode_latents(gs.latents[3][1], [gs.latents[1][1], gs.latents[2][1]])
        decode = _lib.LAUNCHES - before
    expect = (2 + 3) * 66 + 4 * 2 + decode
    print("flowk launches per replay: %d (prior %d, flow decode %d)" % (gs.flowk_launches, expect - decode, decode))
    assert gs.flowk_launches == expect


@pytest.mark.gpu
def test_graphed_mar_sampler_device_noise(no_library, mar_model):
    from flowk.graphs import GraphedSampler
    model = mar_model
    prior = model.flow.c_prior
    gs = GraphedSampler(model, B, (32, 32, 3))
    first = _replay(gs)
    second = _replay(gs)
    torch.cuda.synchronize()
    assert not torch.equal(first, second), "two replays drew the same images"
    assert bool(torch.isfinite(second).all())
    eps = []
    with torch.no_grad():
        for level in (1, 2, 3):
            z1, z2 = gs.latents[level]
            e = recovered_noise(prior.prior_list[level - 1], z1, z2)
            n = gs.noise[level - 1].view(z2.shape[1], z2.shape[0], z2.shape[2], z2.shape[3]).permute(1, 0, 2, 3)
            err = float((e - n).abs().max())
            assert err <= 1e-3, "level %d: recovered noise off by %.3e" % (level, err)
            eps.append(e.flatten())
    eps = torch.cat(eps).double()
    mean, std = float(eps.mean()), float(eps.std())
    print("%d draws: recovered noise mean %.4f std %.4f" % (eps.numel(), mean, std))
    assert abs(mean) <= 0.01 and abs(std - 1) <= 0.01

    # lanes replayed interleaved without synchronising equal their own serial replays
    lanes = [GraphedSampler(model, B, (32, 32, 3), draw_noise=False) for _ in range(3)]
    serial = []
    for i, lane in enumerate(lanes):
        _fill_eager_order(lane, prior, 200 + i)
        serial.append(_replay(lane))
        torch.cuda.synchronize()
    recs = []
    for _ in range(3):
        for lane in lanes:
            lane.run()
            with torch.cuda.stream(lane.stream):
                recs.append(lane.images.clone())
    torch.cuda.synchronize()
    for j, img in enumerate(recs):
        assert torch.equal(img, serial[j % 3]), "interleaved replay %d of lane %d differs" % (j // 3, j % 3)
