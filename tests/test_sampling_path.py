"""The sampling (inverse) path against the fp64 oracle on the inputs sampling produces, and the CUDA-graph lanes that the
headline numbers come from against eager execution.

A round trip decode(encode(x)) only feeds the inverse coupling kernel latents that the forward kernel can reach.  Latents
drawn from N(0, eps_std^2) also reach the u clamp to [1e-5, 1 - 1e-5] (mixlogcdf_coupling.py:44), a sigmoid that
saturates to exactly 0 or 1 in fp32, and the ends of the bisection bracket mu +- 20 sum_k e^{s_k} (log_dist.py:60-62).
`GraphedSampler` replaces NaN by -0.5 and clamps to the data range, so a kernel that returns NaN or garbage there still
gives plausible images: every check below asserts explicitly that the GPU output is finite wherever the oracle's is.

The bisection result is conditioned by 1/pdf, so the transformed half is compared in CDF space, |F(x_gpu) - F(x_ref)|
with the oracle's fp64 mixture, and directly only where the density is not small (pdf > 0.02).  The per-sample log-det
is compared with the oracle's log-det formula evaluated at the kernel's own x: in the flat stretches of a mixture the
CDF pins x only to within a stretch whose log-pdf varies by tens of nats, and the CDF check already bounds that.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from oracle import flow_oracle as O

pytestmark = pytest.mark.gpu
K = 32
CDF_TOL = 5e-6          # |F(x_gpu) - F(x_ref)|
DX_TOL = 3e-4           # |x_gpu - x_ref| where pdf(x_ref) > DENSE
DENSE = 0.02
LDJ_REL = 2e-4          # log-det, |got - ref| <= LDJ_REL * max(1, max|ref|)
T_CLAMP = math.log(O.U_CLAMP) - math.log1p(-O.U_CLAMP)      # sigmoid(T_CLAMP) = 1e-5


def dev():
    return torch.device("cuda:0")


def parity(got, ref, rel, what):
    got, ref = got.detach().double().cpu(), ref.double()
    err = float((got - ref).abs().max())
    assert err <= rel * max(1.0, float(ref.abs().max())), "%s: max abs err %.3e > %.1e" % (what, err, rel)
    return err


def check_inverse(got_y, got_l, xo, raw_params, ref_y, ldj0, what):
    """Inverse coupling output `got_y` / `got_l` (GPU) against the oracle's `ref_y` for the oracle input `xo`
    (cat(v, x_id), fp64) and the oracle's (a, b, pi, mu, s).  Returns the measured errors."""
    a, b, pi, mu, s = raw_params
    c = xo.shape[1] // 2
    xg = got_y[:, :c].detach().cpu().double()
    xr = ref_y[:, :c]
    fin = torch.isfinite(xr)
    assert bool(torch.isfinite(xg)[fin].all()), "%s: %d non-finite GPU outputs where the oracle's are finite" % (
        what, int((~torch.isfinite(xg) & fin).sum()))
    assert torch.equal(got_y[:, c:].cpu(), xo[:, c:].float()), what + ": pass-through half not bit-exact"
    xg_f = torch.where(fin, xg, torch.zeros_like(xg))
    xr_f = torch.where(fin, xr, torch.zeros_like(xr))
    err_cdf = float(((O.mix_log_cdf(xg_f, pi, mu, s).exp() - O.mix_log_cdf(xr_f, pi, mu, s).exp()).abs() * fin).max())
    assert err_cdf <= CDF_TOL, "%s: CDF-space error %.3e" % (what, err_cdf)
    dense = fin & (O.mix_log_pdf(xr_f, pi, mu, s).exp() > DENSE)
    err_dx = float(torch.where(dense, (xg_f - xr_f).abs(), torch.zeros_like(xg)).max())
    assert err_dx <= DX_TOL, "%s: |dx| %.3e where pdf > %g" % (what, err_dx, DENSE)
    t = xo[:, :c] * torch.exp(-a) - b
    ldj_at_gpu_x = ldj0 - (a + Fn.softplus(t) + Fn.softplus(-t) + O.mix_log_pdf(xg_f, pi, mu, s)).flatten(1).sum(-1)
    err_ldj = parity(got_l, ldj_at_gpu_x, LDJ_REL, what + " log-det") / max(1.0, float(ldj_at_gpu_x.abs().max()))
    u = torch.sigmoid(t)
    return {"cdf": err_cdf, "dx": err_dx, "ldj": err_ldj, "dense": int(dense.sum()), "n": xr.numel(),
            "clamped": int(((u < O.U_CLAMP) | (u > 1 - O.U_CLAMP)).sum())}


def report(what, m):
    print("%-34s CDF %.2e  dx(pdf>%.2g) %.2e over %d/%d  log-det rel %.2e  clamped %d"
          % (what, m["cdf"], DENSE, m["dx"], m["dense"], m["n"], m["ldj"], m["clamped"]))


# ---------------------------------------------------------------------------------------------
# 1. the inverse coupling kernel on hand-built parameters
# ---------------------------------------------------------------------------------------------
def edge_case(B, c, H, W, flip, seed):
    """Input x, raw conditioner output [B, 98c, H, W], rescale [c] and ldj0 [B].  Each transformed element draws one of
    six mixture kinds and a t = v e^{-a} - b from a sweep over [-40, 40] that also holds the points where the fp32
    sigmoid is exactly 0 / 1 and points just inside / outside the u clamp."""
    gen = torch.Generator().manual_seed(seed)
    n = B * c * H * W

    def rnd(*shape):
        return torch.rand(*shape, generator=gen)

    special = [-120.0, -100.0, -90.0, 90.0, 100.0, 17.0, 20.0, 30.0, T_CLAMP, -T_CLAMP]
    for d in (1e-4, 1e-3, 1e-2, 1e-1):
        special += [T_CLAMP + d, -T_CLAMP - d, T_CLAMP - d, -T_CLAMP + d]
    rest = max(n - len(special), 0)                  # half of the sweep inside the clamp, half over [-40, 40]
    t = torch.cat([torch.tensor(special), torch.linspace(-40.0, 40.0, rest // 2),
                   torch.linspace(-12.0, 12.0, rest - rest // 2)])[:n]
    kind = torch.randint(0, 6, (n,), generator=gen)
    pi = torch.randn(n, K, generator=gen)
    mu = torch.randn(n, K, generator=gen)
    s = torch.randn(n, K, generator=gen) * 0.7 - 0.5
    # (weights stay near 1/32 in the sharp and the flat kinds: one fp32 ulp of x then moves F by at most ~1e-6)
    m = kind == 1                                    # sharp: at the -7 floor and below it (the floor applies)
    s[m] = torch.where(rnd(int(m.sum()), K) < 0.5, torch.tensor(-7.0), -7.0 - 10.0 * rnd(int(m.sum()), K))
    pi[m] *= 0.3
    mu[m] *= 0.25
    m = kind == 2                                    # broad: sum e^s up to ~600, bracket +-12 000
    s[m] = 1.0 + 2.0 * rnd(int(m.sum()), K)
    m = kind == 3                                    # one dominant broad component over sharp ones
    pi[m, 0] = 25.0
    s[m, 0] = 2.0 * rnd(int(m.sum()))
    s[m, 1:] = -7.0 - 3.0 * rnd(int(m.sum()), K - 1)
    m = kind == 4                                    # near-uniform weights
    pi[m] = 1e-3 * torch.randn(int(m.sum()), K, generator=gen)
    m = kind == 5                                    # components 2 apart and narrow: flat stretches between them
    pi[m] *= 0.3
    mu[m] = -30.0 + 2.0 * torch.stack([torch.randperm(K, generator=gen) for _ in range(int(m.sum()))]).float() \
        + 0.05 * torch.randn(int(m.sum()), K, generator=gen)
    s[m] = -4.0 + 1.5 * rnd(int(m.sum()), K)
    a_raw = 0.4 * torch.randn(n, generator=gen)
    b = torch.randn(n, generator=gen)
    exact = torch.arange(n) < len(special)           # a = b = 0 there, so t is the special value itself
    a_raw[exact] = 0.0
    b[exact] = 0.0
    rescale = rnd(c) + 0.5
    a = rescale.view(1, c, 1, 1).expand(B, c, H, W).reshape(-1) * torch.tanh(a_raw)
    v = ((t + b) * torch.exp(a)).float()
    x_id = torch.randn(n, generator=gen)

    def planes(p):                                   # [n, K] -> [B, K, c, H, W]
        return p.view(B, c, H, W, K).permute(0, 4, 1, 2, 3)
    raw = torch.cat([a_raw.view(B, 1, c, H, W), b.view(B, 1, c, H, W), planes(pi), planes(mu), planes(s)], 1)
    halves = (x_id.view(B, c, H, W), v.view(B, c, H, W)) if flip else (v.view(B, c, H, W), x_id.view(B, c, H, W))
    return torch.cat(halves, 1), raw.reshape(B, -1, H, W).contiguous(), rescale, torch.randn(B, generator=gen)


@pytest.mark.parametrize("flip", [False, True])
@pytest.mark.parametrize("B,c,H,W", [(3, 5, 9, 11), (1, 3, 5, 7), (5, 2, 4, 9), (2, 7, 13, 13)])
def test_inverse_coupling_kernel_edges_vs_fp64_oracle(B, c, H, W, flip):
    """flowk_mixlogcdf_inv on hand-built parameters against the fp64 oracle on the same fp32 inputs.  E = c*H*W is not a
    multiple of 32 (the last warp runs with inactive lanes reading element E - 1); (2, 7, 13, 13) spreads a sample over
    10 CTAs, so the log-det goes through the workspace ticket."""
    from flowk import ops
    from flowk.flow_modules import log_dist
    x, raw, rescale, ldj0 = edge_case(B, c, H, W, flip, seed=1000 + 7 * B + c + int(flip))
    assert (c * H * W) % 32
    y, ldj = ops.mixlogcdf_coupling(x.to(dev()), raw.to(dev()), rescale.to(dev()), ldj0.to(dev()), True, flip, K)
    params = O.mixlogcdf_split_params(raw.double(), rescale.double().view(-1, 1, 1))
    a, b, pi, mu, s = params
    xo = O.tuple_flip(x.double()) if flip else x.double()
    ref_y, _ = O.mixlogcdf_elementwise(xo, a, b, pi, mu, s, ldj0.double(), reverse=True)
    # the sweep reaches what it is meant to reach (fp32 sigmoid of the kernel's form: exactly 0 and exactly 1)
    t32 = (xo[:, :c].float() * torch.exp(-a.float()) - b.float())
    u32 = 1.0 / (1.0 + torch.exp(-t32))
    u64 = torch.sigmoid(xo[:, :c] * torch.exp(-a) - b)
    assert bool((u32 == 0).any()) and bool((u32 == 1).any())
    assert bool(((u64 > O.U_CLAMP) & (u64 < 1.001 * O.U_CLAMP)).any())
    assert bool(((u64 < 1 - O.U_CLAMP) & (u64 > 1 - 1.001 * O.U_CLAMP)).any())
    m = check_inverse(y, ldj, xo, params, ref_y, ldj0.double(), "coupling inv B%d c%d %dx%d flip=%d" % (B, c, H, W, flip))
    report("kernel B%d c%d %dx%d flip=%d" % (B, c, H, W, flip), m)

    # the standalone bisection ([B, K, N] layout) on the same clamped targets and the oracle's (floored) parameters
    u = u64.clamp(O.U_CLAMP, 1 - O.U_CLAMP).float()
    got = log_dist.mixture_inv_cdf(u.to(dev()), *(p.float().contiguous().to(dev()) for p in (pi, mu, s)))
    ref = O.mix_inv_cdf(u.double(), pi, mu, s)
    xg = got.cpu().double()
    assert bool(torch.isfinite(xg).all())
    err_cdf = float((O.mix_log_cdf(xg, pi, mu, s).exp() - O.mix_log_cdf(ref, pi, mu, s).exp()).abs().max())
    dense = O.mix_log_pdf(ref, pi, mu, s).exp() > DENSE
    err_dx = float(((xg - ref).abs() * dense).max())
    print("%-34s CDF %.2e  dx(pdf>%.2g) %.2e" % ("mixture_inv_cdf B%d c%d %dx%d" % (B, c, H, W), err_cdf, DENSE, err_dx))
    assert err_cdf <= CDF_TOL and err_dx <= DX_TOL, (err_cdf, err_dx)


# ---------------------------------------------------------------------------------------------
# 2. sampling at real width, layer by layer against the oracle
# ---------------------------------------------------------------------------------------------
CONFIGS = {   # name: (image HWC, L, K, hidden, batch the ActNorm init sees, seed)
    "cfg2": ((32, 32, 3), 3, 4, 96, 64, 201),
    "cfg4": ((32, 32, 3), 3, 4, 160, 8, 203),
}


def _initialised_model(coupling, image, L, K_, hidden, B, seed, **kw):
    from flowk import marscf
    torch.manual_seed(seed)
    np.random.seed(seed)
    model = marscf.MarScfFlow(B, image, coupling, L, K_, hidden, **kw).to(dev())
    gen = torch.Generator().manual_seed(seed + 1)
    x = torch.rand(B, image[2], image[0], image[1], generator=gen) - 0.5
    noise = torch.rand(B, image[2], image[0], image[1], generator=gen)
    model.train()
    with torch.no_grad():
        model(x.to(dev()), noise=noise.to(dev()))            # ActNorm data-dependent init (first training batch)
        std = 0.02 if hidden <= 96 else 0.005                # wide nets: keep the (2304-term) output sums O(0.1)
        for p in model.parameters():                         # move the zero-initialised output convs off zero
            p.add_((torch.randn(p.shape, generator=gen) * std).to(p.device))
    return model.eval()


_MODELS = {}


def model_for(cfg):
    if cfg not in _MODELS:
        image, L, K_, hidden, B, seed = CONFIGS[cfg]
        _MODELS[cfg] = _initialised_model("mixlogcdf", image, L, K_, hidden, B, seed)
    return _MODELS[cfg]


def latent_shapes(B, image, L):
    """(final latent, [factored-out halves in split order]), as GraphedSampler draws them."""
    h, w, c = image
    halves = []
    for lvl in range(L):
        c, h, w = c * 4, h // 2, w // 2
        if lvl < L - 1:
            c //= 2
            halves.append((B, c, h, w))
    return (B, c, h, w), halves


@pytest.fixture(scope="module", autouse=True)
def _free_models():
    yield
    _MODELS.clear()


@pytest.mark.parametrize("eps_std", [1.0, 2.0])
@pytest.mark.parametrize("cfg", sorted(CONFIGS))
def test_sampling_layer_by_layer_vs_oracle(no_library, cfg, eps_std):
    """Decode drawn latents one sub-layer at a time, feeding the oracle's output (rounded to fp32) to both sides:
    the MixLogCDF coupling (tcgen05 conditioner + flowk_mixlogcdf_inv) and the ActNorm∘InvConv reverse fold
    (flowk_fold_actnorm_invconv + flowk_channel_mix).  Then the whole decode: fused and unfused unsqueeze agree bit for
    bit, and the GPU images are finite wherever the oracle's are."""
    from flowk import ops
    image, L, K_, hidden, _, seed = CONFIGS[cfg]
    model = model_for(cfg)
    B = 8
    sd = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    gen = torch.Generator().manual_seed(seed + int(10 * eps_std))
    zs, hs = latent_shapes(B, image, L)
    z = torch.randn(zs, generator=gen) * eps_std
    z2s = [torch.randn(s_, generator=gen) * eps_std for s_ in hs]

    plan = O.layer_plan(L, K_)
    x = z.double()
    pending = [t.double() for t in z2s]
    worst = {"cdf": 0.0, "dx": 0.0, "ldj": 0.0, "mix": 0.0, "clamped": 0}
    for i in reversed(range(len(plan))):
        if plan[i] == "split":
            x = torch.cat((x, pending.pop()), 1)
            continue
        if plan[i] == "squeeze":
            x = O.unsqueeze2d(x)
            continue
        step, pre = model.flow.layers[i], "flow.layers.%d." % i
        b_, C, H, W = x.shape
        zero = torch.zeros(B, dtype=torch.float64)
        xin = x.float()
        xo = O.tuple_flip(xin.double())
        params = O.mixlogcdf_conditioner(sd, pre + "coupling.nn.", xo[:, C // 2:])
        ref_y, _ = O.mixlogcdf_elementwise(xo, *params, zero, reverse=True)
        with torch.no_grad():
            y, ldj = step.coupling(xin.to(dev()), zero.float().to(dev()), True, flip=True)
        m = check_inverse(y, ldj, xo, params, ref_y, zero, "%s eps %g layer %d coupling" % (cfg, eps_std, i))
        for k in ("cdf", "dx", "ldj"):
            worst[k] = max(worst[k], m[k])
        worst["clamped"] += m["clamped"]

        yin = ref_y.float()
        ic = [sd[pre + "invert_1x1_layer." + n] for n in ("p", "l", "u", "sign_s", "log_s")]
        r, rl = O.invconv(yin.double(), *ic, zero, reverse=True)
        r, rl = O.actnorm(r, sd[pre + "actnormlayer.bias"], sd[pre + "actnormlayer.logs"], rl, reverse=True)
        with torch.no_grad():
            mat, bias, add = step._folded((H, W), True)
            xm, lm = ops.channel_mix(yin.to(dev()), mat, bias, zero.float().to(dev()), add, False, False)
        what = "%s eps %g layer %d ActNorm∘InvConv reverse" % (cfg, eps_std, i)
        worst["mix"] = max(worst["mix"], parity(xm, r, 1e-4, what) / max(1.0, float(r.abs().max())))
        parity(lm, rl, 1e-4, what + " log-det")
        x = r

    with torch.no_grad():
        zd, z2d = z.to(dev()), [t.to(dev()) for t in z2s]
        got, got_l = model.flow.decode_latents(zd, z2d, with_logdet=True)
        model.flow.fuse_squeeze = False
        try:
            got_u = model.flow.decode_latents(zd, z2d)
        finally:
            model.flow.fuse_squeeze = True
    assert torch.equal(got, got_u), "fused and unfused unsqueeze decode differ"
    ref, ref_l = O.flownet_decode(sd, z.double(), [t.double() for t in z2s], L, K_, "mixlogcdf")
    got = got.cpu().double()
    fin = torch.isfinite(ref)
    assert bool(torch.isfinite(got)[fin].all()), "%d non-finite images where the oracle's are finite" % int(
        (~torch.isfinite(got) & fin).sum())
    # reported, not bounded: every flat stretch of a mixture CDF that a layer lands in leaves x loosely pinned, and the
    # layers after it amplify that (the per-layer checks above bound each step)
    e2e = float(torch.where(fin, (got - ref).abs(), torch.zeros_like(ref)).max())
    in_range = fin & (ref.abs() <= 0.5)
    e2e_range = float(torch.where(in_range, (got - ref).abs(), torch.zeros_like(ref)).max())
    print("%s eps %g: worst coupling CDF %.2e dx %.2e log-det %.2e, fold %.2e, clamped %d; decode max|dx| %.2e "
          "(%.2e inside [-0.5, 0.5], max|x| %.3g), log-det %.2e vs %.3g, oracle non-finite %d"
          % (cfg, eps_std, worst["cdf"], worst["dx"], worst["ldj"], worst["mix"], worst["clamped"], e2e, e2e_range,
             float(ref[fin].abs().max()), float((got_l.cpu().double() - ref_l).abs().max()), float(ref_l.abs().max()),
             int((~fin).sum())))


# ---------------------------------------------------------------------------------------------
# 3. the graph lanes behind the headline numbers, replayed concurrently, against eager
# ---------------------------------------------------------------------------------------------
def test_graphed_sampler_lanes_match_eager(no_library):
    """Three GraphedSampler lanes (cfg2, B = 64) replayed interleaved without synchronising between them: every replay
    draws fresh latents in the graph, and its images equal, bit for bit, the eager decode of those latents with the same
    NaN / clamp post-processing."""
    B, image, L = 64, CONFIGS["cfg2"][0], CONFIGS["cfg2"][1]
    from flowk.graphs import GraphedSampler
    model = model_for("cfg2")
    lanes = [GraphedSampler(model, B, image) for _ in range(3)]
    recs = []
    for _ in range(6):
        for lane in lanes:
            lane.run()
            with torch.cuda.stream(lane.stream):            # the graph redraws these static buffers in place
                recs.append((lane.z.clone(), [t.clone() for t in lane.z2s], lane.images.clone()))
    torch.cuda.synchronize()
    for i in range(len(recs)):
        for j in range(i):
            assert not torch.equal(recs[i][0], recs[j][0]), "replays %d and %d drew the same z" % (j, i)
            for a, b in zip(recs[i][1], recs[j][1]):
                assert not torch.equal(a, b), "replays %d and %d drew the same factored-out latents" % (j, i)
    sd = None
    nan_images = 0
    with torch.no_grad():
        for i, (z, z2s, images) in enumerate(recs):
            x = model.flow.decode_latents(z, z2s)
            nan = torch.isnan(x)
            assert torch.equal(torch.clamp(torch.where(nan, torch.full_like(x, -0.5), x), -0.5, 0.5), images), \
                "replay %d: graphed images differ from the eager decode" % i
            if bool(nan.any()):                          # then the oracle must have them too
                rows = nan.flatten(1).any(1).nonzero().flatten().cpu()
                nan_images += len(rows)
                sd = sd or {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
                ref, _ = O.flownet_decode(sd, z[rows].cpu().double(), [t[rows].cpu().double() for t in z2s], L, 4,
                                          "mixlogcdf")
                assert bool((~torch.isfinite(ref))[nan[rows].cpu()].all()), "replay %d: NaN where the oracle is finite" % i
    print("GraphedSampler: %d replays on 3 lanes bit-identical to eager; images with NaN %d" % (len(recs), nan_images))


def test_density_pipeline_lanes_match_eager(no_library, monkeypatch):
    """DensityPipeline (cfg2, B = 64, three lanes; the path of bench.py's `value`): 8 distinct batches submitted
    round-robin, so the lanes replay concurrently and share the model, its operand caches and the per-(device, stream)
    log-det workspaces.  Each batch's z and bits/dim equal, bit for bit, the eager forward with the dequantisation noise
    that its replay drew, every replay draws fresh noise in [0, 1), and no two lanes share a log-det workspace."""
    from flowk import ops
    from flowk.graphs import DensityPipeline
    model = model_for("cfg2")
    B, image = 64, CONFIGS["cfg2"][0]
    gen = torch.Generator().manual_seed(31)
    xs = [(torch.rand(B, image[2], image[0], image[1], generator=gen) - 0.5).to(dev()) for _ in range(8)]
    captured = []                                          # the noise tensor each lane's graph writes at every replay;
    rand_like = torch.rand_like                            # holding it keeps the graph pool from reusing its memory

    def recording_rand_like(t, *args, **kw):
        out = rand_like(t, *args, **kw)
        if torch.cuda.is_current_stream_capturing():
            captured.append(out)
        return out
    with monkeypatch.context() as mp:
        mp.setattr(torch, "rand_like", recording_rand_like)
        pipe = DensityPipeline(model, xs[0], depth=3)
    assert len(captured) == 3
    # concurrent lanes must not share a log-det workspace (ops._workspace keeps one per (device, stream)): a shared one
    # gives wrong sums only when two lanes' reductions interleave, which the bit-exact check below may not catch
    workspaces = set()
    for stream in [lane.stream for lane in pipe.lanes] + [torch.cuda.current_stream()]:
        with torch.cuda.stream(stream):
            workspaces.add(ops._workspace(dev(), B).data_ptr())
    assert len(workspaces) == 4, "the pipeline's lanes and the eager forward share a log-det workspace"
    results = []

    def after(lane):                                       # runs on the lane's stream, right after its replay
        noise = captured[pipe.lanes.index(lane)]
        results.append((lane.static_z.clone(), lane.static_nll.clone(), noise.clone()))
    for x in xs:
        pipe.submit(x, after=after)
    pipe.drain()
    torch.cuda.synchronize()
    bad = []
    with torch.no_grad():
        for k, (x, (z, nll, noise)) in enumerate(zip(xs, results)):
            assert float(noise.min()) >= 0.0 and float(noise.max()) < 1.0
            for j in range(k):
                assert not torch.equal(noise, results[j][2]), "batches %d and %d drew the same noise" % (j, k)
            z_e, nll_e, _ = model(x, noise=noise)
            if not (torch.equal(z_e, z) and torch.equal(nll_e, nll)):
                bad.append((k, float((z_e - z).abs().max()), float((nll_e - nll).abs().max())))
    assert not bad, "%d of 8 batches differ from eager (batch, max|dz|, max|d bits/dim|): %s" % (len(bad), bad)
    print("DensityPipeline: 8 batches on 3 lanes bit-identical to eager")
