"""CUDA-graph capture of the forward (density) pass: at the named batch sizes every kernel of the
stack runs for microseconds, so the step is launch-bound unless the whole layer sequence is replayed
as one graph (streams and graphs instead of a tracing compiler)."""
import torch

from . import _lib


class GraphedDensity:
    """Captures `model(x)` -> (z, bits/dim) for a fixed input shape.  `run(x)` copies x into the static
    input (device or pinned-host source), replays, and returns the static outputs."""

    def __init__(self, model, example_x, inject_noise=False, warmup=3):
        assert example_x.is_cuda
        self.model = model
        self.static_x = example_x.clone()
        self.static_noise = torch.rand_like(example_x) if inject_noise else None
        self.stream = torch.cuda.Stream()               # replays run here, so several instances can overlap
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream), torch.no_grad():
            for _ in range(warmup):                     # fills the weight caches outside the graph
                model(self.static_x, noise=self.static_noise)
        torch.cuda.current_stream().wait_stream(self.stream)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        before = _lib.LAUNCHES
        with torch.no_grad(), torch.cuda.graph(self.graph, stream=self.stream):
            self.static_z, self.static_nll, _ = model(self.static_x, noise=self.static_noise)
        self.flowk_launches = _lib.LAUNCHES - before      # flowk kernels per replay

    def run(self, x=None):
        """Replay on the current stream."""
        if x is not None:
            self.static_x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.static_z, self.static_nll

    def run_async(self, x=None, out=None, after=None):
        """Replay on this instance's own stream (ordered after the caller's current stream); optionally copy the
        per-image bits/dim into `out` (pinned host tensor) and call `after(self)` on that stream (e.g. the bits/dim
        all-reduce).  Several instances replaying concurrently fill the SMs that one batch's deep-level kernels
        leave idle."""
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            if x is not None:
                self.static_x.copy_(x, non_blocking=True)
            self.graph.replay()
            if out is not None:
                out.copy_(self.static_nll, non_blocking=True)
            if after is not None:
                after(self)
        return self.static_z, self.static_nll


class DensityPipeline:
    """`depth` graph instances on separate streams, used round-robin: consecutive batches overlap on the GPU."""

    def __init__(self, model, example_x, depth=2):
        self.lanes = [GraphedDensity(model, example_x) for _ in range(depth)]
        self.i = 0
        self.flowk_launches = self.lanes[0].flowk_launches

    def submit(self, x, out=None, after=None):
        lane = self.lanes[self.i % len(self.lanes)]
        self.i += 1
        return lane.run_async(x, out, after)

    def drain(self):
        for lane in self.lanes:
            torch.cuda.current_stream().wait_stream(lane.stream)


class GraphedSampler:
    """The inverse pass (sampling, marscf_main.py:167-175 / save_samples :223-231) for a fixed batch size: latents for
    the final level and for every factored-out half are drawn from N(0, eps_std^2) IN the captured graph (fresh samples
    at every replay), pushed through `FlowNet.decode_latents`, NaNs replaced by -0.5 and the result clamped to the data
    range [-0.5, 0.5].  `run(out)` replays on this instance's stream and optionally copies the images to pinned host
    memory.

    With the mAR channel prior (`MarScfFlow(..., prior="mar")`) the latents depend on the decoded images' upper halves, so
    the graph runs the interleaved decode instead (`FlowNet.decode` with this instance's prior): sample the last level, decode
    it, and at every split sample z2 given the decoded z1.  Each level has its own `mar_prior.cuda_path.AncestralSampler`
    (own buffers, so instances replay concurrently) whose standard-normal noise `normal_` redraws in the graph.  That
    prior has no temperature (corr_prior.py:96-101), so eps_std != 1 raises ValueError.  `noise[level - 1]` is the
    [nc, B*H*W] noise buffer of a level, which the caller fills when `draw_noise=False`; `latents[level]` = (z1 or None,
    z2) of the last replay."""

    def __init__(self, model, batch, image_hwc, eps_std=1.0, warmup=2, draw_noise=True):
        from .mar_prior import ChannelPriorMultiScale
        flow = model.flow
        dev = next(model.parameters()).device
        h, w, c = image_hwc
        self.model, self.eps_std = model, float(eps_std)
        self.mar = isinstance(flow.c_prior, ChannelPriorMultiScale)
        if self.mar and self.eps_std != 1.0:
            raise ValueError("the mAR channel prior has no temperature: eps_std must be 1.0, got %g" % self.eps_std)
        self.draw_noise = draw_noise
        self.stream = torch.cuda.Stream()
        self.stream.wait_stream(torch.cuda.current_stream())
        shapes = []                                  # factored-out halves, in split order, then the final latent
        for lvl in range(flow.L):
            c, h, w = c * 4, h // 2, w // 2
            if lvl < flow.L - 1:
                c //= 2
                shapes.append((batch, c, h, w))
        with torch.cuda.stream(self.stream), torch.no_grad():
            if self.mar:
                from .mar_prior import cuda_path
                self.samplers = [cuda_path.AncestralSampler(p, batch, dev) for p in flow.c_prior.prior_list]
                self.noise = [s.noise for s in self.samplers]
                self.latents = {}
            else:
                self.z = torch.empty(batch, c, h, w, device=dev)
                self.z2s = [torch.empty(s, device=dev) for s in shapes]
            for _ in range(warmup):
                self._sample(flow)
        torch.cuda.current_stream().wait_stream(self.stream)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        before = _lib.LAUNCHES
        with torch.no_grad(), torch.cuda.graph(self.graph, stream=self.stream):
            self.images = self._sample(flow)
        self.flowk_launches = _lib.LAUNCHES - before

    def _mar_prior(self, z, level, reverse=True, **kw):
        sampler = self.samplers[level - 1]
        if self.draw_noise:
            sampler.noise.normal_()
        z2 = sampler.sample(z)
        self.latents[level] = (z, z2)
        return z2

    def _sample(self, flow):
        if self.mar:
            x = flow.decode(None, prior=self._mar_prior)
        else:
            for t in [self.z] + self.z2s:
                t.normal_(0.0, self.eps_std)
            x = flow.decode_latents(self.z, self.z2s)
        x = torch.where(torch.isnan(x), torch.full_like(x, -0.5), x)
        return torch.clamp(x, -0.5, 0.5)

    def run(self, out=None):
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            self.graph.replay()
            if out is not None:
                out.copy_(self.images, non_blocking=True)
        return self.images
