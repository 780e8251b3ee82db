"""mAR channel prior (mar_prior/corr_prior.py:7-182) with the reference's names and state-dict keys: every latent
channel is Gaussian with mean / log-std predicted by a ConvLSTM from the previous channels (and, at a split, from an
embedding of the half that continues through the flow).  Plugs into `flowk.marscf.FlowNet(prior=...)`, which calls it
like the reference's `c_prior(z, level, reverse=...)`.

On CUDA tensors with autograd off (evaluation, sampling) the networks run on the flowk tensor-core kernels
(`mar_prior/cuda_path.py`: every conv a tcgen05 implicit GEMM, the LSTM cell fused into the recurrent GEMM's epilogue;
sampling through `AncestralSampler`, 2 + num_layers launches per channel).  Training (autograd on, dp_rate = 0 or eval
mode) runs on them too, with backward through time on flowk kernels (`cuda_path.run_sequence_train`); training with
channel dropout, shapes the kernels do not take and CPU tensors use the torch layers below."""
import numpy as np
import torch
import torch.nn as nn

from . import cuda_path
from .lstm import ConvSeqEncoder

_KERNEL_SIZES = [5, 5, 3, 3, 3, 3, 3]        # corr_prior.py:24-25, indexed by level - 1
_DILATIONS = [2, 1, 1, 1, 1, 1, 1]


class ChannelPriorUniScale(nn.Module):
    def __init__(self, batch_size, nc, height, width, level, tot_levels, hidden_size=32, num_layers=1, dp_rate=0.2,
                 plot=False):
        super().__init__()
        self.batch_size = batch_size
        self.height, self.width = height // (2 ** level), width // (2 ** level)
        self.nc = nc * 2 ** level if level != tot_levels else nc * 2 ** (level + 1)
        self.z1_cond_network = nn.Sequential(nn.Conv2d(self.nc, 32, 5, stride=1, padding=2), nn.ReLU(),
                                             nn.Conv2d(32, 4, 5, stride=1, padding=2))
        self.prior_lstm = ConvSeqEncoder(input_ch=5 if level != tot_levels else 1, out_ch=2,
                                         kernel_size=_KERNEL_SIZES[level - 1], dilation=_DILATIONS[level - 1],
                                         embed_ch=hidden_size, num_layers=num_layers, dropout=dp_rate)
        self.Log2PI = float(np.log(2 * np.pi))
        self.dp_rate, self.level, self.tot_levels = dp_rate, level, tot_levels
        self.cond_dropout = nn.Dropout2d(dp_rate)

    def dropout_in(self, z2):
        """Channel dropout of the teacher-forced inputs (corr_prior.py:48-52); the mask is drawn on the host as in the
        reference, and is a no-op for dp_rate = 0 (the setting marscf_main.py:147 uses)."""
        prob = torch.rand(z2.size(0), z2.size(1))
        if self.dp_rate > 0:
            z2[(prob < self.dp_rate).to(z2.device)] = 0
        return z2

    def likelihood(self, mean, logs, z):
        return -0.5 * (logs * 2. + ((z - mean) ** 2) / torch.exp(logs * 2.) + self.Log2PI)

    def get_likelihood(self, z):
        zz = z[1] if isinstance(z, (tuple, list)) else z
        no_dropout = not (self.training and self.dp_rate > 0)
        fast = cuda_path.usable(self, zz) and no_dropout
        train = not fast and no_dropout and cuda_path.trainable(self, zz)
        if isinstance(z, (tuple, list)):
            z1, z2 = z
            if fast:
                emb = cuda_path.z1_embedding(self.z1_cond_network, z1)
            elif train:
                emb = cuda_path.z1_embedding_train(self.z1_cond_network, z1)
            else:
                emb = self.z1_cond_network(z1)
            z1_embd = emb.unsqueeze(1).repeat(1, z2.size(1), 1, 1, 1)
        else:
            z1_embd, z2 = None, z
        z2 = z2.unsqueeze(2)                                            # [B, T = channels, 1, H, W]
        zero = z2.new_zeros(z2.size(0), 1, 1, z2.size(3), z2.size(4))
        lstm_input = torch.cat([zero, self.dropout_in(z2.clone())[:, :-1]], dim=1)      # teacher forcing
        if z1_embd is not None:
            lstm_input = torch.cat([lstm_input, z1_embd], dim=2)
        if fast:
            out = cuda_path.run_sequence(self.prior_lstm, lstm_input)
        elif train:
            out = cuda_path.run_sequence_train(self.prior_lstm, lstm_input)
        else:
            out, _ = self.prior_lstm(lstm_input, None)
        return torch.sum(self.likelihood(out[:, :, 0:1], out[:, :, 1:2], z2), dim=(1, 2, 3, 4))

    def get_sample(self, z1=None, batch_size=None, device=None):
        with torch.no_grad():
            fast = cuda_path.usable(self, z1 if z1 is not None else
                                    torch.empty(1, 1, self.height, self.width, device=device or next(self.parameters()).device))
            if fast:
                b = z1.size(0) if z1 is not None else batch_size or self.batch_size
                sampler = cuda_path.sampler_for(self, b, z1.device if z1 is not None else device or next(self.parameters()).device)
                # the reference's host-side draws (corr_prior.py:96-101), one per channel in its order, copied once
                noise = torch.stack([torch.randn(b, 1, 1, self.height, self.width) for _ in range(self.nc)])
                return sampler.sample(z1, noise)
            if z1 is not None:
                z1_embd = self.z1_cond_network(z1).unsqueeze(1)
                b, device = z1.size(0), z1.device
                lstm_input = torch.cat([z1.new_zeros(b, 1, 1, self.height, self.width), z1_embd], dim=2)
            else:
                b = batch_size or self.batch_size
                device = device or next(self.parameters()).device
                z1_embd = None
                lstm_input = torch.zeros(b, 1, 1, self.height, self.width, device=device)
            hidden, chans = None, []
            for _ in range(self.nc):
                out, hidden = self.prior_lstm(lstm_input, None, hidden)
                mean, logs = out[:, :, 0:1], out[:, :, 1:2]
                sample = torch.randn(mean.size()).to(device) * torch.exp(logs) + mean       # corr_prior.py:96-101
                chans.append(sample)
                lstm_input = sample if z1_embd is None else torch.cat([sample, z1_embd], dim=2)
            return torch.cat(chans, dim=1).squeeze(2)

    def forward(self, z, reverse=False, **kw):
        if not reverse:
            return self.get_likelihood(z)
        if z is None:
            return self.get_sample(None, **kw)
        return self.get_sample(z[0] if isinstance(z, (tuple, list)) else z)


class ChannelPriorMultiScale(nn.Module):
    def __init__(self, batch_size, nc, height, width, levels, hidden_size=32, dp_rate=0., num_layers=2, mog=False):
        super().__init__()
        if mog:
            raise NotImplementedError
        self.prior_list = nn.ModuleList([
            ChannelPriorUniScale(batch_size, nc, height, width, level, levels, hidden_size=hidden_size,
                                 num_layers=num_layers, dp_rate=dp_rate) for level in range(1, levels + 1)])

    def get_likelihood(self, z, level, hidden=None):
        return self.prior_list[level - 1](z, reverse=False)

    def get_sample(self, z, level, hidden=None, **kw):
        return self.prior_list[level - 1](z, reverse=True, **kw)

    def forward(self, z, level, reverse=False, eps_std=None, batch_size=None, device=None):
        if not reverse:
            return self.get_likelihood(z, level)
        if z is None:
            return self.get_sample(None, level, batch_size=batch_size, device=device)
        return self.get_sample(z, level)
