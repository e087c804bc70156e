"""Drop-in module mirror of the reference's model classes for the NVF path.

Same class names, constructor arguments, state_dict keys/shapes and forward
signatures as the reference (utils/network.py:564-742 conv wrappers, :4490-4545
QuantGaussianLikelihood, :4592-4612 SingleLayerLatentGen, :4648-4799
CompDecoder, gdn_3d.py GDN3d/IGDN3d, NVFPCC.py:32-74 Net), so that
`NVFPCC.py` changes by one import (INTEGRATION.md) and reference checkpoints,
quantised checkpoints (manipulate_weights.py) and pack.pk weight pools load
unchanged.

What runs where:
* the conv stack, IGDN, sigmoid heads, thresholding and their backward run in
  the hand-written CUDA kernels (nvfpcc_b200.ops);
* the tiny parameter-side transforms stay in torch so autograd semantics are
  identical (SURVEY.md 8b): kernel noise / straight-through round16 +
  kernel_init, b + b_init, GDN reparametrisation with LowerBound, the
  24-floats-per-block latent head and both Gaussian rate models.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops

# ---------------------------------------------------------------------------
# shared seed stream (the reference reads SEED3.npy from the CWD at import time,
# utils/network.py:20-22, and advances a module-global pointer while building)
# ---------------------------------------------------------------------------
SEED2: Optional[np.ndarray] = None
seed_ptr = 0


def set_seed(seed, reset_ptr: bool = True) -> None:
    """Install the seed stream (an array or a path to SEED3.npy)."""
    global SEED2, seed_ptr
    SEED2 = np.load(seed) if isinstance(seed, (str, os.PathLike)) else np.asarray(seed)
    if reset_ptr:
        seed_ptr = 0


def _seed() -> np.ndarray:
    global SEED2
    if SEED2 is None:
        if not os.path.isfile("SEED3.npy"):
            raise FileNotFoundError("SEED3.npy not found in the working directory; call nvfpcc_b200.network.set_seed()")
        SEED2 = np.load("SEED3.npy")
    return SEED2


# ---------------------------------------------------------------------------
# straight-through / bounded primitives
# ---------------------------------------------------------------------------
class _STE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, scale):
        return torch.round(x * scale) / scale

    @staticmethod
    def backward(ctx, g):
        return g, None


def bypass_round(x):      # utils/network.py:25-32
    return _STE.apply(x, 1.0)


def bypass_round16(x):    # utils/network.py:43-50
    return _STE.apply(x, 16.0)


class _LowerBoundFn(torch.autograd.Function):
    """clamp(min=bound); gradient passes where x >= bound or it pushes x up (utils/network.py:56-72)."""

    @staticmethod
    def forward(ctx, x, bound):
        ctx.save_for_backward(x)
        ctx.bound = float(bound)
        return x.clamp(min=ctx.bound)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return g * ((x >= ctx.bound) | (g < 0)), None


lower_bound = _LowerBoundFn.apply


def _seeded_uniform(shape, seed_slice, bound):
    s = torch.from_numpy(np.asarray(seed_slice).reshape(shape)).float()
    return (s - 0.5) * 2 * bound


class _SeededConvBase(nn.Module):
    """Parameter container shared by the three conv wrappers: zero-initialised trainable
    `kernel`/`b` (the transmitted delta) + `kernel_init`/`b_init` buffers cut from the seed
    stream (utils/network.py:579-604, 637-667, 704-733)."""

    def __init__(self, kshape, n_bias, bias_fan, SEED, quantised: bool):
        super().__init__()
        n = int(np.prod(kshape))
        fan_in = kshape[1] * int(np.prod(kshape[2:]))          # dim 1, whatever the layout (:377-389)
        bound = math.sqrt(3.0) * math.sqrt(2.0) / math.sqrt(fan_in)
        self.register_buffer("kernel_init", _seeded_uniform(kshape, SEED[:n], bound))
        self.register_parameter("kernel", nn.Parameter(torch.zeros(kshape)))
        self.register_buffer("b_init", _seeded_uniform((n_bias,), SEED[n:n + n_bias], 1 / math.sqrt(bias_fan)))
        self.register_parameter("b", nn.Parameter(torch.zeros(n_bias)))
        self.offset = n + n_bias
        self.quantised = quantised
        self.Q = 1 / 16

    def effective(self, q: int = 0):
        """(W_eff, b_eff): q==1 additive U(-1/32,1/32) noise, q==2 straight-through round16
        (utils/network.py:606-620); IConv3d ignores q (:735-741)."""
        k = self.kernel
        if self.quantised:
            if q == 1:
                k = k + (torch.rand_like(k) - 0.5) * self.Q
            elif q == 2:
                k = bypass_round16(k)
        return k + self.kernel_init, self.b + self.b_init


class QConvTranspose3d(_SeededConvBase):
    def __init__(self, in_channels, out_channels, kernel_size, stride, bias, padding=0, output_padding=0, iQ=16,
                 SEED=None, groups=1, zero_bias=False):
        assert groups == 1 and bias and not zero_bias and iQ == 16
        super().__init__((in_channels, out_channels) + (kernel_size,) * 3, out_channels, in_channels, SEED, True)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding, self.output_padding = kernel_size, stride, padding, output_padding


class QConv3d(_SeededConvBase):
    def __init__(self, in_channels, out_channels, kernel_size, stride, bias, padding=0, iQ=16, SEED=None, groups=1,
                 zero_bias=False):
        assert groups == 1 and bias and not zero_bias and iQ == 16
        super().__init__((out_channels, in_channels) + (kernel_size,) * 3, out_channels, in_channels, SEED, True)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding = kernel_size, stride, padding


class IConv3d(_SeededConvBase):
    def __init__(self, in_channels, out_channels, kernel_size, stride, bias, padding=0, SEED=None, groups=1,
                 zero_bias=False):
        assert groups == 1 and bias and not zero_bias
        super().__init__((out_channels, in_channels) + (kernel_size,) * 3, out_channels, in_channels, SEED, False)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding = kernel_size, stride, padding

    def forward(self, x):
        w, b = self.effective()
        return F.conv3d(x, w, b, self.stride, self.padding)


class _GDNBase(nn.Module):
    """gdn_3d.py:32-69 / 97-134 parameters: beta (ch), gamma (ch,ch), pedestal buffer."""

    def __init__(self, ch, inverse=False, beta_min=1e-6, gamma_init=.1, reparam_offset=2 ** -18):
        super().__init__()
        ped = reparam_offset ** 2
        self.reparam_pedestal = ped
        self.beta_bound = (beta_min + ped) ** .5
        self.gamma_bound = reparam_offset
        self.beta = nn.Parameter(torch.sqrt(torch.ones(ch) + ped))
        self.gamma = nn.Parameter(torch.sqrt(gamma_init * torch.eye(ch) + ped))
        self.register_buffer("pedestal", torch.FloatTensor([ped]))

    def effective(self):
        """(beta_eff, gamma_eff) = (max(beta,bound)^2 - pedestal, max(gamma,bound)^2 - pedestal)."""
        b = lower_bound(self.beta, self.beta_bound) ** 2 - self.pedestal
        g = lower_bound(self.gamma, self.gamma_bound) ** 2 - self.pedestal
        return b, g

    def _norm(self, x):
        b, g = self.effective()
        ch = x.shape[1]
        return torch.sqrt(F.conv3d(x * x, g.view(ch, ch, 1, 1, 1), b))


class GDN3d(_GDNBase):
    def forward(self, x):           # gdn_3d.py:88-92 (24 floats per block: stays in torch)
        return x / self._norm(x)


class IGDN3d(_GDNBase):
    def forward(self, x):           # gdn_3d.py:153-157 (the decoder's IGDN runs inside the CUDA kernels)
        return x * self._norm(x)


class GaussianModel(nn.Module):
    """utils/network.py:139-169."""

    def __init__(self, qp=1):
        super().__init__()
        self.qp = qp

    def forward(self, inputs, sigma, mu):
        half = 0.5 * self.qp
        nd = torch.distributions.normal.Normal(0., 1., validate_args=False)   # argument validation would sync the host
        lik = nd.cdf((inputs - mu + half) / sigma) - nd.cdf((inputs - mu - half) / sigma)
        lik = lower_bound(lik, 1e-8)
        return (-1 * torch.log(lik) / np.log(2)).sum()


class GaussianLikelihoodModel(nn.Module):
    """utils/network.py:287-305: bits of a (quantised) kernel under a scalar Gaussian."""

    def __init__(self, step_size=1):
        super().__init__()
        self.gaussian_model = GaussianModel(step_size)
        self.sigma = nn.Parameter(torch.ones(1))
        self.mu = nn.Parameter(torch.zeros(1))

    def forward(self, x):
        return self.gaussian_model(x.reshape(-1, 1), torch.abs(self.sigma), self.mu).sum()


class QuantGaussianLikelihood(nn.Module):
    """utils/network.py:4490-4545: straight-through rounding of the latent + its rate."""

    def __init__(self, in_channels, step_size=1, iQ=1, assume_zero_mean=False):
        super().__init__()
        assert iQ == 1 and not assume_zero_mean
        self.gaussian_model = GaussianModel(step_size)
        self.sigma = nn.Parameter(torch.ones(1, in_channels, 1, 1, 1))
        self.mu = nn.Parameter(torch.zeros(1, in_channels, 1, 1, 1))
        self.noise_scale = 1.0                    # tests set 0 for run-to-run comparable steps

    def forward(self, x, mode='train'):
        noise = (torch.rand_like(x) - 0.5) * self.noise_scale   # drawn in both modes, like the reference (:4516)
        x_rounded = bypass_round(x)
        x_form = x + noise if mode == 'train' else x_rounded
        return x_rounded, self.gaussian_model(x_form, torch.abs(self.sigma), self.mu)

    def get_bits(self):
        return int(np.prod(self.sigma.shape) * 32 + np.prod(self.mu.shape) * 32)


class SingleLayerLatentGen(nn.Module):
    """utils/network.py:4592-4612: 1x1x1 conv + GDN on the embedding."""

    def __init__(self, in_channels=8, out_channels=4):
        super().__init__()
        global seed_ptr
        self.h_analysis_2 = IConv3d(in_channels, out_channels, 1, 1, True, 0, SEED=_seed()[seed_ptr:])
        seed_ptr += self.h_analysis_2.offset
        self.gdn_2 = GDN3d(out_channels)

    def forward(self, x):
        return self.gdn_2(self.h_analysis_2(x))


class CompDecoder(nn.Module):
    """The NVF decoder (utils/network.py:4648-4799) with its conv stack on the GPU kernels.

    forward(x, q) -> (out, [cls0, cls1, out], net_bits)           (:4758-4779)
    reconstruct(x, q) -> out                  fused decode kernel, no aux heads, no net_bits
    decode_points(x, origins, thh, q) -> dict(coords, counts)     (NVFPCC.py:625-638 batched)
    """

    def __init__(self, args, param_model, in_channels=4, useIGDN=False, channels=(8, 16, 8, 8)):
        super().__init__()
        global seed_ptr
        if not useIGDN:
            raise NotImplementedError("the NVF path is built for useIGDN=True (NVFPCC.py:39)")
        c0, c1, c2, c3 = (int(c) for c in channels)
        self.channels = (c0, c1, c2, c3)
        self.in_channels = int(in_channels)
        self.useIGDN = useIGDN
        self.activation = IGDN3d(c0)
        S = _seed()

        def take(mod):
            global seed_ptr
            seed_ptr += mod.offset
            return mod

        self.up0 = take(QConvTranspose3d(in_channels, c0, 5, 2, True, padding=2, output_padding=1, SEED=S[seed_ptr:]))
        self.conv0 = take(QConvTranspose3d(c0, c1, 5, 2, True, padding=2, output_padding=1, SEED=S[seed_ptr:]))
        self.up1 = take(QConvTranspose3d(c1, c2, 5, 2, True, SEED=S[seed_ptr:]))
        self.conv1 = take(QConv3d(c2, c2, 4, 1, True, padding=0, SEED=S[seed_ptr:]))
        self.up2 = take(QConvTranspose3d(c2, c3, 5, 2, True, SEED=S[seed_ptr:]))
        self.conv2 = take(QConv3d(c3, c3, 4, 1, True, padding=0, SEED=S[seed_ptr:]))
        self.conv2_cls = take(QConv3d(c3, 1, 3, 1, True, padding=1, SEED=S[seed_ptr:]))
        self.conv1_cls = take(IConv3d(c2, 1, 3, 1, True, padding=1, SEED=S[seed_ptr:]))
        self.conv0_cls = take(IConv3d(c1, 1, 3, 1, True, padding=1, SEED=S[seed_ptr:]))
        self.likelihood_model = GaussianLikelihoodModel(step_size=1 / 16)

    # -- effective tensors handed to the C ABI ---------------------------------
    def effective_weights(self, q: int, aux: bool = True) -> Dict[str, torch.Tensor]:
        w: Dict[str, torch.Tensor] = {}
        for key, name in _lib.CONV_MODULES.items():
            if aux or key not in ("cls1", "cls0"):
                w[key + "_w"], w[key + "_b"] = getattr(self, name).effective(q)
        w["igdn_beta"], w["igdn_gamma"] = self.activation.effective()
        return w

    def get_q_params(self) -> List[torch.Tensor]:
        return [getattr(self, name).kernel for name in list(_lib.CONV_MODULES.values())[:_lib.NVF_NUM_QUANT]]

    def net_bits(self) -> torch.Tensor:
        return torch.stack([self.likelihood_model(bypass_round16(p)) for p in self.get_q_params()])

    def raw_tensors(self) -> Dict[str, torch.Tensor]:
        """The trainable tensors + seed buffers the fused parameter kernels read (ops.RAW_FIELDS)."""
        raw: Dict[str, torch.Tensor] = {}
        for key, name in _lib.CONV_MODULES.items():
            m = getattr(self, name)
            raw[key + "_kernel"], raw[key + "_kernel_init"], raw[key + "_b"], raw[key + "_b_init"] = (
                m.kernel, m.kernel_init, m.b, m.b_init)
        raw["igdn_beta"], raw["igdn_gamma"] = self.activation.beta, self.activation.gamma
        raw["lik_sigma"], raw["lik_mu"] = self.likelihood_model.sigma, self.likelihood_model.mu
        return raw

    def forward(self, x, q):
        if x.is_cuda:
            # one fused kernel pair for every parameter-side transform + net_bits (nvf_param_prep)
            w, net_bits = ops.decoder_params(self.in_channels, self.channels, q, self.raw_tensors(),
                                             self.activation.beta_bound, self.activation.gamma_bound,
                                             float(self.activation.reparam_pedestal))
        else:
            w, net_bits = self.effective_weights(q), self.net_bits()
        out, cls1, cls0 = ops.nvf_decoder(self.in_channels, self.channels, x, w)
        return out, [cls0, cls1, out], net_bits

    def _decode_weights(self, q):
        """Effective tensors for the decode-only calls: on the GPU one fused parameter kernel (nvf_param_prep, the same
        arithmetic as `effective_weights`: round(k*16)/16 + kernel_init is exact) instead of ~150 elementwise launches."""
        if self.up0.kernel.is_cuda and q != 1:
            w, _ = ops.decoder_params(self.in_channels, self.channels, q, self.raw_tensors(), self.activation.beta_bound,
                                      self.activation.gamma_bound, float(self.activation.reparam_pedestal))
            return w
        return self.effective_weights(q, aux=False)

    @torch.no_grad()
    def reconstruct(self, x, q=2):
        r = ops.decode_blocks(self.in_channels, self.channels, self._decode_weights(q), x, None, 2.0,
                              return_prob=True, return_host=False)
        return r["prob"]

    @torch.no_grad()
    def decode_points(self, x, origins, thh, q=2, return_prob=False, return_host=None, timing=None):
        return ops.decode_blocks(self.in_channels, self.channels, self._decode_weights(q), x, origins,
                                 thh, return_prob=return_prob, return_host=return_host, timing=timing)

    def get_bits(self):
        aux_bits = sum(self.channels[i] * 2 for i in (1, 2, 3)) * 32 + 32 + (self.channels[1] ** 2 + self.channels[1]) * 32
        return self.net_bits().sum().item() + aux_bits


class Net(nn.Module):
    """NVFPCC.py:32-74."""

    def __init__(self, args, param_model, ch=4, channel_str='8,16,8,8') -> None:
        super().__init__()
        channels = tuple(int(c) for c in str(channel_str).split(','))
        self.latent_gen = SingleLayerLatentGen(in_channels=ch, out_channels=ch)
        self.entropy_coder = QuantGaussianLikelihood(in_channels=ch)
        self.reconstructor = CompDecoder(args, param_model, useIGDN=True, in_channels=ch, channels=channels)

    def latent_raw(self) -> Dict[str, torch.Tensor]:
        """The tensors the fused latent-head kernels read (_lib.LATENT_FIELDS)."""
        h, g, e = self.latent_gen.h_analysis_2, self.latent_gen.gdn_2, self.entropy_coder
        return dict(kernel=h.kernel, kernel_init=h.kernel_init, b=h.b, b_init=h.b_init, gdn_beta=g.beta,
                    gdn_gamma=g.gamma, sigma=e.sigma, mu=e.mu)

    def latent_head(self, emb, mode):
        """latent_gen -> entropy_coder: (rounded latent, summed rate).  One fused kernel on the GPU."""
        ch = self.reconstructor.in_channels
        if emb.is_cuda and ch <= 4:
            g = self.latent_gen.gdn_2
            noise = torch.rand_like(emb)                       # drawn in both modes, like the reference (:4516)
            return ops.latent_head(ch, emb, self.latent_raw(), mode, noise, self.entropy_coder.noise_scale,
                                   g.beta_bound, g.gamma_bound, float(g.reparam_pedestal))
        return self.entropy_coder(self.latent_gen(emb), mode)

    def forward(self, emb, mode, q):
        latent_rounded, latent_likelihood = self.latent_head(emb, mode)
        out, out_cls_list, net_bits = self.reconstructor(latent_rounded, q)
        return out, out_cls_list, net_bits, latent_likelihood

    def reconstruct(self, latent, q):
        return self.reconstructor.reconstruct(latent, q)

    def decode_points(self, latent, origins, thh, q=2, **kw):
        """Batched replacement of the loop body of decode() (NVFPCC.py:625-638)."""
        return self.reconstructor.decode_points(latent, origins, thh, q, **kw)

    def get_network_bits(self):
        return self.entropy_coder.get_bits() + self.reconstructor.get_bits()

    def get_latent_bits(self, all_emb):
        _, lik = self.entropy_coder(self.latent_gen(all_emb), mode='eval')
        return lik.sum()

    def get_latent_code(self, all_emb):
        q, lik = self.entropy_coder(self.latent_gen(all_emb), mode='eval')
        return {'quantized_latent': q, 'sigma': torch.abs(self.entropy_coder.sigma), 'mu': self.entropy_coder.mu,
                'latent_likelihood': lik}

    def get_bits(self, all_emb):
        return self.get_latent_bits(all_emb), self.get_network_bits()


class MultiscaleProcessor(nn.Module):
    """NVFPCC.py:76-88 (kept for callers that still want the GT pyramid; ops.rd_distortion pools in-kernel)."""

    def forward(self, x):
        x1 = F.max_pool3d(x, 2, 2)
        return [F.max_pool3d(x1, 2, 2), x1, x]
