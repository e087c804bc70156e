"""Public ops of the B200 NVF path (PyTorch-facing side of the C ABI).

* `decode_blocks`   - batched replacement of the per-block loop in decode()/encode()
                      (NVFPCC.py:625-638, :505-539): latents -> ordered points.
* `nvf_decoder`     - differentiable CompDecoder.forward on effective tensors
                      (utils/network.py:4758-4768) -> (out, cls1, cls0).
* `rd_distortion`   - differentiable fused distortion losses + metrics
                      (utils/loss.py:61-121, NVFPCC.py:76-88,166-184).

All ops run hand-written sm_100a kernels through `libnvf_b200.so`; there is no
CPU implementation and no fallback: without a CUDA device they raise.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import torch

from . import _lib
from ._lib import WEIGHT_FIELDS, NvfError


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise NvfError("nvfpcc_b200 needs a CUDA (sm_100a) device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _to_dev(t: Optional[torch.Tensor], dev: torch.device, dtype=None):
    if t is None:
        return None
    return t.to(device=dev, dtype=dtype if dtype is not None else t.dtype, non_blocking=True)


def decode_blocks(ch: int, channels: Sequence[int], weights: Dict[str, torch.Tensor], latents: torch.Tensor,
                  origins: Optional[torch.Tensor], thh: float, return_prob: bool = False,
                  return_host: Optional[bool] = None, timing: Optional[list] = None):
    """latents [N,ch,2,2,2] (rounded), origins [N,3] -> dict(coords int32 [K,3], counts int32 [N], prob?).

    Inputs may live on the host (ideally pinned) or on the device; host inputs are
    copied in and, unless `return_host=False`, results are copied back.  Point
    order: block order, then row-major (i,j,k), as NVFPCC.py:631-638 emits."""
    dev = _device()
    b = _lib.cuda_binding()
    host_in = latents.device.type != "cuda"
    if return_host is None:
        return_host = host_in
    w = {k: _to_dev(v, dev, torch.float32) for k, v in weights.items()}
    r = b.decode(b.desc(ch, channels), w, _to_dev(latents, dev, torch.float32),
                 _to_dev(origins, dev, torch.int32), thh, want_prob=return_prob, timing=timing)
    out = dict(coords=r["coords"], counts=r["counts"], prob=r["prob"], mask=r["mask"])
    if return_host:
        out = {k: (None if v is None else v.cpu()) for k, v in out.items()}
    return out


class _NvfDecoderFn(torch.autograd.Function):
    """forward: nvf_train_forward; backward: nvf_train_backward.  Inputs: latent, then the 20
    effective tensors in WEIGHT_FIELDS order (plus two python flags)."""

    @staticmethod
    def forward(ctx, ch, channels, latent, *ws):
        b = _lib.cuda_binding()
        if latent.device.type != "cuda":
            raise NvfError("nvf_decoder needs CUDA tensors; there is no CPU fallback")
        weights = dict(zip(WEIGHT_FIELDS, ws))
        desc = b.desc(ch, channels)
        out, cls1, cls0, wsbuf, _ = b.train_forward(desc, weights, latent)
        ctx.desc_args = (ch, tuple(channels))
        ctx.wsbuf = wsbuf
        ctx.save_for_backward(latent, *ws)
        return out, cls1, cls0

    @staticmethod
    def backward(ctx, g_out, g_cls1, g_cls0):
        b = _lib.cuda_binding()
        latent, *ws = ctx.saved_tensors
        weights = dict(zip(WEIGHT_FIELDS, ws))
        need_lat = ctx.needs_input_grad[2]
        need_w = any(ctx.needs_input_grad[3:])
        ch, channels = ctx.desc_args
        g_lat, grads = b.train_backward(b.desc(ch, channels), weights, latent, ctx.wsbuf, g_out, g_cls1, g_cls0,
                                        need_w, need_lat)
        ctx.wsbuf = None
        gw = tuple(grads.get(k) if ctx.needs_input_grad[3 + i] else None for i, k in enumerate(WEIGHT_FIELDS))
        return (None, None, g_lat) + gw


def nvf_decoder(ch: int, channels: Sequence[int], latent: torch.Tensor, weights: Dict[str, torch.Tensor]):
    """Differentiable decoder on effective tensors -> (out [N,1,32^3], cls1 [N,1,16^3], cls0 [N,1,8^3])."""
    return _NvfDecoderFn.apply(int(ch), tuple(int(c) for c in channels), latent, *[weights[k] for k in WEIGHT_FIELDS])


class _RdDistortionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, out, cls1, cls0, gt, dist, alpha_main, alpha_aux, thh_metric):
        b = _lib.cuda_binding()
        if out.device.type != "cuda":
            raise NvfError("rd_distortion needs CUDA tensors; there is no CPU fallback")
        need = any(t.requires_grad for t in (out, cls1, cls0))
        sums, seeds = b.loss_seeds(out, cls1, cls0, gt, dist, alpha_main, alpha_aux, thh_metric, want_seeds=need)
        ctx.save_for_backward(*[s for s in seeds if s is not None])
        ctx.have = need
        ctx.mark_non_differentiable(sums)
        f = sums[:3].to(torch.float32)
        return f[0], f[1], f[2], sums

    @staticmethod
    def backward(ctx, g_bce, g_ms0, g_ms1, _g_sums):
        if not ctx.have:
            return (None,) * 8
        s_out, s_cls1, s_cls0 = ctx.saved_tensors
        return s_out * g_bce, s_cls1 * g_ms1, s_cls0 * g_ms0, None, None, None, None, None


def rd_distortion(out, cls1, cls0, gt, dist, alpha_main: float = 0.9, alpha_aux: float = 0.85,
                  thh_metric: float = 0.6):
    """-> (bce, ms0, ms1, sums[20] float64).  bce = get_surf_focal_dense(out, gt, dist, beta=1, alpha_main);
    ms0/ms1 = get_focal_dense on the 8^3 / 16^3 heads against max-pooled GT (NVFPCC.py:166-184);
    sums: see include/nvf_b200.h (sse/denom at thh_metric, tp/ap/tn/an of each head at 0.5)."""
    return _RdDistortionFn.apply(out, cls1, cls0, gt, dist, float(alpha_main), float(alpha_aux), float(thh_metric))


class _LatentHeadFn(torch.autograd.Function):
    """forward: nvf_latent_forward; backward: nvf_latent_backward.  Inputs after the python
    arguments: emb, then the 8 raw tensors in _lib.LATENT_FIELDS order."""

    @staticmethod
    def forward(ctx, ch, train, noise_scale, bounds, noise, emb, *raw):
        b = _lib.cuda_binding()
        if emb.device.type != "cuda":
            raise NvfError("latent_head needs CUDA tensors; there is no CPU fallback")
        rawd = dict(zip(_lib.LATENT_FIELDS, raw))
        latent, bits = b.latent_forward(ch, rawd, emb, noise, noise_scale, train, bounds)
        ctx.args = (ch, train, noise_scale, bounds)
        ctx.noise = noise
        ctx.save_for_backward(emb, *raw)
        return latent, bits.reshape(())

    @staticmethod
    def backward(ctx, g_latent, g_bits):
        b = _lib.cuda_binding()
        emb, *raw = ctx.saved_tensors
        rawd = dict(zip(_lib.LATENT_FIELDS, raw))
        ch, train, noise_scale, bounds = ctx.args
        want_emb = ctx.needs_input_grad[5]
        want_params = any(ctx.needs_input_grad[6:])
        if g_bits is None:
            g_bits = torch.zeros(1, device=emb.device)
        grads, g_emb = b.latent_backward(ch, rawd, emb, ctx.noise, noise_scale, train, bounds, g_latent, g_bits,
                                         want_params, want_emb)
        ctx.noise = None
        out = []
        for i, f in enumerate(_lib.LATENT_FIELDS):
            g = None
            if grads is not None and f in grads and ctx.needs_input_grad[6 + i]:
                g = grads[f].view_as(raw[i])
            out.append(g)
        return (None, None, None, None, None, g_emb) + tuple(out)


def latent_head(ch: int, emb: torch.Tensor, raw: Dict[str, torch.Tensor], mode: str, noise: Optional[torch.Tensor],
                noise_scale: float, beta_bound: float, gamma_bound: float, pedestal: float):
    """Fused SingleLayerLatentGen + QuantGaussianLikelihood (see include/nvf_b200.h nvf_latent_forward):
    emb [N,ch,2,2,2] -> (rounded latent [N,ch,2,2,2], summed rate in bits); differentiable w.r.t. emb and the
    six trainable tensors.  raw: dict over _lib.LATENT_FIELDS; noise: U(0,1) samples shaped like emb or None."""
    return _LatentHeadFn.apply(int(ch), mode == "train", float(noise_scale),
                               (float(beta_bound), float(gamma_bound), float(pedestal)), noise, emb,
                               *[raw[k] for k in _lib.LATENT_FIELDS])


class _RdTotalFn(torch.autograd.Function):
    """loss = bce + ms0 + ms1 + lmbda (w1 latent_bits / n_pts + w2 sum(net_bits) / n_total) in one launch
    (NVFPCC.py:161-164,196); backward in one launch."""

    @staticmethod
    def forward(ctx, sums, bce, ms0, ms1, latent_bits, net_bits, n_pts, n_total, lmbda, w1, w2, w2_grad):
        b = _lib.cuda_binding()
        loss, stats = b.rd_total(sums, latent_bits, net_bits, n_pts, n_total, lmbda, w1, w2)
        ctx.consts = (n_total, lmbda, w1, w2_grad)
        ctx.save_for_backward(n_pts)
        ctx.mark_non_differentiable(stats)
        return loss.reshape(()), stats

    @staticmethod
    def backward(ctx, g_loss, _g_stats):
        b = _lib.cuda_binding()
        (n_pts,) = ctx.saved_tensors
        g_dist, g_lb, g_nb = b.rd_total_backward(g_loss, n_pts, *ctx.consts)
        return None, g_dist[0], g_dist[1], g_dist[2], g_lb.reshape(()), g_nb, None, None, None, None, None, None


def rd_total(sums, bce, ms0, ms1, latent_bits, net_bits, n_pts, n_total: float, lmbda: float, w1: float, w2: float,
             w2_grad=None):
    """-> (loss, stats[7] = loss bce ms0 ms1 b_latent b_net n_pts).  `sums`/`bce`/`ms0`/`ms1` as returned by
    rd_distortion (the three scalars only carry the autograd edges; values are read from `sums`).
    w2_grad: weight of the network-rate term in the BACKWARD pass only (default w2).  Data-parallel training sums
    the ranks' gradients, and the network-rate term lmbda*w2*sum(net_bits)/n_total does not depend on the rank's
    blocks: it must enter the summed gradient once, so every rank but one passes 0 (trainer._loss_terms)."""
    return _RdTotalFn.apply(sums, bce, ms0, ms1, latent_bits, net_bits, n_pts, float(n_total), float(lmbda),
                            float(w1), float(w2), float(w2 if w2_grad is None else w2_grad))


RAW_FIELDS = tuple("%s_%s" % (l, f) for l in _lib.CONV_LAYERS for f in ("kernel", "kernel_init", "b", "b_init")) + (
    "igdn_beta", "igdn_gamma", "lik_sigma", "lik_mu")


class _ParamPrepFn(torch.autograd.Function):
    """forward: nvf_param_prep; backward: nvf_param_prep_backward.  Inputs: the raw tensors in RAW_FIELDS
    order; outputs: the 20 effective tensors in WEIGHT_FIELDS order + net_bits[7]."""

    @staticmethod
    def forward(ctx, ch, channels, q, noise, beta_bound, gamma_bound, pedestal, *raw):
        b = _lib.cuda_binding()
        rawd = dict(zip(RAW_FIELDS, raw))
        if rawd["lik_sigma"].device.type != "cuda":
            raise NvfError("decoder_params needs CUDA tensors; there is no CPU fallback")
        eff, bits = b.param_prep(b.desc(ch, channels), rawd, q, noise, beta_bound, gamma_bound, pedestal)
        ctx.args = (ch, tuple(channels), beta_bound, gamma_bound)
        ctx.save_for_backward(*raw)
        return tuple(eff[k] for k in WEIGHT_FIELDS) + (bits,)

    @staticmethod
    def backward(ctx, *grads):
        b = _lib.cuda_binding()
        raw = ctx.saved_tensors
        rawd = dict(zip(RAW_FIELDS, raw))
        ch, channels, beta_bound, gamma_bound = ctx.args
        g_eff = {}
        for k, g in zip(WEIGHT_FIELDS, grads[:-1]):
            if g is None:   # shaped like its raw tensor: <key>_kernel for <key>_w, the namesake for the others
                g = torch.zeros_like(rawd[k[:-1] + "kernel" if k.endswith("_w") else k],
                                     memory_format=torch.contiguous_format)
            g_eff[k] = g.contiguous()
        dev = rawd["lik_sigma"].device
        g_bits = grads[-1] if grads[-1] is not None else torch.zeros(_lib.NVF_NUM_QUANT, device=dev)
        out = b.param_prep_backward(b.desc(ch, channels), rawd, beta_bound, gamma_bound, g_eff, g_bits)
        res = []
        for i, name in enumerate(RAW_FIELDS):
            g = None
            if ctx.needs_input_grad[7 + i]:
                g = out.get(name)
            res.append(g)
        return (None,) * 7 + tuple(res)


def decoder_params(ch: int, channels: Sequence[int], q: int, raw: Dict[str, torch.Tensor], beta_bound: float,
                   gamma_bound: float, pedestal: float):
    """Fused parameter-side transforms (see include/nvf_b200.h nvf_param_prep): raw tensors ->
    (effective tensors dict, net_bits[7]); differentiable w.r.t. kernel / b / IGDN beta,gamma / likelihood sigma,mu."""
    noise = None
    if q == 1:
        n = sum(raw[l + "_kernel"].numel() for l in _lib.CONV_LAYERS[:_lib.NVF_NUM_QUANT])
        noise = torch.rand(n, device=raw["lik_sigma"].device, dtype=torch.float32)
    outs = _ParamPrepFn.apply(int(ch), tuple(int(c) for c in channels), int(q), noise, float(beta_bound),
                              float(gamma_bound), float(pedestal), *[raw[k] for k in RAW_FIELDS])
    return dict(zip(WEIGHT_FIELDS, outs[:-1])), outs[-1]
