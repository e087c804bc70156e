"""Shared parity checks: the same assertions run against the CPU emulator
(non-GPU tests) and against the CUDA library (`-m gpu` tests)."""
import numpy as np
import torch

from oracle import nvf_oracle as O
from oracle.gen_golden import TRAIN_HP

LOGIT_RTOL = 1e-4   # BASELINE.json north_star: logits within 1e-4 relative
THH_BAND = 1e-4     # occupancy mismatches only within 1e-4 of thh


def eff_weights(sd, q, dev, grad=False):
    with torch.set_grad_enabled(grad):
        w = O.effective_decoder_weights(sd, q)
    return {k: v.detach().to(dev).contiguous() for k, v in w.items() if k in _FIELDS or True} | {
        "cls2_w": w["conv2_cls_w"].detach().to(dev), "cls2_b": w["conv2_cls_b"].detach().to(dev),
        "cls1_w": w["conv1_cls_w"].detach().to(dev), "cls1_b": w["conv1_cls_b"].detach().to(dev),
        "cls0_w": w["conv0_cls_w"].detach().to(dev), "cls0_b": w["conv0_cls_b"].detach().to(dev)}


_FIELDS = ()


def run_without_gpu(code):
    """Runs `code` in a child Python that sees no CUDA device, from the repository root, so that what the package
    does without a GPU is checked on a machine with one as well.  Fails when the child exits non-zero."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


def logit_of(p):
    p = p.double().clamp(1e-12, 1 - 1e-12)
    return torch.log(p) - torch.log1p(-p)


def assert_prob_close(p_got, logit_ref, what=""):
    """|logit - logit_ref| <= 1e-4 * max(1, |logit_ref|) evaluated through the sigmoid:
    compare probabilities with the tolerance the logit band implies."""
    lr = logit_ref.double()
    band = LOGIT_RTOL * torch.clamp(lr.abs(), min=1.0)
    lo, hi = torch.sigmoid(lr - band), torch.sigmoid(lr + band)
    pg = p_got.double().cpu()
    slack = 2e-7  # fp32 rounding of the sigmoid itself
    bad = (pg < lo - slack) | (pg > hi + slack)
    assert not bad.any(), "%s: %d probabilities outside the 1e-4 logit band (max |dp| %.3e)" % (
        what, int(bad.sum()), float((pg - torch.sigmoid(lr)).abs().max()))


def check_decode_against_oracle(binding, fx, latents, thh, golden, dev):
    desc = binding.desc(fx["ch"], fx["channels"])
    w = eff_weights(fx["sd"], 2, dev)
    n = latents.shape[0]
    origins = torch.arange(n * 3, dtype=torch.int32).reshape(n, 3) * 32
    r = binding.decode(desc, w, latents.to(dev), origins.to(dev), thh, want_prob=True)
    with torch.no_grad():
        wo = O.effective_decoder_weights(fx["sd"], 2)
        out_ref, _, _, logit_ref, _ = O.decoder_forward(latents, wo, aux=False)
    prob = r["prob"].cpu()
    assert_prob_close(prob, logit_ref, "decode")
    # golden: the first fixture latents are the reference's own run
    ng = golden["dec_logit"].shape[0]
    if torch.equal(latents[:ng], fx["latents"][:ng]):
        assert_prob_close(prob[:ng], torch.from_numpy(golden["dec_logit"]), "decode vs golden")
    # occupancy: equal except within THH_BAND of thh (in probability)
    occ = prob > thh
    occ_ref = out_ref > thh
    diff = occ != occ_ref
    assert diff.float().mean().item() <= 1e-4
    assert ((out_ref[diff] - thh).abs() <= THH_BAND).all()
    # mask bits == occupancy of the returned probabilities, exactly
    mask = r["mask"].cpu().numpy().view(np.uint32).reshape(n, 32, 32)
    bits = (mask[..., None] >> np.arange(32, dtype=np.uint32)) & 1
    np.testing.assert_array_equal(bits.astype(bool), occ.numpy().reshape(n, 32, 32, 32))
    # points: block order, row-major in-block order, + origin  (NVFPCC.py:631-637)
    pts_ref, counts_ref = O.threshold_points(prob, origins.numpy(), thh)
    np.testing.assert_array_equal(r["counts"].cpu().numpy(), counts_ref)
    np.testing.assert_array_equal(r["coords"].cpu().numpy(), pts_ref)
    assert int(r["total"]) == pts_ref.shape[0]
    return r


def check_train_against_oracle(binding, fx, golden, dev, blocks=None):
    """forward (3 heads) + loss sums/seeds + backward (all effective-weight grads + d_latent)
    against torch autograd on the oracle, on the golden training inputs."""
    desc = binding.desc(fx["ch"], fx["channels"])
    gt = torch.from_numpy(golden["tr_gt"]).float()
    dist = torch.from_numpy(golden["tr_dist"]).float()
    if blocks is not None:
        gt, dist = gt[blocks], dist[blocks]
    n = gt.shape[0]
    g = torch.Generator().manual_seed(5)
    latent = torch.round(torch.randn(n, fx["ch"], 2, 2, 2, generator=g) * 3)
    # oracle with autograd w.r.t. effective tensors and latent
    wo = {k: v.clone().requires_grad_(True) for k, v in O.effective_decoder_weights(fx["sd"], 2).items()}
    lat_o = latent.clone().requires_grad_(True)
    out_o, cls0_o, cls1_o, logit_o, _ = O.decoder_forward(lat_o, wo, aux=True)
    gts = O.gt_pyramid(gt)
    bce = O.surf_focal_dense(out_o, gt, dist, beta=1, alpha=0.9)
    ms0 = O.focal_dense(cls0_o, gts[0], alpha=0.85)
    ms1 = O.focal_dense(cls1_o, gts[1], alpha=0.85)
    (bce + ms0 + ms1).backward()

    w = {k: v.to(dev) for k, v in eff_weights(fx["sd"], 2, dev).items()}
    out, cls1, cls0, ws, keep = binding.train_forward(desc, w, latent.to(dev))
    assert_prob_close(out, logit_o.detach(), "train out")
    np.testing.assert_allclose(cls1.cpu().numpy(), cls1_o.detach().numpy(), rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(cls0.cpu().numpy(), cls0_o.detach().numpy(), rtol=2e-4, atol=2e-6)
    sums, seeds = binding.loss_seeds(out, cls1, cls0, gt.to(dev), dist.to(dev), 0.9, 0.85, 0.6)
    sums = sums.cpu().numpy()
    np.testing.assert_allclose(sums[0], bce.item(), rtol=2e-5)
    np.testing.assert_allclose(sums[1], ms0.item(), rtol=2e-5)
    np.testing.assert_allclose(sums[2], ms1.item(), rtol=2e-5)
    # metrics are thresholded counts: evaluate the oracle's metric code on the SAME probabilities
    sse, denom = O.sse1(out.cpu(), dist, 0.6)
    np.testing.assert_allclose(sums[3], sse.item(), rtol=1e-5, atol=1e-6)
    assert sums[4] == denom.item()
    _, _, (tp, ap, tn, an) = O.acc_dense(out.cpu(), gt)
    assert [sums[5], sums[6], sums[7], sums[8]] == [tp.item(), ap.item(), tn.item(), an.item()]
    _, _, c0 = O.acc_dense(cls0.cpu(), gts[0])
    assert [sums[9], sums[10], sums[11], sums[12]] == [c.item() for c in c0]
    _, _, c1 = O.acc_dense(cls1.cpu(), gts[1])
    assert [sums[13], sums[14], sums[15], sums[16]] == [c.item() for c in c1]

    g_lat, grads = binding.train_backward(desc, w, latent.to(dev), ws, seeds[0], seeds[1], seeds[2], True, True)
    name_map = {"cls2_w": "conv2_cls_w", "cls2_b": "conv2_cls_b", "cls1_w": "conv1_cls_w", "cls1_b": "conv1_cls_b",
                "cls0_w": "conv0_cls_w", "cls0_b": "conv0_cls_b"}

    def close(got, ref, what):
        got = got.cpu().double()
        ref = ref.double()
        scale = float(ref.abs().max()) + 1e-30
        err = float((got - ref).abs().max()) / scale
        assert err <= 2e-4, "%s: max err / max|ref| = %.3e" % (what, err)

    close(g_lat, lat_o.grad, "d_latent")
    for k, gv in grads.items():
        close(gv, wo[name_map.get(k, k)].grad, "grad " + k)
    return sums


# binding field (include/nvf_b200.h NvfWeights) -> key of O.effective_decoder_weights
ORACLE_NAME = {"cls2_w": "conv2_cls_w", "cls2_b": "conv2_cls_b", "cls1_w": "conv1_cls_w", "cls1_b": "conv1_cls_b",
               "cls0_w": "conv0_cls_w", "cls0_b": "conv0_cls_b"}


class _ConvRecorder:
    """Stands in for torch.nn.functional inside the oracle module: conv3d / conv_transpose3d / relu run unchanged, and
    each convolution's input, weight, bias, arguments and output (with retain_grad) are kept, as is the output of a
    ReLU applied to it, so that the gradients reaching both are available after backward."""

    def __init__(self):
        import torch.nn.functional as F
        self._F = F
        self.calls = []
        self.relus = []      # ReLU inputs, in call order
        self.relu_of = {}    # id(convolution output) -> the ReLU's output

    def relu(self, x):
        y = self._F.relu(x)
        y.retain_grad()
        self.relu_of[id(x)] = y
        self.relus.append(x)
        return y

    def _rec(self, fn, x, w, b, args):
        y = fn(x, w, b, *args)
        y.retain_grad()
        self.calls.append((fn, x, w, b, args, y))
        return y

    def conv3d(self, x, w, b=None, *args):
        return self._rec(self._F.conv3d, x, w, b, args)

    def conv_transpose3d(self, x, w, b=None, *args):
        return self._rec(self._F.conv_transpose3d, x, w, b, args)


# bound on the float32 forward's error in an activation, relative to that activation's forward scale (the same
# convolution of |input| with |weight|, plus |bias|): see oracle_train64's S_fwd
FWD_BAND = 1e-5


def oracle_train64(sd, latent, gt=None, dist=None, cot=None):
    """The float64 oracle of nvf_train_forward -> nvf_loss_seeds -> nvf_train_backward, with autograd.

    The loss is the training loss on (gt, dist) or, with `cot` = (g_out, g_cls1, g_cls0), the sum of the three heads'
    probabilities weighted by those cotangents.  Besides the heads (probabilities and logits), the loss terms, the
    gradients of the 20 effective tensors (binding names) and d_latent, it returns `S`, the elementwise scale of each
    gradient: the same weight-gradient operation (autograd of the oracle's own conv / convT) applied to |input| and
    |output gradient| (bias: the sum of |output gradient|; d_latent: the data gradient of |output gradient| through
    |weight|).  |gradient| <= S holds exactly, and S adds up over blocks.

    S bounds what rounding in the gradient's own sums does.  A float32 kernel also works from a float32 forward,
    whose activations are off by up to FWD_BAND of their forward scale F (the same convolution of |input| with
    |weight|, plus |bias|).  `S_fwd` bounds what that does to a weight or bias gradient, to first order: the
    weight-gradient operation applied to FWD_BAND * F of the input (F = |input| where the input is not a ReLU of a
    convolution) and |output gradient|, plus the full terms of the outputs whose ReLU input lies within FWD_BAND * F
    of zero, which may fall on the other side of the ReLU (taken with the gradient at the ReLU's output).  It
    dominates the few entries whose S comes from a handful of activations that are themselves the small remainder of
    a cancelling sum.  A float32 training step is compared against this oracle within tau * S + S_fwd."""
    from nvfpcc_b200._lib import WEIGHT_FIELDS
    wo = {k: v.detach().double().requires_grad_(True) for k, v in O.effective_decoder_weights(sd, 2).items()}
    lat = latent.detach().double().requires_grad_(True)
    rec = _ConvRecorder()
    f0, O.F = O.F, rec
    try:
        out, cls0, cls1, logit, _ = O.decoder_forward(lat, wo, aux=True)
    finally:
        O.F = f0
    sums = None
    if cot is None:
        gt, dist = gt.double(), dist.double()
        gts = O.gt_pyramid(gt)
        sums = (O.surf_focal_dense(out, gt, dist, beta=1, alpha=0.9), O.focal_dense(cls0, gts[0], alpha=0.85),
                O.focal_dense(cls1, gts[1], alpha=0.85))
        loss = sums[0] + sums[1] + sums[2]
    else:
        loss = sum((p * c.double()).sum() for p, c in zip((out, cls1, cls0), cot))
    loss.backward()
    by_ptr = {wo[ORACLE_NAME.get(k, k)].data_ptr(): k for k in WEIGHT_FIELDS}
    S, S_fwd, logits = {}, {}, {}
    fscale = {}    # id(convolution output) -> its forward scale F

    def wgrad_of_abs(fn, x, w, args, gy):
        wd = torch.zeros_like(w.detach()).requires_grad_(True)
        fn(x.detach().abs(), wd, None, *args).backward(gy)
        return wd.grad

    with torch.enable_grad():
        for fn, x, w, b, args, y in rec.calls:
            with torch.no_grad():
                fscale[id(y)] = fn(x.abs(), w.abs(), b.abs(), *args)
        relu_in = {id(rec.relu_of[id(y)]): y for y in rec.relus}    # id(ReLU output) -> its input
        for fn, x, w, b, args, y in rec.calls:
            gy = y.grad.detach().abs()
            kw, kb = by_ptr[w.data_ptr()], by_ptr[b.data_ptr()]
            shape = wo[ORACLE_NAME.get(kw, kw)].shape
            logits[kw] = y.detach()
            S[kw] = wgrad_of_abs(fn, x, w, args, gy).reshape(shape)
            S[kb] = gy.sum(dim=(0, 2, 3, 4))
            x_scale = fscale[id(relu_in[id(x)])] if id(x) in relu_in else x.detach()
            S_fwd[kw] = FWD_BAND * wgrad_of_abs(fn, x_scale, w, args, gy).reshape(shape)
            S_fwd[kb] = torch.zeros_like(S[kb])
            if id(y) in rec.relu_of:   # outputs that may fall on the other side of the ReLU
                g_act = rec.relu_of[id(y)].grad.detach().abs() * (y.detach().abs() <= FWD_BAND * fscale[id(y)])
                S_fwd[kw] = S_fwd[kw] + wgrad_of_abs(fn, x, w, args, g_act).reshape(shape)
                S_fwd[kb] = S_fwd[kb] + g_act.sum(dim=(0, 2, 3, 4))
            if x is lat:
                xd = torch.zeros_like(lat.detach()).requires_grad_(True)
                fn(xd, w.detach().abs(), None, *args).backward(gy)
                S["d_latent"] = xd.grad
    assert set(S) == set(WEIGHT_FIELDS) | {"d_latent"}
    return dict(out=out.detach(), cls1=cls1.detach(), cls0=cls0.detach(), logit2=logit.detach(),
                logit1=logits["cls1_w"], logit0=logits["cls0_w"],
                sums=None if sums is None else [float(s.detach()) for s in sums],
                grads={k: wo[ORACLE_NAME.get(k, k)].grad.detach() for k in WEIGHT_FIELDS},
                d_latent=lat.grad.detach(), S=S, S_fwd=S_fwd)


def scaled_err(got, ref, S):
    """max over elements of |got - ref| / S; an element whose scale S is zero must match exactly (else inf)."""
    err = (got.detach().cpu().double() - ref.detach().cpu().double()).abs()
    S = S.detach().cpu().double().reshape(err.shape)
    if bool(((S == 0) & (err > 0)).any()):
        return float("inf")
    return float(torch.where(S > 0, err / torch.where(S > 0, S, torch.ones_like(S)), torch.zeros_like(S)).max())
