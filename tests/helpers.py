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
