"""Generate tests/golden/*.npz from the UNMODIFIED reference (run in the build
container only: needs /root/reference).

    python oracle/gen_golden.py

TEST INFRASTRUCTURE ONLY.  The fixtures pin oracle/nvf_oracle.py (and through
it the CUDA path) to the reference's own PyTorch modules:

* nvf_A.npz  chanstr 8,16,8,8 ch=3: decode of 2 blocks (q=2, quantised
  deltas), one weight-loop training step (NVFPCC.py:149-197) on 2 real
  synthetic leaf blocks incl. every parameter/embedding gradient.
* nvf_B.npz  chanstr 16,32,16,16 ch=3: decode of 1 block.
* nvf_train2_A.npz / nvf_train2_B.npz  two more weight-loop steps of the reference: config A at q=1
  (the noisy-kernel phase the bench runs; the uniform noises the reference drew
  are stored so the step can be replayed exactly) and config B at q=2.

Inputs are rebuilt by `fixture_inputs()` from fixed seeds (shared with the
tests); a checksum of the rebuilt state is stored so RNG drift is detected.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import nvf_oracle as O  # noqa: E402
from oracle import ref_import  # noqa: E402
from nvfpcc_b200 import synth  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
TRAIN_HP = dict(lmbda=200.0, w1=10.0, w2=57.0)
# intra-op threads of the generating run: the CPU convolutions split their sums by thread count, so the float32
# outputs stored here are bit-exact only under this count (tests/test_oracle_golden.py runs the oracle with it)
GOLDEN_THREADS = 8


def perturbed_state(ch, channels, seed=1234):
    """A non-trivial state: seeded perturbation of every trainable tensor on
    top of the constructor state (kernel deltas ~N(0,0.05), quantised to 1/16
    for the 7 Q-kernels so q=2 and the '4-bit' path are exercised)."""
    sd = O.make_state(ch, channels, synth.synthetic_seed())
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, v in sd.items():
        if k.startswith("_"):
            continue
        if k.endswith("_init") or k.endswith("pedestal"):
            out[k] = v.clone()
        elif k.endswith(".kernel"):
            d = torch.randn(v.shape, generator=g) * 0.05
            layer = k.split(".")[-2]
            out[k] = torch.round(d * 16) / 16 if layer in O.Q_KERNEL_LAYERS else d
        elif k.endswith(".b"):
            out[k] = torch.randn(v.shape, generator=g) * 0.05
        elif k.endswith("beta"):
            out[k] = v + torch.rand(v.shape, generator=g) * 0.2
        elif k.endswith("gamma"):
            out[k] = v + torch.rand(v.shape, generator=g) * 0.05
        elif k.endswith("sigma"):
            out[k] = v + torch.rand(v.shape, generator=g) * 0.5
        elif k.endswith("mu"):
            out[k] = v + (torch.rand(v.shape, generator=g) - 0.5) * 0.2
        else:
            raise KeyError(k)
    return out


def state_checksum(sd):
    return float(sum(v.double().abs().sum().item() for v in sd.values()))


_cloud_cache = {}


def fixture_blocks(block_ids):
    """gt/dist/origins of a few real leaf blocks of the synthetic vox10 shell."""
    if "pts" not in _cloud_cache:
        pts = synth.sphere_shell_points(1024)
        _cloud_cache["pts"] = pts
        _cloud_cache["origins"] = synth.leaf_origins(pts)
    pts, origins = _cloud_cache["pts"], _cloud_cache["origins"]
    o = origins[list(block_ids)]
    gt, dist = synth.gt_and_dist(pts, o, workers=1)
    return o, gt, dist


def fixture_inputs(tag):
    if tag == "A":
        ch, channels = 3, (8, 16, 8, 8)
        nb = 2
    else:
        ch, channels = 3, (16, 32, 16, 16)
        nb = 1
    sd = perturbed_state(ch, channels)
    latents = torch.from_numpy(synth.random_latents(nb, ch, seed=7))
    g = torch.Generator().manual_seed(99)
    emb = torch.ones(nb, ch, 2, 2, 2) + torch.randn(nb, ch, 2, 2, 2, generator=g) * 2.0
    latent_noise = torch.rand(nb, ch, 2, 2, 2, generator=g)
    return dict(ch=ch, channels=channels, sd=sd, latents=latents, emb=emb, latent_noise=latent_noise)


Q_LAYERS_FWD = ("up0", "conv0", "up1", "conv1", "up2", "conv2", "conv2_cls")   # torch.rand_like order at q=1


def reference_train_step(net, RL, fx, gt, dist, q, seed, n_total=849338.0):
    """One weight-loop step of train() (NVFPCC.py:149-197) on the reference modules -> dict of everything the
    tests compare.  The RNG draws are replayed first so they can be stored: entropy_coder draws rand_like(latent)
    (utils/network.py:4516), then at q=1 every Q-layer draws rand_like(kernel) in forward order (:610, :679)."""
    gt_t, dist_t = torch.from_numpy(gt).float(), torch.from_numpy(dist).float()
    emb = fx["emb"].clone().requires_grad_(True)
    torch.manual_seed(seed)
    noise_lat = torch.rand_like(emb)
    noise_k = {}
    if q == 1:
        for name in Q_LAYERS_FWD:
            noise_k[name] = torch.rand_like(getattr(net.reconstructor, name).kernel)
    torch.manual_seed(seed)
    net.train()
    net.zero_grad()
    out, out_cls, net_bits, latent_bits = net(emb, "train", q)
    n_pts = gt_t.sum()
    gts = O.gt_pyramid(gt_t)
    bpp_loss = latent_bits.sum() / n_pts * TRAIN_HP["w1"] + net_bits.sum() / n_total * TRAIN_HP["w2"]
    ms0 = RL.get_focal_dense(out_cls[0], gts[0], alpha=0.85)
    ms1 = RL.get_focal_dense(out_cls[1], gts[1], alpha=0.85)
    bce = RL.get_surf_focal_dense(out, gt_t, dist_t, beta=1, alpha=0.9)
    loss = bce + ms0 + ms1 + TRAIN_HP["lmbda"] * bpp_loss
    loss.backward()
    r = dict(latent_noise=noise_lat.numpy(), out=out.detach().numpy(), cls0=out_cls[0].detach().numpy(),
             cls1=out_cls[1].detach().numpy(), net_bits=net_bits.detach().numpy(),
             latent_bits=np.float64(latent_bits.item()), loss=np.float64(loss.item()), bce=np.float64(bce.item()),
             ms0=np.float64(ms0.item()), ms1=np.float64(ms1.item()), grad_emb=emb.grad.numpy())
    for name, t in noise_k.items():
        r["knoise::" + name] = t.numpy()
    for k, p_ in net.named_parameters():
        r["grad::" + k] = (p_.grad if p_.grad is not None else torch.zeros_like(p_)).numpy()
    return r


def gen_train2(RL):
    for tag, q, blocks, seed in (("A", 1, (0, 600), 777), ("B", 2, (300,), 778)):
        save = {}
        fx = fixture_inputs(tag)
        net = ref_import.build_net(fx["ch"], fx["channels"])
        net.load_state_dict(fx["sd"], strict=True)
        origins, gt, dist = fixture_blocks(blocks)
        r = reference_train_step(net, RL, fx, gt, dist, q, seed)
        pre = "%sq%d_" % (tag, q)
        save[pre + "gt"] = gt
        save[pre + "dist"] = dist.astype(np.float32)
        for k, v in r.items():
            save[pre + k] = v
        path = os.path.join(GOLDEN, "nvf_train2_%s.npz" % tag)        # one file per step: each stays under 1 MB
        np.savez_compressed(path, **save)
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def _load_into_reference(net, sd):
    missing = net.load_state_dict(sd, strict=True)
    return missing


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    torch.set_num_threads(GOLDEN_THREADS)
    _, RL, _ = ref_import.load()
    if "--train2-only" in sys.argv:
        return gen_train2(RL)
    for tag in ("A", "B"):
        fx = fixture_inputs(tag)
        sd = fx["sd"]
        net = ref_import.build_net(fx["ch"], fx["channels"])
        # the constructor-state of the reference must equal the oracle's make_state
        ref_sd0 = net.state_dict()
        mk = O.make_state(fx["ch"], fx["channels"], synth.synthetic_seed())
        for k, v in ref_sd0.items():
            assert torch.equal(v, mk[k]), "constructor state mismatch: " + k
        _load_into_reference(net, sd)
        net.eval()
        save = dict(state_checksum=np.float64(state_checksum(sd)),
                    seed_consumed=np.int64(int(mk["_seed_consumed"])))
        with torch.no_grad():
            out = net.reconstruct(fx["latents"], q=2)
            # logits: re-run the last layer input through the reference modules
            rec = net.reconstructor
            a = rec.activation(rec.up0(fx["latents"], 2))
            a1 = rec.relu(rec.conv0(a, 2))
            a2 = rec.relu(rec.up1(a1, 2))
            a3 = rec.relu(rec.conv1(a2, 2))
            a4 = rec.relu(rec.up2(a3, 2))
            a5 = rec.relu(rec.conv2(a4, 2))
            logit = rec.conv2_cls(a5, 2)
            assert torch.equal(torch.sigmoid(logit), out)
        save["dec_out"] = out.numpy()
        save["dec_logit"] = logit.numpy()
        for name, t in (("a1", a1), ("a2", a2), ("a3", a3), ("a4", a4), ("a5", a5)):
            save["dec_" + name + "_sum"] = np.float64(t.double().sum().item())
            save["dec_" + name + "_abs"] = np.float64(t.double().abs().sum().item())
        if tag == "A":
            origins, gt, dist = fixture_blocks((0, 600))
            gt_t = torch.from_numpy(gt).float()
            dist_t = torch.from_numpy(dist).float()
            emb = fx["emb"].clone().requires_grad_(True)
            # replay the reference's RNG draw: entropy_coder draws rand_like(latent) first
            # (utils/network.py:4516); q=2 draws nothing else.
            torch.manual_seed(4242)
            noise_ref = torch.rand_like(emb)
            torch.manual_seed(4242)
            net.train()
            out, out_cls, net_bits, latent_bits = net(emb, "train", 2)
            n_pts = gt_t.sum()
            n_total = 849338.0
            gts = O.gt_pyramid(gt_t)
            b_latent = latent_bits.sum() / n_pts
            b_net = net_bits.sum() / n_total
            bpp_loss = b_latent * TRAIN_HP["w1"] + b_net * TRAIN_HP["w2"]
            ms0 = RL.get_focal_dense(out_cls[0], gts[0], alpha=0.85)
            ms1 = RL.get_focal_dense(out_cls[1], gts[1], alpha=0.85)
            bce = RL.get_surf_focal_dense(out, gt_t, dist_t, beta=1, alpha=0.9)
            loss = bce + ms0 + ms1 + TRAIN_HP["lmbda"] * bpp_loss
            loss.backward()
            sse, denom = RL.get_sse1(out, gt_t, dist_t, 0.6)
            pacc, nacc = RL.get_acc_dense(out, gt_t)
            save.update(
                tr_origins=origins.astype(np.int32), tr_gt=gt, tr_dist=dist, tr_latent_noise=noise_ref.numpy(),
                tr_out=out.detach().numpy(), tr_cls0=out_cls[0].detach().numpy(), tr_cls1=out_cls[1].detach().numpy(),
                tr_net_bits=net_bits.detach().numpy(), tr_latent_bits=np.float64(latent_bits.item()),
                tr_loss=np.float64(loss.item()), tr_bce=np.float64(bce.item()), tr_ms0=np.float64(ms0.item()),
                tr_ms1=np.float64(ms1.item()), tr_sse=np.float64(sse.item()), tr_denom=np.float64(denom.item()),
                tr_pacc=np.float64(pacc.item()), tr_nacc=np.float64(nacc.item()),
                tr_grad_emb=emb.grad.numpy())
            for k, p in net.named_parameters():
                save["tr_grad::" + k] = (p.grad if p.grad is not None else torch.zeros_like(p)).numpy()
        path = os.path.join(GOLDEN, "nvf_%s.npz" % tag)
        np.savez_compressed(path, **save)
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")
    gen_train2(RL)


if __name__ == "__main__":
    main()
