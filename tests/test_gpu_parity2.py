"""GPU parity, second tier (round 2): reference-generated training steps in the phase the bench runs (q=1) and for
the wide config, the fused latent-head / parameter kernels against the ORACLE (not the torch mirror), whole-cloud
decode parity on the BASELINE configurations with D1 and D2 PSNR, and the data-parallel weight step (two ranks on
one GPU) against the single-process step."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import nvf_oracle as O
from oracle.gen_golden import TRAIN_HP, fixture_inputs
from tests.conftest import GOLDEN
from tests.helpers import THH_BAND, assert_prob_close, logit_of

pytestmark = pytest.mark.gpu
N_TOTAL = 849338.0


@pytest.fixture(scope="module")
def golden_train2():
    return {tag: np.load(os.path.join(GOLDEN, "nvf_train2_%s.npz" % tag)) for tag in "AB"}


def _net(tag, fx):
    from nvfpcc_b200 import network, synth
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=fx["ch"], channel_str=",".join(str(c) for c in fx["channels"]))
    net.load_state_dict(fx["sd"])
    return net.cuda()


def _product_step(net, fx, emb, gt, dist, q, latent_noise, kernel_noise):
    """Net.forward + the weight-loop loss through the product ops, with the noises handed in (the product draws
    them with torch.rand on the device; the tests replay the reference's draws instead)."""
    from nvfpcc_b200 import _lib, ops
    rec, gd = net.reconstructor, net.latent_gen.gdn_2
    lat, lbits = ops.latent_head(fx["ch"], emb, net.latent_raw(), "train", latent_noise, 1.0, gd.beta_bound,
                                 gd.gamma_bound, float(gd.reparam_pedestal))
    raw = rec.raw_tensors()
    outs = ops._ParamPrepFn.apply(fx["ch"], tuple(fx["channels"]), q, kernel_noise, float(rec.activation.beta_bound),
                                  float(rec.activation.gamma_bound), float(rec.activation.reparam_pedestal),
                                  *[raw[k] for k in ops.RAW_FIELDS])
    w, net_bits = dict(zip(_lib.WEIGHT_FIELDS, outs[:-1])), outs[-1]
    out, cls1, cls0 = ops.nvf_decoder(fx["ch"], fx["channels"], lat, w)
    bce, ms0, ms1, sums = ops.rd_distortion(out, cls1, cls0, gt, dist, 0.9, 0.85, 0.6)
    loss, stats = ops.rd_total(sums, bce, ms0, ms1, lbits, net_bits, gt.sum(), N_TOTAL, TRAIN_HP["lmbda"],
                               TRAIN_HP["w1"], TRAIN_HP["w2"])
    return dict(out=out, cls1=cls1, cls0=cls0, net_bits=net_bits, latent_bits=lbits, loss=loss, stats=stats, sums=sums,
                latent=lat, w=w)


def _close(got, ref, what, tol=2e-4):
    got, ref = torch.as_tensor(got).detach().cpu().double(), torch.as_tensor(ref).double()
    scale = float(ref.abs().max()) + 1e-30
    err = float((got - ref).abs().max()) / scale
    assert err <= tol, "%s: max err / max|ref| = %.3e" % (what, err)


@pytest.mark.parametrize("tag,q", [("A", 1), ("B", 2)])
def test_reference_train_step_q1_A_and_q2_B(gpu, golden_train2, tag, q):
    """One weight-loop step (NVFPCC.py:149-197) of the UNMODIFIED reference modules, stored by oracle/gen_golden.py:
    config A at q=1 (noisy kernels: the phase bench.py times) and config B at q=2.  Probabilities within the 1e-4
    logit band, every loss term, every parameter gradient and d/d-emb."""
    g, pre = golden_train2[tag], "%sq%d_" % (tag, q)
    fx = fixture_inputs(tag)
    net = _net(tag, fx)
    emb = fx["emb"].clone().cuda().requires_grad_(True)
    gt, dist = torch.from_numpy(g[pre + "gt"]).float().cuda(), torch.from_numpy(g[pre + "dist"]).float().cuda()
    kn = None
    if q == 1:
        kn = torch.cat([torch.from_numpy(g[pre + "knoise::" + n]).reshape(-1) for n in O.Q_KERNEL_LAYERS]).cuda()
    r = _product_step(net, fx, emb, gt, dist, q, torch.from_numpy(g[pre + "latent_noise"]).cuda(), kn)
    r["loss"].backward()
    assert_prob_close(r["out"], logit_of(torch.from_numpy(g[pre + "out"])), "train out vs reference")
    np.testing.assert_allclose(r["cls1"].detach().cpu().numpy(), g[pre + "cls1"], rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(r["cls0"].detach().cpu().numpy(), g[pre + "cls0"], rtol=2e-4, atol=2e-6)
    np.testing.assert_allclose(r["net_bits"].detach().cpu().numpy(), g[pre + "net_bits"], rtol=2e-5)
    assert r["latent_bits"].item() == pytest.approx(float(g[pre + "latent_bits"]), rel=2e-5)
    assert r["loss"].item() == pytest.approx(float(g[pre + "loss"]), rel=2e-5)
    st = r["stats"].cpu()
    for i, k in ((1, "bce"), (2, "ms0"), (3, "ms1")):
        assert st[i].item() == pytest.approx(float(g[pre + k]), rel=2e-5), k
    _close(emb.grad, g[pre + "grad_emb"], "d_emb")
    n = 0
    for name, p in net.named_parameters():
        ref = g[pre + "grad::" + name]
        got = p.grad if p.grad is not None else torch.zeros_like(p)
        if float(np.abs(ref).max()) == 0.0:
            assert float(got.abs().max()) == 0.0, name
        else:
            _close(got, ref, "grad " + name)
        n += 1
    assert n == 28


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_latent_head_kernel_matches_oracle(gpu, mode):
    """nvf_latent_forward / backward against oracle.nvf_oracle (latent_gen + entropy_coder, utils/network.py:4610-4612,
    4514-4539; gdn_3d.py:78-92) incl. autograd w.r.t. emb and the six trainable tensors, on a perturbed state whose
    LowerBound / abs branches carry signal."""
    from nvfpcc_b200 import ops
    fx = fixture_inputs("A")
    sd = {k: v.clone() for k, v in fx["sd"].items()}
    sd["latent_gen.gdn_2.gamma"][0, 1] = 1e-7
    sd["latent_gen.gdn_2.beta"][2] = 1e-4
    sd["entropy_coder.sigma"][0, 1] = -0.7
    sd["entropy_coder.mu"][0, 2] = 0.3
    fx = dict(fx, sd=sd)
    net = _net("A", fx)
    g = torch.Generator().manual_seed(3)
    emb_o = (torch.randn(41, 3, 2, 2, 2, generator=g) * 3).requires_grad_(True)
    noise = torch.rand(41, 3, 2, 2, 2, generator=g)
    cot = torch.randn(41, 3, 2, 2, 2, generator=g)
    names = ("latent_gen.h_analysis_2.kernel", "latent_gen.h_analysis_2.b", "latent_gen.gdn_2.beta",
             "latent_gen.gdn_2.gamma", "entropy_coder.sigma", "entropy_coder.mu")
    # forward values against the fp32 oracle; gradients against the SAME oracle evaluated in float64 (the eval-mode
    # rate is a difference of nearby CDF values: in fp32 the oracle's own bias gradient is off by 5e-4 of its
    # maximum against float64, more than the kernel is)
    with torch.no_grad():
        lat_o, bits_o = O.entropy_coder(O.latent_gen(emb_o.detach(), sd), sd, mode, noise)
    sd_o = {k: (v.double().requires_grad_(True) if k in names else v.double()) for k, v in sd.items()}
    emb_o = emb_o.detach().double().requires_grad_(True)
    lat_d, bits_d = O.entropy_coder(O.latent_gen(emb_o, sd_o), sd_o, mode, noise.double())
    ((lat_d * cot.double()).sum() + 0.37 * bits_d.sum()).backward()
    emb_f = emb_o.detach().float().cuda().requires_grad_(True)
    gd = net.latent_gen.gdn_2
    lat_f, bits_f = ops.latent_head(3, emb_f, net.latent_raw(), mode, noise.cuda(), 1.0, gd.beta_bound, gd.gamma_bound,
                                    float(gd.reparam_pedestal))
    ((lat_f * cot.cuda()).sum() + 0.37 * bits_f).backward()
    assert torch.equal(lat_f.detach().cpu(), lat_o.detach())
    assert bits_f.item() == pytest.approx(bits_o.sum().item(), rel=2e-5)
    _close(emb_f.grad, emb_o.grad, "d_emb", 3e-4)
    pf = dict(net.named_parameters())
    for k in names:
        # the rate gradients w.r.t. sigma / mu are sums of differences of nearby fp32 CDF / PDF values
        _close(pf[k].grad, sd_o[k].grad, k, 2e-3 if k.startswith("entropy_coder") else 5e-4)


@pytest.mark.parametrize("q", [0, 1, 2])
def test_param_prep_kernel_matches_oracle(gpu, q):
    """nvf_param_prep (+ backward) against oracle.nvf_oracle.effective_decoder_weights / net_bits
    (utils/network.py:606-620, 669-686, 735-740, 4777-4778; gdn_3d.py:143-150) incl. autograd."""
    from nvfpcc_b200 import _lib, ops
    fx = fixture_inputs("A")
    sd = {k: v.clone() for k, v in fx["sd"].items()}
    sd["reconstructor.activation.gamma"][0, 1] = 1e-7
    sd["reconstructor.activation.gamma"][2, 3] = -0.5
    sd["reconstructor.activation.beta"][1] = 1e-4
    fx = dict(fx, sd=sd)
    rec = _net("A", fx).reconstructor
    g = torch.Generator().manual_seed(5)
    noises = {n: torch.rand(sd["reconstructor.%s.kernel" % n].shape, generator=g) for n in O.Q_KERNEL_LAYERS}
    sd_o = {k: (v.clone().requires_grad_(True) if not k.endswith(("_init", "pedestal")) else v.clone())
            for k, v in sd.items()}
    w_o = O.effective_decoder_weights(sd_o, q, noises if q == 1 else None)
    bits_o = O.net_bits(sd_o)
    name_map = {"cls2_w": "conv2_cls_w", "cls2_b": "conv2_cls_b", "cls1_w": "conv1_cls_w", "cls1_b": "conv1_cls_b",
                "cls0_w": "conv0_cls_w", "cls0_b": "conv0_cls_b"}
    cot = {k: torch.randn(w_o[name_map.get(k, k)].shape, generator=g) for k in _lib.WEIGHT_FIELDS}
    cb = torch.rand(7, generator=g) + 0.1
    (sum((w_o[name_map.get(k, k)] * cot[k]).sum() for k in _lib.WEIGHT_FIELDS) + (bits_o * cb).sum()).backward()
    kn = torch.cat([noises[n].reshape(-1) for n in O.Q_KERNEL_LAYERS]).cuda() if q == 1 else None
    raw = rec.raw_tensors()
    outs = ops._ParamPrepFn.apply(3, (8, 16, 8, 8), q, kn, float(rec.activation.beta_bound),
                                  float(rec.activation.gamma_bound), float(rec.activation.reparam_pedestal),
                                  *[raw[k] for k in ops.RAW_FIELDS])
    w_f, bits_f = dict(zip(_lib.WEIGHT_FIELDS, outs[:-1])), outs[-1]
    (sum((w_f[k] * cot[k].cuda()).sum() for k in _lib.WEIGHT_FIELDS) + (bits_f * cb.cuda()).sum()).backward()
    for k in _lib.WEIGHT_FIELDS:
        np.testing.assert_allclose(w_f[k].detach().cpu().numpy(), w_o[name_map.get(k, k)].detach().numpy(), rtol=1e-6,
                                   atol=1e-7, err_msg=k)
    np.testing.assert_allclose(bits_f.detach().cpu().numpy(), bits_o.detach().numpy(), rtol=2e-5)
    for name, p in rec.named_parameters():
        ref = sd_o["reconstructor." + name].grad
        assert ref is not None and p.grad is not None, name
        _close(p.grad, ref, name, 3e-4)


# ---------------------------------------------------------------------------------------------- whole clouds
def _sphere_normals(p, centre):
    v = np.asarray(p, np.float64) - centre
    return v / np.maximum(np.linalg.norm(v, axis=1, keepdims=True), 1e-12)


def psnr_d1_d2(rec, src, centre, peak):
    """Symmetric point-to-point (D1) and point-to-plane (D2) PSNR of `rec` against the source cloud `src`, as
    MPEG's pc_error defines them: both directions, the worse mean wins; plane normals always come from the SOURCE
    (analytic for the synthetic sphere shell); PSNR = 10 log10(3 peak^2 / mse)."""
    from scipy.spatial import cKDTree
    rec, src = np.asarray(rec, np.float64), np.asarray(src, np.float64)
    n_src = _sphere_normals(src, centre)
    d_sr, j_sr = cKDTree(rec).query(src)            # source -> reconstruction
    d_rs, j_rs = cKDTree(src).query(rec)            # reconstruction -> source
    d1 = max(float((d_sr ** 2).mean()), float((d_rs ** 2).mean()))
    e_sr = np.einsum("ij,ij->i", src - rec[j_sr], n_src)
    e_rs = np.einsum("ij,ij->i", rec - src[j_rs], n_src[j_rs])
    d2 = max(float((e_sr ** 2).mean()), float((e_rs ** 2).mean()))
    f = lambda mse: 10.0 * np.log10(3.0 * peak * peak / max(mse, 1e-12))
    return f(d1), f(d2)


def _whole_cloud_case(chanstr, resolution, n_blocks, thh, oracle_batch):
    from nvfpcc_b200 import network, synth
    import bench
    channels = [int(c) for c in chanstr.split(",")]
    pts = synth.sphere_shell_points(resolution)
    origins = synth.leaf_origins(pts)
    n_all = origins.shape[0]
    sel = np.arange(n_all) if n_blocks is None else np.linspace(0, n_all - 1, n_blocks).astype(np.int64)
    origins = origins[sel]
    n = origins.shape[0]
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=3, channel_str=chanstr).cuda()
    lat = torch.from_numpy(synth.random_latents(n_all, 3, seed=0)[sel])
    bench.calibrate_threshold_bias(net, lat.cuda(), thh)
    org = torch.from_numpy(origins.astype(np.int32))
    got = net.decode_points(lat.cuda(), org.cuda(), thh, return_prob=True, return_host=True)
    sd_cpu = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    n_diff, n_vox, ref_pts = 0, 0, []
    with torch.no_grad():
        for s in range(0, n, oracle_batch):
            ref = O.reconstruct(lat[s:s + oracle_batch], sd_cpu, q=2)
            p = got["prob"][s:s + oracle_batch]
            diff = (p > thh) != (ref > thh)
            n_diff += int(diff.sum())
            n_vox += diff.numel()
            assert ((ref[diff] - thh).abs() <= THH_BAND).all(), "occupancy mismatch outside the thh band"
            assert_prob_close(p, logit_of(ref), "whole-cloud probabilities")
            ref_pts.append(O.threshold_points(ref, origins[s:s + oracle_batch], thh)[0])
    assert n_diff <= 1e-4 * n_vox, (n_diff, n_vox)                 # >= 99.99 % of voxels agree
    ref_pts = np.concatenate(ref_pts, 0)
    centre = np.array([resolution / 2.0] * 3)
    key = lambda a: (np.asarray(a, np.int64) // 32) @ np.array([1 << 40, 1 << 20, 1])
    src = pts[np.isin(key(pts), key(origins))]
    peak = float(resolution - 1)
    d1g, d2g = psnr_d1_d2(got["coords"].numpy(), src, centre, peak)
    d1r, d2r = psnr_d1_d2(ref_pts, src, centre, peak)
    assert abs(d1g - d1r) <= 0.01 and abs(d2g - d2r) <= 0.01, (d1g, d1r, d2g, d2r)   # north_star: within 0.01 dB
    assert got["coords"].shape[0] == int(got["counts"].sum()) and 0.005 < got["coords"].shape[0] / (n * 32768.0) < 0.06
    return n, n_diff, (d1g, d2g)


def test_whole_vox10_cloud_decode_parity_A(gpu):
    """BASELINE.json configs[0]/[1] cloud: ALL 1247 vox10 leaves through the fused decode kernel against the oracle:
    occupancy equal on >= 99.99 % of the 40.9 M voxels, every mismatch within 1e-4 of thh, D1 and D2 PSNR of the
    two reconstructions against the source cloud within 0.01 dB."""
    n, _, _ = _whole_cloud_case("8,16,8,8", 1024, None, 0.65, 64)
    assert n == 1247


def test_vox11_wide_decode_parity_B(gpu):
    """BASELINE.json configs[3]: 256 leaves spread over the vox11 cloud, chanstr 16,32,16,16, same bars."""
    n, _, _ = _whole_cloud_case("16,32,16,16", 2048, 256, 0.65, 32)
    assert n == 256


# ---------------------------------------------------------------------------------------------- data parallel
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dp_worker(rank, world, port, ret):
    """Two ranks on ONE GPU over gloo (NCCL refuses two ranks per device): the host logic and the kernels are the
    product's, only the transport differs."""
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from nvfpcc_b200 import network, synth, trainer
        g = np.load(os.path.join(GOLDEN, "nvf_A.npz"))
        gt, dst = torch.from_numpy(g["tr_gt"]).float().cuda(), torch.from_numpy(g["tr_dist"]).float().cuda()
        network.set_seed(synth.synthetic_seed())
        net = network.Net(None, "Gaussian", ch=3, channel_str="8,16,8,8").cuda()
        net.entropy_coder.noise_scale = 0.0
        opt = trainer.FusedAdam(net.parameters(), lr=1e-3)
        ws = trainer.WeightStep(net, opt, 1, N_TOTAL, 200.0, 10.0, 57.0, use_graph=False)
        emb = torch.ones(1, 3, 2, 2, 2).cuda()
        n_pts = gt.sum().reshape(1)                         # global batch = both blocks
        ws.step(emb, gt[rank:rank + 1], dst[rank:rank + 1], q=2, n_pts=n_pts)
        ret[rank] = (opt.flat_grad.cpu().numpy().copy(), opt.flat.detach().cpu().numpy().copy())
    finally:
        dist.destroy_process_group()


def test_two_rank_weight_step_equals_single_process(gpu):
    """Data-parallel weight step (2 ranks x 1 block, gradients summed) == the single-process step on the same global
    batch of 2: same all-reduced gradient (incl. the network-rate term entering once, not once per rank) and
    bit-identical weights on both ranks after Adam."""
    import torch.multiprocessing as mp
    from nvfpcc_b200 import network, synth, trainer
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    ps = [ctx.Process(target=_dp_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in ps:
        p.start()
    for p in ps:
        p.join(300)
        assert p.exitcode == 0
    g = np.load(os.path.join(GOLDEN, "nvf_A.npz"))
    gt, dst = torch.from_numpy(g["tr_gt"]).float().cuda(), torch.from_numpy(g["tr_dist"]).float().cuda()
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=3, channel_str="8,16,8,8").cuda()
    net.entropy_coder.noise_scale = 0.0
    opt = trainer.FusedAdam(net.parameters(), lr=1e-3)
    ws = trainer.WeightStep(net, opt, 2, N_TOTAL, 200.0, 10.0, 57.0, use_graph=False)
    ws.step(torch.ones(2, 3, 2, 2, 2).cuda(), gt, dst, q=2)
    ref = opt.flat_grad.cpu().numpy()
    g0, w0 = ret[0]
    g1, w1 = ret[1]
    assert np.array_equal(g0, g1) and np.array_equal(w0, w1)
    scale = float(np.abs(ref).max())
    assert float(np.abs(g0 - ref).max()) <= 2e-5 * scale, float(np.abs(g0 - ref).max()) / scale
