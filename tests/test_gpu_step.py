"""The fused weight-loop step (nvf_train_step, trainer.FusedStepCall / WeightStep(fused=True)) against the autograd
path over the individual ops, against the reference-generated golden steps, and its in-kernel noise generator."""
import os

import numpy as np
import pytest
import torch

from oracle import nvf_oracle as O
from oracle.gen_golden import TRAIN_HP, fixture_inputs
from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu
N_TOTAL = 849338.0


def _net(fx):
    from nvfpcc_b200 import network, synth
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=fx["ch"], channel_str=",".join(str(c) for c in fx["channels"]))
    net.load_state_dict(fx["sd"])
    return net.cuda()


def test_philox_known_answer_and_distribution(gpu):
    """Philox4x32-10 known-answer vector of Random123 (counter 0, key 0) through nvf_rng_uniform, then the
    properties the noise needs: [0,1), mean 1/2, variance 1/12, streams / steps / seeds decorrelated, replayable."""
    kat = np.array([0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8], dtype=np.uint64)
    got = gpu.rng_uniform(0, 0, 0, 0, 4, "cuda").cpu().numpy()
    np.testing.assert_array_equal(got, ((kat >> 8).astype(np.float64) / 16777216.0).astype(np.float32))
    a = gpu.rng_uniform(1234, 7, 2, 0, 1 << 20, "cuda")
    assert float(a.min()) >= 0.0 and float(a.max()) < 1.0
    assert abs(float(a.mean()) - 0.5) < 2e-3 and abs(float(a.var()) - 1.0 / 12.0) < 1e-3
    assert torch.equal(a, gpu.rng_uniform(1234, 7, 2, 0, 1 << 20, "cuda"))
    assert torch.equal(a[1000:2000], gpu.rng_uniform(1234, 7, 2, 1000, 1000, "cuda"))
    for other in (gpu.rng_uniform(1234, 8, 2, 0, 1 << 20, "cuda"), gpu.rng_uniform(1234, 7, 1, 0, 1 << 20, "cuda"),
                  gpu.rng_uniform(1235, 7, 2, 0, 1 << 20, "cuda")):
        c = float(((a - 0.5) * (other - 0.5)).mean()) * 12.0
        assert abs(c) < 5e-3


def _steps(fused, graph, q=2, n=3, lr=1e-3):
    from nvfpcc_b200 import network, synth, trainer
    g = np.load(os.path.join(GOLDEN, "nvf_A.npz"))
    gt, dist = torch.from_numpy(g["tr_gt"]).float().cuda(), torch.from_numpy(g["tr_dist"]).float().cuda()
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=3, channel_str="8,16,8,8")
    net.load_state_dict(fixture_inputs("A")["sd"])
    net = net.cuda()
    net.entropy_coder.noise_scale = 0.0
    opt = trainer.FusedAdam(net.parameters(), lr=lr)
    ws = trainer.WeightStep(net, opt, 2, N_TOTAL, 200.0, 10.0, 57.0, use_graph=graph, fused=fused)
    emb = (torch.ones(2, 3, 2, 2, 2) + torch.arange(48).reshape(2, 3, 2, 2, 2) * 0.1).cuda()
    hist, grads = [], []
    for i in range(n):
        a, b = (gt, dist) if i % 2 == 0 else (gt.flip(0), dist.flip(0))
        hist.append(ws.step(emb, a, b, q=q).clone().cpu())
        grads.append(opt.flat_grad.clone().cpu())
    return torch.stack(hist), grads, opt.flat.detach().clone().cpu(), ws, net


def test_fused_step_equals_autograd_step(gpu):
    """Same state, same batches, q = 2, zero latent noise: the fused call and the autograd graph over the individual
    ops give the same logged scalars, the same flat gradient and the same weights after three Adam steps."""
    hs_a, gr_a, w_a, _, _ = _steps(False, False)
    hs_f, gr_f, w_f, ws, _ = _steps(True, False)
    assert ws.fused
    np.testing.assert_allclose(hs_f.numpy(), hs_a.numpy(), rtol=2e-6, atol=1e-7)
    for a, f in zip(gr_a, gr_f):
        scale = float(a.abs().max())
        assert float((a - f).abs().max()) <= 2e-6 * scale
    np.testing.assert_allclose(w_f.numpy(), w_a.numpy(), rtol=0, atol=2e-6)
    # and the graph replay of the fused step walks the same trajectory as its eager form
    hs_g, gr_g, w_g, ws_g, _ = _steps(True, True)
    assert 20 < ws_g.launches_per_step < 60
    np.testing.assert_allclose(hs_g.numpy(), hs_f.numpy(), rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(w_g.numpy(), w_f.numpy(), rtol=0, atol=1e-6)


def test_fused_step_indexed_rows_equal_gathered_batch(gpu):
    """Blocks read their dataset rows through idx (no gather): bit-identical to handing the gathered batch in."""
    from nvfpcc_b200 import trainer
    fx = fixture_inputs("A")
    g = np.load(os.path.join(GOLDEN, "nvf_A.npz"))
    gt2, dist2 = torch.from_numpy(g["tr_gt"]).float().cuda(), torch.from_numpy(g["tr_dist"]).float().cuda()
    gt_all = torch.cat([gt2, gt2.flip(0), gt2]).contiguous()
    dist_all = torch.cat([dist2, dist2.flip(0) * 0.5, dist2 * 2]).contiguous()
    emb_all = torch.randn(6, 3, 2, 2, 2, generator=torch.Generator().manual_seed(1)).cuda()
    idx = torch.tensor([4, 1], device="cuda")
    out = []
    for mode in ("batch", "indexed", "packed"):
        net = _net(fx)
        net.entropy_coder.noise_scale = 0.0
        opt = trainer.FusedAdam(net.parameters(), lr=1e-3)
        ws = trainer.WeightStep(net, opt, 2, N_TOTAL, 200.0, 10.0, 57.0, use_graph=(mode == "packed"))
        n_pts = gt_all[idx].sum().reshape(1)
        if mode == "batch":
            st = ws.step(emb_all[idx], gt_all[idx], dist_all[idx], q=2, n_pts=n_pts)
        elif mode == "indexed":
            st = ws.step_indexed(emb_all, gt_all, dist_all, idx, q=2, n_pts=n_pts)
        else:
            st = ws.step_indexed(emb_all, gt_all, dist_all, idx, q=2, packed=ws.pack_schedule(idx, n_pts))
        out.append((st.clone().cpu(), opt.flat_grad.clone().cpu()))
        ws.check_status()
    for st, gr in out[1:]:
        assert torch.equal(st, out[0][0]) and torch.equal(gr, out[0][1])
    # an out-of-range row is clamped and reported, not read out of bounds
    bad = torch.tensor([4, 99], device="cuda")
    ws.step_indexed(emb_all, gt_all, dist_all, bad, q=2, n_pts=n_pts)
    with pytest.raises(Exception):
        ws.check_status()


@pytest.mark.parametrize("tag,q", [("A", 1), ("B", 2)])
def test_fused_step_matches_reference_golden(gpu, tag, q):
    """nvf_train_step with the reference's own noise draws handed in, against the golden steps produced by the
    UNMODIFIED reference modules (oracle/gen_golden.py gen_train2): loss terms and every raw-parameter gradient."""
    from nvfpcc_b200 import trainer
    g, pre = np.load(os.path.join(GOLDEN, "nvf_train2_%s.npz" % tag)), "%sq%d_" % (tag, q)
    fx = fixture_inputs(tag)
    net = _net(fx)
    gt, dist = torch.from_numpy(g[pre + "gt"]).float().cuda(), torch.from_numpy(g[pre + "dist"]).float().cuda()
    n = gt.shape[0]
    call = trainer.FusedStepCall(net, n, N_TOTAL, TRAIN_HP["lmbda"], TRAIN_HP["w1"], TRAIN_HP["w2"], 0.9, None, "cuda",
                                 want_wgrad=True, want_demb=True)
    kn = None
    if q == 1:
        kn = torch.cat([torch.from_numpy(g[pre + "knoise::" + k]).reshape(-1) for k in O.Q_KERNEL_LAYERS]).cuda()
    stats, sums = torch.zeros(7, device="cuda"), torch.zeros(20, dtype=torch.float64, device="cuda")
    emb = fx["emb"].clone().cuda().contiguous()
    call.run(emb, gt, dist, None, 0, gt.sum().reshape(1), stats, sums, q,
             noise_latent=torch.from_numpy(g[pre + "latent_noise"]).cuda().contiguous(), noise_kernel=kn)
    st = stats.cpu()
    assert st[0].item() == pytest.approx(float(g[pre + "loss"]), rel=2e-5)
    for i, k in ((1, "bce"), (2, "ms0"), (3, "ms1")):
        assert st[i].item() == pytest.approx(float(g[pre + k]), rel=2e-5), k

    def close(got, ref, what):
        got, ref = got.detach().cpu().double().reshape(-1), torch.from_numpy(np.asarray(ref)).double().reshape(-1)
        scale = float(ref.abs().max())
        if scale == 0.0:
            assert float(got.abs().max()) == 0.0, what
        else:
            assert float((got - ref).abs().max()) <= 2e-4 * scale, (what, float((got - ref).abs().max()) / scale)

    close(call.g_emb, g[pre + "grad_emb"], "d_emb")
    k = 0
    for name, p in net.named_parameters():
        close(call.grads[id(p)], g[pre + "grad::" + name], name)
        k += 1
    assert k == 28


def test_fused_step_noise_is_the_philox_stream_and_advances(gpu):
    """q = 1 / train mode with in-kernel noise: (a) the step reproduces exactly when the SAME values, fetched through
    nvf_rng_uniform at the step's counter, are handed in as explicit noise tensors (so the in-kernel noise is the
    verified Philox stream, element for element); (b) in a captured graph the device-resident counter advances:
    replays on the same batch with lr = 0 differ; (c) with lr > 0 the loss goes down."""
    from nvfpcc_b200 import trainer
    fx = fixture_inputs("A")
    net = _net(fx)
    g = np.load(os.path.join(GOLDEN, "nvf_A.npz"))
    gt, dist = torch.from_numpy(g["tr_gt"]).float().cuda(), torch.from_numpy(g["tr_dist"]).float().cuda()
    emb = fx["emb"].clone().cuda().contiguous()
    res = []
    for explicit in (False, True):
        call = trainer.FusedStepCall(net, 2, N_TOTAL, 200.0, 10.0, 57.0, 0.9, None, "cuda", want_wgrad=True,
                                     want_demb=True, seed=4711)
        call.rng_counter.fill_(5)
        nl = nk = None
        if explicit:
            nq = sum(p.numel() for p in net.reconstructor.get_q_params())
            nl = gpu.rng_uniform(4711, 5, 1, 0, emb.numel(), "cuda")
            nk = gpu.rng_uniform(4711, 5, 2, 0, nq, "cuda")
        stats, sums = torch.zeros(7, device="cuda"), torch.zeros(20, dtype=torch.float64, device="cuda")
        call.run(emb, gt, dist, None, 0, gt.sum().reshape(1), stats, sums, 1, noise_latent=nl, noise_kernel=nk)
        res.append((stats.clone(), call.g_emb.clone(), [call.grads[id(p)].clone() for p in net.parameters()],
                    int(call.rng_counter.item())))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    assert all(torch.equal(a, b) for a, b in zip(res[0][2], res[1][2]))
    assert res[0][3] == 6 and res[1][3] == 5            # the counter advances only when the kernels drew from it
    hs, _, w, ws, _ = _steps(True, True, q=1, n=4, lr=0.0)
    assert hs[0, 0] != hs[2, 0] and hs[1, 0] != hs[3, 0] and torch.isfinite(hs).all()
    hs2, _, _, _, _ = _steps(True, True, q=1, n=12, lr=1e-3)
    assert torch.isfinite(hs2).all() and hs2[8:, 0].mean() < hs2[:4, 0].mean()
