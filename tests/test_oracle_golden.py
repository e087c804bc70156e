"""Pins oracle/nvf_oracle.py to the golden vectors produced from the unmodified
reference modules (oracle/gen_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import nvf_oracle as O
from oracle.gen_golden import GOLDEN_THREADS, TRAIN_HP, fixture_inputs, state_checksum


@pytest.fixture(autouse=True, scope="module")
def golden_threads():
    """The golden float32 outputs are bit-exact only under the summation order they were made with, and the CPU
    convolutions split their work - and so their sums - by the number of threads: run the oracle with that count."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("tag", ["A", "B"])
def test_fixture_inputs_reproducible(tag, golden_A, golden_B):
    g = golden_A if tag == "A" else golden_B
    fx = fixture_inputs(tag)
    assert state_checksum(fx["sd"]) == pytest.approx(float(g["state_checksum"]), rel=0, abs=0)
    sd0 = O.make_state(fx["ch"], fx["channels"], __import__("nvfpcc_b200.synth", fromlist=["x"]).synthetic_seed())
    assert int(sd0["_seed_consumed"]) == int(g["seed_consumed"])
    assert int(g["seed_consumed"]) == (52127 if tag == "A" else 200623)  # SURVEY.md 8(a) a16


@pytest.mark.parametrize("tag", ["A", "B"])
def test_decode_matches_reference(tag, golden_A, golden_B):
    g = golden_A if tag == "A" else golden_B
    fx = fixture_inputs(tag)
    with torch.no_grad():
        w = O.effective_decoder_weights(fx["sd"], q=2)
        out, _, _, logit, inter = O.decoder_forward(fx["latents"], w, aux=False, keep=True)
    np.testing.assert_array_equal(out.numpy(), g["dec_out"])
    np.testing.assert_array_equal(logit.numpy(), g["dec_logit"])
    for name in ("a1", "a2", "a3", "a4", "a5"):
        assert inter[name].double().sum().item() == pytest.approx(float(g["dec_" + name + "_sum"]), rel=1e-12)


def test_train_step_matches_reference(golden_A):
    g = golden_A
    fx = fixture_inputs("A")
    sd = {k: v.clone().requires_grad_(not (k.endswith("_init") or k.endswith("pedestal"))) for k, v in fx["sd"].items()}
    emb = fx["emb"].clone().requires_grad_(True)
    gt = torch.from_numpy(g["tr_gt"]).float()
    dist = torch.from_numpy(g["tr_dist"]).float()
    res = O.net_forward(emb, sd, "train", 2, latent_noise=torch.from_numpy(g["tr_latent_noise"]))
    L = O.train_loss(res, gt, dist, n_pts=gt.sum(), n_total=849338.0, **TRAIN_HP)
    L["loss"].backward()
    np.testing.assert_allclose(res["out"].detach().numpy(), g["tr_out"], rtol=0, atol=0)
    np.testing.assert_allclose(res["cls"][0].detach().numpy(), g["tr_cls0"], rtol=0, atol=0)
    np.testing.assert_allclose(res["cls"][1].detach().numpy(), g["tr_cls1"], rtol=0, atol=0)
    np.testing.assert_allclose(res["net_bits"].detach().numpy(), g["tr_net_bits"], rtol=1e-6)
    assert res["latent_bits"].item() == pytest.approx(float(g["tr_latent_bits"]), rel=1e-6)
    for k in ("loss", "bce", "ms0", "ms1"):
        assert L[k].item() == pytest.approx(float(g["tr_" + k]), rel=1e-6), k
    np.testing.assert_allclose(emb.grad.numpy(), g["tr_grad_emb"], rtol=1e-5, atol=1e-7)
    n = 0
    for key in g.files:
        if not key.startswith("tr_grad::"):
            continue
        name = key[len("tr_grad::"):]
        got = sd[name].grad
        got = torch.zeros_like(sd[name]) if got is None else got
        ref = g[key]
        scale = max(1e-6, float(np.abs(ref).max()))
        np.testing.assert_allclose(got.numpy(), ref, rtol=1e-4, atol=1e-5 * scale, err_msg=name)
        n += 1
    assert n == 28
    sse, denom = O.sse1(res["out"].detach(), dist, 0.6)
    assert sse.item() == pytest.approx(float(g["tr_sse"]), rel=1e-6)
    assert denom.item() == float(g["tr_denom"])
    pacc, nacc, _ = O.acc_dense(res["out"].detach(), gt)
    assert pacc.item() == pytest.approx(float(g["tr_pacc"]), rel=1e-6)
    assert nacc.item() == pytest.approx(float(g["tr_nacc"]), rel=1e-6)


def test_threshold_points_order():
    p = torch.zeros(2, 1, 32, 32, 32)
    p[0, 0, 1, 2, 3] = 0.9
    p[0, 0, 0, 31, 31] = 0.7
    p[1, 0, 5, 0, 0] = 0.66
    p[1, 0, 5, 0, 1] = 0.65  # strict '>' (NVFPCC.py:632)
    pts, counts = O.threshold_points(p, np.array([[32, 64, 96], [0, 0, 0]]), 0.65)
    assert counts.tolist() == [2, 1]
    assert pts.tolist() == [[32, 95, 127], [33, 66, 99], [5, 0, 0]]


@pytest.fixture(scope="module")
def golden_train2():
    import os
    from tests.conftest import GOLDEN
    return {tag: np.load(os.path.join(GOLDEN, "nvf_train2_%s.npz" % tag)) for tag in "AB"}


@pytest.mark.parametrize("tag,q", [("A", 1), ("B", 2)])
def test_train_step_q1_A_and_q2_B_match_reference(golden_train2, tag, q):
    """The two extra reference steps (oracle/gen_golden.py gen_train2): config A in the noisy-kernel phase
    (q=1, the phase bench.py runs) with the reference's own uniform draws replayed, and config B at q=2."""
    g, pre = golden_train2[tag], "%sq%d_" % (tag, q)
    fx = fixture_inputs(tag)
    sd = {k: v.clone().requires_grad_(not (k.endswith("_init") or k.endswith("pedestal"))) for k, v in fx["sd"].items()}
    emb = fx["emb"].clone().requires_grad_(True)
    gt, dist = torch.from_numpy(g[pre + "gt"]).float(), torch.from_numpy(g[pre + "dist"]).float()
    noises = {n: torch.from_numpy(g[pre + "knoise::" + n]) for n in O.Q_KERNEL_LAYERS} if q == 1 else None
    res = O.net_forward(emb, sd, "train", q, latent_noise=torch.from_numpy(g[pre + "latent_noise"]),
                        kernel_noises=noises)
    L = O.train_loss(res, gt, dist, n_pts=gt.sum(), n_total=849338.0, **TRAIN_HP)
    L["loss"].backward()
    np.testing.assert_allclose(res["out"].detach().numpy(), g[pre + "out"], rtol=0, atol=0)
    np.testing.assert_allclose(res["net_bits"].detach().numpy(), g[pre + "net_bits"], rtol=1e-6)
    for k in ("loss", "bce", "ms0", "ms1"):
        assert L[k].item() == pytest.approx(float(g[pre + k]), rel=1e-6), k
    np.testing.assert_allclose(emb.grad.numpy(), g[pre + "grad_emb"], rtol=1e-5, atol=1e-7)
    n = 0
    for key in g.files:
        if not key.startswith(pre + "grad::"):
            continue
        name = key[len(pre + "grad::"):]
        got = sd[name].grad
        got = torch.zeros_like(sd[name]) if got is None else got
        ref = g[key]
        np.testing.assert_allclose(got.numpy(), ref, rtol=1e-4, atol=1e-5 * max(1e-6, float(np.abs(ref).max())),
                                   err_msg=name)
        n += 1
    assert n == 28
