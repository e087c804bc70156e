"""The training kernels at the batch sizes where their work schedules change, up to the product batch (16 per GPU).

At one or two blocks every split-K weight-gradient kernel (k_wgrad4_s1 for conv1 / conv2, k_convT5_wgrad for up1 /
up2) gives each persistent CTA at most one work item.  From the batch sizes below on, CTAs loop over several items
and carry their accumulators from one to the next, and the convT grid is rounded to a multiple of the SM count.
These tests run the training path there and check it

1. against the same blocks run one at a time (bit-identical heads and d_latent; each weight gradient equal to the
   float64 sum of the per-block gradients within TAU_SPLIT * S, S the elementwise scale of helpers.oracle_train64),
2. against the float64 oracle at the product batch (TAU_ORACLE * S + S_fwd, S_fwd the part that a float32 forward
   alone can move),
3. through the fused step (nvf_train_step) as the weight loop runs it, against the float64 oracle's raw-parameter
   gradients,
4. in the full-cloud embedding update, where the stem forward switches to its persistent kernel.

test_schedules_loop_at_the_chosen_batches recomputes the launchers' item and grid counts, so that a change of the
dispatch that moves these thresholds fails here instead of silently leaving the loops untested."""
import numpy as np
import pytest
import torch

from oracle import nvf_oracle as O
from oracle.gen_golden import TRAIN_HP, fixture_inputs
from tests import helpers as H

pytestmark = pytest.mark.gpu

N_TOTAL = 849338.0
N_LEAVES = 16                                   # the product batch per GPU (bench.py, trainer.fit)
BATCHES = {"A": (3, 10, 16), "B": (2, 3, 5, 16)}
# The batch decomposition compares the kernels with themselves: only the order of the float32 sums differs, and one
# lost or misrouted work item out of the 2048 of conv2 moves entries by far more than TAU_SPLIT * S.  Against the
# float64 oracle the kernels also carry the error of their float32 forward and data-gradient chain: a float32 CPU
# run of the oracle itself reaches 2.3e-4 * S in config B (up2), and a layout, index or scale error moves entries by
# O(S).  The fused step's raw-parameter gradients (max-normalised) reach 8e-5 in that float32 CPU run.
TAU_SPLIT = 1e-5
TAU_ORACLE = 1e-3
TAU_FUSED = 2e-4                                # raw-parameter gradients of the fused step, against max |ref|

# The split-K weight-gradient kernels of the two shipped configurations (DevLauncher::fast_wgrad in nvf_capi.cu):
# layer -> (kernel, template arguments).  k_wgrad4_s1<C, DG, TYG, MINB>, k_convT5_wgrad<CI, CO, DIN, TYB, CIB, MINB>.
WGRAD_KERNELS = {
    "A": {"conv2": ("wgrad4", (8, 32, 8, 2)), "conv1": ("wgrad4", (8, 16, 8, 2)),
          "up2": ("convT", (8, 8, 16, 4, 8, 3)), "up1": ("convT", (16, 8, 8, 4, 16, 2))},
    "B": {"conv2": ("wgrad4", (16, 32, 4, 2)), "conv1": ("wgrad4", (16, 16, 4, 2)),
          "up2": ("convT", (16, 16, 16, 4, 16, 2)), "up1": ("convT", (32, 16, 8, 4, 16, 2))},
}
K_MAX_PARTIAL_CTAS = 304                        # nvf_api_impl.h kMaxPartialCtas


def schedule(kind, targs, n, sms):
    """(work items, CTAs per channel group, channel groups) of one launch: DevLauncher::wgrad4 / convT_wgrad."""
    if kind == "wgrad4":
        _, dg, tyg, minb = targs
        items = n * dg * (dg // tyg)
        return items, min(sms * minb, items), 1
    ci, co, din, tyb, cib, minb = targs
    groups = (co // 8) * (ci // cib)
    items = n * din * (din // tyb)
    grid = min((sms * minb + groups - 1) // groups, items)
    if grid * groups > K_MAX_PARTIAL_CTAS:
        grid = K_MAX_PARTIAL_CTAS // groups
    if grid * groups > sms:
        grid = (grid * groups // sms) * sms // groups
    return items, grid, groups


def stem_persistent(ch, c0, c1, n, sms):
    """DevLauncher::fast_stem_fwd: whether the stem forward runs its persistent kernel for n blocks."""
    smem = (ch * 8 + 2 * c0 * 64 + c0 * c0 + c0 + ((ch * 125 * c0 + 3) & ~3) + c0 * 75 * c1) * 4
    per_sm = 1 if smem > 110 * 1024 else (2 if smem > 56 * 1024 else 4)
    return n * 8 > sms * per_sm * 2


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


EMB_LEAVES = {"A": 1247, "B": 48}               # A: every leaf of the vox10 shell; B: past its stem threshold (37)


def test_schedules_loop_at_the_chosen_batches(gpu):
    sms = _sms()
    for tag, kernels in WGRAD_KERNELS.items():
        for layer, (kind, targs) in kernels.items():
            loops = [n for n in range(1, N_LEAVES + 1) if schedule(kind, targs, n, sms)[0] > schedule(kind, targs, n, sms)[1]]
            assert loops, (tag, layer)
            assert 1 not in loops, (tag, layer)                            # the one-block reference never loops
            assert min(loops) in BATCHES[tag], (tag, layer, min(loops))    # the first batch where CTAs loop is tested
            assert N_LEAVES in loops, (tag, layer)
        # the convT grid rounding to a multiple of the SM count happens at some tested batch, and so does an uneven
        # tail (some CTAs own one item more than others)
        rounded, uneven = False, False
        for n in BATCHES[tag]:
            for kind, targs in kernels.values():
                items, grid, groups = schedule(kind, targs, n, sms)
                if kind == "convT" and grid * groups % sms == 0 and grid < items:
                    rounded = True
                uneven |= items > grid and items % grid != 0
        assert rounded and uneven, tag
    for tag, (c0, c1) in (("A", (8, 16)), ("B", (16, 32))):
        assert stem_persistent(3, c0, c1, EMB_LEAVES[tag], sms) and not stem_persistent(3, c0, c1, 1, sms), tag


# --------------------------------------------------------------------------------------------------- inputs
_CASES = {}


def _case(tag):
    """Per configuration: the perturbed fixture state, 16 real leaves spread over the vox10 shell (gt / dist from the
    host cKDTree), integer latents, fixed random cotangents of the three heads, and the float64 oracle of each block
    alone under those cotangents (its gradients and scales S add up to any batch of them)."""
    if tag in _CASES:
        return _CASES[tag]
    from nvfpcc_b200 import synth
    fx = fixture_inputs(tag)
    pts = synth.sphere_shell_points(1024)
    origins = synth.leaf_origins(pts)
    pick = np.unique(np.linspace(0, origins.shape[0] - 1, N_LEAVES).round().astype(np.int64))
    assert pick.shape[0] == N_LEAVES
    gt, dist = synth.gt_and_dist(pts, origins[pick])
    g = torch.Generator().manual_seed(11)
    latent = torch.round(torch.randn(N_LEAVES, fx["ch"], 2, 2, 2, generator=g) * 3)
    cot = [torch.randn(N_LEAVES, 1, d, d, d, generator=g) for d in (32, 16, 8)]
    per_block = [H.oracle_train64(fx["sd"], latent[b:b + 1], cot=[c[b:b + 1] for c in cot]) for b in range(N_LEAVES)]
    c = dict(fx=fx, w=H.eff_weights(fx["sd"], 2, "cuda"), latent=latent, cot=cot,
             gt=torch.from_numpy(gt).float(), dist=torch.from_numpy(dist).float(),
             S_block=[r["S"] for r in per_block])
    _CASES[tag] = c
    return c


def _run(gpu, c, latent, cot, wgrad=True):
    desc = gpu.desc(c["fx"]["ch"], c["fx"]["channels"])
    lat = latent.cuda()
    out, cls1, cls0, ws, _ = gpu.train_forward(desc, c["w"], lat)
    g_lat, grads = gpu.train_backward(desc, c["w"], lat, ws, *[t.cuda() for t in cot], wgrad, True)
    return out, cls1, cls0, g_lat, grads, ws


_BLOCKS = {}


def _one_at_a_time(gpu, tag, c):
    """Every leaf run alone (n = 1: no kernel loops): heads, d_latent and weight gradients."""
    if tag not in _BLOCKS:
        res = []
        for b in range(N_LEAVES):
            out, cls1, cls0, g_lat, grads, _ = _run(gpu, c, c["latent"][b:b + 1], [t[b:b + 1] for t in c["cot"]])
            res.append(dict(out=out.cpu(), cls1=cls1.cpu(), cls0=cls0.cpu(), g_lat=g_lat.cpu(),
                            grads={k: v.double().cpu() for k, v in grads.items()}))
        _BLOCKS[tag] = res
    return _BLOCKS[tag]


# --------------------------------------------------------------------------------------------------- 1.
@pytest.mark.parametrize("tag,n", [(t, n) for t in "AB" for n in BATCHES[t]])
def test_batch_equals_its_blocks_one_at_a_time(gpu, tag, n):
    """A batch of n leaves against the same leaves one at a time: heads and d_latent bit-identical, every weight
    gradient equal to the float64 sum of the per-leaf gradients within TAU_SPLIT * S, and a second backward over the
    same forward bit-identical to the first (the split-K partials are summed in a fixed order)."""
    c = _case(tag)
    blocks = _one_at_a_time(gpu, tag, c)
    lat, cot = c["latent"][:n], [t[:n] for t in c["cot"]]
    out, cls1, cls0, g_lat, grads, ws = _run(gpu, c, lat, cot)
    desc = gpu.desc(c["fx"]["ch"], c["fx"]["channels"])
    g_lat2, grads2 = gpu.train_backward(desc, c["w"], lat.cuda(), ws, *[t.cuda() for t in cot], True, True)
    torch.cuda.synchronize()
    assert torch.equal(g_lat, g_lat2)
    for k in grads:
        assert torch.equal(grads[k], grads2[k]), "backward is not repeatable: " + k
    for name, t in (("out", out), ("cls1", cls1), ("cls0", cls0), ("g_lat", g_lat)):
        t = t.cpu()
        for b in range(n):
            assert torch.equal(t[b:b + 1], blocks[b][name]), "%s of leaf %d differs from its one-leaf run" % (name, b)
    worst = {}
    for k, gv in grads.items():
        ref = sum(blocks[b]["grads"][k] for b in range(n))
        S = sum(c["S_block"][b][k] for b in range(n))
        worst[k] = H.scaled_err(gv, ref, S)
    print("split %s n=%d worst |err|/S: %s" % (tag, n, " ".join("%s=%.2e" % kv for kv in worst.items())))
    bad = {k: v for k, v in worst.items() if not v <= TAU_SPLIT}
    assert not bad, "batch of %d against its leaves one at a time, |err| / S above %g: %s" % (n, TAU_SPLIT, bad)


# --------------------------------------------------------------------------------------------------- 2.
@pytest.mark.parametrize("tag", ["A", "B"])
def test_product_batch_matches_float64_oracle(gpu, tag):
    """nvf_train_forward, nvf_loss_seeds and nvf_train_backward on 16 real leaves against the float64 oracle of the
    training loss: probabilities of the three heads within the logit band, the loss sums, every effective-weight
    gradient per element within TAU_ORACLE * S + S_fwd and d_latent within TAU_ORACLE * S."""
    c = _case(tag)
    desc = gpu.desc(c["fx"]["ch"], c["fx"]["channels"])
    lat = c["latent"].cuda()
    out, cls1, cls0, ws, _ = gpu.train_forward(desc, c["w"], lat)
    sums, seeds = gpu.loss_seeds(out, cls1, cls0, c["gt"].cuda(), c["dist"].cuda(), 0.9, 0.85, 0.6)
    g_lat, grads = gpu.train_backward(desc, c["w"], lat, ws, seeds[0], seeds[1], seeds[2], True, True)
    r = H.oracle_train64(c["fx"]["sd"], c["latent"], c["gt"], c["dist"])
    H.assert_prob_close(out, r["logit2"], "out")
    H.assert_prob_close(cls1, r["logit1"], "cls1")
    H.assert_prob_close(cls0, r["logit0"], "cls0")
    sums = sums.cpu().numpy()
    rel = [abs(sums[i] - r["sums"][i]) / abs(r["sums"][i]) for i in range(3)]
    per_s = {k: H.scaled_err(gv, r["grads"][k], r["S"][k]) for k, gv in grads.items()}
    per_s["d_latent"] = H.scaled_err(g_lat, r["d_latent"], r["S"]["d_latent"])
    used = {k: H.scaled_err(gv, r["grads"][k], TAU_ORACLE * r["S"][k] + r["S_fwd"][k]) for k, gv in grads.items()}
    used["d_latent"] = per_s["d_latent"] / TAU_ORACLE
    print("oracle %s n=%d loss rel err %s worst |err|/S: %s; share of the bound: %s" % (
        tag, N_LEAVES, ["%.2e" % e for e in rel], " ".join("%s=%.2e" % kv for kv in per_s.items()),
        " ".join("%s=%.2f" % kv for kv in used.items())))
    assert max(rel) <= 2e-5, rel
    bad = {k: v for k, v in used.items() if not v <= 1.0}
    assert not bad, "16 leaves against the float64 oracle, |err| above TAU_ORACLE * S + S_fwd (share): %s" % bad


# --------------------------------------------------------------------------------------------------- 3.
@pytest.mark.parametrize("tag", ["A", "B"])
def test_fused_step_at_product_batch_matches_float64_oracle(gpu, tag):
    """nvf_train_step through trainer.FusedStepCall at 16 leaves, q = 1 with explicit latent and kernel noise (the
    phase bench.py runs), against O.net_forward + O.train_loss in float64: the loss and its bce / ms0 / ms1 terms,
    d_emb and all 28 raw-parameter gradients.  At 16 leaves the loss kernel runs 256 CTAs, the last of which
    finalises the sums."""
    from nvfpcc_b200 import network, synth, trainer
    c = _case(tag)
    fx = c["fx"]
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=fx["ch"], channel_str=",".join(str(x) for x in fx["channels"]))
    net.load_state_dict(fx["sd"])
    net = net.cuda()
    g = torch.Generator().manual_seed(23)
    emb = torch.ones(N_LEAVES, fx["ch"], 2, 2, 2) + torch.randn(N_LEAVES, fx["ch"], 2, 2, 2, generator=g) * 2.0
    nl = torch.rand(emb.shape, generator=g)
    kn = {k: torch.rand(fx["sd"]["reconstructor.%s.kernel" % k].shape, generator=g) for k in O.Q_KERNEL_LAYERS}
    gt, dist = c["gt"], c["dist"]
    call = trainer.FusedStepCall(net, N_LEAVES, N_TOTAL, TRAIN_HP["lmbda"], TRAIN_HP["w1"], TRAIN_HP["w2"], 0.9, None,
                                 "cuda", want_wgrad=True, want_demb=True)
    stats, sums = torch.zeros(7, device="cuda"), torch.zeros(20, dtype=torch.float64, device="cuda")
    call.run(emb.cuda(), gt.cuda(), dist.cuda(), None, 0, gt.sum().reshape(1).cuda(), stats, sums, 1,
             noise_latent=nl.cuda(), noise_kernel=torch.cat([kn[k].reshape(-1) for k in O.Q_KERNEL_LAYERS]).cuda())
    st = stats.cpu().double()

    sd = {k: v.double().requires_grad_(not (k.endswith("_init") or k.endswith("pedestal"))) for k, v in fx["sd"].items()}
    emb_o = emb.double().requires_grad_(True)
    res = O.net_forward(emb_o, sd, "train", 1, latent_noise=nl.double(), kernel_noises={k: v.double() for k, v in kn.items()})
    L = O.train_loss(res, gt.double(), dist.double(), n_pts=gt.double().sum(), n_total=N_TOTAL, **TRAIN_HP)
    L["loss"].backward()
    rel = {k: abs(float(st[i]) - float(L[k])) / abs(float(L[k])) for i, k in enumerate(("loss", "bce", "ms0", "ms1"))}

    def err(got, ref):
        got, ref = got.detach().cpu().double().reshape(-1), ref.detach().double().reshape(-1)
        scale = float(ref.abs().max())
        return float((got - ref).abs().max()) / scale if scale > 0 else (0.0 if float(got.abs().max()) == 0 else 1.0)

    worst = {"d_emb": err(call.g_emb, emb_o.grad)}
    k = 0
    for name, p in net.named_parameters():
        ref = sd[name].grad
        worst[name] = err(call.grads[id(p)], torch.zeros_like(sd[name]) if ref is None else ref)
        k += 1
    assert k == 28
    print("fused %s n=%d loss rel err %s worst err/max|ref|: %s" % (
        tag, N_LEAVES, {a: "%.2e" % b for a, b in rel.items()}, " ".join("%s=%.2e" % kv for kv in worst.items())))
    assert max(rel.values()) <= 2e-5, rel
    bad = {a: b for a, b in worst.items() if not b <= TAU_FUSED}
    assert not bad, "fused step at 16 leaves against the float64 oracle, err / max|ref| above %g: %s" % (TAU_FUSED, bad)


# --------------------------------------------------------------------------------------------------- 4.
@pytest.mark.parametrize("tag", ["A", "B"])
def test_embedding_update_over_the_whole_cloud(gpu, tag):
    """The once-per-epoch embedding update (trainer.EmbeddingStep): forward and d_latent-only backward over the whole
    cloud at once, where the stem forward runs persistent CTAs.  Nothing is summed across blocks, so a sample of
    blocks (first, last and 14 between) is checked bit-for-bit against one-block runs and against the float64
    oracle (probabilities in the logit band, d_latent within TAU_ORACLE * S)."""
    c = _case(tag)
    fx = c["fx"]
    n = EMB_LEAVES[tag]
    g = torch.Generator().manual_seed(31)
    latent = torch.round(torch.randn(n, fx["ch"], 2, 2, 2, generator=g) * 3)
    cot = [torch.randn(n, 1, d, d, d, generator=g) for d in (32, 16, 8)]
    out, cls1, cls0, g_lat, grads, _ = _run(gpu, c, latent, cot, wgrad=False)
    assert not grads
    got = [t.cpu() for t in (out, cls1, cls0, g_lat)]
    pick = np.unique(np.linspace(0, n - 1, 16).round().astype(np.int64))
    for b in pick:
        one = _run(gpu, c, latent[b:b + 1], [t[b:b + 1] for t in cot], wgrad=False)
        for name, t, o in zip(("out", "cls1", "cls0", "d_latent"), got, one[:4]):
            assert torch.equal(t[b:b + 1], o.cpu()), "%s of block %d of %d differs from its one-block run" % (name, b, n)
    idx = torch.from_numpy(pick)
    r = H.oracle_train64(fx["sd"], latent[idx], cot=[t[idx] for t in cot])
    H.assert_prob_close(got[0][idx], r["logit2"], "out")
    H.assert_prob_close(got[1][idx], r["logit1"], "cls1")
    H.assert_prob_close(got[2][idx], r["logit0"], "cls0")
    e = H.scaled_err(got[3][idx], r["d_latent"], r["S"]["d_latent"])
    print("embedding %s n=%d worst d_latent |err|/S: %.2e" % (tag, n, e))
    assert e <= TAU_ORACLE, e
