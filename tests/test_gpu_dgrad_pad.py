"""The x pitch of the conv2 / conv1 data gradients g4 = [n][c3][35][35][36] and g2 = [n][c2][19][19][20] is padded
to a multiple of four.  k_convT5_dgrad, k_convT5_wgrad and k_chansum_fast read whole float4 rows of them, so the pad
column has to be exactly zero after the backward, whatever the buffer held before.  This test fills both tensors
with NaN between the forward and the backward and checks the pad column and the data columns afterwards.

The offsets mirror TrainWs / Stash / GenericPacked (nvf_api_impl.h, nvf_layers.h): the workspace starts with the
packed weights, then the activation stash, then the gradient stash of the same layout."""
import pytest
import torch

from oracle.gen_golden import fixture_inputs
from tests import helpers as H

pytestmark = pytest.mark.gpu

CONV_W = ("up0_w", "conv0_w", "up1_w", "conv1_w", "up2_w", "conv2_w", "cls2_w", "cls1_w", "cls0_w")


def _align(v):
    return (v + 255) // 256 * 256


def _r4(v):
    return (v + 3) // 4 * 4


def _grad_views(ws, w, channels, n):
    c0, c1, c2, c3 = channels
    packed = sum(2 * _r4(w[k].numel()) for k in CONV_W) + _r4(c3 * 36)
    a2 = 2 * c0 * 64 + c1 * 512
    a4 = a2 + c2 * 19 * 19 * 20 + c2 * 4096
    per_block = a4 + c3 * 35 * 35 * 36 + c3 * 32768
    off_grad = _align(4 * packed) + _align(4 * per_block * n)
    grad = ws[off_grad:off_grad + 4 * per_block * n].view(torch.float32)
    g2 = grad[a2 * n:a2 * n + n * c2 * 19 * 19 * 20].view(n, c2, 19, 19, 20)
    g4 = grad[a4 * n:a4 * n + n * c3 * 35 * 35 * 36].view(n, c3, 35, 35, 36)
    return g2, g4


@pytest.mark.parametrize("tag", ["A", "B"])
def test_dgrad_pad_column_is_zero(gpu, tag):
    dev = torch.device("cuda:0")
    fx = fixture_inputs(tag)
    desc = gpu.desc(fx["ch"], fx["channels"])
    w = H.eff_weights(fx["sd"], 2, dev)
    n = 3
    g = torch.Generator().manual_seed(17)
    latent = torch.round(torch.randn(n, fx["ch"], 2, 2, 2, generator=g) * 3).to(dev)
    cot = [torch.randn(n, 1, d, d, d, generator=g).to(dev) for d in (32, 16, 8)]
    out, cls1, cls0, ws, keep = gpu.train_forward(desc, w, latent)
    g2, g4 = _grad_views(ws, w, fx["channels"], n)
    g2.fill_(float("nan"))
    g4.fill_(float("nan"))
    gpu.train_backward(desc, w, latent, ws, cot[0], cot[1], cot[2], True, True)
    torch.cuda.synchronize()
    for name, t, d in (("g2", g2, 19), ("g4", g4, 35)):
        assert torch.equal(t[..., d:], torch.zeros_like(t[..., d:])), name + " pad column"
        assert torch.isfinite(t[..., :d]).all(), name + " data columns"
        assert t[..., :d].abs().max() > 0, name
    del keep
