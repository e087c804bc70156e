"""Kernel-logic tests on the CPU emulator (tests/emu): the same generic layer kernels,
point emission and host orchestration as the CUDA library, executed sequentially,
checked against the oracle.  Decode runs layer-wise here for every configuration
(the fused decode head is CUDA-only).  The `-m gpu` tests repeat these checks on
the real device."""
import numpy as np
import pytest
import torch

from oracle import nvf_oracle as O
from oracle.gen_golden import TRAIN_HP, fixture_inputs
from tests.emu import emu_backend
from tests.helpers import eff_weights, check_decode_against_oracle, check_train_against_oracle


@pytest.fixture(scope="module")
def emu():
    return emu_backend.binding()


def test_decode_layerwise_A_matches_oracle_and_golden(emu, golden_A):
    fx = fixture_inputs("A")
    lat = torch.cat([fx["latents"], fx["latents"].flip(0) * 0.5 + 1, fx["latents"][:1] * -1.0], 0).round()
    check_decode_against_oracle(emu, fx, lat, thh=0.5, golden=golden_A, dev="cpu")


def test_decode_layerwise_B_matches_oracle_and_golden(emu, golden_B):
    fx = fixture_inputs("B")
    check_decode_against_oracle(emu, fx, fx["latents"], thh=0.5, golden=golden_B, dev="cpu")


def test_decode_empty_and_cap_overflow(emu):
    fx = fixture_inputs("A")
    desc = emu.desc(fx["ch"], fx["channels"])
    w = eff_weights(fx["sd"], 2, "cpu")
    r = emu.decode(desc, w, torch.zeros(0, 3, 2, 2, 2), torch.zeros(0, 3, dtype=torch.int32), 0.5)
    assert r["coords"].shape == (0, 3) and int(r["total"]) == 0
    lat = fx["latents"][:1]
    full = emu.decode(desc, w, lat, None, 0.3)
    small = emu.decode(desc, w, lat, None, 0.3, cap=5)  # forces the nvf_emit_points retry path
    assert int(full["total"]) > 5
    assert torch.equal(full["coords"], small["coords"])


def test_train_forward_backward_A(emu, golden_A):
    check_train_against_oracle(emu, fixture_inputs("A"), golden_A, dev="cpu")
