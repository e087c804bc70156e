"""CPU tier for the ground-truth grid / distance-field builder (SURVEY.md 8f row 1):
the oracle against the fixture produced by the unmodified reference script, the host-side
file front end, and the C-ABI exports of include/nvf_prep_b200.h (no compute calls)."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import grids_oracle as GO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "grids_small.npz"))


def golden_dist(g):
    n = g["origins"].shape[0]
    dist = np.sqrt(g["d2"].astype(np.float64)).reshape(n, 1, 32, 32, 32)
    gt = np.unpackbits(g["gt"])[: n * 32768].reshape(n, 1, 32, 32, 32)
    return gt, dist


def test_fixture_is_what_the_reference_writes(golden):
    assert str(golden["dist_dtype"]) == "float64" and str(golden["gt_dtype"]) == "uint8"
    assert str(golden["origins_saved_dtype"]) == "float64"          # np.loadtxt -> np.save, util_get_grids.py:16-17
    assert np.array_equal(golden["origins_saved"], golden["origins"].astype(np.float64))
    gt, dist = golden_dist(golden)
    assert np.array_equal(gt, (dist == 0).astype(np.uint8))
    assert dist.max() > 32.0                                        # a nearest point beyond the own leaf is exercised


def test_kdtree_oracle_matches_reference_output(golden):
    gt, dist = GO.build_grids(golden["points"], golden["origins"])
    gt_ref, dist_ref = golden_dist(golden)
    assert dist.dtype == np.float64 and gt.dtype == np.uint8
    assert np.array_equal(dist, dist_ref)                           # bit-exact float64
    assert np.array_equal(gt, gt_ref)


def test_bruteforce_oracle_matches_reference_output(golden):
    sel = [4]                                                      # the sparse leaf: 3 candidate points matter
    pts = golden["points"]
    near = pts[np.abs(pts - (golden["origins"][4] + 16)).max(1) < 16 + 54]
    gt, dist = GO.build_grids_bruteforce(near, golden["origins"][sel])
    gt_ref, dist_ref = golden_dist(golden)
    assert np.array_equal(dist, dist_ref[sel]) and np.array_equal(gt, gt_ref[sel])


def test_ply_reader_ascii_and_binary(tmp_path):
    from nvfpcc_b200 import grids
    pts = np.array([[1, 2, 3], [400, 5, 6], [7, 800, 1023]], dtype=np.float64)
    a = tmp_path / "a.ply"
    a.write_text("ply\nformat ascii 1.0\ncomment x\nelement vertex 3\nproperty float x\nproperty float y\n"
                 "property float z\nproperty uchar red\nend_header\n" +
                 "".join("%d %d %d 9\n" % tuple(p) for p in pts))
    assert np.array_equal(grids.read_ply_xyz(str(a)), pts)
    rec = np.zeros(3, dtype=[("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("red", "u1")])
    rec["x"], rec["y"], rec["z"] = pts[:, 0], pts[:, 1], pts[:, 2]
    b = tmp_path / "b.ply"
    b.write_bytes(b"ply\nformat binary_little_endian 1.0\nelement vertex 3\nproperty float x\nproperty float y\n"
                  b"property float z\nproperty uchar red\nelement face 0\nproperty list uchar int vertex_indices\n"
                  b"end_header\n" + rec.tobytes())
    assert np.array_equal(grids.read_ply_xyz(str(b)), pts)


def declared_functions():
    src = open(os.path.join(ROOT, "include", "nvf_prep_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nvf_[a-z0-9_]+)\s*\(", src)))


def test_prep_header_symbols_are_exported_and_bound():
    from nvfpcc_b200 import build, entropy, grids, trainer
    names = declared_functions()
    assert sorted(grids.EXPORTS + entropy.EXPORTS + trainer.EXPORTS) == names
    lib = ctypes.CDLL(build.build())
    for n in names:
        assert hasattr(lib, n), n
    out = ctypes.c_size_t(0)
    lib.nvf_grids_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.POINTER(ctypes.c_size_t)]
    assert lib.nvf_grids_workspace_bytes(1247, ctypes.byref(out)) == 0 and out.value > 1247 * 4096
    assert lib.nvf_grids_workspace_bytes(0, ctypes.byref(out)) == -1


def test_grids_have_no_cpu_fallback():
    from tests.helpers import run_without_gpu
    run_without_gpu("import numpy as np, pytest, torch\n"
                    "from nvfpcc_b200 import grids\n"
                    "assert not torch.cuda.is_available()\n"
                    "with pytest.raises(RuntimeError):\n"
                    "    grids.build_grids(np.zeros((1, 3), np.int32), np.zeros((1, 3), np.int32))\n")
