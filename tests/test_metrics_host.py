"""CPU tier of the distortion metrics: the C-ABI exports of include/nvf_metrics_b200.h and its workspace queries
(no device needed), the oracle against its brute-force form and against the host helpers, the PLY vertex reader,
and the absence of a CPU fallback."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import metrics_oracle as MO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "nvf_metrics_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nvf_[a-z0-9_]+)\s*\(", src)))


def test_metrics_header_symbols_are_exported_and_bound():
    from nvfpcc_b200 import build, metrics
    names = declared_functions()
    assert sorted(metrics.EXPORTS) == names
    lib = ctypes.CDLL(build.build())
    for n in names:
        assert hasattr(lib, n), n


def test_workspace_queries_need_no_device():
    from nvfpcc_b200 import build
    lib = ctypes.CDLL(build.build())
    sz = ctypes.c_size_t
    lib.nvf_nn_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.POINTER(sz)]
    lib.nvf_distortion_workspace_bytes.argtypes = [ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(sz)]
    out = sz(0)
    assert lib.nvf_nn_workspace_bytes(849338, ctypes.byref(out)) == 0 and out.value > 849338 * 24
    small = out.value
    assert lib.nvf_distortion_workspace_bytes(849338, 800000, ctypes.byref(out)) == 0 and out.value > small
    assert lib.nvf_nn_workspace_bytes(1, ctypes.byref(out)) == 0 and out.value > 0
    for bad in (0, -1, 1 << 31):
        assert lib.nvf_nn_workspace_bytes(bad, ctypes.byref(out)) == -1
        assert lib.nvf_distortion_workspace_bytes(bad, 10, ctypes.byref(out)) == -1
        assert lib.nvf_distortion_workspace_bytes(10, bad, ctypes.byref(out)) == -1
    assert lib.nvf_nn_workspace_bytes(10, None) == -1


def tie_heavy_cloud(rng, n, lo=-3, hi=3):
    """Points in a 6^3 box (negative coordinates included) with duplicates."""
    p = rng.integers(lo, hi, size=(n, 3))
    dup = rng.integers(0, n, size=max(1, n // 5))
    return np.concatenate([p, p[dup]], 0)


def unit_normals(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_bruteforce_on_tie_heavy_clouds(seed):
    rng = np.random.default_rng(seed)
    src = tie_heavy_cloud(rng, int(rng.integers(1, 60)))
    rec = tie_heavy_cloud(rng, int(rng.integers(1, 60)))
    if seed == 0:
        rec = rec[:1]                                              # n_target = 1
    nrm = unit_normals(rng, src.shape[0])
    for k in (1, 2, 8):                                            # small k: the ball-query fallback runs often
        for t, q in ((rec, src), (src, rec)):
            a, b = MO.nearest(t, q, k=k), MO.nearest_bruteforce(t, q)
            for key in ("index", "d2", "ties", "offsets", "members"):
                assert np.array_equal(a[key], b[key]), key
    assert (MO.nearest_bruteforce(rec, src)["ties"] > 1).any() or seed == 0
    r, rb = MO.distortion(src, rec, 6.0, nrm), MO.distortion(src, rec, 6.0, nrm, nn=MO.nearest_bruteforce)
    for key in ("d1_sum", "hausdorff_d2", "d2_sum"):
        assert r[key] == rb[key], key
    assert MO.nearest(rec, np.zeros((0, 3), np.int64))["d2"].shape == (0,)


def test_oracle_agrees_with_host_helpers():
    """D1 equals a plain cKDTree D1; with no ties anywhere, D2 equals the tests' existing psnr_d1_d2 formula."""
    from scipy.spatial import cKDTree

    from tests.test_gpu_parity2 import _sphere_normals, psnr_d1_d2
    rng = np.random.default_rng(7)
    centre = np.array([200.0, 200.0, 200.0])
    v = rng.normal(size=(3000, 3))
    src = np.rint(centre + 150 * v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.int64)
    src = np.unique(src, axis=0)
    rec = src + rng.integers(-2, 3, size=src.shape)
    nrm = _sphere_normals(src, centre)
    for _ in range(10):                                            # drop the queries with ties until none is left
        r = MO.distortion(src, rec, 1023.0, nrm)
        a, b = r["nn"]
        if (a["ties"] == 1).all() and (b["ties"] == 1).all():
            break
        keep_s, keep_r = a["ties"] == 1, b["ties"] == 1
        src, nrm, rec = src[keep_s], nrm[keep_s], rec[keep_r]
    assert (a["ties"] == 1).all() and (b["ties"] == 1).all() and src.shape[0] > 2500
    d_sr = cKDTree(rec).query(src)[0]
    d_rs = cKDTree(src).query(rec)[0]
    assert r["d1"] == pytest.approx(max((d_sr ** 2).mean(), (d_rs ** 2).mean()), rel=1e-12)
    d1_ref, d2_ref = psnr_d1_d2(rec, src, centre, 1023.0)
    assert abs(r["d1_psnr"] - d1_ref) <= 1e-9
    assert abs(r["d2_psnr"] - d2_ref) <= 1e-9


def test_ply_vertex_reader_ascii_and_binary(tmp_path):
    from nvfpcc_b200 import grids
    pts = np.array([[1, 2, 3], [400, 5, 6], [7, 800, 1023]], dtype=np.float64)
    nrm = np.array([[1, 0, 0], [0, 0.6, 0.8], [0, -1, 0]], dtype=np.float64)
    a = tmp_path / "a.ply"
    a.write_text("ply\nformat ascii 1.0\nelement vertex 3\nproperty float x\nproperty float y\nproperty float z\n"
                 "property float nx\nproperty float ny\nproperty float nz\nend_header\n" +
                 "".join("%d %d %d %g %g %g\n" % (tuple(p) + tuple(n)) for p, n in zip(pts, nrm)))
    rec = np.zeros(3, dtype=[("x", "<i4"), ("y", "<i4"), ("z", "<i4"), ("nx", "<f8"), ("ny", "<f8"), ("nz", "<f8")])
    for i, k in enumerate("xyz"):
        rec[k] = pts[:, i]
        rec["n" + k] = nrm[:, i]
    b = tmp_path / "b.ply"
    b.write_bytes(b"ply\nformat binary_little_endian 1.0\nelement vertex 3\nproperty int x\nproperty int y\n"
                  b"property int z\nproperty double nx\nproperty double ny\nproperty double nz\nend_header\n" +
                  rec.tobytes())
    for path in (a, b):
        v = grids.read_ply_vertex(str(path))
        assert sorted(v) == ["nx", "ny", "nz", "x", "y", "z"]
        assert np.array_equal(np.stack([v[k] for k in "xyz"], 1), pts)
        assert np.array_equal(np.stack([v[k] for k in ("nx", "ny", "nz")], 1), nrm)
        assert np.array_equal(grids.read_ply_xyz(str(path)), pts)


def test_metrics_have_no_cpu_fallback():
    from tests.helpers import run_without_gpu
    run_without_gpu("import numpy as np, pytest, torch\n"
                    "from nvfpcc_b200 import metrics\n"
                    "assert not torch.cuda.is_available()\n"
                    "p = np.zeros((2, 3), np.int32)\n"
                    "with pytest.raises(RuntimeError):\n"
                    "    metrics.nearest_neighbours(p, p)\n"
                    "with pytest.raises(RuntimeError):\n"
                    "    metrics.distortion(p, p, peak=1023)\n")
