"""GPU tier of the distortion metrics (nvfpcc_b200.metrics): exact nearest neighbours and D1 / D2 sums against the
float64 / int64 oracle (oracle/metrics_oracle.py), tie rule included, on small tie-heavy clouds, far queries, the
whole vox10 sphere shell and the decoded vox10 cloud; determinism, order independence and argument errors."""
import json

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

PEAK = 1023.0


def check_nn(target, query, k=8):
    from nvfpcc_b200 import metrics
    got = metrics.nearest_neighbours(target, query)
    host = lambda a: a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    ref = MO.nearest(host(target), host(query), k=k)
    for key in ("index", "d2", "ties"):
        assert np.array_equal(got[key].cpu().numpy().astype(np.int64), ref[key]), key
    assert int(got["status"].item()) == 0
    return got, ref


def check_distortion(src, rec, nrm, peak=PEAK, k=8):
    from nvfpcc_b200 import metrics
    got = metrics.distortion(src, rec, peak=peak, source_normals=nrm)
    ref = MO.distortion(src, rec, peak, nrm, nn=lambda t, q: MO.nearest(t, q, k=k))
    assert got["n"] == ref["n"]
    assert got["d1_sum"] == ref["d1_sum"] and got["hausdorff_d2"] == ref["hausdorff_d2"]
    assert got["d1_psnr"] == pytest.approx(ref["d1_psnr"], abs=1e-9)
    if nrm is not None:
        for g, r in zip(got["d2_sum"], ref["d2_sum"]):
            assert g == pytest.approx(r, rel=1e-12, abs=1e-300)
        assert got["d2_psnr"] == pytest.approx(ref["d2_psnr"], abs=1e-9)
    else:
        assert "d2" not in got
    return got, ref


def unit_normals(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


@pytest.mark.parametrize("seed", range(8))
def test_small_clouds_match_oracle(gpu, seed):
    rng = np.random.default_rng(seed)
    lo, hi = [(-3, 3), (-40, -20), (1000, 1004), (-3, 3)][seed % 4]
    src = rng.integers(lo, hi, size=(int(rng.integers(1, 400)), 3))
    rec = rng.integers(lo, hi, size=(int(rng.integers(1, 400)), 3))
    rec = np.concatenate([rec, rec[rng.integers(0, rec.shape[0], size=rec.shape[0] // 3)]])   # duplicates
    nrm = unit_normals(rng, src.shape[0])
    got, ref = check_nn(rec, src)
    assert (ref["ties"] > 1).any()
    check_nn(src, rec)
    check_distortion(src, rec, nrm)
    check_distortion(src, rec, None)


def test_single_target_empty_query_and_many_bins(gpu):
    rng = np.random.default_rng(11)
    q = rng.integers(-500, 500, size=(3000, 3))
    check_nn(np.array([[7, -3, 12]]), q)                            # n_target = 1: everything ties to it
    got, _ = check_nn(q, np.zeros((0, 3), np.int64))                # n_query = 0
    assert got["index"].numel() == 0
    wide = rng.integers(-2000, 2000, size=(20000, 3))               # sparse, many tree levels, unaligned
    check_nn(wide, rng.integers(-2100, 2100, size=(20000, 3)))
    check_distortion(wide[:5000], wide[5000:9000] + 1, unit_normals(rng, 5000))
    src = rng.integers(0, 8, size=(500, 3)).astype(np.float64)      # integral floats and torch input
    check_nn(torch.from_numpy(src).cuda(), torch.from_numpy(src[::-1].copy()))


def test_far_queries_are_exact(gpu):
    rng = np.random.default_rng(3)
    cluster = rng.integers(0, 16, size=(4000, 3)) + np.array([200, -300, 50])
    far = []
    for d in (100, 317, 1000, 2500, 5000):
        for axis in np.eye(3, dtype=np.int64):
            far += [cluster[0] + d * axis, cluster[0] - d * axis]
        far += [cluster[0] + d * np.array([1, 1, 1]), cluster[0] - d * np.array([1, -1, 1])]
    far = np.array(far)
    got, ref = check_nn(cluster, far)
    assert int(ref["d2"].max()) >= 3 * 4985 ** 2
    check_distortion(far, cluster, unit_normals(rng, far.shape[0]))   # disjoint clouds


def shell_case(resolution, seed=0, drop=0.05, remove_leaf=True):
    """Sphere shell against its +-1-jittered copy with `drop` of the points dropped and one 32^3 leaf removed."""
    from nvfpcc_b200 import synth
    src = synth.sphere_shell_points(resolution).astype(np.int64)
    rng = np.random.default_rng(seed)
    rec = src + rng.integers(-1, 2, size=src.shape)
    rec = rec[rng.random(rec.shape[0]) >= drop]
    if remove_leaf:
        leaf = synth.leaf_origins(src)[len(synth.leaf_origins(src)) // 3] // 32
        rec = rec[~np.all(rec // 32 == leaf, axis=1)]
    centre = np.array([resolution / 2.0] * 3)
    return src, rec, centre


def test_whole_vox10_shell_matches_oracle(gpu):
    from tests.test_gpu_parity2 import _sphere_normals
    src, rec, centre = shell_case(1024)
    nrm = _sphere_normals(src, centre)
    _, ref0 = check_nn(rec, src, k=16)
    _, ref1 = check_nn(src, rec, k=16)
    assert (ref1["ties"] > 1).mean() > 0.2 and ref0["d2"].max() > 100   # tie-heavy, and the removed leaf is far
    check_distortion(src, rec, nrm, k=16)


def decoded_vox10():
    """All 1247 vox10 leaves decoded through net.decode_points, calibrated as the whole-cloud parity test does;
    returns (source points inside the decoded leaves, decoded points, sphere centre)."""
    import bench
    from nvfpcc_b200 import network, synth
    pts = synth.sphere_shell_points(1024)
    origins = synth.leaf_origins(pts)
    network.set_seed(synth.synthetic_seed())
    net = network.Net(None, "Gaussian", ch=3, channel_str="8,16,8,8").cuda()
    lat = torch.from_numpy(synth.random_latents(origins.shape[0], 3, seed=0)).cuda()
    bench.calibrate_threshold_bias(net, lat, 0.65)
    got = net.decode_points(lat, torch.from_numpy(origins.astype(np.int32)).cuda(), 0.65, return_host=True)
    key = lambda a: (np.asarray(a, np.int64) // 32) @ np.array([1 << 40, 1 << 20, 1])
    src = pts[np.isin(key(pts), key(origins))]
    return src, got["coords"].numpy(), np.array([512.0] * 3)


def test_decoded_vox10_cloud_matches_oracle_and_host_helper(gpu):
    from tests.test_gpu_parity2 import _sphere_normals, psnr_d1_d2
    src, rec, centre = decoded_vox10()
    assert src.shape[0] > 800000 and rec.shape[0] > 500000
    nrm = _sphere_normals(src, centre)
    check_nn(rec, src, k=16)
    check_nn(src, rec, k=16)
    got, _ = check_distortion(src, rec, nrm, k=16)
    d1_ref, _ = psnr_d1_d2(rec, src, centre, PEAK)
    assert got["d1_psnr"] == pytest.approx(d1_ref, abs=1e-9)


def test_deterministic_and_order_independent(gpu):
    from nvfpcc_b200 import metrics
    from tests.test_gpu_parity2 import _sphere_normals
    src, rec, centre = shell_case(512, seed=1)
    nrm = _sphere_normals(src, centre)
    a = metrics.distortion(src, rec, peak=511.0, source_normals=nrm)
    b = metrics.distortion(src, rec, peak=511.0, source_normals=nrm)
    assert a == b                                                   # bit-identical, every field
    na, nb = metrics.nearest_neighbours(rec, src), metrics.nearest_neighbours(rec, src)
    for k in ("index", "d2", "ties"):
        assert torch.equal(na[k], nb[k])
    perm = np.random.default_rng(5).permutation(src.shape[0])
    permr = np.random.default_rng(6).permutation(rec.shape[0])
    c = metrics.distortion(src[perm], rec[permr], peak=511.0, source_normals=nrm[perm])
    assert c["d1_sum"] == a["d1_sum"] and c["hausdorff_d2"] == a["hausdorff_d2"]
    for x, y in zip(c["d2_sum"], a["d2_sum"]):
        assert x == pytest.approx(y, rel=1e-12)


def test_argument_errors(gpu):
    from nvfpcc_b200 import _lib, metrics
    p = np.zeros((4, 3), np.int32)
    with pytest.raises(ValueError):
        metrics.nearest_neighbours(np.zeros((4, 2), np.int32), p)
    with pytest.raises(ValueError):
        metrics.nearest_neighbours(p, np.zeros(3, np.int32))
    with pytest.raises(ValueError):
        metrics.nearest_neighbours(p, p + 0.5)
    with pytest.raises(ValueError):
        metrics.nearest_neighbours(np.zeros((0, 3), np.int32), p)
    with pytest.raises(ValueError):
        metrics.distortion(p, p, peak=1.0, source_normals=np.zeros((3, 3)))
    with pytest.raises(ValueError):
        metrics.distortion(p, np.zeros((0, 3), np.int32), peak=1.0)
    big = p.copy()
    big[2] = [1 << 20, 0, 0]                                        # first coordinate outside the cell key's range
    with pytest.raises(_lib.NvfError):
        metrics.nearest_neighbours(big, p)
    with pytest.raises(_lib.NvfError):
        metrics.nearest_neighbours(p, big)
    with pytest.raises(_lib.NvfError):
        metrics.distortion(big, p, peak=1.0)
    r = metrics.nearest_neighbours(p, -big, check=False)            # -2^20 is still inside
    assert int(r["status"].item()) == 0
    assert metrics.distortion(p, p, peak=1.0)["d1_psnr"] == float("inf")


def test_command_line(gpu, tmp_path, capsys):
    from nvfpcc_b200 import metrics
    from tests.test_gpu_parity2 import _sphere_normals
    src, rec, centre = shell_case(256, seed=2)
    nrm = _sphere_normals(src, centre)
    rows = np.zeros(src.shape[0], dtype=[("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("nx", "<f8"), ("ny", "<f8"),
                                         ("nz", "<f8")])
    for i, k in enumerate("xyz"):
        rows[k], rows["n" + k] = src[:, i], nrm[:, i]
    hdr = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\n"
           "property float z\nproperty double nx\nproperty double ny\nproperty double nz\nend_header\n" % src.shape[0])
    (tmp_path / "s.ply").write_bytes(hdr.encode() + rows.tobytes())
    (tmp_path / "r.ply").write_text("ply\nformat ascii 1.0\nelement vertex %d\nproperty int x\nproperty int y\n"
                                    "property int z\nend_header\n" % rec.shape[0] +
                                    "".join("%d %d %d\n" % tuple(p) for p in rec))
    assert metrics.main([str(tmp_path / "s.ply"), str(tmp_path / "r.ply"), "--peak", "255"]) == 0
    out = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    ref = MO.distortion(src, rec, 255.0, nrm)
    assert out["d1_psnr"] == pytest.approx(ref["d1_psnr"], abs=1e-9)
    assert out["d2_psnr"] == pytest.approx(ref["d2_psnr"], abs=1e-9)
    assert metrics.main([str(tmp_path / "r.ply"), str(tmp_path / "s.ply"), "--peak", "255"]) == 0
    out = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert "d2_psnr" not in out and out["d1_psnr"] == pytest.approx(ref["d1_psnr"], abs=1e-9)
