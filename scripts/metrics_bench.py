"""Timing of the GPU distortion metrics (nvfpcc_b200.metrics) against the host cKDTree baseline.

    python scripts/metrics_bench.py [--reps 30] [--out result.json]

Prints one JSON line.  Cases: the vox10 and vox11 sphere shells against their +-1-jittered copies (5 % of the points
dropped, one 32^3 leaf removed) and the decoded vox10 cloud (all 1247 leaves through net.decode_points).  Per case:
  - device time from CUDA events, median over `reps` runs after warm-up, of nearest_neighbours (one direction,
    source -> reconstruction, inputs already on the device) and of distortion with normals (both directions);
  - host-to-host time of distortion, numpy in to the dict out;
  - the host baseline: the two cKDTree(workers=-1) passes of one D1 evaluation;
and once per run an equality check of the vox10 shell against oracle/metrics_oracle.py.  The card name and power
limit are read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    name, limit = torch.cuda.get_device_name(0), None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        if out:
            name, limit = [s.strip() for s in out.split(",")[:2]]
    except (OSError, subprocess.SubprocessError):
        pass
    return {"name": name, "power_limit": limit}


def shell_case(resolution, seed=0):
    from nvfpcc_b200 import synth
    src = synth.sphere_shell_points(resolution).astype(np.int64)
    rng = np.random.default_rng(seed)
    rec = src + rng.integers(-1, 2, size=src.shape)
    rec = rec[rng.random(rec.shape[0]) >= 0.05]
    origins = synth.leaf_origins(src)
    rec = rec[~np.all(rec // 32 == origins[len(origins) // 3] // 32, axis=1)]
    return src, rec, np.array([resolution / 2.0] * 3)


def decoded_vox10():
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
    return pts[np.isin(key(pts), key(origins))].astype(np.int64), got["coords"].numpy().astype(np.int64), \
        np.array([512.0] * 3)


def sphere_normals(p, centre):
    v = np.asarray(p, np.float64) - centre
    return v / np.maximum(np.linalg.norm(v, axis=1, keepdims=True), 1e-12)


def device_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), float(np.min(times)), float(np.max(times))


def host_ms(fn, reps):
    times = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t) * 1e3)
    return float(np.median(times))


def run_case(name, src, rec, centre, peak, reps):
    from scipy.spatial import cKDTree

    from nvfpcc_b200 import metrics
    nrm = sphere_normals(src, centre)
    s_d, r_d = torch.from_numpy(src.astype(np.int32)).cuda(), torch.from_numpy(rec.astype(np.int32)).cuda()
    n_d = torch.from_numpy(nrm).cuda()
    nn = device_ms(lambda: metrics.nearest_neighbours(r_d, s_d, check=False), reps)
    dist = device_ms(lambda: metrics.distortion(s_d, r_d, peak=peak, source_normals=n_d), reps)
    h2h = host_ms(lambda: metrics.distortion(src, rec, peak=peak, source_normals=nrm), max(5, reps // 4))
    s64, r64 = src.astype(np.float64), rec.astype(np.float64)

    def kdtree_d1():
        cKDTree(r64).query(s64, workers=-1)
        cKDTree(s64).query(r64, workers=-1)
    host = host_ms(kdtree_d1, 3)
    r = metrics.distortion(src, rec, peak=peak, source_normals=nrm)
    return {"case": name, "n_source": int(src.shape[0]), "n_rec": int(rec.shape[0]),
            "nn_device_ms": {"median": nn[0], "min": nn[1], "max": nn[2]},
            "distortion_device_ms": {"median": dist[0], "min": dist[1], "max": dist[2]},
            "distortion_host_to_host_ms": h2h, "ckdtree_d1_host_ms": host,
            "speedup_distortion_h2h_vs_ckdtree": host / h2h,
            "d1_psnr": r["d1_psnr"], "d2_psnr": r["d2_psnr"], "hausdorff_d2": r["hausdorff_d2"]}


def oracle_check(src, rec, centre, peak):
    from nvfpcc_b200 import metrics
    from oracle import metrics_oracle as MO
    nrm = sphere_normals(src, centre)
    got = metrics.distortion(src, rec, peak=peak, source_normals=nrm)
    ref = MO.distortion(src, rec, peak, nrm, nn=lambda t, q: MO.nearest(t, q, k=16))
    nn = metrics.nearest_neighbours(rec, src)
    a = ref["nn"][0]
    per_point = all(np.array_equal(nn[k].cpu().numpy().astype(np.int64), a[k]) for k in ("index", "d2", "ties"))
    d2_rel = max(abs(g - r) / max(abs(r), 1e-300) for g, r in zip(got["d2_sum"], ref["d2_sum"]))
    return {"per_point_equal": bool(per_point), "d1_sum_equal": got["d1_sum"] == ref["d1_sum"],
            "hausdorff_equal": got["hausdorff_d2"] == ref["hausdorff_d2"], "d2_sum_max_rel_err": d2_rel,
            "ok": bool(per_point and got["d1_sum"] == ref["d1_sum"] and d2_rel <= 1e-12)}


def main(argv=None) -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise RuntimeError("metrics_bench needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"card": card(), "reps": a.reps, "host_cpus": os.cpu_count(), "cases": []}
    s10 = shell_case(1024)
    res["oracle_vox10"] = oracle_check(*s10, 1023.0)
    res["cases"].append(run_case("vox10_shell_vs_jittered", *s10, 1023.0, a.reps))
    res["cases"].append(run_case("vox11_shell_vs_jittered", *shell_case(2048), 2047.0, a.reps))
    res["cases"].append(run_case("vox10_decoded", *decoded_vox10(), 1023.0, a.reps))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
