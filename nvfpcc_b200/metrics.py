"""Point-cloud distortion on the GPU: exact nearest neighbours and D1 / D2 PSNR.

    python -m nvfpcc_b200.metrics source.ply reconstruction.ply --peak 1023

prints one JSON line with the D1 (point-to-point) PSNR of the reconstruction against the source and, when the
source PLY carries nx / ny / nz, the D2 (point-to-plane) PSNR.  Both directions are measured, the worse mean wins,
and PSNR = 10 log10(3 peak^2 / mse), as MPEG's pc_error defines them.

Nearest neighbours are exact on the integer lattice at any distance (`nvf_nearest_points`,
include/nvf_metrics_b200.h, csrc/nvf_metrics.cuh).  Ties are common on the lattice; the rule is:
  - `index` is the LOWEST target index at the nearest distance (what np.argmin over exact distances returns);
  - D2 averages the squared plane error over ALL target points at the nearest distance, so it does not depend on
    the order of the points.
Sums run in a fixed order without float atomics: two calls give bit-identical results.

There is no CPU fallback: the functions need a CUDA device and the built library.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import sys
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .grids import as_i32, read_ply_vertex

STATUS_RANGE, STATUS_SUM_OVERFLOW = 1, 2
COORD_LIMIT = 1 << 20
EXPORTS = ("nvf_nn_workspace_bytes", "nvf_nearest_points", "nvf_distortion_workspace_bytes", "nvf_pc_distortion")

_bound = None


def _binding():
    """The product library with the nvf_metrics_b200.h signatures attached."""
    global _bound
    if _bound is None:
        b = _lib.cuda_binding()
        L = b.lib
        for name in EXPORTS:
            if not hasattr(L, name):
                raise _lib.NvfError("%s does not export %s" % (b.path, name))
        vp, i64, sz = C.c_void_p, C.c_int64, C.c_size_t
        L.nvf_nn_workspace_bytes.argtypes = [i64, C.POINTER(sz)]
        L.nvf_nearest_points.argtypes = [vp, i64, vp, i64, vp, vp, vp, vp, vp, sz, vp]
        L.nvf_distortion_workspace_bytes.argtypes = [i64, i64, C.POINTER(sz)]
        L.nvf_pc_distortion.argtypes = [vp, i64, vp, vp, i64, vp, vp, vp, sz, vp]
        _bound = b
    return _bound


def _device(*arrays) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("nvfpcc_b200.metrics needs a CUDA device (no CPU fallback)")
    for a in arrays:
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a.device
    return torch.device("cuda", torch.cuda.current_device())


def _raise_status(s: int, what: str) -> None:
    if s & STATUS_RANGE:
        raise _lib.NvfError("%s: a coordinate lies outside [-2^20, 2^20)" % what)
    if s & STATUS_SUM_OVERFLOW:
        raise _lib.NvfError("%s: a sum of squared distances does not fit int64" % what)


def psnr(mse: float, peak: float) -> float:
    """10 log10(3 peak^2 / mse); inf when mse == 0."""
    return math.inf if mse == 0 else 10.0 * math.log10(3.0 * peak * peak / mse)


def nearest_neighbours(target, query, *, check: bool = True) -> Dict[str, torch.Tensor]:
    """Nearest target point of every query point, exactly.

    target (T,3), query (Q,3): integer voxel coordinates (numpy or torch, integer or integral float), T >= 1.
    Returns CUDA tensors 'index' int32 [Q] (lowest index at the nearest distance), 'd2' int64 [Q] (exact squared
    distance), 'ties' int32 [Q] (number of target points at that distance) and 'status' int32 [1].  With check=True
    (one host sync) a non-zero status raises NvfError."""
    dev = _device(target, query)
    b = _binding()
    t = as_i32(target, "target", dev)
    q = as_i32(query, "query", dev)
    nt, nq = int(t.shape[0]), int(q.shape[0])
    if nt == 0:
        raise ValueError("target is empty: the nearest neighbour is undefined")
    nbytes = C.c_size_t(0)
    b.check(b.lib.nvf_nn_workspace_bytes(nt, C.byref(nbytes)), "nvf_nn_workspace_bytes")
    ws = b.cached_workspace(int(nbytes.value), dev, "metrics")
    out = {"index": torch.empty(nq, dtype=torch.int32, device=dev),
           "d2": torch.empty(nq, dtype=torch.int64, device=dev),
           "ties": torch.empty(nq, dtype=torch.int32, device=dev),
           "status": torch.empty(1, dtype=torch.int32, device=dev)}
    with torch.cuda.device(dev):
        rc = b.lib.nvf_nearest_points(_lib._ptr(t), nt, _lib._ptr(q) if nq else None, nq, _lib._ptr(out["index"]),
                                      _lib._ptr(out["d2"]), _lib._ptr(out["ties"]), _lib._ptr(out["status"]),
                                      _lib._ptr(ws), int(nbytes.value), b._stream(dev))
    b.check(rc, "nvf_nearest_points")
    if check:
        _raise_status(int(out["status"].item()), "nvf_nearest_points")
    return out


def distortion(source, reconstruction, *, peak: float, source_normals=None, check: bool = True) -> Dict:
    """D1 (and with `source_normals`, D2) of `reconstruction` against `source`.

    source (S,3), reconstruction (R,3): integer voxel coordinates, both non-empty; source_normals (S,3) unit normals
    of the source, used as given in float64.  `peak` is the signal peak of the PSNR (1023 for vox10).
    Pairs are (source -> reconstruction, reconstruction -> source).  Returns
      'd1_mse' (pair), 'd1' = max of the pair, 'd1_psnr', 'hausdorff_d2' (pair of largest squared distances),
      'n' (pair of query counts) and, with normals, 'd2_mse' (pair), 'd2', 'd2_psnr'."""
    dev = _device(source, reconstruction)
    b = _binding()
    src = as_i32(source, "source", dev)
    rec = as_i32(reconstruction, "reconstruction", dev)
    ns, nr = int(src.shape[0]), int(rec.shape[0])
    if ns == 0 or nr == 0:
        raise ValueError("source and reconstruction must both hold at least one point")
    nrm = None
    if source_normals is not None:
        nrm = torch.as_tensor(np.ascontiguousarray(source_normals) if isinstance(source_normals, np.ndarray)
                              else source_normals)
        if tuple(nrm.shape) != (ns, 3):
            raise ValueError("source_normals must have shape (%d,3), got %s" % (ns, tuple(nrm.shape)))
        nrm = nrm.to(device=dev, dtype=torch.float64).contiguous()
    nbytes = C.c_size_t(0)
    b.check(b.lib.nvf_distortion_workspace_bytes(ns, nr, C.byref(nbytes)), "nvf_distortion_workspace_bytes")
    ws = b.cached_workspace(int(nbytes.value), dev, "metrics")
    res = torch.empty(8, dtype=torch.int64, device=dev)          # NvfDistortion: n, d1_sum, d1_max (int64), d2_sum
    status = torch.empty(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = b.lib.nvf_pc_distortion(_lib._ptr(src), ns, _lib._ptr(nrm), _lib._ptr(rec), nr, _lib._ptr(res),
                                     _lib._ptr(status), _lib._ptr(ws), int(nbytes.value), b._stream(dev))
    b.check(rc, "nvf_pc_distortion")
    host = torch.cat([res, status.to(torch.int64)]).cpu().numpy()
    if check:
        _raise_status(int(host[8]), "nvf_pc_distortion")
    n = (int(host[0]), int(host[1]))
    d1_sum = (int(host[2]), int(host[3]))
    d2_sum = tuple(float(v) for v in host[6:8].view(np.float64))
    d1_mse = (d1_sum[0] / n[0], d1_sum[1] / n[1])
    out = {"n": n, "d1_sum": d1_sum, "d1_mse": d1_mse, "d1": max(d1_mse), "d1_psnr": psnr(max(d1_mse), peak),
           "hausdorff_d2": (int(host[4]), int(host[5])), "status": int(host[8])}
    if nrm is not None:
        d2_mse = (d2_sum[0] / n[0], d2_sum[1] / n[1])
        out.update(d2_sum=d2_sum, d2_mse=d2_mse, d2=max(d2_mse), d2_psnr=psnr(max(d2_mse), peak))
    return out


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m nvfpcc_b200.metrics",
                                 description="D1 / D2 PSNR of a reconstructed point cloud against its source.")
    ap.add_argument("source")
    ap.add_argument("reconstruction")
    ap.add_argument("--peak", type=float, required=True, help="signal peak, e.g. 1023 for vox10")
    a = ap.parse_args(argv)
    sv, rv = read_ply_vertex(a.source), read_ply_vertex(a.reconstruction)
    for path, v in ((a.source, sv), (a.reconstruction, rv)):
        if not all(k in v for k in "xyz"):
            raise ValueError("PLY vertex element of %s has no x/y/z" % path)
    src = np.stack([sv[k] for k in "xyz"], 1)
    rec = np.stack([rv[k] for k in "xyz"], 1)
    normals = np.stack([sv[k] for k in ("nx", "ny", "nz")], 1) if all(k in sv for k in ("nx", "ny", "nz")) else None
    r = distortion(src, rec, peak=a.peak, source_normals=normals)
    keys = ["n", "d1_mse", "d1", "d1_psnr", "hausdorff_d2"] + (["d2_mse", "d2", "d2_psnr"] if normals is not None else [])
    print(json.dumps({"source": a.source, "reconstruction": a.reconstruction, "peak": a.peak,
                      **{k: r[k] for k in keys}}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
