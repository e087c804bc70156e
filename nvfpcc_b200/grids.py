"""Ground-truth occupancy grids and exact distance fields of the leaf blocks on the GPU.

Drop-in for the reference's preprocessing script util_get_grids.py:

    python -m nvfpcc_b200.grids longdress_vox10_1300.ply 5

reads `{fid}_l5_origins.txt` (written by get_octree) and the PLY, and writes
`{fid}_l5_origins.npy`, `{fid}_l5_gt_grid.npy` (uint8) and `{fid}_l5_dist.npy` (float64) with
the reference's shapes and dtypes (util_get_grids.py:16-17, 42-46) - the files
LoadedVoxelDataset loads (utils/dataloader.py:152-160).  The reference asks an open3d KD-tree
once per grid voxel from Python; here `nvf_build_grids` (include/nvf_prep_b200.h,
csrc/nvf_grids.cuh) runs an exact integer distance transform, one CTA per leaf.

There is no CPU fallback: the functions need a CUDA device and the built library.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib

LEAF = 32
MAX_RADIUS = 53
STATUS_CELL_OVERFLOW, STATUS_NOT_FOUND = 1, 2
EXPORTS = ("nvf_grids_workspace_bytes", "nvf_build_grids")

_bound = None


def _binding():
    """The product library with the nvf_prep_b200.h signatures attached."""
    global _bound
    if _bound is None:
        b = _lib.cuda_binding()
        L = b.lib
        for name in EXPORTS:
            if not hasattr(L, name):
                raise _lib.NvfError("%s does not export %s" % (b.path, name))
        vp = C.c_void_p
        L.nvf_grids_workspace_bytes.argtypes = [C.c_int64, C.POINTER(C.c_size_t)]
        L.nvf_build_grids.argtypes = [vp, C.c_int64, vp, C.c_int64, C.c_int64, C.c_int32, vp, vp, vp, vp, vp, vp,
                                      C.c_size_t, vp]
        _bound = b
    return _bound


def as_i32(a, what: str, dev: torch.device) -> torch.Tensor:
    """(n,3) integer voxel coordinates (numpy or torch, integer or integral float) as a contiguous int32 tensor
    on `dev`; raises ValueError for another shape or a non-integral coordinate."""
    t = torch.as_tensor(np.ascontiguousarray(a) if isinstance(a, np.ndarray) else a)
    if t.dim() != 2 or t.shape[1] != 3:
        raise ValueError("%s must have shape (n,3)" % what)
    if t.is_floating_point():
        r = torch.round(t)
        if not torch.equal(r, t):
            raise ValueError("%s must be integer voxel coordinates" % what)
        t = r
    return t.to(device=dev, dtype=torch.int32).contiguous()


def workspace_bytes(max_cells: int) -> int:
    b = _binding()
    out = C.c_size_t(0)
    b.check(b.lib.nvf_grids_workspace_bytes(int(max_cells), C.byref(out)), "nvf_grids_workspace_bytes")
    return int(out.value)


def build_grids(points, origins, *, max_cells: Optional[int] = None, max_radius: int = MAX_RADIUS,
                want_gt: bool = True, want_dist64: bool = True, want_dist32: bool = False, want_d2: bool = False,
                check: bool = True, device: Optional[torch.device] = None) -> Dict[str, torch.Tensor]:
    """util_get_grids.py:26-44 for all leaves at once.

    points  (P,3) integer voxel coordinates (numpy or torch); origins (N,3) leaf origins.
    Returns CUDA tensors: 'gt' uint8 / 'dist' float64 / 'dist32' float32, each [N,1,32,32,32],
    'd2' uint16 [N,32768], and 'status' (int32 [1]).  max_cells=None counts the cloud's occupied 32^3 cells
    first (one small sort + host sync); pass it to stay asynchronous.  With check=True (one host sync) a
    non-zero status raises: leaves without any point, or more occupied cells than max_cells.
    """
    if not torch.cuda.is_available():
        raise RuntimeError("nvfpcc_b200.grids needs a CUDA device (no CPU fallback)")
    b = _binding()
    dev = torch.device(device) if device is not None else (
        points.device if isinstance(points, torch.Tensor) and points.is_cuda else torch.device("cuda", torch.cuda.current_device()))

    pts = as_i32(points, "points", dev)
    org = as_i32(origins, "origins", dev)
    n, npts = int(org.shape[0]), int(pts.shape[0])
    if max_cells is None:                    # distinct (point >> 5) cells of the cloud, counted on the device
        c = (pts.to(torch.int64) >> 5) + (1 << 20)
        max_cells = max(int(torch.unique((c[:, 0] << 42) | (c[:, 1] << 21) | c[:, 2]).numel()), 64) if npts else 64
    nbytes = workspace_bytes(max_cells)
    ws = b.cached_workspace(nbytes, dev, "grids")
    out: Dict[str, torch.Tensor] = {}
    shape = (n, 1, LEAF, LEAF, LEAF)
    if want_gt:
        out["gt"] = torch.empty(shape, dtype=torch.uint8, device=dev)
    if want_dist64:
        out["dist"] = torch.empty(shape, dtype=torch.float64, device=dev)
    if want_dist32:
        out["dist32"] = torch.empty(shape, dtype=torch.float32, device=dev)
    if want_d2:
        out["d2"] = torch.empty((n, LEAF ** 3), dtype=torch.int16, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = b.lib.nvf_build_grids(_lib._ptr(pts), npts, _lib._ptr(org), n, int(max_cells), int(max_radius),
                                   _lib._ptr(out.get("gt")), _lib._ptr(out.get("dist")), _lib._ptr(out.get("dist32")),
                                   _lib._ptr(out.get("d2")), _lib._ptr(status), _lib._ptr(ws), nbytes, b._stream(dev))
    b.check(rc, "nvf_build_grids")
    if want_d2:
        out["d2"] = out["d2"].view(torch.uint16)
    out["status"] = status
    if check:
        s = int(status.item())
        if s & STATUS_CELL_OVERFLOW:
            raise _lib.NvfError("nvf_build_grids: more occupied 32^3 cells than max_cells=%d" % max_cells)
        if s & STATUS_NOT_FOUND:
            raise _lib.NvfError("nvf_build_grids: a leaf has no cloud point within %d voxels (empty leaf?)" % max_radius)
    return out


_host_bufs: Dict[str, torch.Tensor] = {}


def build_grids_host(points, origins, copy: bool = False, **kw) -> Dict[str, np.ndarray]:
    """build_grids with HOST results (what the file front end and any caller that stores the grids needs):
    {'gt': uint8 [N,1,32,32,32], 'dist': float64 [N,1,32,32,32]} as numpy arrays.

    The float64 distances are 8 bytes per voxel (368 MB for vox10) and `tensor.cpu()` into pageable memory was 98 %
    of the host-to-host time.  Here the results land in reusable PINNED staging buffers (one asynchronous copy each at
    full PCIe rate); with copy=False the returned arrays are views of those buffers - valid until the next call -
    which is all `np.save` needs.  (Taking the square root of the exact 16-bit squared distances on the host instead
    was measured and rejected: a correctly rounded float64 sqrt of 41 M values costs the host cores 0.4 s.)"""
    r = build_grids(points, origins, want_gt=True, want_dist64=True, want_dist32=False, want_d2=False, **kw)

    def staged(name, src):
        buf = _host_bufs.get(name)
        if buf is None or buf.numel() < src.numel() or buf.dtype != src.dtype:
            buf = torch.empty(src.numel(), dtype=src.dtype).pin_memory()
            _host_bufs[name] = buf
        out = buf[:src.numel()].view(src.shape)
        out.copy_(src, non_blocking=True)
        return out

    gt_h, dist_h = staged("gt", r["gt"]), staged("dist", r["dist"])
    torch.cuda.current_stream(r["gt"].device).synchronize()
    gt, dist = gt_h.numpy(), dist_h.numpy()
    return {"gt": gt.copy(), "dist": dist.copy()} if copy else {"gt": gt, "dist": dist}


# ----------------------------------------------------------------------------- file front end
_PLY_TYPES = {"char": "i1", "uchar": "u1", "short": "i2", "ushort": "u2", "int": "i4", "uint": "u4", "float": "f4",
              "double": "f8", "int8": "i1", "uint8": "u1", "int16": "i2", "uint16": "u2", "int32": "i4",
              "uint32": "u4", "float32": "f4", "float64": "f8"}


def read_ply_vertex(path: str) -> Dict[str, np.ndarray]:
    """Every scalar vertex property of an ASCII or binary PLY, by name, as float64 arrays of length N."""
    with open(path, "rb") as f:
        if f.readline().strip() != b"ply":
            raise ValueError("%s is not a PLY file" % path)
        fmt, n_vertex, props, in_vertex = None, 0, [], False
        while True:
            line = f.readline()
            if not line:
                raise ValueError("PLY header of %s is truncated" % path)
            tok = line.decode("ascii", "replace").split()
            if not tok:
                continue
            if tok[0] == "format":
                fmt = tok[1]
            elif tok[0] == "element":
                in_vertex = tok[1] == "vertex"
                if in_vertex:
                    n_vertex = int(tok[2])
            elif tok[0] == "property" and in_vertex:
                if tok[1] == "list":
                    raise ValueError("list property on the vertex element is not supported")
                props.append((tok[2], _PLY_TYPES[tok[1]]))
            elif tok[0] == "end_header":
                break
        names = [p[0] for p in props]
        if fmt == "ascii":
            rows = np.loadtxt(f, max_rows=n_vertex, ndmin=2, dtype=np.float64)
            return {nm: rows[:, i] for i, nm in enumerate(names)}
        order = "<" if fmt == "binary_little_endian" else ">"
        dt = np.dtype([(nm, order + ty) for nm, ty in props])
        rec = np.frombuffer(f.read(n_vertex * dt.itemsize), dtype=dt, count=n_vertex)
        return {nm: rec[nm].astype(np.float64) for nm in names}


def read_ply_xyz(path: str) -> np.ndarray:
    """Vertex x,y,z of an ASCII or binary PLY as float64 (N,3) - what
    np.asarray(o3d.io.read_point_cloud(path).points) holds (util_get_grids.py:32,40)."""
    v = read_ply_vertex(path)
    if not all(a in v for a in "xyz"):
        raise ValueError("PLY vertex element has no x/y/z")
    return np.stack([v[a] for a in "xyz"], 1)


def main(argv=None) -> int:
    """Same command line and output files as util_get_grids.py:9-17, 42-46."""
    argv = sys.argv if argv is None else argv
    if len(argv) < 2:
        print("usage: python -m nvfpcc_b200.grids cloud.ply [level=5]")
        return 2
    qstr = ""
    fid = argv[1].split("/")[-1][:-4]
    lx = int(argv[2]) if len(argv) == 3 else 5
    origins = np.loadtxt(f"{fid}_l{lx}{qstr}_origins.txt", delimiter=",", ndmin=2)
    np.save(f"{fid}_l{lx}{qstr}_origins", origins)
    pts = read_ply_xyz(argv[1])
    r = build_grids_host(pts, origins)
    np.save(f"{fid}_l{lx}{qstr}_gt_grid", r["gt"])
    np.save(f"{fid}_l{lx}{qstr}_dist", r["dist"])
    return 0


if __name__ == "__main__":
    sys.exit(main())
