"""CPU oracle of the point-cloud distortion metrics (nvfpcc_b200.metrics, include/nvf_metrics_b200.h).

TEST INFRASTRUCTURE ONLY: a float64 / int64 numpy + scipy restatement of the contract, tie rule included.  Only
`tests/`, `__graft_entry__.smoke()` and `scripts/metrics_bench.py` import it; the product package never does.

For a target cloud T and a query point q (integer voxel coordinates):
  d2(q)    = min over t in T of |q - t|^2 (exact int64);
  ties(q)  = the target points at exactly d2(q), duplicates counted separately;
  index(q) = the lowest index in ties(q).
D1 per direction = mean d2(q); D2 per direction = mean over queries of the squared plane error averaged over ties(q)
(direction 0, source -> reconstruction: ((s_i - r_t) . n_i)^2; direction 1: ((r_i - s_t) . n_t)^2).

`nearest` asks cKDTree for K candidates, recomputes their exact integer squared distances and falls back to
`query_ball_point` for the rows where all K candidates tie; `nearest_bruteforce` computes all pairs (small inputs)
so that the oracle itself can be checked.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional

import numpy as np


def _i64(a) -> np.ndarray:
    a = np.asarray(a)
    r = np.rint(a)
    if a.ndim != 2 or a.shape[1] != 3 or not np.array_equal(r, a):
        raise ValueError("expected (n,3) integer voxel coordinates")
    return r.astype(np.int64)


def _csr(rows: np.ndarray, members: np.ndarray, n: int):
    """Tie lists as CSR (offsets [n+1], members sorted by row, then by index)."""
    order = np.lexsort((members, rows))
    rows, members = rows[order], members[order]
    counts = np.bincount(rows, minlength=n)
    offsets = np.zeros(n + 1, np.int64)
    np.cumsum(counts, out=offsets[1:])
    return offsets, members.astype(np.int64)


def _result(offsets, members, d2):
    ties = np.diff(offsets)
    index = np.minimum.reduceat(members, offsets[:-1]) if members.size else np.zeros(0, np.int64)
    return {"index": index.astype(np.int64), "d2": d2.astype(np.int64), "ties": ties.astype(np.int64),
            "offsets": offsets, "members": members}


def nearest(target, query, k: int = 8, workers: int = -1) -> Dict[str, np.ndarray]:
    """Exact nearest neighbours with the tie rule: {'index', 'd2', 'ties', 'offsets', 'members'} (int64);
    members[offsets[i]:offsets[i+1]] are the tied target indices of query i in ascending order."""
    from scipy.spatial import cKDTree
    T, Q = _i64(target), _i64(query)
    nt, nq = T.shape[0], Q.shape[0]
    if nt == 0:
        raise ValueError("empty target")
    if nq == 0:
        return _result(np.zeros(1, np.int64), np.zeros(0, np.int64), np.zeros(0, np.int64))
    K = min(k, nt)
    tree = cKDTree(T.astype(np.float64))
    _, idx = tree.query(Q.astype(np.float64), k=K, workers=workers)
    idx = np.asarray(idx, np.int64).reshape(nq, K)
    diff = Q[:, None, :] - T[idx]
    d2c = (diff * diff).sum(-1)                                   # exact int64
    d2 = d2c.min(1)
    mask = d2c == d2[:, None]
    full = mask.all(1) & (K < nt)                                 # every candidate ties: more may exist
    mask[full] = False
    rows, cols = np.nonzero(mask)
    rows_l, mem_l = [rows], [idx[rows, cols]]
    for i in np.nonzero(full)[0]:
        r = math.sqrt(float(d2[i]))
        cand = np.asarray(tree.query_ball_point(Q[i].astype(np.float64), r * (1 + 1e-9) + 1e-6), np.int64)
        dd = Q[i] - T[cand]
        m = cand[(dd * dd).sum(-1) == d2[i]]
        rows_l.append(np.full(m.size, i, np.int64))
        mem_l.append(m)
    offsets, members = _csr(np.concatenate(rows_l), np.concatenate(mem_l), nq)
    return _result(offsets, members, d2)


def nearest_bruteforce(target, query) -> Dict[str, np.ndarray]:
    """Same result from all pairs (small inputs only)."""
    T, Q = _i64(target), _i64(query)
    if T.shape[0] == 0:
        raise ValueError("empty target")
    diff = Q[:, None, :] - T[None, :, :]
    d = (diff * diff).sum(-1)
    d2 = d.min(1) if Q.shape[0] else np.zeros(0, np.int64)
    rows, members = np.nonzero(d == d2[:, None])
    offsets, members = _csr(rows.astype(np.int64), members.astype(np.int64), Q.shape[0])
    return _result(offsets, members, d2)


def psnr(mse: float, peak: float) -> float:
    return math.inf if mse == 0 else 10.0 * math.log10(3.0 * peak * peak / mse)


def _plane(query, target, normals, nn, query_normals: bool) -> np.ndarray:
    """Per-query squared plane error averaged over the tied neighbours."""
    nq = query.shape[0]
    rows = np.repeat(np.arange(nq), np.diff(nn["offsets"]))
    t = nn["members"]
    n = normals[rows] if query_normals else normals[t]
    e = ((query[rows] - target[t]).astype(np.float64) * n).sum(1)
    return np.bincount(rows, e * e, minlength=nq) / np.maximum(nn["ties"], 1)


def distortion(source, reconstruction, peak: float, source_normals=None,
               nn: Callable = nearest) -> Dict:
    """D1 / D2 of `reconstruction` against `source`, with the same keys as nvfpcc_b200.metrics.distortion, plus the
    per-direction nearest-neighbour results 'nn' (source -> reconstruction, reconstruction -> source)."""
    S, R = _i64(source), _i64(reconstruction)
    a, b = nn(R, S), nn(S, R)
    n = (S.shape[0], R.shape[0])
    d1_sum = (int(a["d2"].sum()), int(b["d2"].sum()))
    d1_mse = (d1_sum[0] / n[0], d1_sum[1] / n[1])
    out = {"n": n, "d1_sum": d1_sum, "d1_mse": d1_mse, "d1": max(d1_mse), "d1_psnr": psnr(max(d1_mse), peak),
           "hausdorff_d2": (int(a["d2"].max()), int(b["d2"].max())), "nn": (a, b)}
    if source_normals is not None:
        N = np.asarray(source_normals, np.float64)
        e0 = _plane(S, R, N, a, True)
        e1 = _plane(R, S, N, b, False)
        d2_sum = (math.fsum(e0), math.fsum(e1))
        d2_mse = (d2_sum[0] / n[0], d2_sum[1] / n[1])
        out.update(d2_sum=d2_sum, d2_mse=d2_mse, d2=max(d2_mse), d2_psnr=psnr(max(d2_mse), peak), plane=(e0, e1))
    return out
