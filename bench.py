#!/usr/bin/env python
"""Benchmark of the NVF leaf-block decoder hot path (BASELINE.json metric:
"NVF decoded voxels/sec & train blocks/sec at 1/2/4/8 B200; % of roofline").

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Primary line = BASELINE.json configs[1]: weight-loop training steps
(NVFPCC.py:149-223) at batchsize 16 on synthetic vox10 leaf blocks, lambda 200,
lr 1e-3, chanstr 8,16,8,8 -> train blocks/s.  The same JSON line carries the
decode half of the metric under "decode" (all 1247 vox10 blocks, thh 0.65 ->
decoded voxels/s), each with its own roofline / e2e numbers.

A "step" is one pass of the hot path over one batch: train = forward + fused
rate-distortion loss + backward + Adam on 16 blocks per rank; decode = all of
the rank's blocks through the fused decode kernel to an ordered point list.
`value` is measured with inputs resident in HBM; `e2e` goes through the public
API with pinned HOST buffers (H2D of the step's inputs and D2H of its result
inside the timed region).

--steps K sets the timed steps of the train loop and, unless --decode-steps is
given, of each decode workload.  --dump-outputs DIR writes, on rank 0, what the
last timed steps computed: the train step's stats and the weights it left
(train_*.npy), and the point list and per-block counts of each decode workload
(decode_*.npy; with --gpus N these cover rank 0's share of the blocks).  Inputs and seeds
are fixed, so two builds run with the same arguments can be compared output
for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

# algorithmic work per block, SURVEY.md section 8(d) / BASELINE.md section 3
F_DEC = {"8,16,8,8": 398_481_616, "16,32,16,16": 1_567_314_848}
F_TRAIN = {"8,16,8,8": 1_201_139_184, "16,32,16,16": 4_713_333_216}
FP32_PEAK_THEORETICAL = 148 * 128 * 2 * 1.965e9 / 1e12   # TFLOP/s at the 1965 MHz max clock
HP = dict(lmbda=200.0, w1=10.0, w2=57.0, lr=1e-3, batch=16, thh=0.65)


_JSON_FD = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner on rank 0),
    so keep a private duplicate of the real stdout for the result line and point fd 1 at stderr for everything else."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _round(o, sig=6):
    if isinstance(o, float):
        return float("%.*g" % (sig, o))
    if isinstance(o, dict):
        return {k: _round(v, sig) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_round(v, sig) for v in o]
    return o


def emit(line, detail=None):
    """ONE compact JSON line on stdout (floats to 6 significant digits, no prose beyond `config.workload`).  The
    long-form record (notes, sample descriptions, the rows either side of the path) goes to stderr, so that the
    result line stays short enough for any log tail and the benchmark writes nothing into the source tree."""
    sys.stdout.flush()
    if detail is not None:
        sys.stderr.write("[bench detail] " + json.dumps(detail) + "\n")
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(_round(line), separators=(",", ":")) + "\n").encode())


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--chanstr", default="8,16,8,8")
    ap.add_argument("--resolution", type=int, default=1024, help="1024 = vox10, 2048 = vox11")
    ap.add_argument("--train-blocks", type=int, default=0,
                    help="distinct leaf blocks (per rank) cycled by the train steps; 0 = every leaf of the cloud (vox10: 1247 "
                         "leaves = 326 MB of gt + dist, larger than the 126 MB L2, so no flush is needed between steps)")
    ap.add_argument("--flush-l2", action="store_true", help="rewrite a 512 MB buffer before every timed train step")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--decode-steps", type=int, default=None,
                    help="timed steps of each decode workload (default: --steps)")
    ap.add_argument("--no-graph", action="store_true", help="run the train step eagerly (no CUDA graph)")
    ap.add_argument("--skip-epoch", action="store_true", help="skip the embedding-loop / epoch measurement")
    ap.add_argument("--skip-prep", action="store_true", help="skip the grid-builder and encode/decode-driver measurements")
    ap.add_argument("--skip-wide", action="store_true", help="skip the vox11 / chanstr 16,32,16,16 decode (BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed train and decode steps computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the native path computed; the reference arm has nothing to dump")
    if args.decode_steps is None:
        args.decode_steps = args.steps
    return args


# ----------------------------------------------------------------------------- data
def make_cloud(resolution):
    from nvfpcc_b200 import synth
    pts = synth.sphere_shell_points(resolution)
    return pts, synth.leaf_origins(pts)


def make_net(chanstr, device):
    from nvfpcc_b200 import network, synth
    network.set_seed(synth.synthetic_seed())
    return network.Net(None, "Gaussian", ch=3, channel_str=chanstr).to(device)


def calibrate_threshold_bias(net, latents, thh, target_occ=0.021, sample=64):
    """Random-init weights never cross thh (SURVEY.md 8d): shift conv2_cls.b so that the
    (1 - target_occ) quantile of p equals thh, giving a realistic ~2 % occupancy."""
    with torch.no_grad():
        p = net.reconstruct(latents[:sample], 2)
        logit = torch.log(p) - torch.log1p(-p)
        qv = torch.quantile(logit.flatten()[:: 7].float(), 1 - target_occ)
        want = float(np.log(thh / (1 - thh)))
        net.reconstructor.conv2_cls.b += (want - qv)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled through NVML from a background thread every ~2 ms
    (nvidia-smi -lms cannot resolve a timed region of a few tens of milliseconds)."""

    def __init__(self, gpu_index=0):
        import threading
        self.idx, self.rows, self._stop, self._t = gpu_index, [], threading.Event(), None
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                  int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)),
                                  nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is None:
            return
        import threading
        self.rows, self._stop = [], threading.Event()
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.nv is None or self._t is None:
            return out
        self._stop.set()
        self._t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        if self.rows:
            bits = 0
            for _, r, _ in self.rows:
                bits |= r
            out.update(sm_mhz=statistics.median(r[0] for r in self.rows), sm_max_mhz=self.sm_max,
                       reasons=sorted(n for n, b in names.items() if bits & b), samples=len(self.rows),
                       power_w_max=max(r[2] for r in self.rows))
        return out


# ----------------------------------------------------------------------------- timing helpers
def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier_sync(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world):
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed(fn, steps, world, pre=None):
    """device time (CUDA events on the launching stream) of `steps` calls, summed over the calls
    (an optional untimed `pre` hook - the L2 flush - runs before each), max over ranks, in ms."""
    barrier_sync(world)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        if pre is not None:
            pre()
        ev[i][0].record()
        fn(i)
        ev[i][1].record()
    barrier_sync(world)
    return max_over_ranks(sum(a.elapsed_time(b) for a, b in ev), world)


def flush_l2(buf):
    buf.add_(1.0)  # 512 MB read+write: larger than the 126 MB L2


def ffma_peak(binding):
    sink = torch.empty(148 * 4 * 256 * 2, device="cuda")
    best = {}
    for variant in (0, 1):
        for _ in range(2):
            binding.ffma_microbench(variant, 2000, sink)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        flops = binding.ffma_microbench(variant, 40000, sink)
        e1.record()
        torch.cuda.synchronize()
        best["ffma" if variant == 0 else "ffma2"] = flops / (e0.elapsed_time(e1) * 1e-3) / 1e12
    return best


DUMP_MAX_ELEMS = 4 << 20       # per array: 16 MB as float32, so that a whole dump stays well under 64 MB


def dump_outputs(dirname, arrays):
    """DIR/<name>.npy for every array (float64 stays float64, everything else becomes float32; coordinates and counts
    are exact).  An array of more than DUMP_MAX_ELEMS elements is replaced by a fixed, seeded sample of its rows,
    kept in their original order, so that two runs with the same arguments write the same rows.  The sample is
    drawn from the array's row count: when two builds emit different numbers of points (only the wide decode is
    large enough to be sampled), compare the per-block counts first, since the sampled rows then differ throughout."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.size > DUMP_MAX_ELEMS:
            keep = DUMP_MAX_ELEMS // (a.size // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


# ----------------------------------------------------------------------------- workloads
class TrainWorkload:
    """Weight-loop steps of train() (NVFPCC.py:149-223) on the fused path."""

    def __init__(self, args, rank, world, pts, origins):
        from nvfpcc_b200 import synth
        self.args, self.rank, self.world = args, rank, world
        nb = min(args.train_blocks, origins.shape[0]) if args.train_blocks > 0 else origins.shape[0]
        sel = (np.arange(nb) + rank * (origins.shape[0] // max(1, world))) % origins.shape[0]
        from nvfpcc_b200 import grids
        g = grids.build_grids(pts, origins[sel], want_gt=True, want_dist64=False, want_dist32=True)   # util_get_grids.py on the GPU
        self.n_total = float(pts.shape[0])
        self.gt_dev = g["gt"].float()
        self.dist_dev = g["dist32"]
        self.gt_host = g["gt"].cpu().pin_memory()          # uint8, as *_gt_grid.npy stores it; converted on the device
        self.dist_host = self.dist_dev.cpu().pin_memory()
        self.nb = nb
        self.net = make_net(args.chanstr, "cuda")
        from nvfpcc_b200 import trainer
        self.opt = trainer.FusedAdam(self.net.parameters(), lr=HP["lr"])
        self.emb = torch.ones(nb, 3, 2, 2, 2, device="cuda")
        self.B = HP["batch"]
        self.ws = trainer.WeightStep(self.net, self.opt, self.B, self.n_total, HP["lmbda"], HP["w1"], HP["w2"],
                                     use_graph=not args.no_graph)
        self.idx_dev = [self.batch_idx(i).cuda() for i in range(max(1, nb // self.B))]
        # batch-global n_pts (NVFPCC.py:154) of every batch of the cycle from the per-block point counts, summed over
        # the ranks ONCE here (as trainer.fit does): the timed step has no gt reduction and no scalar all-reduce
        cnt = self.gt_dev.reshape(nb, -1).sum(1)
        npts = torch.stack([cnt[i].sum() for i in self.idx_dev])
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(npts)
        self.npts = npts.reshape(-1, 1)
        self.packed = [self.ws.pack_schedule(i, n) for i, n in zip(self.idx_dev, self.npts)]
        self.last_loss = None

    def batch_idx(self, i):
        s = (i * self.B) % self.nb
        return (torch.arange(self.B) + s) % self.nb

    def step(self, i, host_inputs):
        """One weight-loop step (NVFPCC.py:149-223): batch -> static buffers -> fused fwd + loss + bwd +
        all-reduce + Adam (one CUDA-graph replay), inputs resident in HBM."""
        k = i % len(self.idx_dev)
        st = self.ws.step_indexed(self.emb, self.gt_dev, self.dist_dev, self.idx_dev[k], q=1, n_pts=self.npts[k],
                                  packed=self.packed[k])
        self.last_loss = st[0]
        return st

    def e2e_loop(self, first, steps):
        """`steps` weight-loop steps fed from HOST memory through the public API (trainer.HostBatchFeeder +
        trainer.WeightStep): every step's gt/dist batch is gathered from the host dataset into pinned memory,
        copied H2D, and every step's loss is read back D2H - the reference's DataLoader / .to(device) / .item()
        path (NVFPCC.py:149-223) - with the copies of step i+1 overlapping the kernels of step i."""
        from nvfpcc_b200 import trainer
        if not hasattr(self, "feeder"):
            self.feeder = trainer.HostBatchFeeder(self.gt_host, self.dist_host, self.B)
            self.emb_batches = [self.emb[self.batch_idx(i).cuda()] for i in range(max(1, self.nb // self.B))]
            # schedule rows (slot's row indices + the batch's n_pts) for the in-place read of the feeder's slots
            self.packed_e2e = [[self.ws.pack_schedule(self.feeder.slot_rows(s), n) for n in self.npts] for s in range(2)]
        f = self.feeder
        f.submit(self.batch_idx(first))
        for i in range(first, first + steps):
            (gt, dst), slot = f.take()
            k = i % len(self.emb_batches)
            # the fused step reads the slot in place (rows of the feeder's device buffers): no copy of the batch
            st = self.ws.step_indexed(f.emb_stage(self.emb_batches[k], slot), f.gt_all, f.dist_all, f.slot_rows(slot),
                                      q=1, n_pts=self.npts[k], packed=self.packed_e2e[slot][k])
            f.release(slot)
            if i + 1 < first + steps:
                f.submit(self.batch_idx(i + 1))        # overlaps the kernels of step i
            prev = f.read_stats(st)                     # D2H of this step's result; returns the previous step's
            if prev is not None:
                self.last_loss = float(prev[0])
        self.last_loss = float(f.drain()[0])

    h2d_bytes = 16 * 32768 * (1 + 4)      # gt uint8 + dist float32 per block
    d2h_bytes = 7 * 4


class DecodeWorkload:
    """All leaf blocks of a cloud through nvf_decode (NVFPCC.py:625-638 batched), block-sharded over the ranks."""

    def __init__(self, chanstr, rank, world, pts, origins, thh):
        from nvfpcc_b200 import dist as D
        from nvfpcc_b200 import synth
        self.rank, self.world, self.thh, self.chanstr = rank, world, thh, chanstr
        self.n_all = origins.shape[0]
        lo, hi = D.block_range(self.n_all, rank, world)
        lat = synth.random_latents(self.n_all, 3, seed=0)
        self.lat_host = torch.from_numpy(lat[lo:hi]).pin_memory()
        self.org_host = torch.from_numpy(origins[lo:hi].astype(np.int32)).pin_memory()
        self.lat_dev, self.org_dev = self.lat_host.cuda(), self.org_host.cuda()
        self.net = make_net(chanstr, "cuda")
        calibrate_threshold_bias(self.net, torch.from_numpy(lat).cuda(), thh)
        self.n_local = hi - lo
        self.points = 0
        self.checksum = None
        self.kernel_events = []
        self._host = None

    def finish(self):
        """Order-sensitive checksum of the last gathered cloud: equal across GPU counts <=> identical point lists."""
        if self._host is not None and self.points:
            c_host = self._host[:self.points].long()
            w = torch.arange(1, self.points + 1, dtype=torch.int64) % 1000003
            self.checksum = int(((c_host * torch.tensor([1, 1 << 11, 1 << 22])).sum(1) * w).sum() % (1 << 61))

    def step(self, i, host_inputs):
        from nvfpcc_b200 import dist as D
        if host_inputs:
            r = self.net.decode_points(self.lat_host, self.org_host, self.thh, return_host=False)
            c, n = D.gather_points(r["coords"], r["counts"])     # coordinate gather to rank 0
            if c is not None:
                # device -> host read of the result into a pinned buffer (grown on demand), as a caller writing the
                # cloud out would do; the verification checksum is computed outside the timed region (finish())
                k = c.shape[0]
                if self._host is None or self._host.shape[0] < k:
                    self._host = torch.empty((max(k, 1) * 5 // 4, 3), dtype=torch.int32).pin_memory()
                self._host[:k].copy_(c, non_blocking=True)
                torch.cuda.current_stream().synchronize()
                self.points = k
        else:
            r = self.net.decode_points(self.lat_dev, self.org_dev, self.thh, return_host=False,
                                       timing=self.kernel_events)
            self.last = r               # the device-resident result of the latest timed step (--dump-outputs)
        return r


def decode_bench(args, chanstr, resolution, rank, world, local, binding, pts, origins, flush, thh, steps):
    """-> (compact dict, DecodeWorkload) on rank 0; device-resident `value`, host-to-host `e2e`, kernel roofline."""
    dw = DecodeWorkload(chanstr, rank, world, pts, origins, thh)
    for i in range(3):
        dw.step(i, False)
    dl0 = binding.launch_count()
    dw.kernel_events = []
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total = timed(lambda i: dw.step(i, False), steps, world, pre=lambda: flush_l2(flush))
    clocks = sampler.stop() if rank == 0 else None
    launches = binding.launch_count() - dl0
    ms = ms_total / steps
    # the nvf_decode launch sequence alone: CUDA events on its stream
    kernel_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in dw.kernel_events) / max(1, len(dw.kernel_events)), world)
    for i in range(2):
        dw.step(i, True)
    barrier_sync(world)
    t0 = time.perf_counter()
    for i in range(steps):
        dw.step(i, True)
    barrier_sync(world)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world) / steps
    dw.finish()
    out = dict(metric="decoded_voxels_per_sec", value=dw.n_all * 32768 / (ms * 1e-3), unit="voxels/s", ms_per_step=ms,
               ms_kernel=kernel_ms, blocks=int(dw.n_all), blocks_rank0=int(dw.n_local), points=int(dw.points),
               points_checksum=dw.checksum, gpu_launches=int(launches), steps=steps, clocks=clocks,
               workload="vox%d %s thh %.2f" % (10 if resolution == 1024 else 11, chanstr, thh),
               e2e=dict(value=dw.n_all * 32768 / (e2e_ms * 1e-3), unit="voxels/s",
                        h2d_bytes_per_step=int(dw.n_all * (96 + 12)), d2h_bytes_per_step=int(dw.points * 12)))
    return out, dw


def embedding_loop(tw, args, world, n_blocks, flush):
    """The once-per-epoch embedding update (NVFPCC.py:225-251): ONE full-batch forward + backward over all of the
    rank's leaf blocks w.r.t. the embeddings (weight gradients skipped: the reference discards them) + Adam on
    the embeddings.  gt/dist of the `train_blocks` distinct synthetic blocks are tiled to `n_blocks`."""
    from nvfpcc_b200 import _lib, trainer
    bind = _lib.cuda_binding()
    per_block = bind.workspace_bytes(bind.desc(3, [int(c) for c in args.chanstr.split(",")]), 64, _lib.NVF_MODE_TRAIN) / 64
    n_full, scale = n_blocks, 1.0
    if n_blocks * per_block > 40e9:            # bound the activation stash: measure a slice, scale linearly
        n_blocks = int(40e9 / per_block)
        scale = n_full / n_blocks
    reps = (n_blocks + tw.nb - 1) // tw.nb
    gt = tw.gt_dev.repeat(reps, 1, 1, 1, 1)[:n_blocks].contiguous()
    dst = tw.dist_dev.repeat(reps, 1, 1, 1, 1)[:n_blocks].contiguous()
    emb = torch.ones(n_blocks, 3, 2, 2, 2, device="cuda", requires_grad=True)
    opt_emb = torch.optim.Adam([emb], lr=HP["lr"] * 5.0)                       # lr * wemb (NVFPCC.py:124)
    es = trainer.EmbeddingStep(tw.net, emb, opt_emb, tw.n_total, HP["lmbda"], HP["w1"], HP["w2"])
    es.step(gt, dst, 1)
    ms = timed(lambda i: es.step(gt, dst, 1), 2, world, pre=lambda: flush_l2(flush)) / 2 * scale
    del es, opt_emb, emb, gt, dst
    torch.cuda.empty_cache()
    return ms


# ----------------------------------------------------------------------------- rows either side of the path (SURVEY 8f)
def measured_traffic(kind, **match):
    """roofline.traffic: DRAM bytes per launch from the committed ncu capture (profiles/r02_traffic.json), only
    when this run's workload is the captured one; otherwise None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            e = json.load(f)[kind]
        return e["dram_bytes"] if all(e.get(k) == v for k, v in match.items()) else None
    except Exception:
        return None


def hbm_peak_gbs():
    """Measured copy bandwidth of this pool's B200s (driver-written MEASURED_PEAKS.json), else the
    profiling guide's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6550.0, "B200_PROFILING.md fallback (MEASURED_PEAKS.json absent)"


def grids_bench(args, rank, world, pts, origins, flush, with_cpu):
    """util_get_grids.py:19-46 for the rank's leaves: nvf_build_grids (cells + per-leaf exact distance
    transform), inputs resident in HBM; e2e = host points/origins in, uint8 gt + float64 dist out to host."""
    from nvfpcc_b200 import dist as D
    from nvfpcc_b200 import grids
    lo, hi = D.block_range(origins.shape[0], rank, world)
    p_dev = torch.from_numpy(pts).cuda()
    o_dev = torch.from_numpy(origins[lo:hi].astype(np.int32)).cuda()
    # aligned octree leaves: the occupied 32^3 cells of the cloud ARE the leaves
    kw = dict(want_gt=True, want_dist64=True, want_dist32=True, check=False, max_cells=int(origins.shape[0]))
    for _ in range(2):
        grids.build_grids(p_dev, o_dev, **kw)
    reps = 5
    ms = timed(lambda i: grids.build_grids(p_dev, o_dev, **kw), reps, world, pre=lambda: flush_l2(flush)) / reps
    barrier_sync(world)
    t0 = time.perf_counter()
    grids.build_grids_host(pts, origins[lo:hi])                # warm-up: pinned staging buffers, lazy init
    barrier_sync(world)
    t0 = time.perf_counter()
    rh = grids.build_grids_host(pts, origins[lo:hi])           # host points in, uint8 gt + float64 dist on the host out
    gt_h = torch.from_numpy(rh["gt"])
    barrier_sync(world)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
    n_all = origins.shape[0]
    vox = n_all * 32768
    bytes_per_vox = 1 + 8 + 4                                  # gt u8 + dist f64 + dist f32 written per grid voxel
    alg_bytes = (hi - lo) * 32768 * bytes_per_vox + pts.shape[0] * 12 + (hi - lo) * 12
    peak, src = hbm_peak_gbs()
    ach = alg_bytes / (ms * 1e-3) / 1e9
    out = dict(metric="grid_voxels_per_sec", value=vox / (ms * 1e-3), unit="voxels/s", ms_per_step=ms, blocks=int(n_all),
               points=int(pts.shape[0]), gpu_launches=3 * reps, occupied=int(gt_h.sum()) if world == 1 else None,
               workload="gt_grid + dist of all %d leaves of the synthetic cloud (util_get_grids.py), exact, float64" % n_all,
               e2e=dict(value=vox / (e2e_ms * 1e-3), unit="voxels/s", h2d_bytes_per_step=int(pts.shape[0] * 12 + (hi - lo) * 12),
                        d2h_bytes_per_step=int((hi - lo) * 32768 * 9)),
               roofline=dict(bound="hbm", achieved=ach, peak=peak, unit="GB/s", frac=ach / peak,
                             traffic=measured_traffic("grids", blocks=int(hi - lo)),
                             per_gpu=True, algorithmic_bytes_per_block=32768 * bytes_per_vox, peak_source=src,
                             kernel="k_edt_blocks", note="integer shared-memory work per plane, not HBM, limits this "
                                                         "kernel today (DESIGN.md section 3)"))
    if with_cpu:
        from oracle import grids_oracle as GO
        nb = min(48, n_all)
        t0 = time.perf_counter()
        GO.build_grids(pts, origins[:nb], workers=-1)
        el = time.perf_counter() - t0
        out["cpu_baseline"] = dict(value=nb * 32768 / el, unit="voxels/s", cores=os.cpu_count(), kind="port",
                                   sample="%d leaves (%.1f s) of the oracle port: scipy cKDTree queries on all host "
                                          "threads (the reference itself calls open3d's KD-tree once per voxel from "
                                          "Python, util_get_grids.py:37-39)" % (nb, el))
    return out


def codec_bench(args, rank, world, origins, with_cpu):
    """encode() / decode() of the reference (NVFPCC.py:395-652) through nvfpcc_b200.codec: wall time from the
    embeddings / the pack in HOST memory to the reconstructed cloud in host memory, entropy coding included."""
    from nvfpcc_b200 import codec, entropy, network, synth
    net = make_net(args.chanstr, "cpu")
    sd = net.state_dict()
    sd.update(synth.random_kernel_deltas(sd, seed=1, sigma=0.05, quantize=True))
    net.load_state_dict(sd)
    net = net.cuda()
    n = origins.shape[0]
    emb = torch.from_numpy(synth.random_latents(n, 3, seed=3)) * 0.7
    with torch.no_grad():
        lat = net.get_latent_code(emb[:64].cuda())["quantized_latent"]
    calibrate_threshold_bias(net, lat, 0.64)
    state = codec.quantize_state({k: v.detach().cpu() for k, v in net.state_dict().items()}, 16)
    net.load_state_dict(state, strict=False)
    codec.encode(net, emb[:64], origins[:64], 0.64, weights_state=state)       # warm-up
    barrier_sync(world)
    t0 = time.perf_counter()
    enc = codec.encode(net, emb, origins, 0.64, weights_state=state)
    barrier_sync(world)
    enc_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
    network.set_seed(synth.synthetic_seed())
    t0 = time.perf_counter()
    dec = codec.decode(enc["total_pack"], 3, args.chanstr, 0.64)
    barrier_sync(world)
    dec_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
    if rank != 0:
        return None
    lp = enc["total_pack"]["latent_pack"]
    out = dict(metric="decoded_voxels_per_sec", workload="encode() -> pack -> decode() of all %d leaves, 1/16-quantised "
               "weights, thh 0.64, host to host (BASELINE.json configs[2])" % n,
               encode_ms=enc_ms, decode_ms=dec_ms, value=n * 32768 / (dec_ms * 1e-3), unit="voxels/s",
               points=int(dec.shape[0]), rc_enc_equals_rc_dec=bool(np.array_equal(dec, enc["points"])),
               latent_stream_bytes=len(lp["latent_byte_stream"]),
               weight_stream_bytes=len(enc["total_pack"]["net_weight_pack"]["bit_stream"]),
               bpp=(enc["latent_bits"] + enc["net_bits"]) / max(1, dec.shape[0]))
    # entropy coder alone: in-process coder vs the reference's helper binary (when compiled into oracle/_ref)
    s = tuple(lp["shape"])
    mu = (np.broadcast_to(lp["mu"].numpy().astype(np.float32), s).reshape(-1) + np.float32(512)).astype(np.float32)
    sg = np.broadcast_to(lp["sigma"].numpy().astype(np.float32), s).reshape(-1).astype(np.float32)
    sym = (entropy.decode_latents(lp).reshape(-1) + 512).astype(np.int16)
    t0 = time.perf_counter()
    for _ in range(5):
        stream = entropy.arithmetic_encode(sym, mu, sg)
        entropy.arithmetic_decode(stream, mu, sg)
    el = (time.perf_counter() - t0) / 5
    out["entropy"] = dict(symbols=int(sym.size), value=sym.size / el, unit="symbols/s (encode + decode)")
    exe = os.path.join(ROOT, "oracle", "_ref", "module_arithmeticcoding")
    if with_cpu and os.path.isfile(exe):
        length = np.array([sym.size], dtype=np.int64)
        t0 = time.perf_counter()
        r = subprocess.run([exe, "e", "1", "1"], input=length.tobytes() + sym.tobytes() + mu.tobytes() + sg.tobytes(),
                           stdout=subprocess.PIPE).stdout
        subprocess.run([exe, "d", "1", "1"], input=length.tobytes() + mu.tobytes() + sg.tobytes() + r, stdout=subprocess.PIPE)
        el_ref = time.perf_counter() - t0
        out["entropy"]["cpu_baseline"] = dict(value=sym.size / el_ref, unit="symbols/s (encode + decode)", cores=1,
                                              kind="reference", same_stream=bool(r == stream),
                                              sample="the reference's module_arithmeticcoding helper (oracle/_ref), "
                                                     "all %d latent symbols, subprocess as in NVFPCC.py:461-470" % sym.size)
    return out


# ----------------------------------------------------------------------------- reference arm
def oracle_state(chanstr):
    from nvfpcc_b200 import synth
    from oracle import nvf_oracle as O
    return O.make_state(3, [int(c) for c in chanstr.split(",")], synth.synthetic_seed())


def cpu_train_baseline(args, pts, origins, budget_s=20.0, max_steps=None, warmup=1):
    """The reference algorithm (oracle port, torch CPU fp32, all host threads) on the same train
    workload: one weight-loop step = forward + losses + backward + Adam at batch 16."""
    from nvfpcc_b200 import synth
    from oracle import nvf_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    sd = {k: v.clone() for k, v in oracle_state(args.chanstr).items() if not k.startswith("_")}
    params = {k: v.requires_grad_(True) for k, v in sd.items() if not k.endswith(("_init", "pedestal"))}
    opt = torch.optim.Adam(list(params.values()), lr=HP["lr"])
    B = HP["batch"]
    gt, dist_ = synth.gt_and_dist(pts, origins[:B])
    gt, dist_ = torch.from_numpy(gt).float(), torch.from_numpy(dist_).float()
    emb = torch.ones(B, 3, 2, 2, 2, requires_grad=True)
    n_total = float(pts.shape[0])

    def one():
        opt.zero_grad()
        res = O.net_forward(emb, sd, "train", 1)
        L = O.train_loss(res, gt, dist_, gt.sum(), n_total, HP["lmbda"], HP["w1"], HP["w2"])
        L["loss"].backward()
        opt.step()

    for _ in range(max(1, warmup)):
        one()
    t0 = time.perf_counter()
    n = 0
    while True:
        one()
        n += 1
        el = time.perf_counter() - t0
        if (max_steps and n >= max_steps) or (not max_steps and (el > budget_s or n >= 64)):
            break
    return dict(value=n * B / el, unit="blocks/s", cores=torch.get_num_threads(), kind="port",
                sample="%d weight-loop steps at batch %d (%.1f s) of the oracle port, torch CPU fp32" % (n, B, el)), el / n


def cpu_decode_baseline(args, origins, budget_s=12.0):
    """decode() as shipped: one block per iteration, batch 1 (NVFPCC.py:625-638)."""
    from nvfpcc_b200 import synth
    from oracle import nvf_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    sd = {k: v for k, v in oracle_state(args.chanstr).items() if not k.startswith("_")}
    lat = torch.from_numpy(synth.random_latents(256, 3, seed=0))
    n = 0
    with torch.no_grad():
        O.reconstruct(lat[:1], sd, 2)
        t0 = time.perf_counter()
        while n < 256:
            p = O.reconstruct(lat[n:n + 1], sd, 2)
            O.threshold_points(p, origins[n:n + 1], HP["thh"])
            n += 1
            if time.perf_counter() - t0 > budget_s:
                break
        el = time.perf_counter() - t0
    return dict(value=n * 32768 / el, unit="voxels/s", cores=torch.get_num_threads(), kind="port",
                sample="%d blocks at batch 1 (%.1f s) of the oracle port, torch CPU fp32" % (n, el))


def torch_cuda_baseline(args, pts, origins, budget_s=6.0):
    """The reference's op sequence (oracle port = plain torch ops -> cuDNN / ATen kernels) on THIS B200 with TF32
    off: the 'same box, stock framework' bar of SURVEY.md 8d.  Not the product path - a reported baseline.
    train: weight-loop steps at batch 16 with the per-step `.item()` read of train() (NVFPCC.py:190-221);
    decode: the batch-1 loop of decode() (NVFPCC.py:625-638) incl. the per-block device->host reads."""
    from nvfpcc_b200 import synth
    from oracle import nvf_oracle as O
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        dev = torch.device("cuda")
        sd = {k: v.clone().to(dev) for k, v in oracle_state(args.chanstr).items() if not k.startswith("_")}
        params = {k: v.requires_grad_(True) for k, v in sd.items() if not k.endswith(("_init", "pedestal"))}
        opt = torch.optim.Adam(list(params.values()), lr=HP["lr"])
        B = HP["batch"]
        gt, dist_ = synth.gt_and_dist(pts, origins[:B])
        gt, dist_ = torch.from_numpy(gt).float().to(dev), torch.from_numpy(dist_).float().to(dev)
        emb = torch.ones(B, 3, 2, 2, 2, device=dev, requires_grad=True)
        n_total = float(pts.shape[0])

        def one():
            opt.zero_grad()
            res = O.net_forward(emb, sd, "train", 1)
            L = O.train_loss(res, gt, dist_, gt.sum(), n_total, HP["lmbda"], HP["w1"], HP["w2"])
            L["loss"].backward()
            opt.step()
            return float(L["loss"].item())

        for _ in range(3):
            one()
        torch.cuda.synchronize()
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < budget_s and n < 200:
            one()
            n += 1
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        train = dict(value=n * B / el, unit="blocks/s", sample="%d weight-loop steps at batch %d (%.1f s)" % (n, B, el))
        lat = torch.from_numpy(synth.random_latents(256, 3, seed=0)).to(dev)
        sd_d = {k: v.detach() for k, v in sd.items()}
        with torch.no_grad():
            O.reconstruct(lat[:1], sd_d, 2)
            torch.cuda.synchronize()
            t0, m = time.perf_counter(), 0
            while m < 256 and time.perf_counter() - t0 < budget_s:
                pr = O.reconstruct(lat[m:m + 1], sd_d, 2)
                O.threshold_points(pr.cpu(), origins[m:m + 1], HP["thh"])
                m += 1
            torch.cuda.synchronize()
            el = time.perf_counter() - t0
        dec = dict(value=m * 32768 / el, unit="voxels/s", sample="%d blocks at batch 1 (%.1f s)" % (m, el))
        # batch 256 "for fairness" (BASELINE.md section 4): the same ops on 256 blocks per call, thresholded on the
        # device, one D2H of the points per call
        lat_b = torch.from_numpy(synth.random_latents(1024, 3, seed=0)).to(dev)
        org_b = torch.from_numpy(np.resize(origins, (1024, 3)).astype(np.int64)).to(dev)
        with torch.no_grad():
            def call(s):
                pr = O.reconstruct(lat_b[s:s + 256], sd_d, 2)
                idx = torch.nonzero(pr[:, 0] > HP["thh"])
                return (idx[:, 1:] + org_b[s:s + 256][idx[:, 0]]).cpu()
            call(0)
            torch.cuda.synchronize()
            t0, m = time.perf_counter(), 0
            while time.perf_counter() - t0 < budget_s and m < 64:
                call((m % 4) * 256)
                m += 1
            torch.cuda.synchronize()
            el = time.perf_counter() - t0
        dec256 = dict(value=m * 256 * 32768 / el, unit="voxels/s", sample="%d calls at batch 256 (%.1f s)" % (m, el))
        return dict(kind="port on torch-CUDA (cuDNN/ATen, TF32 off) on the same B200", train=train, decode=dec,
                    decode_b256=dec256)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pts, origins = make_cloud(args.resolution)
    cb, sec_per = cpu_train_baseline(args, pts, origins, max_steps=args.steps, warmup=args.warmup)
    dec = cpu_decode_baseline(args, origins)
    # rows either side of the path, CPU side: the grid oracle (scipy cKDTree, all threads) and the reference's own
    # arithmetic-coding helper (oracle/_ref) on seeded latents of the cloud's size
    from oracle import grids_oracle as GO
    nb = min(48, origins.shape[0])
    t0 = time.perf_counter()
    GO.build_grids(pts, origins[:nb], workers=-1)
    el = time.perf_counter() - t0
    grids_ref = dict(metric="grid_voxels_per_sec", value=nb * 32768 / el, unit="voxels/s",
                     cpu_baseline=dict(value=nb * 32768 / el, unit="voxels/s", cores=os.cpu_count(), kind="port",
                                       sample="%d leaves (%.1f s), scipy cKDTree restatement of util_get_grids.py" % (nb, el)))
    entropy_ref = None
    exe = os.path.join(ROOT, "oracle", "_ref", "module_arithmeticcoding")
    if os.path.isfile(exe):
        rng = np.random.default_rng(0)
        n = origins.shape[0] * 24
        sym = (np.clip(np.rint(rng.normal(0, 3, n)), -512, 511) + 512).astype(np.int16)
        mu, sg = np.full(n, 512, np.float32), np.full(n, 3, np.float32)
        length = np.array([n], dtype=np.int64)
        t0 = time.perf_counter()
        r = subprocess.run([exe, "e", "1", "1"], input=length.tobytes() + sym.tobytes() + mu.tobytes() + sg.tobytes(),
                           stdout=subprocess.PIPE).stdout
        subprocess.run([exe, "d", "1", "1"], input=length.tobytes() + mu.tobytes() + sg.tobytes() + r, stdout=subprocess.PIPE)
        el = time.perf_counter() - t0
        entropy_ref = dict(value=n / el, unit="symbols/s (encode + decode)", cores=1, kind="reference", symbols=int(n),
                           sample="module_arithmeticcoding compiled from the reference source, subprocess as in NVFPCC.py:461-470")
    line = dict(impl="reference", metric="train_blocks_per_sec", value=cb["value"], unit="blocks/s",
                n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=sec_per * 1e3,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                config=workload_config(args, args.gpus), cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit="blocks/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                decode=dict(metric="decoded_voxels_per_sec", value=dec["value"], unit="voxels/s", cpu_baseline=dec,
                            e2e=dict(value=dec["value"], unit="voxels/s", h2d_bytes_per_step=0,
                                     d2h_bytes_per_step=0)),
                grids=grids_ref, codec=dict(entropy=entropy_ref))
    compact = {k: v for k, v in line.items() if k not in ("grids", "codec", "decode")}
    compact["grids"] = dict(value=grids_ref["value"], unit=grids_ref["unit"])
    compact["decode"] = line["decode"]
    emit(compact, line)


def workload_config(args, world):
    return {"workload": "BASELINE configs[1]: NVFPCC.py train weight-loop steps, synthetic vox%d leaf blocks, batch 16/GPU, "
                        "lambda=200 lr=1e-3 q=1, chanstr %s ch=3" % (10 if args.resolution == 1024 else 11, args.chanstr),
            "chanstr": args.chanstr, "batch_per_gpu": HP["batch"], "global_batch": HP["batch"] * world,
            "parallelism": "dp%d" % world, "l2": "512 MB flush between timed steps"}


# ----------------------------------------------------------------------------- main
def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        return run_reference(args)
    from nvfpcc_b200 import _lib
    rank, world, local = dist_setup(args.gpus)
    # a fixed seed per rank: the in-kernel noise of the train steps, and with it every output, repeats from run to run
    torch.manual_seed(rank)
    binding = _lib.cuda_binding()
    pts, origins = make_cloud(args.resolution)
    flush = torch.zeros(128 * 1024 * 1024, device="cuda")
    sampler = ClockSampler(local)

    # ---------------- train (primary) ----------------
    tw = TrainWorkload(args, rank, world, pts, origins)
    for i in range(args.warmup):
        tw.step(i, False)
    launches0 = binding.launch_count()
    if rank == 0:
        sampler.start()

    # L2: the cycled dataset (gt + dist of tw.nb leaves, float32) is larger than the L2, so a step's inputs are never
    # cache-resident while weights and workspace are as warm as in a real epoch; small datasets get the explicit flush
    dataset_mb = tw.nb * 2 * 32768 * 4 / 1e6
    use_flush = args.flush_l2 or dataset_mb < 1.5 * 126
    ms_total = timed(lambda i: tw.step(args.warmup + i, False), args.steps, world,
                     pre=(lambda: flush_l2(flush)) if use_flush else None)
    clocks = sampler.stop() if rank == 0 else None
    # replayed graphs do not pass through the library's host-side launch counter
    launches = (binding.launch_count() - launches0) if args.no_graph else tw.ws.launches_per_step * args.steps
    ms_step = ms_total / args.steps
    train_value = HP["batch"] * world / (ms_step * 1e-3)
    outputs = {}
    if args.dump_outputs and rank == 0:
        # the last timed step's stats (trainer.STAT_NAMES) and the weights it left; the e2e steps below train on
        outputs["train_stats"] = tw.ws.stats.cpu().numpy()
        outputs.update(("train_" + k, v.cpu().numpy()) for k, v in tw.net.state_dict().items() if v.is_floating_point())
    tw.e2e_loop(0, 3)
    barrier_sync(world)
    t0 = time.perf_counter()
    tw.e2e_loop(args.warmup, args.steps)
    barrier_sync(world)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world) / args.steps
    train_e2e = HP["batch"] * world / (e2e_ms * 1e-3)

    # ---------------- embedding loop / whole epoch ----------------
    epoch = None
    if not args.skip_epoch:
        from nvfpcc_b200 import dist as D
        lo, hi = D.block_range(origins.shape[0], rank, world)
        emb_ms = embedding_loop(tw, args, world, hi - lo, flush)
        n_all = origins.shape[0]
        steps_a = (n_all + HP["batch"] * world - 1) // (HP["batch"] * world)     # weight-loop steps per epoch
        epoch_ms = steps_a * ms_step + emb_ms
        f_emb = F_TRAIN[args.chanstr] * 2.0 / 3.0                                # forward + data gradients
        epoch = dict(blocks=int(n_all), weight_loop_steps=int(steps_a), weight_loop_ms=steps_a * ms_step,
                     embedding_loop_ms=emb_ms, epoch_ms=epoch_ms, epochs_per_sec=1e3 / epoch_ms,
                     block_passes_per_sec=2.0 * n_all / (epoch_ms * 1e-3),
                     embedding_loop_tflops=(hi - lo) * f_emb / (emb_ms * 1e-3) / 1e12,
                     note="one epoch of train() (NVFPCC.py:128-254) = weight loop over all blocks at batch 16 per GPU "
                          "(measured per step above, x steps) + one full-batch embedding update (measured); "
                          "embedding_loop_tflops counts forward + data-gradient FLOPs only (2/3 of F_train)")

    # ---------------- decode (second half of the metric) ----------------
    dec, dw = decode_bench(args, args.chanstr, args.resolution, rank, world, local, binding, pts, origins, flush,
                           HP["thh"], args.decode_steps)
    # BASELINE.json configs[3]: vox11 cloud, wide chanstr, block-sharded decode (same commit at every N)
    dec_wide = dw_wide = None
    if not args.skip_wide:
        pts11, origins11 = make_cloud(2048)
        dec_wide, dw_wide = decode_bench(args, "16,32,16,16", 2048, rank, world, local, binding, pts11, origins11, flush,
                                         HP["thh"], args.decode_steps)
    if args.dump_outputs and rank == 0:
        for tag, w in (("decode", dw), ("decode_wide", dw_wide)):
            if w is not None:
                outputs.update((tag + "_" + k, w.last[k].cpu().numpy()) for k in ("coords", "counts"))
        dump_outputs(args.dump_outputs, outputs)

    # ---------------- rows either side of the path: grid builder, encode/decode drivers ----------------
    prep = None
    if not args.skip_prep:
        with_cpu = (not args.skip_cpu_baseline) and world == 1
        prep = dict(grids=grids_bench(args, rank, world, pts, origins, flush, with_cpu),
                    codec=codec_bench(args, rank, world, origins, with_cpu))

    if rank != 0:
        return
    peaks = ffma_peak(binding)
    peak = min(FP32_PEAK_THEORETICAL, max(peaks.values()))
    cs = args.chanstr
    t_ach = train_value / world * F_TRAIN[cs] / 1e12
    peak_source = ("live nvf_ffma_microbench (MEASURED_PEAKS.json has no fp32 figure): ffma %.1f, ffma2 %.1f TFLOP/s; "
                   "theoretical 74.4 at 1965 MHz; denominator = min" % (peaks["ffma"], peaks["ffma2"]))

    def dec_roofline(d, w, chanstr):
        ach = w.n_local * F_DEC[chanstr] / (d["ms_kernel"] * 1e-3) / 1e12    # rank 0's blocks / its kernel time
        tr = measured_traffic("decode", chanstr=chanstr, blocks=int(w.n_local))
        return dict(bound="fp32", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak, traffic=tr,
                    kernel="nvf_decode: stem layer kernels + k_decode_head (fused up2-conv2-cls-threshold, 78 % of the time)"
                    if binding.has_fused_decode(chanstr) else "layer-wise kernels")

    dec["roofline"] = dec_roofline(dec, dw, cs)
    if dec_wide is not None:
        dec_wide["roofline"] = dec_roofline(dec_wide, dw_wide, "16,32,16,16")
    traffic = measured_traffic("train", chanstr=cs, blocks_per_step=HP["batch"])
    line = dict(
        metric="train_blocks_per_sec", value=train_value, unit="blocks/s", n_gpus=world, steps=args.steps,
        warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None,
        dtype="f32", data="synthetic", config=dict(workload_config(args, world), l2=(
            "512 MB flush between timed steps" if use_flush else
            "inputs larger than L2: %d-leaf dataset, %.0f MB of gt + dist cycled, no flush" % (tw.nb, dataset_mb))),
        clocks=clocks,
        e2e=dict(value=train_e2e, unit="blocks/s", h2d_bytes_per_step=TrainWorkload.h2d_bytes,
                 d2h_bytes_per_step=TrainWorkload.d2h_bytes),
        gpu_launches=int(launches),
        roofline=dict(bound="fp32", achieved=t_ach, peak=peak, unit="TFLOP/s", frac=t_ach / peak, traffic=traffic,
                      kernel="whole train step"))
    detail = dict(line)
    detail["roofline"] = dict(line["roofline"], per_gpu=True, algorithmic_flop_per_block=F_TRAIN[cs],
                              peak_source=peak_source, hbm_gbs=(traffic or 0) / (ms_step * 1e-3) / 1e9,
                              hbm=dict(algorithmic_bytes_per_block=164032,
                                       achieved_gbs=train_value / world * 164032 / 1e9, peak_gbs=hbm_peak_gbs()[0],
                                       note="96 B emb + 32 KB gt + 128 KB dist + 96 B d_emb per block: the path is "
                                            "FP32-FMA bound, HBM is <0.1 % utilised by algorithmic bytes"))
    if not args.skip_cpu_baseline and world == 1:
        tcb = torch_cuda_baseline(args, pts, origins)
        cb, _ = cpu_train_baseline(args, pts, origins, budget_s=15.0)
        dcb = cpu_decode_baseline(args, origins, budget_s=10.0)
        detail["torch_cuda_baseline"], detail["cpu_baseline"] = tcb, cb
        line["cpu_baseline"] = cb
        line["torch_cuda_baseline"] = dict(train=tcb["train"]["value"], decode_b1=tcb["decode"]["value"],
                                           decode_b256=tcb["decode_b256"]["value"])
        dec["cpu_baseline"] = dcb
    if epoch is not None:
        epoch["embedding_loop_frac_of_peak"] = epoch["embedding_loop_tflops"] / peak
        detail["epoch"] = epoch
        line["epoch"] = dict(epoch_ms=epoch["epoch_ms"], embedding_loop_ms=epoch["embedding_loop_ms"],
                             embedding_loop_frac_of_peak=epoch["embedding_loop_frac_of_peak"])
    if prep is not None:
        detail["grids"], detail["codec"] = prep["grids"], prep["codec"]
        gr, cd = prep["grids"], prep["codec"] or {}
        line["grids"] = dict(value=gr["value"], unit=gr["unit"], ms_per_step=gr["ms_per_step"], e2e=gr["e2e"]["value"],
                             hbm_frac=gr["roofline"]["frac"])
        line["codec"] = dict(encode_ms=cd.get("encode_ms"), decode_ms=cd.get("decode_ms"),
                             rc_enc_equals_rc_dec=cd.get("rc_enc_equals_rc_dec"),
                             same_stream=(cd.get("entropy", {}).get("cpu_baseline") or {}).get("same_stream"))
    detail["decode"] = dec
    if dec_wide is not None:
        detail["decode_wide"] = dec_wide
        line["decode_wide"] = {k: v for k, v in dec_wide.items() if k != "clocks"}
    line["decode"] = dec                          # the second half of the metric: LAST, so that a log tail keeps it
    emit(line, detail)


if __name__ == "__main__":
    main()
