"""Host-sync-free training steps for the NVF path (SURVEY.md 8f-2).

`WeightStep` is the body of the reference's weight loop (train(), NVFPCC.py:149-223)
and `EmbeddingStep` the once-per-epoch embedding update (NVFPCC.py:225-251), with

* every scalar the reference reads back with `.item()` (NVFPCC.py:190-221) kept on the
  device in one small `stats` tensor that the caller may read whenever it wants,
* the whole step - fused decoder forward, fused rate-distortion loss, fused backward,
  the tiny parameter-side torch ops, the NCCL all-reduce of the shared-weight gradient
  and Adam - captured once in a CUDA graph and replayed (launch-bound otherwise: a
  16-block step is ~0.3 ms of FP32 work but ~800 kernel launches),
* results-neutral skipping of gradients the reference computes and then discards
  (SURVEY.md 3.3: d/d-emb in the weight loop, all weight gradients in the embedding loop).

The optimisation trajectory is the reference's: same loss, same Adam, same RNG
distributions (the RNG *stream* differs, as it does between any two runs of the reference).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import dist as D
from . import ops

STAT_NAMES = ("loss", "bce", "ms0", "ms1", "b_latent", "b_net", "n_pts")
EXPORTS = ("nvf_gather_batch",)          # include/nvf_prep_b200.h entry points bound here
_gather_bound = None
_last_opt = None


def _gather_batch(emb_all, gt_all, dist_all, idx, emb_out, gt_out, dist_out, status=None) -> None:
    """nvf_gather_batch: rows `idx` of the three device-resident tensors -> the static batch buffers, one launch.
    status: optional int32 device word; bit 0 is set by the kernel when an index is out of range."""
    import ctypes as C
    global _gather_bound
    b = ops._lib.cuda_binding()
    if _gather_bound is None:
        vp = C.c_void_p
        b.lib.nvf_gather_batch.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_int64, C.c_int32, vp, vp, vp, vp, vp]
        _gather_bound = b
    n_rows = int(gt_all.shape[0])
    for t, per_row in ((emb_all, int(emb_out[0].numel())), (gt_all, 32768), (dist_all, 32768)):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape[0] == n_rows and
                t[0].numel() == per_row):
            raise ops.NvfError("nvf_gather_batch needs contiguous float32 CUDA tensors with %d rows" % n_rows)
    p = ops._lib._ptr
    rc = b.lib.nvf_gather_batch(p(emb_all), p(gt_all), p(dist_all), p(idx), int(idx.numel()), n_rows,
                                int(emb_all[0].numel()), p(emb_out), p(gt_out), p(dist_out), p(status),
                                b._stream(gt_all.device))
    b.check(rc, "nvf_gather_batch")


def _loss_terms(net, emb, gt, dst, q, n_total, lmbda, w1, w2, focal_alpha, n_pts=None):
    """NVFPCC.py:154-196 on the fused ops.  Returns (loss, stats[7], sums[20])."""
    if n_pts is None:
        n_pts = D.allreduce_sum_(gt.sum())                       # batch-global (NVFPCC.py:154,161)
    out, cls_list, net_bits, latent_bits = net(emb, "train", q)
    bce, ms0, ms1, sums = ops.rd_distortion(out, cls_list[1], cls_list[0], gt, dst, focal_alpha, 0.85, 0.6)
    # total loss + the logged scalars in one launch (forward) / one launch (backward).  Under data parallelism the
    # ranks' weight gradients are SUMMED: the bce / ms / latent-rate terms are sums over the rank's own blocks, but
    # the network-rate term lmbda*w2*sum(net_bits)/n_total is the same on every rank, so only rank 0 back-propagates it.
    rank, _ = D.world()
    loss, stats = ops.rd_total(sums, bce, ms0, ms1, latent_bits, net_bits, n_pts, n_total, lmbda, w1, w2,
                               w2_grad=w2 if rank == 0 else 0.0)
    return loss, stats, sums


def forward_loss(net, emb, gt, dist_, q, n_total, lmbda, w1, w2, focal_alpha=0.9, n_pts=None):
    """SURVEY.md 8b `forward_loss`: Net.forward + the rate-distortion loss of train() in one call ->
    (loss, stats[7] on the device (STAT_NAMES), sums[20]); differentiable w.r.t. emb and the network."""
    return _loss_terms(net, emb, gt, dist_, q, n_total, lmbda, w1, w2, focal_alpha, n_pts=n_pts)


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam (defaults of train(), NVFPCC.py:116,124: betas (0.9, 0.999), eps 1e-8, no weight decay,
    no amsgrad) over ONE flat buffer: all parameters are re-pointed to views of `flat`, the moments are flat too,
    and step() is a single kernel (nvf_adam_step) instead of ~70 launches.  Learning-rate schedulers work as
    usual (they edit param_groups[0]['lr']); the value is mirrored to a device scalar by sync_lr() so that a
    captured CUDA graph follows the schedule.  One param group."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        params = list(params)
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdam supports a single param group")
        self.ps = [p for p in self.param_groups[0]["params"]]
        dev = self.ps[0].device
        if dev.type != "cuda":
            raise ops.NvfError("FusedAdam needs CUDA parameters; there is no CPU fallback")
        n = sum(p.numel() for p in self.ps)
        self.flat = torch.empty(n, dtype=torch.float32, device=dev)
        o = 0
        with torch.no_grad():
            for p in self.ps:
                k = p.numel()
                self.flat[o:o + k].copy_(p.detach().reshape(-1))
                p.data = self.flat[o:o + k].view(p.shape)
                o += k
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self.step_t = torch.zeros(1, dtype=torch.float32, device=dev)
        self.lr_t = torch.full((1,), float(lr), dtype=torch.float32, device=dev)
        self._lr_host = float(lr)
        self._symm = None            # peer-mapped gradient buffers (enable_peer_allreduce)
        self._symm_tried = False

    def enable_peer_allreduce(self) -> bool:
        """Data parallel with one process per GPU of ONE node (NCCL backend): allocate this rank's symmetric gradient
        buffer, exchange the CUDA IPC handles and map the peers' buffers, so that step_allreduce() is ONE kernel
        (nvf_adam_allreduce_step: all-reduce over NVLink fused with Adam) instead of an NCCL all-reduce + Adam.
        COLLECTIVE: every rank must call it.  Returns False - and the NCCL path stays - when the process group is not
        NCCL / spans several hosts / has more than 16 ranks, NVF_PEER_ALLREDUCE=0, or any rank could not map its peers
        (decided by all ranks together; the reason goes to stderr)."""
        import os, socket, sys
        import torch.distributed as tdist
        self._symm_tried = True
        if not D.is_dist() or os.environ.get("NVF_PEER_ALLREDUCE", "1") == "0":
            return False
        if tdist.get_backend() != "nccl":
            return False
        rank, ws = D.world()
        dev = self.flat.device
        b = ops._lib.cuda_binding()
        ok, own, handle, why = 1, None, b"", ""
        if ws > 16:
            ok, why = 0, "more than 16 ranks"
        else:
            try:
                with torch.cuda.device(dev):
                    own, handle = b.symm_alloc(self.flat.numel())
            except ops.NvfError as e:
                ok, why = 0, str(e)
        infos = [None] * ws
        tdist.all_gather_object(infos, (socket.gethostname(), handle if ok else b""))
        peers = []
        if ok and len({h for h, _ in infos}) != 1:
            ok, why = 0, "ranks on several hosts"
        if ok and not all(len(hd) == 64 for _, hd in infos):
            ok, why = 0, "a peer could not allocate its buffer"
        if ok:
            try:
                with torch.cuda.device(dev):
                    for r, (_, hd) in enumerate(infos):
                        peers.append(own if r == rank else b.symm_open(hd))
            except ops.NvfError as e:
                ok, why = 0, str(e)
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        tdist.all_reduce(flag, op=tdist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            for r, ptr in enumerate(peers):
                if r != rank:
                    b.symm_close(ptr)
            if own is not None:
                b.symm_free(own)
            if rank == 0:
                print("nvfpcc_b200: peer-memory all-reduce unavailable (%s); using the NCCL all-reduce" % (why or "a peer failed"),
                      file=sys.stderr)
            return False
        self._symm = dict(own=own, peers=peers, rank=rank, ctl=torch.zeros(4, dtype=torch.int32, device=dev))
        tdist.barrier()
        return True

    @torch.no_grad()
    def step_allreduce(self):
        """Sum flat_grad over the ranks and apply Adam: the fused peer-memory kernel when enabled, else ONE NCCL
        all-reduce followed by nvf_adam_step.  Single process: plain step."""
        if self._symm is None:
            D.allreduce_sum_(self.flat_grad)
            return self.step(gathered=True)
        if not torch.cuda.is_current_stream_capturing():
            self.sync_lr()
        g, sy = self.param_groups[0], self._symm
        ops._lib.cuda_binding().adam_allreduce_step(self.flat, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_t,
                                                    self.lr_t, sy["peers"], sy["rank"], sy["ctl"], g["betas"][0],
                                                    g["betas"][1], g["eps"])

    def sync_lr(self):
        """Mirror param_groups[0]['lr'] to the device scalar (call outside graph capture)."""
        lr = float(self.param_groups[0]["lr"])
        if lr != self._lr_host:
            self.lr_t.fill_(lr)
            self._lr_host = lr

    def gather_grads(self) -> torch.Tensor:
        """p.grad of every parameter -> flat_grad (one concatenation); missing grads count as zero."""
        parts = [(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in self.ps]
        torch.cat(parts, out=self.flat_grad)
        return self.flat_grad

    @torch.no_grad()
    def step(self, closure=None, gathered: bool = False):
        if not torch.cuda.is_current_stream_capturing():
            self.sync_lr()
        if not gathered:
            self.gather_grads()
        g = self.param_groups[0]
        ops._lib.cuda_binding().adam_step(self.flat, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_t,
                                          self.lr_t, g["betas"][0], g["betas"][1], g["eps"])

    def snapshot(self):
        return [t.clone() for t in (self.flat, self.exp_avg, self.exp_avg_sq, self.step_t)]

    def restore(self, snap):
        for t, s in zip((self.flat, self.exp_avg, self.exp_avg_sq, self.step_t), snap):
            t.copy_(s)


class FusedStepCall:
    """Argument block of nvf_train_step for one (net, batch size) pair: raw-parameter pointers, gradient destinations
    (slices of FusedAdam.flat_grad when an optimizer is given, else private buffers), the step's workspace and the
    device-resident noise counter.  Built once; `run()` is one C call (about 45 kernel launches, no framework op)."""

    def __init__(self, net, n: int, n_total: float, lmbda: float, w1: float, w2: float, focal_alpha: float,
                 opt: Optional["FusedAdam"], dev, want_wgrad: bool = True, want_demb: bool = False, seed: int = 0):
        import ctypes as C
        L = ops._lib
        self.b = L.cuda_binding()
        dev = torch.device(dev)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.net, self.dev, self.n = net, dev, int(n)
        rec = net.reconstructor
        ch = rec.in_channels
        if ch > 4:
            raise ops.NvfError("the fused step supports ch <= 4")
        self.desc = self.b.desc(ch, rec.channels)
        self.ws = self.b.train_step_workspace(self.desc, n, dev)
        self.rng_counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.g_emb = torch.zeros(n, ch, 2, 2, 2, device=dev) if want_demb else None
        a = L.NvfStepArgs()
        a.desc, a.n = self.desc, int(n)
        a.flags = (L.NVF_BWD_WGRAD if want_wgrad else 0) | (L.NVF_BWD_DLATENT if want_demb else 0)
        self._keep = []

        def ptr(t):
            if not t.is_cuda or (torch.device(dev).index not in (None, t.device.index)):
                raise ops.NvfError("fused step: every tensor must live on %s" % (dev,))
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise ops.NvfError("fused step: float32 contiguous tensors required")
            self._keep.append(t)
            return t.data_ptr()

        # gradient destinations: views of the optimizer's flat gradient buffer (no gather before the all-reduce / Adam)
        if want_wgrad:
            if opt is not None:
                off, o = {}, 0
                for p_ in opt.ps:
                    off[id(p_)] = o
                    o += p_.numel()
                gdst = lambda p_: opt.flat_grad[off[id(p_)]:off[id(p_)] + p_.numel()]
            else:
                self.grads = {}
                def gdst(p_):
                    g = torch.zeros(p_.numel(), device=dev)
                    self.grads[id(p_)] = g
                    return g
        raw = rec.raw_tensors()
        a.params = L.param_set(raw, lambda t: ptr(t.detach()))
        if want_wgrad:
            for i, name in enumerate(L.CONV_LAYERS):
                a.g_params.kernel[i] = ptr(gdst(raw[name + "_kernel"]))
                a.g_params.b[i] = ptr(gdst(raw[name + "_b"]))
            for field in ("igdn_beta", "igdn_gamma", "lik_sigma", "lik_mu"):
                setattr(a.g_params, field, ptr(gdst(raw[field])))
        lraw = net.latent_raw()
        for field in L.LATENT_FIELDS:
            setattr(a.latent, field, ptr(lraw[field].detach()))
        if want_wgrad:
            for field in L.LATENT_GRAD_FIELDS:
                setattr(a.g_latent, field, ptr(gdst(lraw[field])))
        if want_demb:
            a.g_emb = ptr(self.g_emb)
        a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        a.rng_counter = self.rng_counter.data_ptr()
        a.n_total, a.lmbda, a.w1, a.w2 = float(n_total), float(lmbda), float(w1), float(w2)
        a.alpha_main, a.alpha_aux, a.thh_metric = float(focal_alpha), 0.85, 0.6
        g, act = net.latent_gen.gdn_2, rec.activation
        a.latent_beta_bound, a.latent_gamma_bound, a.latent_pedestal = (float(g.beta_bound), float(g.gamma_bound),
                                                                         float(g.reparam_pedestal))
        a.igdn_beta_bound, a.igdn_gamma_bound, a.igdn_pedestal = (float(act.beta_bound), float(act.gamma_bound),
                                                                  float(act.reparam_pedestal))
        self.args = a

    def run(self, emb, gt, dist_, idx, n_rows, n_pts, stats, sums, q: int, mode: str = "train", status=None,
            noise_latent=None, noise_kernel=None):
        """emb / gt / dist_: the batch (idx None) or the resident dataset with rows idx (int64, device)."""
        a = self.args
        p = ops._lib._ptr
        a.q, a.train_mode = int(q), 1 if mode == "train" else 0
        a.emb, a.gt, a.dist = emb.data_ptr(), gt.data_ptr(), dist_.data_ptr()
        a.idx = None if idx is None else idx.data_ptr()
        a.n_rows = int(n_rows)
        a.status = None if status is None else status.data_ptr()
        a.n_pts = n_pts.data_ptr()
        a.noise_scale = float(self.net.entropy_coder.noise_scale)
        rank, _ = D.world()
        a.w2_grad = a.w2 if rank == 0 else 0.0
        a.noise_latent = None if noise_latent is None else noise_latent.data_ptr()
        a.noise_kernel = None if noise_kernel is None else noise_kernel.data_ptr()
        a.stats, a.sums = stats.data_ptr(), sums.data_ptr()
        self.b.train_step(a, self.ws, self.dev)


class WeightStep:
    """One minibatch update of the shared decoder weights (NVFPCC.py:149-223).

    step(emb_batch, gt, dist) copies the batch into static device buffers (host tensors are
    fine - pinned memory makes the copies asynchronous), replays the captured graph and returns
    the device-resident stats tensor (see STAT_NAMES) - no host synchronisation."""

    def __init__(self, net, opt: torch.optim.Optimizer, batch: int, n_total: float, lmbda: float, w1: float,
                 w2: float, focal_alpha: float = 0.9, use_graph: bool = True, device=None, fused: Optional[bool] = None,
                 seed: Optional[int] = None):
        """fused: run the step through nvf_train_step (one C call: in-kernel gather and noise, one-launch loss,
        gradients written straight into the flat buffer) instead of the autograd graph over the individual ops.
        Default: on whenever the optimizer is a FusedAdam.  Same kernels for the heavy layers, same results up to
        summation order; the noise of the q = 1 / train phases comes from the in-kernel Philox streams (seeded by
        `seed`, default torch.initial_seed()) instead of torch.rand."""
        self.net, self.opt = net, opt
        self.hp = dict(n_total=float(n_total), lmbda=float(lmbda), w1=float(w1), w2=float(w2),
                       focal_alpha=float(focal_alpha))
        dev = device if device is not None else next(net.parameters()).device
        ch = net.reconstructor.in_channels
        self.emb = torch.zeros(batch, ch, 2, 2, 2, device=dev)
        self.gt = torch.zeros(batch, 1, 32, 32, 32, device=dev)
        self.dist = torch.zeros(batch, 1, 32, 32, 32, device=dev)
        self.stats = torch.zeros(len(STAT_NAMES), device=dev)
        self.sums = torch.zeros(ops._lib.NVF_LOSS_SUMS, dtype=torch.float64, device=dev)
        # [0:batch] minibatch row indices, [batch] the batch-global point count (float32 bits in the low half): one
        # small buffer so that a precomputed schedule row (pack_schedule) reaches the step with ONE async copy
        self._hdr = torch.zeros(batch + 1, dtype=torch.int64, device=dev)
        self._idx_buf = self._hdr[:batch]
        self.n_pts = self._hdr[batch:].view(torch.float32)[:1]   # batch-global point count handed in by the caller
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)   # sticky: bit 0 = a gather index was out of range
        self.use_graph = use_graph
        self.launches_per_step = 0
        self._graphs: Dict[tuple, torch.cuda.CUDAGraph] = {}
        self.fused_opt = isinstance(opt, FusedAdam)
        self.fused = self.fused_opt and net.reconstructor.in_channels <= 4 if fused is None else bool(fused)
        if self.fused and not self.fused_opt:
            raise ValueError("WeightStep(fused=True) needs a FusedAdam optimizer (gradients go to its flat buffer)")
        self._warming = False           # graph-capture warm-up runs: no collectives (see _capture)
        if self.fused_opt and D.is_dist() and not opt._symm_tried:
            opt.enable_peer_allreduce()        # collective: every rank builds its steps in the same order
        self._call = None
        self._idx_src = None           # (emb_all, gt_all, dist_all) of the pending step_indexed call
        self._seed = int(torch.initial_seed() if seed is None else seed)
        if use_graph and not self.fused_opt:
            for g in opt.param_groups:
                if not g.get("capturable", False):
                    raise ValueError("WeightStep(use_graph=True) needs FusedAdam or an optimizer built with capturable=True")

    def _body(self, q: int, ext_npts: bool = False, indexed: bool = False):
        """ext_npts: the batch-global point count was put into self.n_pts by the caller (known from the per-block
        counts and the deterministic batch schedule: no reduction, no collective); otherwise it is gt.sum(),
        all-reduced over the ranks (NVFPCC.py:154).  indexed (fused path only): the blocks read rows self._idx_buf
        of the resident dataset self._idx_src directly - no gather."""
        if self.fused:
            return self._body_fused(q, ext_npts, indexed)
        self.opt.zero_grad(set_to_none=True)
        loss, stats, sums = _loss_terms(self.net, self.emb, self.gt, self.dist, q,
                                        n_pts=self.n_pts if ext_npts else (self.gt.sum() if self._warming else None),
                                        **self.hp)
        loss.backward()
        self._reduce_and_step()
        self.stats.copy_(stats)
        self.sums.copy_(sums)

    def _body_fused(self, q: int, ext_npts: bool, indexed: bool = False):
        if self._call is None:
            hp = self.hp
            self._call = FusedStepCall(self.net, self.emb.shape[0], hp["n_total"], hp["lmbda"], hp["w1"], hp["w2"],
                                       hp["focal_alpha"], self.opt, self.emb.device, seed=self._seed)
        if not ext_npts:
            n = self.gt.sum()
            self.n_pts.copy_((n if self._warming else D.allreduce_sum_(n)).reshape(1))   # batch-global (NVFPCC.py:154,161)
        if indexed:
            emb_all, gt_all, dist_all = self._idx_src
            self._call.run(emb_all, gt_all, dist_all, self._idx_buf, gt_all.shape[0], self.n_pts, self.stats, self.sums,
                           q, status=self.status)
        else:
            self._call.run(self.emb, self.gt, self.dist, None, 0, self.n_pts, self.stats, self.sums, q)
        if self._warming:
            self.opt.step(gathered=True)
        else:
            self.opt.step_allreduce()         # all-reduce of the flat gradient + Adam (one fused kernel over NVLink)

    def _reduce_and_step(self):
        if self.fused_opt:
            self.opt.gather_grads()
            if self._warming:
                self.opt.step(gathered=True)
            else:
                self.opt.step_allreduce()                        # ONE exchange of the flat shared-weight gradient
        else:
            if not self._warming:
                D.allreduce_grads_(self.net.parameters())
            self.opt.step()

    def empty_step(self) -> torch.Tensor:
        """A step of a rank whose share of the minibatch is empty (short last batch of an epoch): it contributes a
        zero gradient to the all-reduce and applies the same Adam update as the other ranks."""
        if self.fused_opt:
            for p in self.opt.ps:
                p.grad = None
        else:
            for p in self.net.parameters():
                p.grad = torch.zeros_like(p)
        self._reduce_and_step()
        self.stats.zero_()
        return self.stats

    def _capture(self, key, q: int, ext_npts: bool = False, indexed: bool = False):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            state = self._snapshot()
            # warm-up (allocator, lazy init, kernel attributes) WITHOUT the collectives: a rank captures a graph the
            # first time it meets a (batch size, q) pair, which need not be the step at which its peers do (uneven
            # shards, short last batches) - every rank must still issue exactly one gradient exchange per global
            # step.  The state is restored afterwards, so a local Adam update is as good as the real one here.
            self._warming = True
            try:
                for _ in range(3):
                    self._body(q, ext_npts, indexed)
            finally:
                self._warming = False
            self._restore(state)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        self.opt.zero_grad(set_to_none=True)
        b = ops._lib.cuda_binding()
        n0 = b.launch_count()
        with torch.cuda.graph(g):
            self._body(q, ext_npts, indexed)
        self.launches_per_step = b.launch_count() - n0           # hand-written kernels inside one replay
        self._restore(state)                                     # capture does not run, but keep state exact
        self._graphs[key] = g

    def _snapshot(self):
        import copy
        if self.fused_opt:
            extra = [self._call.rng_counter.clone()] if self._call is not None else []
            return self.opt.snapshot() + extra
        return [p.detach().clone() for p in self.net.parameters()], copy.deepcopy(self.opt.state_dict())

    def _restore(self, state):
        if self.fused_opt:
            with torch.no_grad():
                self.opt.restore(state[:4])
                if len(state) > 4 and self._call is not None:
                    self._call.rng_counter.copy_(state[4])
            return
        params, opt_sd = state
        with torch.no_grad():
            for p, s in zip(self.net.parameters(), params):
                p.copy_(s)
        # restore optimizer tensors IN PLACE (the captured graph holds their addresses)
        cur = self.opt.state_dict()
        for k, st in opt_sd["state"].items():
            for name, v in st.items():
                if torch.is_tensor(v) and k in cur["state"]:
                    cur["state"][k][name].copy_(v)
        if not opt_sd["state"]:
            for st in self.opt.state.values():
                for name, v in st.items():
                    if torch.is_tensor(v):
                        v.zero_()

    def pack_schedule(self, idx: torch.Tensor, n_pts: torch.Tensor) -> torch.Tensor:
        """One schedule row for step_indexed(packed=...): the minibatch indices and the batch-global point count in
        the layout of the step's header buffer (built once per run by trainer.fit / bench.py)."""
        row = torch.zeros(self._hdr.shape[0], dtype=torch.int64, device=self._hdr.device)
        row[:-1] = idx.to(row.device)
        row[-1:].view(torch.float32)[0] = n_pts.reshape(()).to(row.device, torch.float32)
        return row

    def step_indexed(self, emb_all: torch.Tensor, gt_all: torch.Tensor, dist_all: torch.Tensor, idx: torch.Tensor,
                     q: int = 1, n_pts: Optional[torch.Tensor] = None, packed: Optional[torch.Tensor] = None) -> torch.Tensor:
        """step() for device-resident float32 datasets.  Fused path: the step's kernels read rows `idx` (int64,
        device) of the three tensors in place - nothing is gathered; `packed` (pack_schedule(idx, n_pts)) delivers
        indices and n_pts with one 136-byte copy.  Autograd path: the rows are gathered into the static buffers by
        ONE launch (nvf_gather_batch; advanced indexing + copy_ is six launches).  n_pts: see step()."""
        n_rows = int(gt_all.shape[0])
        ok = all(t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape[0] == n_rows
                 for t in (emb_all, gt_all, dist_all))
        ok = (ok and gt_all[0].numel() == 32768 and dist_all[0].numel() == 32768 and
              emb_all[0].numel() == self.emb[0].numel() and idx.dtype == torch.int64 and idx.is_cuda and
              idx.numel() == self.emb.shape[0] and idx.device == gt_all.device == self.emb.device)
        if not ok:
            idx_d = idx.to(emb_all.device)
            return self.step(emb_all.detach()[idx_d], gt_all[idx.to(gt_all.device)], dist_all[idx.to(dist_all.device)],
                             q, n_pts=n_pts)
        if self.fused:
            self._idx_src = (emb_all.detach(), gt_all, dist_all)
            if packed is not None:
                self._hdr.copy_(packed, non_blocking=True)
                return self._run(q, None, indexed=True, ext=True)
            self._idx_buf.copy_(idx, non_blocking=True)
            if n_pts is None:          # batch-global count from the rows themselves (one reduction + all-reduce)
                n_pts = D.allreduce_sum_(gt_all[idx].sum())
            return self._run(q, n_pts, indexed=True)
        _gather_batch(emb_all.detach(), gt_all, dist_all, idx.contiguous(), self.emb, self.gt, self.dist, self.status)
        return self._run(q, n_pts)

    def step(self, emb_batch: torch.Tensor, gt: torch.Tensor, dist_: torch.Tensor, q: int = 1,
             n_pts: Optional[torch.Tensor] = None) -> torch.Tensor:
        """n_pts: optional 1-element tensor, the number of occupied voxels of the GLOBAL minibatch (NVFPCC.py:154);
        when given, the step neither reduces gt nor all-reduces the scalar (the caller knows it from the per-block
        counts of its dataset and the deterministic batch schedule, as trainer.fit does)."""
        self.emb.copy_(emb_batch.detach(), non_blocking=True)
        self.gt.copy_(gt, non_blocking=True)
        self.dist.copy_(dist_, non_blocking=True)
        return self._run(q, n_pts)

    def _run(self, q: int, n_pts: Optional[torch.Tensor] = None, indexed: bool = False, ext: bool = False) -> torch.Tensor:
        if n_pts is not None:
            ext = True
            self.n_pts.copy_(n_pts.reshape(1), non_blocking=True)
        if not self.use_graph:
            self._body(q, ext, indexed)
            return self.stats
        if self.fused_opt:
            self.opt.sync_lr()
        # a captured step holds the addresses of what it reads: the resident dataset is part of the key
        key = (q, ext, tuple(t.data_ptr() for t in self._idx_src)) if indexed else (q, ext)
        if key not in self._graphs:
            self._capture(key, q, ext, indexed)
        self._graphs[key].replay()
        return self.stats

    def check_status(self) -> None:
        """Host read of the sticky status word (one synchronisation; call it when results are read anyway)."""
        if int(self.status.item()) & 1:
            raise ops.NvfError("nvf_gather_batch: a minibatch index was outside the dataset")


class HostBatchFeeder:
    """Host -> device input pipeline for the weight loop (the reference's DataLoader + `.to(device)`,
    NVFPCC.py:109-111,152-153, and its per-step `.item()` read, :190-221), double buffered:

    * `submit(idx)` gathers the batch's gt / dist rows from the host dataset into one of two PINNED staging
      buffers and enqueues their H2D copies on a dedicated copy stream (no allocation, no host sync);
    * `take()` makes the compute stream wait for the oldest submitted batch and returns its device tensors;
    * `read_stats(stats)` enqueues an asynchronous D2H copy of a step's stats into pinned memory and returns the
      stats of the PREVIOUS step (already landed), so the host reads every step's result without draining the GPU.

    With this, the copies and the CPU-side gather of step i+1 overlap the kernels of step i."""

    def __init__(self, gt_host: torch.Tensor, dist_host: torch.Tensor, batch: int, device=None):
        dev = torch.device(device if device is not None else "cuda")
        self.gt_host, self.dist_host = gt_host, dist_host
        shape = (batch,) + tuple(gt_host.shape[1:])
        self.pin = [(torch.empty(shape, dtype=gt_host.dtype).pin_memory(), torch.empty(shape, dtype=dist_host.dtype).pin_memory())
                    for _ in range(2)]
        # the two device slots are the halves of ONE [2 * batch] tensor per input, so that the fused step can read a
        # slot in place as rows of a resident "dataset" (WeightStep.step_indexed with slot_rows(slot)): no copy of the
        # batch into the step's static buffers
        self.batch = int(batch)
        self.gt_all = torch.empty((2 * batch,) + tuple(gt_host.shape[1:]), dtype=torch.float32, device=dev)
        self.dist_all = torch.empty((2 * batch,) + tuple(gt_host.shape[1:]), dtype=torch.float32, device=dev)
        self.dev = [(self.gt_all[s * batch:(s + 1) * batch], self.dist_all[s * batch:(s + 1) * batch]) for s in range(2)]
        self._rows = [torch.arange(s * batch, (s + 1) * batch, dtype=torch.int64, device=dev) for s in range(2)]
        self.emb_all = None
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.h2d_done = [torch.cuda.Event() for _ in range(2)]
        self._head = self._tail = 0
        self.stats_pin = [torch.zeros(len(STAT_NAMES)).pin_memory() for _ in range(2)]
        self.stats_ev = [None, None]
        self._stat_i = 0
        self.bytes_per_batch = sum(t.numel() * t.element_size() for t in self.pin[0])

    def submit(self, idx: torch.Tensor) -> None:
        s = self._head & 1
        if self._head >= 2:
            self.h2d_done[s].synchronize()           # the pinned buffer's previous H2D has finished
        torch.index_select(self.gt_host, 0, idx, out=self.pin[s][0])
        torch.index_select(self.dist_host, 0, idx, out=self.pin[s][1])
        with torch.cuda.stream(self.copy_stream):
            if self._head >= 2:
                self.copy_stream.wait_event(self.consumed[s])   # the device buffer's previous consumer is done
            self.dev[s][0].copy_(self.pin[s][0], non_blocking=True)
            self.dev[s][1].copy_(self.pin[s][1], non_blocking=True)
            self.h2d_done[s].record(self.copy_stream)
            self.ready[s].record(self.copy_stream)
        self._head += 1

    def take(self):
        s = self._tail & 1
        torch.cuda.current_stream().wait_event(self.ready[s])
        self._tail += 1
        return self.dev[s], s

    def slot_rows(self, slot: int) -> torch.Tensor:
        """Row indices (int64, device) of `slot` inside gt_all / dist_all / emb_stage()."""
        return self._rows[slot]

    def emb_stage(self, emb_batch: torch.Tensor, slot: int) -> torch.Tensor:
        """Copy the batch's embedding rows (device tensor, 96 bytes per block) next to the slot's gt / dist rows and
        return the [2 * batch, ...] staging tensor, so that one index vector addresses all three inputs."""
        if self.emb_all is None:
            self.emb_all = torch.zeros((2 * self.batch,) + tuple(emb_batch.shape[1:]), dtype=torch.float32,
                                       device=self.gt_all.device)
        self.emb_all[slot * self.batch:(slot + 1) * self.batch].copy_(emb_batch.detach(), non_blocking=True)
        return self.emb_all

    def release(self, slot: int) -> None:
        """Call after the consumer of `slot` has been enqueued on the compute stream."""
        self.consumed[slot].record(torch.cuda.current_stream())

    def read_stats(self, stats: torch.Tensor) -> Optional[torch.Tensor]:
        i = self._stat_i & 1
        self.stats_pin[i].copy_(stats, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self.stats_ev[i] = ev
        self._stat_i += 1
        prev = self.stats_ev[i ^ 1]
        if prev is None:
            return None
        prev.synchronize()
        return self.stats_pin[i ^ 1]

    def drain(self) -> torch.Tensor:
        """Stats of the most recent step (blocks until it has finished)."""
        i = (self._stat_i - 1) & 1
        self.stats_ev[i].synchronize()
        return self.stats_pin[i]


class EmbeddingStep:
    """The once-per-epoch update of all embeddings (NVFPCC.py:225-251): one full-batch forward +
    backward w.r.t. the embeddings only (the weight gradients of this pass are discarded by the
    reference, so they are not computed), rank-local: no collective (SURVEY.md 8e)."""

    def __init__(self, net, emb: torch.Tensor, opt_emb: torch.optim.Optimizer, n_total: float, lmbda: float,
                 w1: float, w2: float, focal_alpha: float = 0.9):
        self.net, self.emb, self.opt = net, emb, opt_emb
        self.hp = dict(n_total=float(n_total), lmbda=float(lmbda), w1=float(w1), w2=float(w2),
                       focal_alpha=float(focal_alpha))

    def step(self, gt: torch.Tensor, dist_: torch.Tensor, q: int, n_pts: Optional[torch.Tensor] = None):
        self.opt.zero_grad(set_to_none=True)
        req = [p.requires_grad for p in self.net.parameters()]
        for p in self.net.parameters():
            p.requires_grad_(False)
        try:
            if n_pts is None:
                n_pts = torch.as_tensor(self.hp["n_total"], device=gt.device)   # NVFPCC.py:230,319
            loss, stats, _ = _loss_terms(self.net, self.emb, gt, dist_, q, n_pts=n_pts, **self.hp)
            loss.backward()
        finally:
            for p, r in zip(self.net.parameters(), req):
                p.requires_grad_(r)
        self.opt.step()
        return stats


def dataset_index(i: int, n_leaf: int, shuffle: bool = True) -> int:
    """LoadedVoxelDataset.__getitem__ (utils/dataloader.py:163-167): the 'shuffle' of the reference's
    dataset is the fixed stride permutation (i * 2113) % N_leaf."""
    return (i * 2113) % n_leaf if shuffle else i


def epoch_schedule(n_leaf_all: int, rank: int, world_size: int, batch_per_rank: int, shuffle: bool = True):
    """Minibatch schedule of one epoch of the weight loop for `rank`: a list (one entry per step) of lists of
    indices into the rank's OWN contiguous leaf range (dist.block_range).  Single process: exactly the batches of
    DataLoader(dataset, batch_size, shuffle=False, drop_last=False) over LoadedVoxelDataset (NVFPCC.py:109-111,
    utils/dataloader.py:163-167) - full batches, then one SHORT batch.  Every rank runs the step count of the
    longest range; a rank whose range is exhausted gets empty batches at the end."""
    lo, hi = D.block_range(n_leaf_all, rank, world_size)
    n_leaf, B = hi - lo, int(batch_per_rank)
    steps = (D.block_range(n_leaf_all, 0, world_size)[1] + B - 1) // B       # rank 0 holds the longest range
    order = [dataset_index(i, n_leaf, shuffle) for i in range(n_leaf)]
    return [order[s * B:min(n_leaf, (s + 1) * B)] for s in range(steps)]


def fit(net, gt: torch.Tensor, dist_: torch.Tensor, *, epochs: int, batchsize: int, lr: float, lmbda: float,
        w1: float = 1.0, w2: float = 1.0, wemb: float = 5.0, phase_change: int = 100, focal_alpha: float = 0.9,
        emb: Optional[torch.Tensor] = None, n_total: Optional[float] = None, start_epoch: int = 0,
        milestones=(300, 400, 450), checkpoint_dir: Optional[str] = None, save_every: int = 10,
        dataset_shuffle: bool = True, use_graph: bool = True, log=None):
    """The epoch loop of train() (NVFPCC.py:103-296) on the sync-free steps above.

    gt / dist_: the whole dataset, [N_leaf,1,32,32,32] (uint8 / float, host or device) - kept resident
    in HBM (vox10: 1247 x 256 KB = 0.33 GB; SURVEY.md 8f-2), so the weight loop has no H2D traffic.
    Per epoch: the weight loop over all leaves at `batchsize` (drop_last=False: the last batch of an epoch is
    short, exactly as the reference's DataLoader emits it; it runs through its own captured graph), then ONE
    full-batch embedding update, then both schedulers step on the WEIGHT optimizer (NVFPCC.py:126:
    sch_emb wraps `opt`, so the weight LR decays by 0.01 per milestone and the embedding LR never decays).
    Under torch.distributed each rank owns a contiguous range of leaves (embedding rows, gt/dist shards);
    its minibatches come from that range and the shared-weight gradient is all-reduced once per step.
    Checkpoints are the reference's files: '%04d.ckpt' (state_dict) and '%04d_emb.ckpt' (the embedding tensor).
    Returns (emb, history) where history[e] holds the epoch means of STAT_NAMES (one D2H read per epoch)."""
    import os
    import warnings

    dev = next(net.parameters()).device
    if dev.type != "cuda":
        raise ops.NvfError("trainer.fit needs the network on a CUDA device; there is no CPU fallback")
    rank, ws = D.world()
    n_leaf_all = int(gt.shape[0])
    lo, hi = D.block_range(n_leaf_all, rank, ws)
    gt_d = gt[lo:hi].to(dev, torch.float32)
    dist_d = dist_[lo:hi].to(dev, torch.float32)
    n_leaf = hi - lo
    if n_total is None:
        n_total = float(D.allreduce_sum_(gt_d.sum().double()).item())              # train_data.N (utils/dataloader.py:159)
    ch = net.reconstructor.in_channels
    if emb is None:
        emb = torch.ones((n_leaf_all, ch, 2, 2, 2), dtype=torch.float32)            # NVFPCC.py:120-122
    emb_local = emb[lo:hi].detach().to(dev, torch.float32).clone().requires_grad_(True)
    opt = FusedAdam(net.parameters(), lr=lr)
    global _last_opt
    _last_opt = opt                    # introspection for the multi-GPU check (peer all-reduce on / off)
    opt_emb = torch.optim.Adam([emb_local], lr=lr * wemb)
    sch = torch.optim.lr_scheduler.MultiStepLR(opt, list(milestones), 0.1)
    sch_emb = torch.optim.lr_scheduler.MultiStepLR(opt, list(milestones), 0.1)      # sic: wraps opt (NVFPCC.py:126)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        for _ in range(start_epoch):
            sch_emb.step()
            sch.step()
    if batchsize % ws != 0:
        raise ValueError("batchsize must be a multiple of the number of ranks")
    B = batchsize // ws
    estep = EmbeddingStep(net, emb_local, opt_emb, n_total, lmbda, w1, w2, focal_alpha)
    # minibatch schedule of one epoch, built once.  DataLoader(drop_last=False) (NVFPCC.py:109-111): the last batch
    # of an epoch is SHORT, not padded - a second step object (own static buffers + graph) handles its size.  Under
    # torch.distributed every rank runs the step count of the longest range; a rank whose range is exhausted
    # contributes a zero gradient (WeightStep.empty_step).
    batches = [torch.tensor(b, dtype=torch.int64, device=dev)
               for b in epoch_schedule(n_leaf_all, rank, ws, B, dataset_shuffle)]
    steps = len(batches)
    wsteps: Dict[int, WeightStep] = {}
    for nb in sorted({int(b.numel()) for b in batches} | {B}, reverse=True):
        if nb > 0:
            wsteps[nb] = WeightStep(net, opt, nb, n_total, lmbda, w1, w2, focal_alpha, use_graph=use_graph, device=dev)
    wstep = wsteps[B]
    # batch-global n_pts of every step (NVFPCC.py:154) from the per-block point counts: one all-reduce of a
    # `steps`-long vector at set-up instead of a reduction + a scalar all-reduce inside every step
    cnt = gt_d.reshape(n_leaf, -1).sum(1)
    npts_steps = torch.stack([cnt[b].sum() if b.numel() else cnt.new_zeros(()) for b in batches])
    npts_steps = D.allreduce_sum_(npts_steps).reshape(steps, 1)
    packed = [wsteps[int(b.numel())].pack_schedule(b, npts_steps[s]) if b.numel() else None for s, b in enumerate(batches)]
    history = []
    acc = torch.zeros(len(STAT_NAMES), device=dev)
    q = 1 if start_epoch < phase_change else 2
    for epoch in range(start_epoch, epochs):
        if epoch == phase_change:
            q = 2
        acc.zero_()
        for s in range(steps):
            nb = int(batches[s].numel())
            if nb == 0:
                wstep.empty_step()
                continue
            acc += wsteps[nb].step_indexed(emb_local, gt_d, dist_d, batches[s], q=q, n_pts=npts_steps[s],
                                           packed=packed[s])
        est = estep.step(gt_d, dist_d, q)
        with warnings.catch_warnings():          # the graph replays opt.step(); the schedulers cannot see it
            warnings.simplefilter("ignore", UserWarning)
            sch_emb.step()
            sch.step()
        for w_ in wsteps.values():
            w_.check_status()
        rec = dict(zip(STAT_NAMES, (acc / steps).tolist()))                         # the epoch's only host read
        rec.update(epoch=epoch, q=q, emb_loss=float(est[0]), lr=float(opt.param_groups[0]["lr"]))
        history.append(rec)
        if log is not None:
            log(rec)
        if checkpoint_dir is not None and epoch % save_every == 0:
            full = _gather_emb(emb_local, n_leaf_all, lo, hi, ws)
            if rank == 0:
                os.makedirs(checkpoint_dir, exist_ok=True)
                torch.save(net.state_dict(), os.path.join(checkpoint_dir, '%04d.ckpt' % epoch))
                torch.save(full, os.path.join(checkpoint_dir, '%04d_emb.ckpt' % epoch))
    return _gather_emb(emb_local, n_leaf_all, lo, hi, ws), history


def _gather_emb(emb_local: torch.Tensor, n_all: int, lo: int, hi: int, ws: int) -> torch.Tensor:
    """All embedding rows on every rank (N x ch x 8 floats: the only time embeddings cross ranks)."""
    e = emb_local.detach()
    if ws == 1:
        return e.clone().requires_grad_(True)
    full = torch.zeros((n_all,) + tuple(e.shape[1:]), dtype=e.dtype, device=e.device)
    full[lo:hi] = e
    D.allreduce_sum_(full)
    return full.requires_grad_(True)
