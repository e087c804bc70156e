"""ctypes binding of the C ABI in include/nvf_b200.h.

The product library is `nvfpcc_b200/libnvf_b200.so` (built in-tree by
`__graft_entry__.build()` / `nvfpcc_b200/build.py` with nvcc for sm_100a).
There is no CPU fallback: `cuda_binding()` raises if the library is missing or
cannot be loaded, and every op in `nvfpcc_b200.ops` requires CUDA tensors.

`Binding` itself is device-agnostic plumbing (it passes `tensor.data_ptr()`), so
the test suite can also point it at the test-only emulator build under
tests/emu/ to check kernel logic on CPU tensors; the package never does that.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Callable, Dict, Optional, Sequence

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libnvf_b200.so"

WEIGHT_FIELDS = (
    "up0_w", "up0_b", "igdn_beta", "igdn_gamma", "conv0_w", "conv0_b", "up1_w", "up1_b", "conv1_w", "conv1_b",
    "up2_w", "up2_b", "conv2_w", "conv2_b", "cls2_w", "cls2_b", "cls1_w", "cls1_b", "cls0_w", "cls0_b",
)
NVF_MODE_DECODE, NVF_MODE_TRAIN = 0, 1
NVF_BWD_WGRAD, NVF_BWD_DLATENT, NVF_BWD_DLOGIT = 1, 2, 4
NVF_LOSS_SUMS = 20
NVF_LOSS_CHUNKS = 16   # CTAs per block of nvf_loss_seeds (workspace: 8 * NVF_LOSS_SUMS * (NVF_LOSS_CHUNKS * n + 1) bytes)
EXPORTS = (
    "nvf_abi_version", "nvf_strerror", "nvf_last_cuda_error", "nvf_launch_count", "nvf_has_fused_decode", "nvf_workspace_bytes",
    "nvf_decode", "nvf_emit_points", "nvf_train_forward", "nvf_loss_seeds", "nvf_train_backward",
    "nvf_ffma_microbench", "nvf_param_prep", "nvf_param_prep_backward",
    "nvf_latent_forward", "nvf_latent_backward", "nvf_rd_total", "nvf_rd_total_backward", "nvf_adam_step",
    "nvf_train_step_workspace_bytes", "nvf_train_step", "nvf_rng_uniform",
    "nvf_symm_bytes", "nvf_symm_alloc", "nvf_symm_open", "nvf_symm_close", "nvf_symm_free", "nvf_adam_allreduce_step",
)
LATENT_FIELDS = ("kernel", "kernel_init", "b", "b_init", "gdn_beta", "gdn_gamma", "sigma", "mu")   # NvfLatentParams
LATENT_GRAD_FIELDS = ("kernel", "b", "gdn_beta", "gdn_gamma", "sigma", "mu")                         # NvfLatentGrads
NVF_LATENT_WS_BYTES = 128 * 1024
# The decoder's nine convolutions in NvfParamSet order: ABI key -> CompDecoder attribute.  The first NVF_NUM_QUANT
# are the quantised ones.
CONV_MODULES = {"up0": "up0", "conv0": "conv0", "up1": "up1", "conv1": "conv1", "up2": "up2", "conv2": "conv2",
                "cls2": "conv2_cls", "cls1": "conv1_cls", "cls0": "conv0_cls"}
CONV_LAYERS = tuple(CONV_MODULES)
NVF_NUM_CONV, NVF_NUM_QUANT, NVF_PARAM_WS_BYTES = 9, 7, 64 * 1024


class NvfDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("ch", "c0", "c1", "c2", "c3")]


class NvfWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in WEIGHT_FIELDS]


class NvfWeightGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in WEIGHT_FIELDS]


class NvfParamSet(C.Structure):
    _fields_ = [("kernel", C.c_void_p * 9), ("kernel_init", C.c_void_p * 9), ("b", C.c_void_p * 9),
                ("b_init", C.c_void_p * 9), ("igdn_beta", C.c_void_p), ("igdn_gamma", C.c_void_p),
                ("lik_sigma", C.c_void_p), ("lik_mu", C.c_void_p)]


class NvfParamGrads(C.Structure):
    _fields_ = [("kernel", C.c_void_p * 9), ("b", C.c_void_p * 9), ("igdn_beta", C.c_void_p),
                ("igdn_gamma", C.c_void_p), ("lik_sigma", C.c_void_p), ("lik_mu", C.c_void_p)]


class NvfLatentParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in LATENT_FIELDS]


class NvfLatentGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in LATENT_GRAD_FIELDS]


class NvfStepArgs(C.Structure):
    """include/nvf_b200.h NvfStepArgs (field order is the ABI)."""
    _fields_ = ([("desc", NvfDesc)] + [(n, C.c_int32) for n in ("n", "q", "flags", "train_mode")] +
                [("emb", C.c_void_p), ("gt", C.c_void_p), ("dist", C.c_void_p), ("idx", C.c_void_p),
                 ("n_rows", C.c_int64), ("status", C.c_void_p),
                 ("latent", NvfLatentParams), ("params", NvfParamSet), ("g_latent", NvfLatentGrads),
                 ("g_params", NvfParamGrads), ("g_emb", C.c_void_p), ("noise_latent", C.c_void_p),
                 ("noise_kernel", C.c_void_p), ("seed", C.c_uint64), ("rng_counter", C.c_void_p), ("n_pts", C.c_void_p)] +
                [(n, C.c_float) for n in ("n_total", "lmbda", "w1", "w2", "w2_grad", "alpha_main", "alpha_aux", "thh_metric",
                                          "noise_scale", "latent_beta_bound", "latent_gamma_bound", "latent_pedestal",
                                          "igdn_beta_bound", "igdn_gamma_bound", "igdn_pedestal")] +
                [("stats", C.c_void_p), ("sums", C.c_void_p)])


class NvfError(RuntimeError):
    pass


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def param_set(raw: Dict[str, torch.Tensor], ptr: Callable[[torch.Tensor], int]) -> NvfParamSet:
    """NvfParamSet over the raw tensors of ops.RAW_FIELDS; ptr(tensor) -> the device address to pass."""
    ps = NvfParamSet()
    for i, key in enumerate(CONV_LAYERS):
        for field in ("kernel", "kernel_init", "b", "b_init"):
            getattr(ps, field)[i] = ptr(raw["%s_%s" % (key, field)])
    for field in ("igdn_beta", "igdn_gamma", "lik_sigma", "lik_mu"):
        setattr(ps, field, ptr(raw[field]))
    return ps


class Binding:
    """Thin, typed wrapper over one loaded shared library exporting the NVF C ABI."""

    def __init__(self, path: str):
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        for name in EXPORTS:
            if not hasattr(L, name):
                raise NvfError("%s does not export %s" % (path, name))
        L.nvf_abi_version.restype = C.c_int
        L.nvf_strerror.restype = C.c_char_p
        L.nvf_strerror.argtypes = [C.c_int]
        L.nvf_last_cuda_error.restype = C.c_int
        L.nvf_launch_count.restype = C.c_longlong
        L.nvf_has_fused_decode.argtypes = [C.POINTER(NvfDesc)]
        L.nvf_workspace_bytes.argtypes = [C.POINTER(NvfDesc), C.c_int64, C.c_int, C.POINTER(C.c_size_t)]
        vp = C.c_void_p
        L.nvf_decode.argtypes = [C.POINTER(NvfDesc), C.POINTER(NvfWeights), vp, vp, C.c_int64, C.c_float, vp, vp, vp,
                                 vp, C.c_int64, vp, vp, C.c_size_t, vp]
        L.nvf_emit_points.argtypes = [vp, vp, vp, C.c_int64, vp, C.c_int64, vp, vp, C.c_size_t, vp]
        L.nvf_train_forward.argtypes = [C.POINTER(NvfDesc), C.POINTER(NvfWeights), vp, C.c_int64, vp, vp, vp, vp,
                                        C.c_size_t, vp]
        L.nvf_loss_seeds.argtypes = [vp, vp, vp, vp, vp, C.c_int64, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp,
                                     vp, C.c_size_t, vp]
        L.nvf_train_backward.argtypes = [C.POINTER(NvfDesc), C.POINTER(NvfWeights), vp, C.c_int64, vp, vp, vp, C.c_int,
                                         C.POINTER(NvfWeightGrads), vp, vp, C.c_size_t, vp]
        L.nvf_ffma_microbench.argtypes = [C.c_int, C.c_int64, vp, C.POINTER(C.c_double), vp]
        L.nvf_param_prep.argtypes = [C.POINTER(NvfDesc), C.POINTER(NvfParamSet), C.c_int, vp, C.c_float, C.c_float,
                                     C.c_float, C.POINTER(NvfWeightGrads), vp, vp, C.c_size_t, vp]
        L.nvf_param_prep_backward.argtypes = [C.POINTER(NvfDesc), C.POINTER(NvfParamSet), C.c_float, C.c_float,
                                              C.POINTER(NvfWeights), vp, C.POINTER(NvfParamGrads), vp, C.c_size_t, vp]
        f32 = C.c_float
        L.nvf_latent_forward.argtypes = [C.c_int, C.POINTER(NvfLatentParams), vp, vp, f32, C.c_int, C.c_int64, f32, f32,
                                         f32, vp, vp, vp, C.c_size_t, vp]
        L.nvf_latent_backward.argtypes = [C.c_int, C.POINTER(NvfLatentParams), vp, vp, f32, C.c_int, C.c_int64, f32,
                                          f32, f32, vp, vp, C.POINTER(NvfLatentGrads), vp, vp, C.c_size_t, vp]
        L.nvf_rd_total.argtypes = [vp, vp, vp, vp, f32, f32, f32, f32, vp, vp, vp]
        L.nvf_rd_total_backward.argtypes = [vp, vp, f32, f32, f32, f32, vp, vp, vp, vp]
        L.nvf_adam_step.argtypes = [vp, vp, vp, vp, C.c_int64, vp, vp, f32, f32, f32, vp]
        L.nvf_symm_bytes.argtypes, L.nvf_symm_bytes.restype = [C.c_int64], C.c_size_t
        L.nvf_symm_alloc.argtypes = [C.c_size_t, C.POINTER(vp), vp]
        L.nvf_symm_open.argtypes = [vp, C.POINTER(vp)]
        L.nvf_symm_close.argtypes = [vp]
        L.nvf_symm_free.argtypes = [vp]
        L.nvf_adam_allreduce_step.argtypes = [vp, vp, vp, vp, C.c_int64, vp, vp, f32, f32, f32, C.POINTER(vp), C.c_int,
                                              C.c_int, vp, vp]
        L.nvf_train_step_workspace_bytes.argtypes = [C.POINTER(NvfDesc), C.c_int64, C.POINTER(C.c_size_t)]
        L.nvf_train_step.argtypes = [C.POINTER(NvfStepArgs), vp, C.c_size_t, vp]
        L.nvf_rng_uniform.argtypes = [C.c_uint64, C.c_uint64, C.c_int, C.c_int64, C.c_int64, vp, vp]
        if L.nvf_abi_version() != 1:
            raise NvfError("ABI version mismatch in %s" % path)
        self._ws: Dict[tuple, torch.Tensor] = {}

    # ------------------------------------------------------------------ utils
    def check(self, rc: int, what: str) -> None:
        if rc != 0:
            msg = self.lib.nvf_strerror(rc).decode()
            raise NvfError("%s failed: %s (rc=%d, cudaError=%d)" % (what, msg, rc, self.lib.nvf_last_cuda_error()))

    @staticmethod
    def desc(ch: int, channels: Sequence[int]) -> NvfDesc:
        c0, c1, c2, c3 = (int(c) for c in channels)
        return NvfDesc(int(ch), c0, c1, c2, c3)

    @staticmethod
    def _stream(dev: torch.device):
        if dev.type == "cuda":
            return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        return None

    def workspace_bytes(self, desc: NvfDesc, n: int, mode: int) -> int:
        out = C.c_size_t(0)
        self.check(self.lib.nvf_workspace_bytes(C.byref(desc), n, mode, C.byref(out)), "nvf_workspace_bytes")
        return int(out.value)

    def cached_workspace(self, nbytes: int, dev: torch.device, tag: str) -> torch.Tensor:
        """Grow-only scratch buffer per (device, tag); contents need not survive between calls.  Only for calls
        whose size is fixed (parameter-side kernels) or that are never captured in a CUDA graph (decode): a
        superseded buffer is dropped, so its address must not outlive the call."""
        key = (str(dev), tag)
        buf = self._ws.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
            self._ws[key] = buf
        return buf

    @staticmethod
    def pack_weights(weights: Dict[str, torch.Tensor], dev: torch.device, need_aux: bool):
        keep = []
        st = NvfWeights()
        for name in WEIGHT_FIELDS:
            t = weights.get(name)
            if t is None:
                if need_aux or not name.startswith(("cls1", "cls0")):
                    raise NvfError("missing effective tensor " + name)
                setattr(st, name, None)
                continue
            if t.device != dev or t.dtype != torch.float32:
                raise NvfError("%s must be float32 on %s" % (name, dev))
            t = t.detach().contiguous()
            keep.append(t)
            setattr(st, name, t.data_ptr())
        return st, keep

    # ------------------------------------------------------------------ calls
    def decode(self, desc: NvfDesc, weights: Dict[str, torch.Tensor], latent: torch.Tensor,
               origins: Optional[torch.Tensor], thh: float, want_prob: bool = False, want_coords: bool = True,
               cap: Optional[int] = None, timing: Optional[list] = None):
        """timing: optional list; a (start, stop) pair of CUDA events recorded on the launching stream
        immediately around the nvf_decode launch sequence is appended (bench.py roofline)."""
        dev = latent.device
        n = int(latent.shape[0])
        latent = latent.detach().contiguous().float()
        wst, keep = self.pack_weights(weights, dev, need_aux=False)
        if origins is not None:
            origins = origins.to(device=dev, dtype=torch.int32).contiguous()
        nbytes = self.workspace_bytes(desc, n, NVF_MODE_DECODE)
        ws = self.cached_workspace(nbytes, dev, "decode")
        prob = torch.empty((n, 1, 32, 32, 32), dtype=torch.float32, device=dev) if want_prob else None
        mask = torch.empty((n, 1024), dtype=torch.int32, device=dev)
        counts = torch.empty((n,), dtype=torch.int32, device=dev)
        total = torch.zeros((1,), dtype=torch.int64, device=dev)
        if cap is None:
            cap = n * 2048
        coords = torch.empty((cap, 3), dtype=torch.int32, device=dev) if want_coords else None
        if timing is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        rc = self.lib.nvf_decode(C.byref(desc), C.byref(wst), _ptr(latent), _ptr(origins), n, float(thh), _ptr(prob),
                                 _ptr(mask), _ptr(counts), _ptr(coords), cap if want_coords else 0, _ptr(total),
                                 _ptr(ws), nbytes, self._stream(dev))
        if timing is not None:
            ev[1].record()
            timing.append(ev)
        self.check(rc, "nvf_decode")
        del keep
        res = dict(prob=prob, mask=mask, counts=counts, total=total, coords=None)
        if want_coords:
            k = int(total.item())  # the one host sync of the decode path: size of the result
            if k > cap:
                coords = torch.empty((k, 3), dtype=torch.int32, device=dev)
                rc = self.lib.nvf_emit_points(_ptr(mask), _ptr(counts), _ptr(origins), n, _ptr(coords), k, _ptr(total),
                                              _ptr(ws), nbytes, self._stream(dev))
                self.check(rc, "nvf_emit_points")
            res["coords"] = coords[:k]
        return res

    def train_forward(self, desc: NvfDesc, weights: Dict[str, torch.Tensor], latent: torch.Tensor):
        dev = latent.device
        n = int(latent.shape[0])
        latent = latent.detach().contiguous().float()
        wst, keep = self.pack_weights(weights, dev, need_aux=True)
        nbytes = self.workspace_bytes(desc, n, NVF_MODE_TRAIN)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)  # owned by the autograd node until backward
        out = torch.empty((n, 1, 32, 32, 32), dtype=torch.float32, device=dev)
        cls1 = torch.empty((n, 1, 16, 16, 16), dtype=torch.float32, device=dev)
        cls0 = torch.empty((n, 1, 8, 8, 8), dtype=torch.float32, device=dev)
        rc = self.lib.nvf_train_forward(C.byref(desc), C.byref(wst), _ptr(latent), n, _ptr(out), _ptr(cls1),
                                        _ptr(cls0), _ptr(ws), nbytes, self._stream(dev))
        self.check(rc, "nvf_train_forward")
        return out, cls1, cls0, ws, keep

    def train_backward(self, desc: NvfDesc, weights: Dict[str, torch.Tensor], latent: torch.Tensor, ws: torch.Tensor,
                       g_out, g_cls1, g_cls0, need_wgrad: bool, need_dlatent: bool):
        dev = latent.device
        n = int(latent.shape[0])
        latent = latent.detach().contiguous().float()
        wst, keep = self.pack_weights(weights, dev, need_aux=True)
        grads: Dict[str, torch.Tensor] = {}
        gst = NvfWeightGrads()
        if need_wgrad:
            for name in WEIGHT_FIELDS:
                g = torch.empty_like(weights[name], memory_format=torch.contiguous_format)
                grads[name] = g
                setattr(gst, name, g.data_ptr())
        g_latent = torch.empty_like(latent) if need_dlatent else None
        flags = (NVF_BWD_WGRAD if need_wgrad else 0) | (NVF_BWD_DLATENT if need_dlatent else 0)
        cg = [None if g is None else g.detach().contiguous().float() for g in (g_out, g_cls1, g_cls0)]
        rc = self.lib.nvf_train_backward(C.byref(desc), C.byref(wst), _ptr(latent), n, _ptr(cg[0]), _ptr(cg[1]),
                                         _ptr(cg[2]), flags, C.byref(gst), _ptr(g_latent), _ptr(ws), ws.numel(),
                                         self._stream(dev))
        self.check(rc, "nvf_train_backward")
        del keep, cg
        return g_latent, grads

    def loss_seeds(self, out, cls1, cls0, gt, dist, alpha_main=0.9, alpha_aux=0.85, thh_metric=0.6,
                   want_seeds: bool = True):
        dev = out.device
        n = int(out.shape[0])
        ts = [t.detach().contiguous().float() for t in (out, cls1, cls0, gt, dist)]
        sums = torch.empty((NVF_LOSS_SUMS,), dtype=torch.float64, device=dev)   # every entry is written by the finalisation
        # owned by this call: the pointer is baked into captured CUDA graphs (trainer.WeightStep), so it must not come
        # from the shared grow-only cache, which drops a buffer when a later, larger call (the full-batch embedding
        # step) outgrows it.  Inside a capture the allocation comes from the graph's private pool and stays valid.
        ws = torch.empty(8 * NVF_LOSS_SUMS * (NVF_LOSS_CHUNKS * n + 1), dtype=torch.uint8, device=dev)
        g = [torch.empty_like(t) for t in ts[:3]] if want_seeds else [None, None, None]
        rc = self.lib.nvf_loss_seeds(_ptr(ts[0]), _ptr(ts[1]), _ptr(ts[2]), _ptr(ts[3]), _ptr(ts[4]), n,
                                     float(alpha_main), float(alpha_aux), float(thh_metric), _ptr(sums), _ptr(g[0]),
                                     _ptr(g[1]), _ptr(g[2]), _ptr(ws), ws.numel(), self._stream(dev))
        self.check(rc, "nvf_loss_seeds")
        return sums, g

    # ---- fused parameter-side transforms --------------------------------------------------------
    @staticmethod
    def _param_set(raw: Dict[str, torch.Tensor]):
        keep = []

        def ptr(t):
            keep.append(t.detach().contiguous())
            return keep[-1].data_ptr()
        return param_set(raw, ptr), keep

    def param_prep(self, desc: NvfDesc, raw: Dict[str, torch.Tensor], q: int, noise: Optional[torch.Tensor],
                   beta_bound: float, gamma_bound: float, pedestal: float):
        dev = raw["lik_sigma"].device
        ps, keep = self._param_set(raw)
        eff: Dict[str, torch.Tensor] = {}
        est = NvfWeightGrads()
        for name in CONV_LAYERS:
            eff[name + "_w"] = torch.empty_like(raw[name + "_kernel"], memory_format=torch.contiguous_format)
            eff[name + "_b"] = torch.empty_like(raw[name + "_b"])
        eff["igdn_beta"] = torch.empty_like(raw["igdn_beta"])
        eff["igdn_gamma"] = torch.empty_like(raw["igdn_gamma"], memory_format=torch.contiguous_format)
        for name in WEIGHT_FIELDS:
            setattr(est, name, eff[name].data_ptr())
        bits = torch.empty(NVF_NUM_QUANT, dtype=torch.float32, device=dev)
        ws = self.cached_workspace(NVF_PARAM_WS_BYTES, dev, "param")
        rc = self.lib.nvf_param_prep(C.byref(desc), C.byref(ps), int(q), _ptr(noise), float(beta_bound),
                                     float(gamma_bound), float(pedestal), C.byref(est), _ptr(bits), _ptr(ws),
                                     ws.numel(), self._stream(dev))
        self.check(rc, "nvf_param_prep")
        del keep
        return eff, bits

    def param_prep_backward(self, desc: NvfDesc, raw: Dict[str, torch.Tensor], beta_bound: float, gamma_bound: float,
                            g_eff: Dict[str, torch.Tensor], g_bits: torch.Tensor):
        dev = raw["lik_sigma"].device
        ps, keep = self._param_set(raw)
        gst, keep2 = self.pack_weights(g_eff, dev, need_aux=True)
        out: Dict[str, torch.Tensor] = {}
        pg = NvfParamGrads()
        for i, name in enumerate(CONV_LAYERS):
            out[name + "_kernel"] = torch.empty_like(raw[name + "_kernel"], memory_format=torch.contiguous_format)
            out[name + "_b"] = torch.empty_like(raw[name + "_b"])
            pg.kernel[i] = out[name + "_kernel"].data_ptr()
            pg.b[i] = out[name + "_b"].data_ptr()
        for field in ("igdn_beta", "igdn_gamma", "lik_sigma", "lik_mu"):
            out[field] = torch.empty_like(raw[field], memory_format=torch.contiguous_format)
            setattr(pg, field, out[field].data_ptr())
        g_bits = g_bits.detach().contiguous().float()
        ws = self.cached_workspace(NVF_PARAM_WS_BYTES, dev, "param_bwd")
        rc = self.lib.nvf_param_prep_backward(C.byref(desc), C.byref(ps), float(beta_bound), float(gamma_bound),
                                              C.byref(gst), _ptr(g_bits), C.byref(pg), _ptr(ws), ws.numel(),
                                              self._stream(dev))
        self.check(rc, "nvf_param_prep_backward")
        del keep, keep2
        return out

    # ---- fused latent head / total loss / Adam ----------------------------------------------------
    def zeroed_workspace(self, nbytes: int, dev: torch.device, tag: str) -> torch.Tensor:
        """Scratch that the library expects zero-filled on first use and leaves zeroed (ticket counters)."""
        key = (str(dev), tag)
        buf = self._ws.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.zeros(max(nbytes, 1), dtype=torch.uint8, device=dev)
            self._ws[key] = buf
        return buf

    @staticmethod
    def _latent_set(raw: Dict[str, torch.Tensor]):
        ps, keep = NvfLatentParams(), []
        for f in LATENT_FIELDS:
            t = raw[f].detach().contiguous()
            keep.append(t)
            setattr(ps, f, t.data_ptr())
        return ps, keep

    def latent_forward(self, ch: int, raw: Dict[str, torch.Tensor], emb: torch.Tensor, noise: Optional[torch.Tensor],
                       noise_scale: float, train: bool, bounds):
        dev = emb.device
        emb = emb.detach().contiguous().float()
        n = int(emb.shape[0])
        ps, keep = self._latent_set(raw)
        latent = torch.empty_like(emb)
        bits = torch.empty(1, dtype=torch.float32, device=dev)
        ws = self.zeroed_workspace(NVF_LATENT_WS_BYTES, dev, "latent")
        rc = self.lib.nvf_latent_forward(int(ch), C.byref(ps), _ptr(emb), _ptr(noise), float(noise_scale), int(train), n,
                                         float(bounds[0]), float(bounds[1]), float(bounds[2]), _ptr(latent), _ptr(bits),
                                         _ptr(ws), ws.numel(), self._stream(dev))
        self.check(rc, "nvf_latent_forward")
        del keep
        return latent, bits

    def latent_backward(self, ch: int, raw: Dict[str, torch.Tensor], emb: torch.Tensor, noise: Optional[torch.Tensor],
                        noise_scale: float, train: bool, bounds, g_latent: Optional[torch.Tensor],
                        g_bits: torch.Tensor, want_params: bool, want_emb: bool,
                        out: Optional[Dict[str, torch.Tensor]] = None):
        """-> (grads dict over LATENT_GRAD_FIELDS or None, g_emb or None).  `out`: preallocated gradient tensors."""
        dev = emb.device
        emb = emb.detach().contiguous().float()
        n = int(emb.shape[0])
        ps, keep = self._latent_set(raw)
        grads, gst = None, None
        if want_params:
            grads = out if out is not None else {f: torch.empty_like(raw[f], memory_format=torch.contiguous_format)
                                                 for f in LATENT_GRAD_FIELDS}
            gst = NvfLatentGrads()
            for f in LATENT_GRAD_FIELDS:
                setattr(gst, f, grads[f].data_ptr())
        g_emb = torch.empty_like(emb) if want_emb else None
        if g_latent is not None:
            g_latent = g_latent.detach().contiguous().float()
        g_bits = g_bits.detach().reshape(1).float()
        ws = self.zeroed_workspace(NVF_LATENT_WS_BYTES, dev, "latent")
        rc = self.lib.nvf_latent_backward(int(ch), C.byref(ps), _ptr(emb), _ptr(noise), float(noise_scale), int(train), n,
                                          float(bounds[0]), float(bounds[1]), float(bounds[2]), _ptr(g_latent),
                                          _ptr(g_bits), C.byref(gst) if gst is not None else None, _ptr(g_emb), _ptr(ws),
                                          ws.numel(), self._stream(dev))
        self.check(rc, "nvf_latent_backward")
        del keep
        return grads, g_emb

    def rd_total(self, sums, latent_bits, net_bits, n_pts, n_total, lmbda, w1, w2, want_stats=True):
        dev = sums.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        stats = torch.empty(7, dtype=torch.float32, device=dev) if want_stats else None
        lb = latent_bits.detach().reshape(1).float()
        nb = net_bits.detach().contiguous().float()
        npts = n_pts.detach().reshape(1).float()
        rc = self.lib.nvf_rd_total(_ptr(sums), _ptr(lb), _ptr(nb), _ptr(npts), float(n_total), float(lmbda), float(w1),
                                   float(w2), _ptr(loss), _ptr(stats), self._stream(dev))
        self.check(rc, "nvf_rd_total")
        return loss, stats

    def rd_total_backward(self, g_loss, n_pts, n_total, lmbda, w1, w2):
        dev = g_loss.device
        g_dist = torch.empty(3, dtype=torch.float32, device=dev)
        g_lb = torch.empty(1, dtype=torch.float32, device=dev)
        g_nb = torch.empty(NVF_NUM_QUANT, dtype=torch.float32, device=dev)
        gl = g_loss.detach().reshape(1).float()
        npts = n_pts.detach().reshape(1).float()
        rc = self.lib.nvf_rd_total_backward(_ptr(gl), _ptr(npts), float(n_total), float(lmbda), float(w1), float(w2),
                                            _ptr(g_dist), _ptr(g_lb), _ptr(g_nb), self._stream(dev))
        self.check(rc, "nvf_rd_total_backward")
        return g_dist, g_lb, g_nb

    def adam_step(self, param, grad, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8):
        rc = self.lib.nvf_adam_step(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq), int(param.numel()),
                                    _ptr(step), _ptr(lr), float(beta1), float(beta2), float(eps),
                                    self._stream(param.device))
        self.check(rc, "nvf_adam_step")

    # ---- symmetric (peer-mapped) gradient buffers + fused all-reduce / Adam ------------------------
    def symm_alloc(self, n: int):
        """-> (device pointer, 64-byte IPC handle) of a zero-filled symmetric buffer for n gradient floats."""
        ptr, handle = C.c_void_p(), C.create_string_buffer(64)
        self.check(self.lib.nvf_symm_alloc(self.lib.nvf_symm_bytes(int(n)), C.byref(ptr), handle), "nvf_symm_alloc")
        return ptr.value, handle.raw

    def symm_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        self.check(self.lib.nvf_symm_open(C.create_string_buffer(handle, 64), C.byref(ptr)), "nvf_symm_open")
        return ptr.value

    def symm_close(self, ptr: int) -> None:
        self.check(self.lib.nvf_symm_close(ptr), "nvf_symm_close")

    def symm_free(self, ptr: int) -> None:
        self.check(self.lib.nvf_symm_free(ptr), "nvf_symm_free")

    def adam_allreduce_step(self, param, grad, exp_avg, exp_avg_sq, step, lr, peers, rank, ctl, beta1=0.9,
                            beta2=0.999, eps=1e-8):
        arr = (C.c_void_p * len(peers))(*peers)
        rc = self.lib.nvf_adam_allreduce_step(_ptr(param), _ptr(grad), _ptr(exp_avg), _ptr(exp_avg_sq),
                                              int(param.numel()), _ptr(step), _ptr(lr), float(beta1), float(beta2),
                                              float(eps), arr, int(rank), len(peers), _ptr(ctl),
                                              self._stream(param.device))
        self.check(rc, "nvf_adam_allreduce_step")

    # ---- fused weight-loop step -------------------------------------------------------------------
    def train_step_workspace(self, desc: NvfDesc, n: int, dev: torch.device) -> torch.Tensor:
        """Zero-filled workspace of nvf_train_step for n blocks (owned by the caller: its address is baked into
        captured graphs; the ticket words inside must start at zero and are left at zero by every call)."""
        out = C.c_size_t(0)
        self.check(self.lib.nvf_train_step_workspace_bytes(C.byref(desc), int(n), C.byref(out)),
                   "nvf_train_step_workspace_bytes")
        return torch.zeros(int(out.value), dtype=torch.uint8, device=dev)

    def train_step(self, args: "NvfStepArgs", ws: torch.Tensor, dev: torch.device) -> None:
        rc = self.lib.nvf_train_step(C.byref(args), _ptr(ws), ws.numel(), self._stream(dev))
        self.check(rc, "nvf_train_step")

    def rng_uniform(self, seed: int, step: int, stream_id: int, first: int, n: int, dev) -> torch.Tensor:
        out = torch.empty(int(n), dtype=torch.float32, device=dev)
        rc = self.lib.nvf_rng_uniform(int(seed), int(step), int(stream_id), int(first), int(n), _ptr(out),
                                      self._stream(out.device))
        self.check(rc, "nvf_rng_uniform")
        return out

    def launch_count(self) -> int:
        return int(self.lib.nvf_launch_count())

    def has_fused_decode(self, chanstr) -> bool:
        """True when nvf_decode runs the fused per-block kernel for this channel configuration (ch = 3)."""
        ch = [int(c) for c in chanstr.split(",")] if isinstance(chanstr, str) else list(chanstr)
        d = self.desc(3, ch)
        return bool(self.lib.nvf_has_fused_decode(C.byref(d)))

    def ffma_microbench(self, variant: int, iters: int, sink: torch.Tensor) -> float:
        flops = C.c_double(0)
        rc = self.lib.nvf_ffma_microbench(variant, iters, _ptr(sink), C.byref(flops), self._stream(sink.device))
        self.check(rc, "nvf_ffma_microbench")
        return float(flops.value)


_cuda_binding: Optional[Binding] = None


def lib_path() -> str:
    return os.path.join(HERE, LIB_NAME)


def cuda_binding() -> Binding:
    """The product binding.  Fails loudly when the CUDA library is not built."""
    global _cuda_binding
    if _cuda_binding is None:
        p = lib_path()
        if not os.path.isfile(p):
            raise NvfError("%s not found: build it with `python -m nvfpcc_b200.build` (nvcc, sm_100a). "
                           "There is no CPU fallback." % p)
        _cuda_binding = Binding(p)
    return _cuda_binding
