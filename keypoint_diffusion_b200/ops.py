"""Thin Python wrappers over the C ABI (include/kpdiff_b200.h): batch layout, graph build,
denoiser forward, posterior step and the captured sampling loop.

torch is used for device memory and streams only; every computation below is a call into
libkpdiff_b200.so.  All tensors must live on one CUDA device (no CPU fallback).
"""
import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import (KpdBatch, KpdCsr, KpdEgnnConfig, KpdGraphParams, KpdGvpConfig, KpdSamplerConfig, check, lib, ptr)
from . import pack


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("keypoint_diffusion_b200 runs on CUDA tensors only (no CPU fallback)")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32(t):
    return t.contiguous().to(torch.float32)


class DeviceBatch:
    """Node layout of a batch of complexes (replaces the DGL batch bookkeeping read by the hot
    path: g.batch_size, g.batch_num_nodes, utils.get_batch_idxs -- reference utils.py:81-170)."""

    def __init__(self, lig_n: Sequence[int], kp_n: Sequence[int], device, max_lig: int = 0, max_kp: int = 0):
        lig_n = [int(v) for v in lig_n]
        kp_n = [int(v) for v in kp_n]
        if len(lig_n) != len(kp_n) or not lig_n:
            raise ValueError("lig_n and kp_n must be non-empty and of equal length")
        if min(lig_n) < 1 or min(kp_n) < 1:
            raise ValueError("every complex needs at least one ligand atom and one keypoint")
        self.device = torch.device(device)
        self.lig_n, self.kp_n = lig_n, kp_n
        self.B = len(lig_n)
        ln = torch.tensor(lig_n, dtype=torch.int64)
        kn = torch.tensor(kp_n, dtype=torch.int64)
        self.n_lig, self.n_kp = int(ln.sum()), int(kn.sum())
        lp = torch.zeros(self.B + 1, dtype=torch.int32); lp[1:] = torch.cumsum(ln, 0)
        kp = torch.zeros(self.B + 1, dtype=torch.int32); kp[1:] = torch.cumsum(kn, 0)
        ar = torch.arange(self.B, dtype=torch.int32)
        self.lig_ptr = lp.to(self.device)
        self.kp_ptr = kp.to(self.device)
        self.lig_batch = ar.repeat_interleave(ln).to(self.device)
        self.kp_batch = ar.repeat_interleave(kn).to(self.device)
        self.c = KpdBatch(self.B, self.n_lig, self.n_kp, max(max(lig_n), int(max_lig or 0)), max(max(kp_n), int(max_kp or 0)),
                          self.lig_ptr.data_ptr(), self.kp_ptr.data_ptr(), self.lig_batch.data_ptr(),
                          self.kp_batch.data_ptr())

    def set_layout(self, lig_n: Sequence[int], kp_n: Sequence[int]):
        """Overwrite the per-complex sizes IN PLACE (same device arrays, same addresses): the number of complexes and
        the node totals must stay what this object was created with, and no complex may exceed max_lig / max_kp.  This
        is what lets a captured sampler (whose kernels hold these addresses and the totals) run a different batch."""
        lig_n = [int(v) for v in lig_n]
        kp_n = [int(v) for v in kp_n]
        if (len(lig_n) != self.B or len(kp_n) != self.B or sum(lig_n) != self.n_lig or sum(kp_n) != self.n_kp
                or max(lig_n) > self.c.max_lig or max(kp_n) > self.c.max_kp or min(lig_n) < 1 or min(kp_n) < 1):
            raise ValueError("set_layout: the new layout does not fit this batch's fixed totals / maxima")
        if lig_n == self.lig_n and kp_n == self.kp_n:
            return
        self.lig_n, self.kp_n = lig_n, kp_n
        ln = torch.tensor(lig_n, dtype=torch.int64)
        kn = torch.tensor(kp_n, dtype=torch.int64)
        lp = torch.zeros(self.B + 1, dtype=torch.int32); lp[1:] = torch.cumsum(ln, 0)
        kp = torch.zeros(self.B + 1, dtype=torch.int32); kp[1:] = torch.cumsum(kn, 0)
        ar = torch.arange(self.B, dtype=torch.int32)
        self.lig_ptr.copy_(lp, non_blocking=True)
        self.kp_ptr.copy_(kp, non_blocking=True)
        self.lig_batch.copy_(ar.repeat_interleave(ln), non_blocking=True)
        self.kp_batch.copy_(ar.repeat_interleave(kn), non_blocking=True)

    def edge_capacity(self, gp: "GraphParams") -> Tuple[int, int]:
        """(cap_ll, cap_kl): the most edges any configuration of this batch can produce."""
        ll_lim = gp.ll_k if gp.ll_k > 0 else gp.ll_cap
        kl_lim = gp.kl_k if gp.kl_k > 0 else gp.kl_cap
        cap_ll = sum(n * min(n - 1, ll_lim) for n in self.lig_n)
        cap_kl = sum(k * min(n, kl_lim) for n, k in zip(self.lig_n, self.kp_n))
        return max(cap_ll, 1), max(cap_kl, 1)


@dataclass
class GraphParams:
    """How add_lig_edges draws ligand edges (reference models/dynamics.py:393-404)."""
    ll_k: int = 0
    ll_r: float = 5.0
    ll_cap: int = 200
    kl_k: int = 5
    kl_r: float = 8.0
    kl_cap: int = 100

    @property
    def c(self):
        return KpdGraphParams(self.ll_k, self.ll_cap, self.kl_k, self.kl_cap, float(self.ll_r), float(self.kl_r))

    @staticmethod
    def from_module(ll_k, kl_k, graph_cutoffs):
        return GraphParams(ll_k=int(ll_k), ll_r=float(graph_cutoffs.get("ll", 0.0) or 0.0), kl_k=int(kl_k),
                           kl_r=float(graph_cutoffs.get("kl", 0.0) or 0.0))


class Csr:
    """dst-sorted CSR + COO of one edge type on the device."""

    def __init__(self, n_dst: int, cap: int, device):
        self.n_dst, self.cap = int(n_dst), int(cap)
        self.rowptr = torch.zeros(self.n_dst + 1, dtype=torch.int32, device=device)
        self.src = torch.zeros(self.cap + 1, dtype=torch.int32, device=device)
        self.dst = torch.zeros(self.cap + 1, dtype=torch.int32, device=device)
        self.c = KpdCsr(self.n_dst, self.cap, self.rowptr.data_ptr(), self.src.data_ptr(), self.dst.data_ptr())

    @staticmethod
    def from_edges(src: torch.Tensor, dst: torch.Tensor, n_dst: int, device) -> "Csr":
        """Static graph (kk) given as global (src, dst) index lists: stable sort by destination."""
        src = src.to("cpu", torch.int64)
        dst = dst.to("cpu", torch.int64)
        order = torch.sort(dst, stable=True).indices
        out = Csr(n_dst, max(int(src.numel()), 1), device)
        if src.numel():
            out.src[: src.numel()] = src[order].to(torch.int32).to(device)
            out.dst[: src.numel()] = dst[order].to(torch.int32).to(device)
        rp = torch.zeros(n_dst + 1, dtype=torch.int64)
        rp[1:] = torch.cumsum(torch.bincount(dst, minlength=n_dst), 0)
        out.rowptr.copy_(rp.to(torch.int32))
        return out

    def fill_from_edges(self, src: torch.Tensor, dst: torch.Tensor):
        """Rewrite this CSR IN PLACE from global (src, dst) index lists, with device ops only (stable sort by
        destination, bincount, cumsum): no host round trip, addresses unchanged, so a captured sampler that holds this
        CSR sees the new graph.  At most `cap` edges."""
        n = int(src.numel())
        if n > self.cap:
            raise ValueError(f"fill_from_edges: {n} edges exceed the capacity {self.cap}")
        dev = self.rowptr.device
        if n == 0:
            self.rowptr.zero_()
            return self
        src = src.to(dev, non_blocking=True)
        dst = dst.to(dev, non_blocking=True)
        order = torch.sort(dst, stable=True).indices
        self.src[:n] = src[order].to(torch.int32)
        self.dst[:n] = dst[order].to(torch.int32)
        self.rowptr[0] = 0
        self.rowptr[1:] = torch.cumsum(torch.bincount(dst, minlength=self.n_dst), 0).to(torch.int32)
        return self

    def edges(self) -> torch.Tensor:
        """[2, E] int64 (src; dst) on the CPU -- synchronises; for tests and debugging only."""
        e = int(self.rowptr[-1].item())
        return torch.stack([self.src[:e].long().cpu(), self.dst[:e].long().cpu()])


class LigandGraphs:
    """ll / kl / lk graphs of one denoiser call + the scratch kpd_build_graph needs."""

    def __init__(self, batch: DeviceBatch, gp: GraphParams, with_lk: bool):
        self.batch, self.gp, self.with_lk = batch, gp, with_lk
        cap_ll, cap_kl = batch.edge_capacity(gp)
        dev = batch.device
        self.ll = Csr(batch.n_lig, cap_ll, dev)
        self.kl = Csr(batch.n_lig, cap_kl, dev)
        self.lk = Csr(batch.n_kp, cap_kl, dev) if with_lk else None
        self.counts_ll = torch.zeros(batch.B, dtype=torch.int32, device=dev)
        self.counts_kl = torch.zeros(batch.B, dtype=torch.int32, device=dev)
        self.ws = torch.empty(int(lib.kpd_graph_workspace_bytes(C.byref(batch.c))), dtype=torch.uint8, device=dev)

    def build(self, x_lig: torch.Tensor, x_kp: torch.Tensor):
        _require_cuda(x_lig, x_kp)
        assert x_lig.dtype == torch.float32 and x_kp.dtype == torch.float32
        assert x_lig.is_contiguous() and x_kp.is_contiguous()
        gpc = self.gp.c
        check(lib.kpd_build_graph(C.byref(self.batch.c), ptr(x_lig), ptr(x_kp), C.byref(gpc), C.byref(self.ll.c),
                                  C.byref(self.kl.c), C.byref(self.lk.c) if self.lk else None,
                                  ptr(self.counts_ll), ptr(self.counts_kl), ptr(self.ws), _stream()),
              "kpd_build_graph")
        return self


def linear(x, wt, bias=None, residual=None, act=0, n_out=None):
    """Y = act(X @ WT + b) (+R) through kpd_linear (WT K-major, columns padded to x4)."""
    _require_cuda(x, wt)
    M, K = x.shape
    N = n_out if n_out is not None else wt.shape[1]
    y = torch.empty(M, N, dtype=torch.float32, device=x.device)
    check(lib.kpd_linear(ptr(x), x.stride(0), ptr(wt), wt.stride(0), ptr(bias), ptr(residual),
                         residual.stride(0) if residual is not None else 0, ptr(y), y.stride(0), M, K, N, act,
                         _stream()), "kpd_linear")
    return y


def tc_linear(x, w_packed, n_out, bias=None, residual=None, act=0, nsplit=1):
    """Y = act(X @ W^T + b) (+R) on tcgen05 tensor cores, fp32 accumulate.  nsplit=1: bf16 operands, w_packed from
    pack.pack_tc_weight(w); nsplit=2: split (hi, lo) bf16 operands ("bf16x3", fp32-grade), w_packed from
    pack.pack_tc_weight(w, split=True).  Rows of x must be 16-byte aligned."""
    _require_cuda(x, w_packed)
    M, K = x.shape
    if x.stride(0) % 4:
        xp = torch.zeros(M, (K + 3) // 4 * 4, dtype=torch.float32, device=x.device)
        xp[:, :K] = x
        x = xp
    y = torch.empty(M, n_out, dtype=torch.float32, device=x.device)
    check(lib.kpd_tc_linear(ptr(x), x.stride(0), ptr(w_packed), ptr(bias), ptr(residual),
                            residual.stride(0) if residual is not None else 0, ptr(y), y.stride(0), M, K, n_out, act,
                            int(nsplit), _stream()), "kpd_tc_linear")
    return y


class _Model:
    arch = -1

    def __init__(self):
        self.handle = C.c_void_p()
        self._ws: Dict[Tuple, torch.Tensor] = {}

    def _workspace(self, batch: DeviceBatch, caps: Tuple[int, int, int]) -> torch.Tensor:
        # keyed on what the workspace size depends on (values, not id(batch): ids are reused after garbage collection)
        key = (batch.c.B, batch.c.n_lig, batch.c.n_kp, batch.c.max_lig, batch.c.max_kp, tuple(caps), str(batch.device))
        ws = self._ws.get(key)
        if ws is None:
            fn = lib.kpd_egnn_workspace_bytes if self.arch == 0 else lib.kpd_gvp_workspace_bytes
            n = int(fn(self.handle, C.byref(batch.c), *caps))
            ws = torch.empty(n, dtype=torch.uint8, device=batch.device)
            self._ws = {key: ws}          # keep only the latest layout
        return ws


def egnn_has_tc_tiles(hidden_nf: int) -> bool:
    """Whether the EGNN tensor-core modes take this width (csrc/egnn.cu kpd_egnn_attach_tc): H = hidden_nf + 1 <= 257
    and nmain = min(H, 256) rounded down to a multiple of 4 is a non-zero multiple of 8 (the nmain output columns are
    one MMA of N = nmain padded to 16; the H - nmain <= 3 leftover columns run beside it).  Other widths run the fp32
    SIMT kernels."""
    H = hidden_nf + 1
    nmain = min(H, 256) // 4 * 4
    return H <= 257 and nmain >= 8 and nmain % 8 == 0


def gvp_has_tc_tiles(n_hidden_scalars: int) -> bool:
    """Whether the GVP tensor-core modes take this scalar width (csrc/gvp.cu kpd_gvp_attach_tc); other widths the
    library accepts (multiples of 4 up to 256) run the fp32 SIMT kernels."""
    return n_hidden_scalars % 16 == 0


class EgnnModel(_Model):
    """Packed EGNN denoiser weights on the device (kpd_egnn_model)."""
    arch = 0

    def __init__(self, sd: Dict[str, torch.Tensor], *, atom_nf, rec_nf, hidden_nf, n_layers, use_tanh,
                 update_kp_feat, norm, message_norm, device, coords_range=10.0, z_effective=False):
        super().__init__()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("EgnnModel needs a CUDA device (no CPU fallback)")
        self.update_kp_feat = bool(update_kp_feat)
        self.atom_nf, self.rec_nf, self.hidden_nf = atom_nf, rec_nf, hidden_nf
        self.n_layers = n_layers
        has_rec = "rec_encoder.0.weight" in sd
        self.blob, offs = pack.pack_egnn(sd, atom_nf=atom_nf, rec_nf=rec_nf, hidden_nf=hidden_nf, n_layers=n_layers,
                                         update_kp_feat=update_kp_feat, norm=norm, device=self.device)
        cfg = KpdEgnnConfig(atom_nf, rec_nf, hidden_nf, n_layers, int(bool(use_tanh)), int(bool(update_kp_feat)),
                            int(bool(norm)), int(has_rec), float(coords_range), float(message_norm),
                            int(bool(z_effective)))
        arr = (C.c_int64 * len(offs))(*offs)
        check(lib.kpd_egnn_create(C.byref(cfg), ptr(self.blob), arr, len(offs), C.byref(self.handle)), "kpd_egnn_create")
        self.precision = "fp32"
        self.tc_blob = self.tc_blob2 = None
        self._sd_bf16 = None
        if egnn_has_tc_tiles(hidden_nf):
            self.tc_blob2 = self._attach_tc(sd, split=True)
            # the plain-bf16 pack is built on the first set_precision('bf16') (from a reference to sd, not a copy): a
            # model that never uses that mode costs no more to create and holds no more packed weights
            self._sd_bf16 = sd

    PRECISIONS = {"fp32": 0, "bf16": 1, "bf16x3": 2}

    def _attach_tc(self, sd, split: bool) -> torch.Tensor:
        blob, toffs = pack.pack_egnn_tc(sd, hidden_nf=self.hidden_nf, n_layers=self.n_layers,
                                        update_kp_feat=self.update_kp_feat, device=self.device, split=split)
        tarr = (C.c_int64 * len(toffs))(*toffs)
        check(lib.kpd_egnn_attach_tc(self.handle, ptr(blob), tarr, len(toffs), 2 if split else 1), "kpd_egnn_attach_tc")
        return blob

    def set_precision(self, precision: str):
        """'fp32' (SIMT, the reference's arithmetic), 'bf16x3' (tcgen05 tensor cores with split bf16 operands:
        fp32-grade, inside the 1e-4 parity bar) or 'bf16' (tcgen05, plain bf16 operands in the edge kernel: faster,
        within 3e-2 of the fp32 output scale)."""
        if precision not in self.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(self.PRECISIONS)}, got {precision!r}")
        if precision == "bf16" and self.tc_blob is None and self.tc_blob2 is not None:
            self.tc_blob = self._attach_tc(self._sd_bf16, split=False)
            self._sd_bf16 = None
        check(lib.kpd_egnn_set_mode(self.handle, self.PRECISIONS[precision]), "kpd_egnn_set_mode")
        self.precision = precision

    def __del__(self):
        if getattr(self, "handle", None) and self.handle.value and lib is not None:
            lib.kpd_egnn_destroy(self.handle)
            self.handle = C.c_void_p()

    def forward(self, batch: DeviceBatch, graphs: LigandGraphs, kk: Optional[Csr], h_lig, x_lig, h_kp, x_kp, t,
                kp_feat_enc=None):
        """(eps_h, eps_x) for one denoiser call; t: float tensor [1] (shared) or [B] on the device."""
        _require_cuda(h_lig, x_lig, h_kp, x_kp, t)
        eps_h = torch.empty(batch.n_lig, self.atom_nf, dtype=torch.float32, device=self.device)
        eps_x = torch.empty(batch.n_lig, 3, dtype=torch.float32, device=self.device)
        caps = (graphs.ll.cap, graphs.kl.cap, kk.cap if kk is not None else 1)
        ws = self._workspace(batch, caps)
        per_complex = int(t.numel() == batch.B and batch.B > 1)
        # converted copies are bound to locals so they outlive the launch (a temporary would go back to the caching
        # allocator inside the argument list and two arguments could alias)
        h_lig, x_lig, h_kp, x_kp, t = _f32(h_lig), _f32(x_lig), _f32(h_kp), _f32(x_kp), _f32(t)
        check(lib.kpd_egnn_forward(self.handle, C.byref(batch.c), ptr(h_lig), ptr(x_lig), ptr(h_kp),
                                   ptr(x_kp), ptr(kp_feat_enc), ptr(t), per_complex,
                                   C.byref(graphs.ll.c), C.byref(graphs.kl.c),
                                   C.byref(graphs.lk.c) if graphs.lk is not None else None,
                                   C.byref(kk.c) if kk is not None else None, ptr(eps_h), ptr(eps_x), ptr(ws),
                                   _stream()), "kpd_egnn_forward")
        return eps_h, eps_x


class GvpModel(_Model):
    """Packed GVP denoiser weights on the device (kpd_gvp_model)."""
    arch = 1

    def __init__(self, sd: Dict[str, torch.Tensor], *, n_lig_scalars, n_kp_scalars, vector_size, n_convs,
                 n_hidden_scalars, update_kp, n_message_gvps, n_update_gvps, n_noise_gvps, message_norm, device,
                 rbf_dmax=15.0, rbf_dim=16, precision="fp32"):
        super().__init__()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("GvpModel needs a CUDA device (no CPU fallback)")
        self.update_kp = bool(update_kp)
        self.atom_nf, self.vector_size = n_lig_scalars, vector_size
        self.blob, offs = pack.pack_gvp(sd, n_lig_scalars=n_lig_scalars, n_kp_scalars=n_kp_scalars,
                                        vector_size=vector_size, n_convs=n_convs, n_hidden_scalars=n_hidden_scalars,
                                        update_kp=update_kp, n_message_gvps=n_message_gvps,
                                        n_update_gvps=n_update_gvps, n_noise_gvps=n_noise_gvps, device=self.device)
        if message_norm == "mean":
            mode, mn = 1, 1.0
        elif float(message_norm) == 0.0:
            mode, mn = 2, 0.0
        else:
            mode, mn = 0, float(message_norm)
        cfg = KpdGvpConfig(n_lig_scalars, n_kp_scalars, vector_size, n_convs, n_hidden_scalars, n_message_gvps,
                           n_update_gvps, n_noise_gvps, int(bool(update_kp)), mode, mn, float(rbf_dmax), int(rbf_dim))
        arr = (C.c_int64 * len(offs))(*offs)
        check(lib.kpd_gvp_create(C.byref(cfg), ptr(self.blob), arr, len(offs), C.byref(self.handle)), "kpd_gvp_create")
        self.precision = "fp32"
        self.tc_blob = self.tc_blob2 = None
        if gvp_has_tc_tiles(n_hidden_scalars):
            kw = dict(n_convs=n_convs, update_kp=update_kp, n_message_gvps=n_message_gvps, n_update_gvps=n_update_gvps,
                      n_noise_gvps=n_noise_gvps, device=self.device)
            self.tc_blob, toffs = pack.pack_gvp_tc(sd, **kw)
            tarr = (C.c_int64 * len(toffs))(*toffs)
            check(lib.kpd_gvp_attach_tc(self.handle, ptr(self.tc_blob), tarr, len(toffs), 1), "kpd_gvp_attach_tc")
            self.tc_blob2, toffs = pack.pack_gvp_tc(sd, split=True, **kw)
            tarr = (C.c_int64 * len(toffs))(*toffs)
            check(lib.kpd_gvp_attach_tc(self.handle, ptr(self.tc_blob2), tarr, len(toffs), 2), "kpd_gvp_attach_tc")
        if precision != "fp32":
            self.set_precision(precision)

    PRECISIONS = {"fp32": 0, "bf16": 1, "bf16x3": 2}

    def set_precision(self, precision: str):
        """'fp32' (SIMT, the reference's arithmetic), 'bf16x3' (tcgen05 tensor cores with split bf16 operands:
        fp32-grade, inside the 1e-4 parity bar) or 'bf16' (tcgen05, plain bf16 operands, ~2e-3)."""
        if precision not in self.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(self.PRECISIONS)}, got {precision!r}")
        check(lib.kpd_gvp_set_mode(self.handle, self.PRECISIONS[precision]), "kpd_gvp_set_mode")
        self.precision = precision

    def __del__(self):
        if getattr(self, "handle", None) and self.handle.value and lib is not None:
            lib.kpd_gvp_destroy(self.handle)
            self.handle = C.c_void_p()

    def forward(self, batch: DeviceBatch, graphs: LigandGraphs, kk: Optional[Csr], h_lig, x_lig, h_kp, x_kp, v_kp, t):
        _require_cuda(h_lig, x_lig, h_kp, x_kp, v_kp, t)
        eps_h = torch.empty(batch.n_lig, self.atom_nf, dtype=torch.float32, device=self.device)
        eps_x = torch.empty(batch.n_lig, 3, dtype=torch.float32, device=self.device)
        caps = (graphs.ll.cap, graphs.kl.cap, kk.cap if kk is not None else 1)
        ws = self._workspace(batch, caps)
        per_complex = int(t.numel() == batch.B and batch.B > 1)
        h_lig, x_lig, h_kp, x_kp, v_kp, t = _f32(h_lig), _f32(x_lig), _f32(h_kp), _f32(x_kp), _f32(v_kp), _f32(t)
        check(lib.kpd_gvp_forward(self.handle, C.byref(batch.c), ptr(h_lig), ptr(x_lig), ptr(h_kp),
                                  ptr(x_kp), ptr(v_kp), ptr(t), per_complex, C.byref(graphs.ll.c),
                                  C.byref(graphs.kl.c), C.byref(graphs.lk.c) if graphs.lk is not None else None,
                                  C.byref(kk.c) if kk is not None else None, ptr(eps_h), ptr(eps_x), ptr(ws),
                                  _stream()), "kpd_gvp_forward")
        return eps_h, eps_x


def ddpm_step(batch: DeviceBatch, x_lig, h_lig, x_kp, eps_x, eps_h, coef, step: torch.Tensor, noise_x=None,
              noise_h=None, seed=0):
    """In-place reverse step s <- s+1 (reference ligand_diffuser.py:515-536); step: int32 [1] on device."""
    _require_cuda(x_lig, h_lig, x_kp, eps_x, eps_h, coef, step)
    check(lib.kpd_ddpm_step(C.byref(batch.c), ptr(x_lig), ptr(h_lig), ptr(x_kp), ptr(eps_x), ptr(eps_h),
                            h_lig.shape[1], ptr(coef), ptr(step), ptr(noise_x), ptr(noise_h), int(seed), _stream()),
          "kpd_ddpm_step")


def ddpm_multistep_step(batch: DeviceBatch, x_lig, h_lig, x_kp, eps_x, eps_h, coef, ms_coef, step: torch.Tensor,
                        first_row: int, hist_x, hist_h, noise_x=None, noise_h=None, seed=0):
    """In-place DPM-Solver++(2M) reverse step (kpd_ddpm_multistep_step, DESIGN.md section 6.5): the DDIM eta = 0 row of
    coef, plus c (x^ - hist) with row `step` of ms_coef (schedule.multistep_rows) unless step == first_row; hist_x /
    hist_h then hold x^, its positions moved with the ligand COM."""
    _require_cuda(x_lig, h_lig, x_kp, eps_x, eps_h, coef, ms_coef, step, hist_x, hist_h, noise_x, noise_h)
    check(lib.kpd_ddpm_multistep_step(C.byref(batch.c), ptr(x_lig), ptr(h_lig), ptr(x_kp), ptr(eps_x), ptr(eps_h),
                                      h_lig.shape[1], ptr(coef), ptr(ms_coef), ptr(step), int(first_row), ptr(hist_x),
                                      ptr(hist_h), ptr(noise_x), ptr(noise_h), int(seed), _stream()),
          "kpd_ddpm_multistep_step")


def ddpm_inpaint_step(batch: DeviceBatch, x_lig, h_lig, x_kp, eps_x, eps_h, coef, coef2, step: torch.Tensor, u: int,
                      fixed_mask, x_fix, h_fix, init_kp_com, lig_feat_norm_constant=1.0, noise=None, seed=0):
    """In-place fragment-conditioned reverse step, pass u (kpd_ddpm_inpaint_step): the posterior step with the atoms of
    fixed_mask (bool / uint8 [n_lig], or None) replaced by a noised copy of (x_fix, h_fix), aligned to the generated
    part.  noise: None (Philox) or [2, n_lig*(3+F)] injected draws (posterior, known part; x channels first)."""
    _require_cuda(x_lig, h_lig, x_kp, eps_x, eps_h, coef, coef2, step, init_kp_com, fixed_mask, x_fix, h_fix, noise)
    mask = fixed_mask.to(torch.uint8).contiguous() if fixed_mask is not None else None
    check(lib.kpd_ddpm_inpaint_step(C.byref(batch.c), ptr(x_lig), ptr(h_lig), ptr(x_kp), ptr(eps_x), ptr(eps_h),
                                    h_lig.shape[1], ptr(coef), ptr(coef2), ptr(step), int(u), ptr(mask),
                                    ptr(x_fix), ptr(h_fix), ptr(init_kp_com), float(lig_feat_norm_constant), ptr(noise),
                                    int(seed), _stream()), "kpd_ddpm_inpaint_step")


def renoise(batch: DeviceBatch, x_lig, h_lig, x_kp, coef2, step: torch.Tensor, u: int, noise=None, seed=0):
    """In-place re-noise to level t = s+1 after pass u of step s (kpd_renoise); noise: None or [n_lig*(3+F)]."""
    _require_cuda(x_lig, h_lig, x_kp, coef2, step, noise)
    check(lib.kpd_renoise(C.byref(batch.c), ptr(x_lig), ptr(h_lig), ptr(x_kp), h_lig.shape[1], ptr(coef2), ptr(step),
                          int(u), ptr(noise), int(seed), _stream()), "kpd_renoise")


def partial_noise(batch: DeviceBatch, x_start, h_start, x_kp, alpha: float, sigma: float, lig_feat_norm_constant=1.0,
                  noise=None, seed=0):
    """The start of a run from a given ligand (kpd_partial_noise): x_start [n_lig,3] / h_start [n_lig,F] noised to the
    level (alpha, sigma) in the frame of each complex's start-ligand mean, then the ligand COM removed; x_kp is moved
    with the ligand, in place.  noise: None (Philox, the plain loop's initial draw) or [n_lig*(3+F)] (x first).
    -> (x_lig, h_lig)."""
    _require_cuda(x_start, h_start, x_kp, noise)
    x_lig, h_lig = torch.empty_like(x_start), torch.empty_like(h_start)
    check(lib.kpd_partial_noise(C.byref(batch.c), ptr(x_start), ptr(h_start), ptr(x_lig), ptr(h_lig), ptr(x_kp),
                                h_start.shape[1], float(alpha), float(sigma), float(lig_feat_norm_constant), ptr(noise),
                                int(seed), _stream()), "kpd_partial_noise")
    return x_lig, h_lig


def decode_atom_types(h_lig: torch.Tensor) -> torch.Tensor:
    """int32 [n] = argmax over the feature channels of every atom (lowest index wins ties, like torch.argmax on the
    CPU), on the device through kpd_decode_atom_types -- what the reference computes on the host right after sampling
    (test.py:199-203: ``torch.argmax(feat, dim=1)`` then ``lig_atom_idx_to_element``)."""
    _require_cuda(h_lig)
    h_lig = _f32(h_lig)
    out = torch.empty(h_lig.shape[0], dtype=torch.int32, device=h_lig.device)
    check(lib.kpd_decode_atom_types(ptr(h_lig), h_lig.shape[0], h_lig.shape[1], ptr(out), _stream()),
          "kpd_decode_atom_types")
    return out


def remove_com(batch: DeviceBatch, x_lig, x_kp, which: str):
    """In-place remove_com (reference ligand_diffuser.py:185-203); returns the [B,3] means."""
    _require_cuda(x_lig, x_kp)
    com = torch.empty(batch.B, 3, dtype=torch.float32, device=batch.device)
    check(lib.kpd_remove_com(C.byref(batch.c), ptr(x_lig), ptr(x_kp), {"ligand": 0, "receptor": 1}[which], ptr(com),
                             _stream()), "kpd_remove_com")
    return com


class Sampler:
    """The captured reverse-diffusion loop for one (model, batch) pair (kpd_sampler).

    resamplings >= 1 with inpaint_coef (schedule.inpaint_table on the device) makes it a fragment-conditioned
    (inpainting) sampler: every reverse step runs `resamplings` denoiser passes with the atoms given to set_fragment
    pinned, and a captured graph holds steps_per_graph // resamplings steps.  0 (default) = the plain loop.
    Either kind runs from a given ligand after set_start (ligand optimisation by partial noising), and with fewer,
    strided or DDIM steps after set_schedule; neither captures again.  record=True makes it a recording sampler: its
    captured step holds one more launch, and run(record_every=k) returns the trajectory (DESIGN.md section 6.4).
    multistep=True makes it a DPM-Solver++(2M) sampler (DESIGN.md section 6.5; not with resamplings): its captured step
    runs the multistep step kernel, which carries the previous step's clean-ligand estimate in a history the sampler
    allocates for its layout; every run needs DDIM eta = 0 rows (set_schedule) and their set_multistep rows."""

    def __init__(self, model: _Model, batch: DeviceBatch, gp: GraphParams, kk: Optional[Csr], coef: torch.Tensor,
                 T: int, atom_nf: int, steps_per_graph: int = 50, use_cuda_graph: bool = True,
                 lig_feat_norm_constant: float = 1.0, atom_offset: int = 0, caps: Optional[Tuple[int, int]] = None,
                 resamplings: int = 0, inpaint_coef: Optional[torch.Tensor] = None, record: bool = False,
                 multistep: bool = False):
        self.model, self.batch, self.gp, self.kk, self.coef = model, batch, gp, kk, coef
        _require_cuda(coef)
        self.T, self.atom_nf = int(T), int(atom_nf)
        self.resamplings = int(resamplings)
        if self.resamplings < 0 or (self.resamplings > 0) != (inpaint_coef is not None):
            raise ValueError("an inpainting sampler needs resamplings >= 1 and inpaint_coef; a plain one neither")
        if multistep and self.resamplings:
            raise ValueError("a multistep sampler cannot inpaint (resamplings must be 0)")
        self.has_lk = bool(model.update_kp_feat if model.arch == 0 else model.update_kp)
        if self.resamplings:        # about as many graph nodes per captured graph as the plain loop
            steps_per_graph = max(1, int(steps_per_graph) // self.resamplings)
        steps_per_graph = max(1, min(int(steps_per_graph), self.T))
        self.cfg = KpdSamplerConfig(model.arch, self.T, self.atom_nf, steps_per_graph, int(bool(use_cuda_graph)),
                                    float(lig_feat_norm_constant))
        cap_ll, cap_kl = caps if caps is not None else batch.edge_capacity(gp)
        cap_kk = kk.cap if kk is not None else 1
        n = int(lib.kpd_sampler_workspace_bytes(C.byref(self.cfg), model.handle, C.byref(batch.c), cap_ll, cap_kl, cap_kk))
        if n < 0:
            check(-1, "kpd_sampler_workspace_bytes")
        self.ws = torch.empty(n, dtype=torch.uint8, device=batch.device)
        self.handle = C.c_void_p()
        self._gpc = gp.c
        check(lib.kpd_sampler_create(C.byref(self.cfg), model.handle, C.byref(batch.c), C.byref(self._gpc),
                                     C.byref(kk.c) if kk is not None else None, int(self.has_lk), ptr(coef), cap_ll,
                                     cap_kl, ptr(self.ws), n, C.byref(self.handle)), "kpd_sampler_create")
        if atom_offset:     # this sampler holds a slice of a larger batch: keep the noise of the undivided batch
            check(lib.kpd_sampler_set_atom_offset(self.handle, int(atom_offset)), "kpd_sampler_set_atom_offset")
        self.inpaint_coef = inpaint_coef
        self._fragment = None
        self._start = None
        self._schedule = None
        if self.resamplings:
            _require_cuda(inpaint_coef)
            check(lib.kpd_sampler_enable_inpainting(self.handle, self.resamplings, ptr(inpaint_coef)),
                  "kpd_sampler_enable_inpainting")
        self.record = bool(record)
        if self.record:
            check(lib.kpd_sampler_enable_recording(self.handle), "kpd_sampler_enable_recording")
        self.multistep = bool(multistep)
        self._ms_coef = None
        if self.multistep:
            check(lib.kpd_sampler_enable_multistep(self.handle), "kpd_sampler_enable_multistep")
            self.hist_x = torch.empty(batch.n_lig, 3, dtype=torch.float32, device=batch.device)
            self.hist_h = torch.empty(batch.n_lig, self.atom_nf, dtype=torch.float32, device=batch.device)

    def set_multistep(self, ms_coef: torch.Tensor):
        """The DPM-Solver++(2M) rows of the next runs (multistep samplers only; kpd_sampler_set_multistep): ms_coef fp32
        [n,4] on the device, schedule.multistep_rows over the grid of the active schedule, which must hold the DDIM
        eta = 0 rows of that grid (n == schedule_rows, checked by the run).  The tensor must stay alive and in place
        while runs use it (only its address is kept)."""
        if not self.multistep:
            raise ValueError("set_multistep needs a multistep sampler (multistep=True)")
        _require_cuda(ms_coef)
        assert ms_coef.dtype == torch.float32 and ms_coef.is_contiguous() and ms_coef.dim() == 2
        assert ms_coef.shape[1] == 4
        check(lib.kpd_sampler_set_multistep(self.handle, int(ms_coef.shape[0]), ptr(ms_coef), ptr(self.hist_x),
                                            ptr(self.hist_h)), "kpd_sampler_set_multistep")
        self._ms_coef = ms_coef

    def set_fragment(self, fixed_mask: Optional[torch.Tensor], x_fix: Optional[torch.Tensor],
                     h_fix: Optional[torch.Tensor]):
        """The atoms the next runs pin (inpainting samplers only): fixed_mask uint8 [n_lig] (nonzero = fixed; None = no
        fixed atom), x_fix [n_lig,3] in the frame of the keypoints passed to run(), h_fix [n_lig,F] in the returned
        feature space.  The tensors must stay alive and in place while runs use them (only their addresses are kept)."""
        if fixed_mask is not None:
            _require_cuda(fixed_mask, x_fix, h_fix)
            assert fixed_mask.dtype == torch.uint8 and x_fix.dtype == torch.float32 and h_fix.dtype == torch.float32
            assert fixed_mask.shape == (self.batch.n_lig,) and x_fix.shape == (self.batch.n_lig, 3)
            assert h_fix.shape == (self.batch.n_lig, self.atom_nf)
            assert fixed_mask.is_contiguous() and x_fix.is_contiguous() and h_fix.is_contiguous()
        check(lib.kpd_sampler_set_fragment(self.handle, ptr(fixed_mask), ptr(x_fix), ptr(h_fix)),
              "kpd_sampler_set_fragment")
        self._fragment = (fixed_mask, x_fix, h_fix)

    def set_start(self, start_step: Optional[int], x_start: Optional[torch.Tensor] = None,
                  h_start: Optional[torch.Tensor] = None, alpha: float = 0.0, sigma: float = 0.0):
        """The ligand the next runs start from (kpd_sampler_set_start): x_start [n_lig,3] in the frame of the keypoints
        passed to run(), h_start [n_lig,F] in the returned feature space, noised to step start_step in [0, T] with
        (alpha, sigma) = schedule.start_coefficients(gamma, start_step); the runs then take start_step reverse steps.
        start_step=None restores the plain start from pure noise.  The tensors must stay alive and in place while runs
        use them (only their addresses are kept)."""
        if start_step is None:
            check(lib.kpd_sampler_set_start(self.handle, 0, None, None, 0.0, 0.0), "kpd_sampler_set_start")
            self._start = None
            return
        _require_cuda(x_start, h_start)
        assert x_start.dtype == torch.float32 and h_start.dtype == torch.float32
        assert x_start.shape == (self.batch.n_lig, 3) and h_start.shape == (self.batch.n_lig, self.atom_nf)
        assert x_start.is_contiguous() and h_start.is_contiguous()
        check(lib.kpd_sampler_set_start(self.handle, int(start_step), ptr(x_start), ptr(h_start), float(alpha),
                                        float(sigma)), "kpd_sampler_set_start")
        self._start = (int(start_step), x_start, h_start)

    def set_schedule(self, coef: Optional[torch.Tensor] = None, coef2: Optional[torch.Tensor] = None):
        """The coefficient rows of the next runs (kpd_sampler_set_schedule; fewer-step sampling, DESIGN.md section 6.3):
        coef fp32 [n,4] on the device, 1 <= n <= T (schedule.coefficient_rows over a step grid) and, for an inpainting
        sampler, coef2 [n,4] (schedule.inpaint_rows over the same grid).  Runs then take n steps (rows n-1 .. 0), or
        start_step of set_start, which counts rows of this schedule.  coef=None restores the create-time tables.  The
        tensors must stay alive and in place while runs use them (only their addresses are kept)."""
        if coef is None:
            check(lib.kpd_sampler_set_schedule(self.handle, 0, None, None), "kpd_sampler_set_schedule")
            self._schedule = None
            return
        n = int(coef.shape[0])
        for c in (coef, coef2) if self.resamplings else (coef,):
            if c is None:
                raise ValueError("an inpainting sampler needs coef2 with its schedule")
            _require_cuda(c)
            assert c.dtype == torch.float32 and c.is_contiguous() and tuple(c.shape) == (n, 4)
        if not 1 <= n <= self.T:
            raise ValueError(f"a schedule has 1 .. {self.T} rows, got {n}")
        check(lib.kpd_sampler_set_schedule(self.handle, n, ptr(coef), ptr(coef2) if self.resamplings else None),
              "kpd_sampler_set_schedule")
        self._schedule = (coef, coef2)

    @property
    def schedule_rows(self) -> int:
        """Rows of the active schedule: T, or n of set_schedule."""
        return self.T if self._schedule is None else int(self._schedule[0].shape[0])

    @property
    def start_step(self) -> int:
        """The row runs start from: the rows of the active schedule, or the start step of set_start."""
        return self.schedule_rows if self._start is None else self._start[0]

    @property
    def noise_slots(self) -> int:
        """Slots of injected noise run() takes, with t0 = start_step: t0+1 (plain) or 1 + t0*(3r-1) (inpainting with r
        resamplings)."""
        t0 = self.start_step
        return t0 + 1 if not self.resamplings else 1 + t0 * (3 * self.resamplings - 1)

    def __del__(self):
        if getattr(self, "handle", None) and self.handle.value and lib is not None:
            lib.kpd_sampler_destroy(self.handle)
            self.handle = C.c_void_p()

    def run(self, x_kp, h_kp, v_kp, init_lig_pos, noise=None, seed=0, n_steps=None, decode=False, record_every=None,
            pred_coef=None):
        """Returns (x_lig [n_lig,3], h_lig [n_lig,F], x_kp) on the device, in the input frame; with decode=True also
        the atom type of every generated atom (int32 [n_lig] = argmax over the feature channels, the first step of
        the reference's output handling, test.py:199-203), written by a kernel enqueued behind the loop.

        record_every = k (recording samplers only) also returns, last, the trajectory of the n_steps executed steps as a
        dict of device tensors with m = ceil(n_steps / k): 'positions' [m+1, n_lig, 3] and 'features' [m+1, n_lig, F]
        (frame j < m: the state before executed step j*k; frame m: the outputs), 'pred_positions' [m, n_lig, 3] and
        'pred_features' [m, n_lig, F] (the clean-ligand estimate of frame j), all in the frame and feature space of the
        outputs.  pred_coef: fp32 [rows, 2] on the device, schedule.prediction_rows over the active schedule's grid."""
        _require_cuda(x_kp, h_kp, init_lig_pos)
        b = self.batch
        x_kp = _f32(x_kp).clone()
        x_lig = torch.empty(b.n_lig, 3, dtype=torch.float32, device=b.device)
        h_lig = torch.empty(b.n_lig, self.atom_nf, dtype=torch.float32, device=b.device)
        n_steps = self.start_step if n_steps is None else int(n_steps)
        if noise is not None:
            _require_cuda(noise)
            assert noise.shape == (self.noise_slots, b.n_lig * (3 + self.atom_nf)) and noise.dtype == torch.float32
        h_kp, init_lig_pos = _f32(h_kp), _f32(init_lig_pos)
        v_kp = _f32(v_kp) if v_kp is not None else None
        frames = None
        if self.record:
            frames = self._set_recording(n_steps, record_every, pred_coef)
        elif record_every is not None:
            raise ValueError("record_every needs a recording sampler (record=True)")
        check(lib.kpd_sampler_run(self.handle, ptr(x_kp), ptr(h_kp), ptr(v_kp) if v_kp is not None else None,
                                  ptr(init_lig_pos), ptr(x_lig), ptr(h_lig), ptr(noise), int(seed), n_steps,
                                  _stream()), "kpd_sampler_run")
        out = (x_lig, h_lig, x_kp) + ((decode_atom_types(h_lig),) if decode else ())
        return out + (frames,) if frames is not None else out

    def _set_recording(self, n_steps: int, every, pred_coef) -> Optional[Dict[str, torch.Tensor]]:
        """Frame buffers of one run (kpd_sampler_set_recording), or recording off when every is None."""
        if every is None:
            check(lib.kpd_sampler_set_recording(self.handle, 1, 0, None, None, None, None, 0, None),
                  "kpd_sampler_set_recording")
            return None
        if isinstance(every, bool) or int(every) != every or every < 1:
            raise ValueError(f"record_every must be an integer >= 1, got {every!r}")
        if pred_coef is None:
            raise ValueError("recording needs pred_coef (schedule.prediction_rows over the active schedule's grid)")
        _require_cuda(pred_coef)
        assert pred_coef.dtype == torch.float32 and pred_coef.is_contiguous() and pred_coef.shape[1:] == (2,)
        every = int(every)
        m = -(-n_steps // every)
        b, F, dev = self.batch, self.atom_nf, self.batch.device
        fr = {"positions": torch.empty(m + 1, b.n_lig, 3, device=dev),
              "features": torch.empty(m + 1, b.n_lig, F, device=dev),
              "pred_positions": torch.empty(m, b.n_lig, 3, device=dev),
              "pred_features": torch.empty(m, b.n_lig, F, device=dev)}
        check(lib.kpd_sampler_set_recording(self.handle, every, m + 1, ptr(fr["positions"]), ptr(fr["features"]),
                                            ptr(fr["pred_positions"]) if m else None,
                                            ptr(fr["pred_features"]) if m else None, int(pred_coef.shape[0]),
                                            ptr(pred_coef)), "kpd_sampler_set_recording")
        self._pred_coef = pred_coef         # read by every recorded step of the run, on the sampler's stream
        return fr

    @property
    def launches_per_step(self):
        return int(lib.kpd_sampler_launches_per_step(self.handle))


# ------------------------------------------------------------------------------------------------------------------
# Capacity-based sampling: capture once per capacity bucket, run any batch that fits.
#
# A captured loop (Sampler) bakes in three kinds of constants: the addresses of its buffers, the node totals
# (B, n_lig, n_kp -> grids, workspace carving) and the edge capacities.  The per-complex structure, on the other
# hand, is DATA: lig_ptr / kp_ptr / lig_batch / kp_batch and the kk CSR are device arrays the kernels read.  So a
# sampler captured for totals (B, N, K) runs ANY batch whose padded layout has exactly those totals: the real
# complexes come first (their global atom indices, hence their Philox noise, and their tile boundaries are those of
# the unpadded batch), followed by a few filler complexes that absorb the spare atoms / keypoints.  Complexes are
# independent (no cross-complex term anywhere in the loop), so the fillers cannot influence the real ones; their
# results are dropped.  Totals are rounded up to coarse granules, so that the sizes drawn by
# LigandSizeDistribution.sample (reference n_nodes_dist.py:42-60; a new draw per call in
# ligand_diffuser.py:490-495) land in a handful of buckets.

def _round_up(v: int, g: int) -> int:
    return (int(v) + g - 1) // g * g


def _pow2_floor(v: int) -> int:
    g = 1
    while g * 2 <= v:
        g *= 2
    return g


def _geometric_bucket(v: int, lo: int = 512) -> int:
    """The smallest value of {lo, 1.5 lo, 2 lo, 3 lo, 4 lo, ...} that is >= v."""
    b = lo
    while True:
        if v <= b:
            return b
        if v <= b + b // 2:
            return b + b // 2
        b *= 2


@dataclass(frozen=True)
class CapacityPlan:
    key: Tuple                       # (B, N, K, max_lig, max_kp, cap_ll, cap_kl, cap_kk)
    lig_n: Tuple[int, ...]           # padded layout: real complexes first, then fillers
    kp_n: Tuple[int, ...]
    n_real: int                      # real complexes
    n_lig_real: int
    n_kp_real: int


def plan_capacity(lig_n: Sequence[int], kp_n: Sequence[int], n_kk_edges: int, gp: "GraphParams") -> CapacityPlan:
    """Capacity bucket + padded layout for a batch (see the comment above).  The bucket is coarse on purpose: node
    totals round up to a granule of ~1/6 of the total (<= ~8 % filler work on average), per-complex maxima to 64 / 8,
    and the edge capacities are functions of the node totals wherever a bound exists, so that ligand sizes drawn
    afresh for every call (LigandSizeDistribution.sample) fall into a few buckets."""
    lig_n = [int(v) for v in lig_n]
    kp_n = [int(v) for v in kp_n]
    B_r, N_r, K_r = len(lig_n), sum(lig_n), sum(kp_n)
    max_lig, max_kp = _round_up(max(lig_n), 64), _round_up(max(kp_n), 8)
    gN, gK = max(8, _pow2_floor(N_r // 6)), max(8, _pow2_floor(K_r // 6))
    N, K = _round_up(N_r + 1, gN), _round_up(K_r + 1, gK)
    while True:
        f_min = max(-(-(N - N_r) // max_lig), -(-(K - K_r) // max_kp), 1)
        B = _round_up(B_r + f_min, 8)
        f = B - B_r
        if f <= N - N_r and f <= K - K_r:
            break
        if f > N - N_r:
            N += gN
        if f > K - K_r:
            K += gK

    def spread(total, parts):
        q, r = divmod(total, parts)
        return [q + (1 if i < r else 0) for i in range(parts)]

    lig_p = lig_n + spread(N - N_r, f)
    kp_p = kp_n + spread(K - K_r, f)
    ll_lim = gp.ll_k if gp.ll_k > 0 else gp.ll_cap
    kl_lim = gp.kl_k if gp.kl_k > 0 else gp.kl_cap
    need_ll = max(sum(n * min(n - 1, ll_lim) for n in lig_p), 1)
    need_kl = max(sum(k * min(n, kl_lim) for n, k in zip(lig_p, kp_p)), 1)
    if gp.ll_k > 0:
        cap_ll = N * gp.ll_k
    else:                                   # radius graph: ~(mean n + var/mean) edges per atom; two levels, then exact
        cap_ll = next((c for c in (32 * N, 64 * N) if c >= need_ll), _geometric_bucket(need_ll))
    bound_kl = K * min(max_lig, kl_lim)
    cap_kl = bound_kl if bound_kl <= 4 * need_kl else _geometric_bucket(need_kl)
    # kk: keypoint models (<= 64 keypoints per complex) take the complete-graph bound, which does not depend on the
    # pockets at hand (spare capacity only costs CTAs that exit at once); all-atom pockets a geometric bucket
    cap_kk = K * (max_kp - 1) if max_kp <= 64 and K * (max_kp - 1) >= n_kk_edges else _geometric_bucket(max(int(n_kk_edges), 1))
    return CapacityPlan((B, N, K, max_lig, max_kp, cap_ll, cap_kl, cap_kk), tuple(lig_p), tuple(kp_p), B_r, N_r, K_r)


class CapacitySampler:
    """A captured reverse-diffusion loop for one capacity bucket (see plan_capacity): owns its layout arrays, kk CSR and
    input buffers; run() rewrites their CONTENTS for the batch at hand and replays the same CUDA graphs.  With
    resamplings >= 1 (and inpaint_coef) it is an inpainting sampler that also owns zero-filled fragment buffers sized at
    capacity: run(fragment=...) fills the rows of the real atoms; filler complexes and atoms are never fixed.  Likewise
    it owns start-ligand buffers at capacity for run(start=...); filler rows stay zero and filler outputs are dropped.
    record=True: a recording sampler (see Sampler); run(record_every=...) returns the frames of the real atoms.
    multistep=True: a DPM-Solver++(2M) sampler (see Sampler) whose history is sized at capacity; run(multistep=...) takes
    the rows of each run."""

    def __init__(self, model: _Model, plan: CapacityPlan, gp: GraphParams, coef: torch.Tensor, T: int, atom_nf: int,
                 kp_width: int, v_width: int, steps_per_graph: int = 50, use_cuda_graph: bool = True,
                 lig_feat_norm_constant: float = 1.0, resamplings: int = 0, inpaint_coef: Optional[torch.Tensor] = None,
                 record: bool = False, multistep: bool = False):
        B, N, K, max_lig, max_kp, cap_ll, cap_kl, cap_kk = plan.key
        dev = model.device
        self.key, self.model, self.atom_nf, self.T = plan.key, model, int(atom_nf), int(T)
        self.batch = DeviceBatch(plan.lig_n, plan.kp_n, dev, max_lig=max_lig, max_kp=max_kp)
        self.has_lk = bool(model.update_kp_feat if model.arch == 0 else model.update_kp)
        self.kk = Csr(K, cap_kk, dev)
        self.x_kp = torch.zeros(K, 3, dtype=torch.float32, device=dev)
        self.h_kp = torch.zeros(K, kp_width, dtype=torch.float32, device=dev)
        self.v_kp = torch.zeros(K, v_width, 3, dtype=torch.float32, device=dev) if v_width else None
        self.init_pos = torch.zeros(B, 3, dtype=torch.float32, device=dev)
        self.sampler = Sampler(model, self.batch, gp, self.kk, coef, T, atom_nf, steps_per_graph=steps_per_graph,
                               use_cuda_graph=use_cuda_graph, lig_feat_norm_constant=lig_feat_norm_constant,
                               caps=(cap_ll, cap_kl), resamplings=resamplings, inpaint_coef=inpaint_coef,
                               record=record, multistep=multistep)
        if self.sampler.resamplings:
            self.fixed_mask = torch.zeros(N, dtype=torch.uint8, device=dev)
            self.x_fix = torch.zeros(N, 3, dtype=torch.float32, device=dev)
            self.h_fix = torch.zeros(N, self.atom_nf, dtype=torch.float32, device=dev)
            self.sampler.set_fragment(self.fixed_mask, self.x_fix, self.h_fix)
        self.x_start = torch.zeros(N, 3, dtype=torch.float32, device=dev)
        self.h_start = torch.zeros(N, self.atom_nf, dtype=torch.float32, device=dev)
        self.runs = 0

    def run(self, plan: CapacityPlan, x_kp, h_kp, v_kp, kk_src, kk_dst, init_pos, seed: int, atom_offset: int = 0,
            noise: Optional[torch.Tensor] = None, decode: bool = False, fragment: Optional[Tuple] = None,
            start: Optional[Tuple] = None, schedule: Optional[Tuple] = None, record_every: Optional[int] = None,
            pred_coef: Optional[torch.Tensor] = None, multistep: Optional[torch.Tensor] = None):
        """x_kp/h_kp/v_kp: the REAL keypoint rows (host or device tensors; pinned host tensors are uploaded straight
        into the capacity buffers); kk_src/kk_dst: kk edges in this batch's own keypoint numbering; init_pos [B_real,3].
        fragment (inpainting samplers): (fixed_mask [N_real] bool, x_fix [N_real,3], h_fix [N_real,F]) or None.
        start: (x [N_real,3], h [N_real,F], t0, alpha_t0, sigma_t0) -- run t0 reverse steps from that ligand (see
        Sampler.set_start) -- or None for the plain start; injected noise then has the slots of a t0-step run.
        schedule: (coef [n,4], coef2 [n,4] or None) on the device -- run the n rows of that schedule (see
        Sampler.set_schedule; t0 of start then counts its rows) -- or None for the create-time tables.  A run-time
        value like the start: no new capture.  record_every / pred_coef (recording samplers): see Sampler.run; pred_coef
        has the rows of the schedule run.  multistep (multistep samplers, required there): ms_coef [n,4] on the device,
        schedule.multistep_rows over the grid of `schedule`, whose coef must be its DDIM eta = 0 rows.
        -> (x_lig [N_real,3], h_lig [N_real,F], x_kp [K_real,3][, atom_type int32 [N_real]][, frames]) on the device,
        frames holding the real atoms only ([m+1, N_real, .] and [m, N_real, .])."""
        if plan.key != self.key:
            raise ValueError("CapacitySampler.run: the plan belongs to another capacity bucket")
        if fragment is not None and not self.sampler.resamplings:
            raise ValueError("CapacitySampler.run: a fragment needs an inpainting sampler")
        if (multistep is not None) != self.sampler.multistep:
            raise ValueError("CapacitySampler.run: multistep rows go with a multistep sampler, and only there")
        B_r, N_r, K_r = plan.n_real, plan.n_lig_real, plan.n_kp_real
        self.batch.set_layout(plan.lig_n, plan.kp_n)
        if self.sampler.resamplings:     # rows past the real atoms stay zero: fillers are never fixed
            self.fixed_mask.zero_()
            if fragment is not None:
                self.fixed_mask[:N_r].copy_(fragment[0], non_blocking=True)
                self.x_fix[:N_r].copy_(fragment[1], non_blocking=True)
                self.h_fix[:N_r].copy_(fragment[2], non_blocking=True)
        if start is not None:            # rows past the real atoms stay zero: filler complexes start from the origin
            self.x_start.zero_()
            self.h_start.zero_()
            self.x_start[:N_r].copy_(start[0], non_blocking=True)
            self.h_start[:N_r].copy_(start[1], non_blocking=True)
            self.sampler.set_start(int(start[2]), self.x_start, self.h_start, float(start[3]), float(start[4]))
        else:
            self.sampler.set_start(None)
        self.sampler.set_schedule(*(schedule or ()))
        if multistep is not None:
            self.sampler.set_multistep(multistep)
        self.x_kp[:K_r].copy_(x_kp, non_blocking=True)
        self.h_kp[:K_r].copy_(h_kp, non_blocking=True)
        if self.v_kp is not None:
            self.v_kp[:K_r].copy_(v_kp, non_blocking=True)
        self.init_pos[:B_r].copy_(init_pos, non_blocking=True)
        if self.has_lk:
            self.kk.fill_from_edges(kk_src, kk_dst)
        check(lib.kpd_sampler_set_atom_offset(self.sampler.handle, int(atom_offset)), "kpd_sampler_set_atom_offset")
        if noise is not None:            # injected draws are laid out for the real atoms: re-lay them for the padded total
            N, F = self.batch.n_lig, self.atom_nf
            pad = torch.zeros(noise.shape[0], N * (3 + F), dtype=torch.float32, device=noise.device)
            pad[:, : N_r * 3] = noise[:, : N_r * 3]
            pad[:, N * 3: N * 3 + N_r * F] = noise[:, N_r * 3:]
            noise = pad
        out = self.sampler.run(self.x_kp, self.h_kp, self.v_kp, self.init_pos, noise=noise, seed=seed, decode=decode,
                               record_every=record_every, pred_coef=pred_coef)
        self.runs += 1
        res = (out[0][:N_r], out[1][:N_r], out[2][:K_r])
        if decode:
            res = res + (out[3][:N_r],)
        if record_every is not None:
            res = res + ({k: v[:, :N_r] for k, v in out[-1].items()},)
        return res
