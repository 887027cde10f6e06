"""Thin Python wrappers over the C ABI (include/kpdiff_b200.h): batch layout, graph build,
denoiser forward, posterior step and the captured sampling loop.

torch is used for device memory and streams only; every computation below is a call into
libkpdiff_b200.so.  All tensors must live on one CUDA device (no CPU fallback).
"""
import ctypes as C
import os
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
        H = hidden_nf + 1
        if (min(H, 256) // 4 * 4) % 8 == 0 and H <= 257:
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
        if n_hidden_scalars % 16 == 0:
            kw = dict(n_convs=n_convs, update_kp=update_kp, n_message_gvps=n_message_gvps, n_update_gvps=n_update_gvps,
                      n_noise_gvps=n_noise_gvps, device=self.device)
            self.tc_blob, toffs = pack.pack_gvp_tc(sd, **kw)
            tarr = (C.c_int64 * len(toffs))(*toffs)
            check(lib.kpd_gvp_attach_tc(self.handle, ptr(self.tc_blob), tarr, len(toffs), 1), "kpd_gvp_attach_tc")
            # KPD_EDGE_PAIR=1: pair-packed message weights for a library built with -DKPD_EDGE_PAIR (experimental
            # cta_group::2 edge kernel; measured slower than the single-CTA kernel, DESIGN.md 4.3)
            self.tc_blob2, toffs = pack.pack_gvp_tc(sd, split=True, pair=os.environ.get("KPD_EDGE_PAIR", "0") == "1", **kw)
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
    """The captured reverse-diffusion loop for one (model, batch) pair (kpd_sampler)."""

    def __init__(self, model: _Model, batch: DeviceBatch, gp: GraphParams, kk: Optional[Csr], coef: torch.Tensor,
                 T: int, atom_nf: int, steps_per_graph: int = 50, use_cuda_graph: bool = True,
                 lig_feat_norm_constant: float = 1.0, atom_offset: int = 0, caps: Optional[Tuple[int, int]] = None):
        self.model, self.batch, self.gp, self.kk, self.coef = model, batch, gp, kk, coef
        _require_cuda(coef)
        self.T, self.atom_nf = int(T), int(atom_nf)
        self.has_lk = bool(model.update_kp_feat if model.arch == 0 else model.update_kp)
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

    def __del__(self):
        if getattr(self, "handle", None) and self.handle.value and lib is not None:
            lib.kpd_sampler_destroy(self.handle)
            self.handle = C.c_void_p()

    def run(self, x_kp, h_kp, v_kp, init_lig_pos, noise=None, seed=0, n_steps=None, decode=False):
        """Returns (x_lig [n_lig,3], h_lig [n_lig,F], x_kp) on the device, in the input frame; with decode=True also
        the atom type of every generated atom (int32 [n_lig] = argmax over the feature channels, the first step of
        the reference's output handling, test.py:199-203), written by a kernel enqueued behind the loop."""
        _require_cuda(x_kp, h_kp, init_lig_pos)
        b = self.batch
        x_kp = _f32(x_kp).clone()
        x_lig = torch.empty(b.n_lig, 3, dtype=torch.float32, device=b.device)
        h_lig = torch.empty(b.n_lig, self.atom_nf, dtype=torch.float32, device=b.device)
        n_steps = self.T if n_steps is None else int(n_steps)
        if noise is not None:
            _require_cuda(noise)
            assert noise.shape == (self.T + 1, b.n_lig * (3 + self.atom_nf)) and noise.dtype == torch.float32
        h_kp, init_lig_pos = _f32(h_kp), _f32(init_lig_pos)
        v_kp = _f32(v_kp) if v_kp is not None else None
        check(lib.kpd_sampler_run(self.handle, ptr(x_kp), ptr(h_kp), ptr(v_kp) if v_kp is not None else None,
                                  ptr(init_lig_pos), ptr(x_lig), ptr(h_lig), ptr(noise), int(seed), n_steps,
                                  _stream()), "kpd_sampler_run")
        if decode:
            return x_lig, h_lig, x_kp, decode_atom_types(h_lig)
        return x_lig, h_lig, x_kp

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
    input buffers; run() rewrites their CONTENTS for the batch at hand and replays the same CUDA graphs."""

    def __init__(self, model: _Model, plan: CapacityPlan, gp: GraphParams, coef: torch.Tensor, T: int, atom_nf: int,
                 kp_width: int, v_width: int, steps_per_graph: int = 50, use_cuda_graph: bool = True,
                 lig_feat_norm_constant: float = 1.0):
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
                               caps=(cap_ll, cap_kl))
        self.runs = 0

    def run(self, plan: CapacityPlan, x_kp, h_kp, v_kp, kk_src, kk_dst, init_pos, seed: int, atom_offset: int = 0,
            noise: Optional[torch.Tensor] = None, decode: bool = False):
        """x_kp/h_kp/v_kp: the REAL keypoint rows (host or device tensors; pinned host tensors are uploaded straight
        into the capacity buffers); kk_src/kk_dst: kk edges in this batch's own keypoint numbering; init_pos [B_real,3].
        -> (x_lig [N_real,3], h_lig [N_real,F], x_kp [K_real,3][, atom_type int32 [N_real]]) on the device."""
        if plan.key != self.key:
            raise ValueError("CapacitySampler.run: the plan belongs to another capacity bucket")
        B_r, N_r, K_r = plan.n_real, plan.n_lig_real, plan.n_kp_real
        self.batch.set_layout(plan.lig_n, plan.kp_n)
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
        out = self.sampler.run(self.x_kp, self.h_kp, self.v_kp, self.init_pos, noise=noise, seed=seed, decode=decode)
        self.runs += 1
        res = (out[0][:N_r], out[1][:N_r], out[2][:K_r])
        return res + (out[3][:N_r],) if decode else res
