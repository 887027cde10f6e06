"""Weight packer: reference ``state_dict`` -> one fp32 device blob + offsets for the CUDA library.

Setup-time host code (runs once per model).  Layouts are the ones documented at the top of
csrc/egnn.cu and csrc/gvp.cu: every Linear is stored K-major (transposed) with its output width
padded to a multiple of 4 floats, every entry starts on a 16-byte boundary.

EGNN specifics (reference models/dynamics.py):
  * the first Linear of edge_mlp / coord_mlp (:41, :73) acts on cat(h_src, h_dst, dij); it is
    split into W1a (h_src), W1b (h_dst) and w1c (dij) and the two h blocks of every edge type
    that a node type takes part in are concatenated into one per-node GEMM weight (WpreT), with
    the bias folded into the destination role;
  * H = hidden_nf + 1 (:337-339).
"""
from typing import Dict, List, Tuple

import torch


def _r4(n):
    return (n + 3) // 4 * 4


class _Blob:
    def __init__(self):
        self.parts: List[torch.Tensor] = []
        self.n = 0

    def add(self, t: torch.Tensor) -> int:
        t = t.detach().to(torch.float32).contiguous().reshape(-1).cpu()
        off = self.n
        pad = _r4(t.numel()) - t.numel()
        self.parts.append(t)
        if pad or t.numel() == 0:
            z = torch.zeros(pad if t.numel() else 4)
            self.parts.append(z)
            self.n += z.numel()
        self.n += t.numel()
        return off

    def finish(self, device) -> torch.Tensor:
        return torch.cat(self.parts).to(device)


def _padcols(w: torch.Tensor, ncols: int) -> torch.Tensor:
    out = torch.zeros(w.shape[0], ncols, dtype=torch.float32)
    out[:, : w.shape[1]] = w
    return out


def _padvec(v: torch.Tensor, n: int) -> torch.Tensor:
    out = torch.zeros(n, dtype=torch.float32)
    out[: v.numel()] = v.reshape(-1)
    return out


def _linT(sd, name, ncols=None):
    """K-major (transposed) weight + bias of nn.Linear ``name``, output width padded."""
    w = sd[name + ".weight"].detach().float().cpu()
    n = _r4(w.shape[0]) if ncols is None else ncols
    wt = _padcols(w.t().contiguous(), n)
    b = sd.get(name + ".bias")
    bv = _padvec(b.detach().float().cpu(), n) if b is not None else torch.zeros(n)
    return wt, bv


EGNN_ROLES = {
    # node type -> ordered (edge type, 's'|'d') roles; slot = 2*role + branch
    True: {"lig": [("ll", "s"), ("ll", "d"), ("lk", "s"), ("kl", "d")],
           "kp": [("kl", "s"), ("kk", "s"), ("kk", "d"), ("lk", "d")]},
    False: {"lig": [("ll", "s"), ("ll", "d"), ("kl", "d")], "kp": [("kl", "s")]},
}


def pack_egnn(sd: Dict[str, torch.Tensor], *, atom_nf, rec_nf, hidden_nf, n_layers, update_kp_feat, norm,
              device) -> Tuple[torch.Tensor, List[int]]:
    H = hidden_nf + 1
    Hp = _r4(H)
    hidp = _r4(hidden_nf)
    nmain = min(H, 256) // 4 * 4
    nlo = H - nmain
    blob, offs = _Blob(), []

    def put(t):
        offs.append(blob.add(t))

    w, b = _linT(sd, "lig_encoder.0", 64); put(w); put(b)
    w, b = _linT(sd, "lig_encoder.2", hidp); put(w); put(b)
    if "rec_encoder.0.weight" in sd:
        w, b = _linT(sd, "rec_encoder.0", _r4(2 * rec_nf)); put(w); put(b)
        w, b = _linT(sd, "rec_encoder.2", hidp); put(w); put(b)
    else:
        offs.extend([-1, -1, -1, -1])
    w, b = _linT(sd, "lig_decoder.0", _r4(2 * atom_nf)); put(w); put(b)
    w, b = _linT(sd, "lig_decoder.2", _r4(atom_nf)); put(w); put(b)

    etypes = ["ll", "kl", "lk", "kk"] if update_kp_feat else ["ll", "kl"]
    upd = ["lig", "kp"] if update_kp_feat else ["lig"]
    roles = EGNN_ROLES[bool(update_kp_feat)]
    for l in range(n_layers):
        q = f"egnn.conv_layers.{l}."
        for nt in ("lig", "kp"):
            cols, bias = [], []
            for et, sdir in roles[nt]:
                for mlp in ("edge_mlp", "coord_mlp"):
                    W1 = sd[f"{q}{mlp}.{et}.0.weight"].detach().float().cpu()     # [H, 2H+1]
                    blk = W1[:, :H] if sdir == "s" else W1[:, H:2 * H]
                    cols.append(_padcols(blk.t().contiguous(), Hp))              # [H(in), Hp(out)]
                    bias.append(_padvec(sd[f"{q}{mlp}.{et}.0.bias"].detach().float().cpu(), Hp)
                                if sdir == "d" else torch.zeros(Hp))
            put(torch.cat(cols, dim=1))
            put(torch.cat(bias))
        for et in etypes:
            for mlp in ("edge_mlp", "coord_mlp"):
                W1 = sd[f"{q}{mlp}.{et}.0.weight"].detach().float().cpu()
                put(_padvec(W1[:, 2 * H], Hp))                                     # w1c (dij column)
                W2 = sd[f"{q}{mlp}.{et}.2.weight"].detach().float().cpu()         # [H, H]
                put(_padcols(W2.t().contiguous(), Hp))                             # W2T
                put(_padvec(sd[f"{q}{mlp}.{et}.2.bias"].detach().float().cpu(), Hp))
                lo = torch.zeros(max(3, nlo), Hp)       # nlo > 3 is refused by kpd_egnn_create, with its reason
                if nlo:
                    lo[:nlo, :H] = W2[nmain:H, :]
                put(lo)                                                            # W2lo
            put(_padvec(sd[f"{q}soft_attention.{et}.0.weight"].detach().float().cpu(), Hp))
            put(_padvec(sd[f"{q}soft_attention.{et}.0.bias"].detach().float().cpu(), 4))
            put(_padvec(sd[f"{q}coord_mlp.{et}.4.weight"].detach().float().cpu(), Hp))
        for nt in upd:
            w, b = _linT(sd, f"{q}node_mlp.{nt}.0", Hp); put(w); put(b)            # [2H][Hp]
            w, b = _linT(sd, f"{q}node_mlp.{nt}.2", Hp); put(w); put(b)            # [H][Hp]
            if norm:
                put(_padvec(sd[f"{q}layer_norm.{nt}.weight"].detach().float().cpu(), Hp))
                put(_padvec(sd[f"{q}layer_norm.{nt}.bias"].detach().float().cpu(), Hp))
            else:
                offs.extend([-1, -1])
    return blob.finish(device), offs


def gvp_layer_etypes(l, n_convs, update_kp):
    """reference models/dynamics_gvp.py:65-74: the last conv of an update_kp model is lig-only."""
    base = [("lig", "ll", "lig"), ("kp", "kl", "lig")]
    if (not update_kp) or l == n_convs - 1:
        return base
    return base + [("lig", "lk", "kp"), ("kp", "kk", "kp")]


def pack_gvp(sd: Dict[str, torch.Tensor], *, n_lig_scalars, n_kp_scalars, vector_size, n_convs,
             n_hidden_scalars, update_kp, n_message_gvps, n_update_gvps, n_noise_gvps,
             device) -> Tuple[torch.Tensor, List[int]]:
    blob, offs = _Blob(), []

    def put(t):
        offs.append(blob.add(t))

    def put_gvp(name):
        put(sd[name + ".Wh"])
        put(sd[name + ".Wu"])
        w, b = _linT(sd, name + ".to_feats_out.0"); put(w); put(b)
        put(sd[name + ".scalar_to_vector_gates.weight"].detach().float().cpu().t().contiguous())   # [fout][vout]
        put(sd[name + ".scalar_to_vector_gates.bias"])

    for enc in ("lig_encoder", "kp_encoder"):
        w, b = _linT(sd, enc + ".0", n_hidden_scalars); put(w); put(b)
        put(sd[enc + ".2.weight"]); put(sd[enc + ".2.bias"])
    for l in range(n_convs):
        q = f"noise_predictor.conv_layers.{l}."
        etypes = gvp_layer_etypes(l, n_convs, update_kp)
        for et in etypes:
            for i in range(n_message_gvps):
                put_gvp(f"{q}edge_message_fns.{'_'.join(et)}.{i}")
        for nt in (["lig", "kp"] if len(etypes) == 4 else ["lig"]):
            for i in range(n_update_gvps):
                put_gvp(f"{q}node_update_fns.{nt}.{i}")
            put(sd[f"{q}message_layer_norms.{nt}.feat_norm.weight"]); put(sd[f"{q}message_layer_norms.{nt}.feat_norm.bias"])
            put(sd[f"{q}update_layer_norms.{nt}.feat_norm.weight"]); put(sd[f"{q}update_layer_norms.{nt}.feat_norm.bias"])
    q = "noise_predictor.noise_predictor."
    for i in range(n_noise_gvps):
        put_gvp(f"{q}gvps.{i}")
    w, b = _linT(sd, q + "to_scalar_output"); put(w); put(b)
    return blob.finish(device), offs


def pack_egnn_tc(sd: Dict[str, torch.Tensor], *, hidden_nf, n_layers, update_kp_feat, device,
                 split: bool = True) -> Tuple[torch.Tensor, List[int]]:
    """Tensor-core weights of the EGNN (csrc/egnn.cu kpd_egnn_attach_tc), packed with pack_tc_weight: per layer the
    per-node first-layer weight of lig and kp ([slots * Hp, H], same column order as pack_egnn's WpreT), per edge type
    the second Linear of edge_mlp and coord_mlp (output rows [0, nmain)), per updated node type node_mlp.0 / .2."""
    H = hidden_nf + 1
    Hp = _r4(H)
    nmain = min(H, 256) // 4 * 4
    etypes = ["ll", "kl", "lk", "kk"] if update_kp_feat else ["ll", "kl"]
    upd = ["lig", "kp"] if update_kp_feat else ["lig"]
    roles = EGNN_ROLES[bool(update_kp_feat)]
    parts, offs, n = [], [], 0

    def add(w):
        nonlocal n
        t = pack_tc_weight(w, split)
        pad = (-t.numel()) % 64
        offs.append(2 * n)
        parts.append(t)
        if pad:
            parts.append(torch.zeros(pad, dtype=torch.bfloat16))
        n += t.numel() + pad

    for l in range(n_layers):
        q = f"egnn.conv_layers.{l}."
        for nt in ("lig", "kp"):
            rows = []
            for et, sdir in roles[nt]:
                for mlp in ("edge_mlp", "coord_mlp"):
                    W1 = sd[f"{q}{mlp}.{et}.0.weight"].detach().float().cpu()     # [H, 2H+1]
                    blk = torch.zeros(Hp, H)
                    blk[:H] = W1[:, :H] if sdir == "s" else W1[:, H:2 * H]
                    rows.append(blk)                                               # one slot: Hp output rows
            add(torch.cat(rows, dim=0))
        for et in etypes:
            for mlp in ("edge_mlp", "coord_mlp"):
                add(sd[f"{q}{mlp}.{et}.2.weight"].detach().float().cpu()[:nmain, :])
        for nt in upd:
            # the tensor-core node stage stores cat = [h (H) | zero gap up to Hp | h_neigh (H)]: matching zero columns
            W1 = sd[f"{q}node_mlp.{nt}.0.weight"].detach().float().cpu()           # [H, 2H]
            add(torch.cat([W1[:, :H], torch.zeros(H, Hp - H), W1[:, H:]], dim=1))
            add(sd[f"{q}node_mlp.{nt}.2.weight"].detach().float().cpu())
    return torch.cat(parts).to(device), offs


def _tc_block(wp: torch.Tensor, split: bool) -> torch.Tensor:
    """[NB, ks*16] fp32 -> k-step slabs [ks][hi(, lo)][2 k-chunks][NB/8][8 rows][8] bf16."""
    NB, K16 = wp.shape
    ks = K16 // 16

    def slabs(x):
        return x.view(NB // 8, 8, ks, 2, 8).permute(2, 3, 0, 1, 4).contiguous().view(ks, 1, -1)

    hi = wp.to(torch.bfloat16)
    if not split:
        return slabs(hi).reshape(-1)
    lo = (wp - hi.float()).to(torch.bfloat16)
    return torch.cat([slabs(hi), slabs(lo)], dim=1).reshape(-1)


def pack_tc_weight(w: torch.Tensor, split: bool = False) -> torch.Tensor:
    """nn.Linear weight [N, K] -> bf16 "k-step slabs" for the tcgen05 kernels (csrc/tc.cuh):
    for every k-step of 16 input features, 2 k-chunks x (NB/8) row groups x (8 rows x 8 bf16 = 128 B), i.e. the
    no-swizzle K-major canonical UMMA layout, so one slab is one contiguous bulk copy.  K is padded to a multiple
    of 16 with zeros.  Output rows are packed in blocks of 256 (UMMA N <= 256); the last block is padded to a
    multiple of 16 rows (NB).  split=True interleaves, per k-step, the slab of hi = bf16(w) and the slab of
    lo = bf16(w - hi) (the bf16x3 mode)."""
    w = w.detach().float().cpu()
    N, K = w.shape
    ks = (K + 15) // 16
    parts = []
    for n0 in range(0, N, 256):
        n = min(256, N - n0)
        NB = (n + 15) // 16 * 16
        wp = torch.zeros(NB, ks * 16)
        wp[:n, :K] = w[n0:n0 + n]
        parts.append(_tc_block(wp, split))
    return torch.cat(parts)


def pack_gvp_tc(sd: Dict[str, torch.Tensor], *, n_convs, update_kp, n_message_gvps, n_update_gvps, n_noise_gvps,
                device, split: bool = False) -> Tuple[torch.Tensor, List[int]]:
    """bf16 tensor-core weights of every GVP, in the library's creation order (csrc/gvp.cu kpd_gvp_attach_tc):
    per conv the message GVPs per edge type, then the update GVPs per node type; then the noise head.
    Three entries per GVP: to_feats_out (rows padded to 16), scalar_to_vector_gates (rows padded to 16) and the
    shared-memory image of its small fp32 weights (pack_gvp_small).
    split=True packs (hi, lo) slab pairs for the bf16x3 mode.
    Returns one bf16 device blob (every entry 128-byte aligned) and byte offsets."""
    names = []
    for l in range(n_convs):
        q = f"noise_predictor.conv_layers.{l}."
        etypes = gvp_layer_etypes(l, n_convs, update_kp)
        for et in etypes:
            names += [f"{q}edge_message_fns.{'_'.join(et)}.{i}" for i in range(n_message_gvps)]
        for nt in (["lig", "kp"] if len(etypes) == 4 else ["lig"]):
            names += [f"{q}node_update_fns.{nt}.{i}" for i in range(n_update_gvps)]
    names += [f"noise_predictor.noise_predictor.gvps.{i}" for i in range(n_noise_gvps)]
    parts, offs, n = [], [], 0

    def add(t):
        nonlocal n
        pad = (-t.numel()) % 64                      # 64 bf16 = 128 bytes
        offs.append(2 * n)
        parts.append(t)
        if pad:
            parts.append(torch.zeros(pad, dtype=torch.bfloat16))
        n += t.numel() + pad

    for name in names:
        wf = sd[name + ".to_feats_out.0.weight"]
        add(pack_tc_weight(wf, split))
        # gates weight: tcgen05 slabs in the bf16 mode; mma.sync B fragments in the bf16x3 mode (the gates GEMM then
        # runs on the warp-level tensor cores straight from the epilogue registers)
        wg = sd[name + ".scalar_to_vector_gates.weight"]
        # (split: followed by the (hi, lo) tcgen05 slabs of the same weight, which the KS edge kernel streams through its ring)
        add(torch.cat([pack_gates_frag(wg), pack_gates_ks(wg)]) if split else pack_tc_weight(wg, False))
        # message GVP 0 of every edge type takes the unit x_diff as its first input vector channel
        xfirst = ".edge_message_fns." in name and name.endswith(".0")
        img = pack_gvp_small(sd[name + ".Wh"], sd[name + ".Wu"], sd[name + ".to_feats_out.0.bias"],
                             sd[name + ".scalar_to_vector_gates.bias"], xfirst, split)
        if split:       # followed by the plain fp32 image the KS edge kernel's FP32-pipe vector GEMMs read
            img = torch.cat([img, pack_gvp_small_ks(sd[name + ".Wh"], sd[name + ".Wu"], sd[name + ".to_feats_out.0.bias"],
                                                    sd[name + ".scalar_to_vector_gates.bias"], xfirst)])
        add(img.view(torch.bfloat16))                # fp32 image carried in the bf16 blob (two bf16 per float)
    return torch.cat(parts).to(device), offs


def pack_gates_ks(wg: torch.Tensor, n_col_groups: int = 4) -> torch.Tensor:
    """scalar_to_vector_gates.weight for the KS edge kernel (csrc/gvp_ws.inl issue_ks): the (hi, lo) tcgen05 k-step slabs
    of pack_tc_weight(split=True) -- 512 B hi + 512 B lo per k-step -- reordered so that the k-steps over the FIRST halves of
    the epilogue's column groups (256 / n_col_groups columns each) come first: the issuer runs those as soon as epilogue 1
    is half way."""
    slabs = pack_tc_weight(wg, True).view(-1, 512)          # [ks][512 bf16 = 1 KB]
    cpw = 256 // n_col_groups
    first = [j for j in range(slabs.shape[0]) if (16 * j) % cpw < cpw // 2]
    rest = [j for j in range(slabs.shape[0]) if j not in first]
    return slabs[first + rest].reshape(-1)


def pack_gates_frag(wg: torch.Tensor) -> torch.Tensor:
    """scalar_to_vector_gates.weight [vout <= 16, fout] -> m16n8k16 bf16 B fragments for csrc/gvp_ws.inl gates_mma:
    [hi | lo][k16 step S][t][n'][2 words], word 0 = (W[n][16S+2t], W[n][16S+2t+1]), word 1 = (W[n][16S+2t+8], +9) as bf16
    pairs (low half = even k), n' = (n + 4t) & 15 (bank swizzle); hi = bf16(W), lo = bf16(W - hi).  Same byte size as
    the tcgen05 packing (ksg * 512 B per plane)."""
    w = wg.detach().float().cpu()
    vout, fout = w.shape
    ks = (fout + 15) // 16
    full = torch.zeros(16, ks * 16)
    full[:vout, :fout] = w
    hi = full.to(torch.bfloat16).float()
    planes = []
    for plane in (hi, full - hi):
        b = plane.to(torch.bfloat16).view(torch.int16).to(torch.int64) & 0xFFFF          # [16][ks*16] bf16 bits
        words = torch.zeros(ks, 4, 16, 2, dtype=torch.int64)
        for t in range(4):
            for n in range(16):
                nsw = (n + 4 * t) & 15
                for half in range(2):
                    k = 2 * t + 8 * half
                    words[:, t, nsw, half] = b[n, k::16] | (b[n, k + 1::16] << 16)
        words = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)
        planes.append(words.reshape(-1))
    return torch.cat(planes).view(torch.bfloat16)


# shared-memory image of the small fp32 weights of one GVP (csrc/gvp_ws.inl: ws::WH_LD, WU_LD, wsm_floats)
_WH_LD, _WU_LD = 36, 20
_WH_SZ, _WU_SZ = 12 * _WH_LD * 2, 12 * _WU_LD * 2


def _tf32_rna(x: torch.Tensor) -> torch.Tensor:
    """cvt.rna.tf32.f32: round to nearest, ties away, keeping 10 mantissa bits."""
    b = x.contiguous().view(torch.int32)
    mag = (b & 0x7FFFFFFF) + 0x1000
    return ((mag & ~0x1FFF) | (b & -0x80000000)).view(torch.float32)


_WH_LD_KS, _WU_LD_KS = 28, 20


def pack_gvp_small_ks(Wh, Wu, bf, bg, xfirst: bool) -> torch.Tensor:
    """The small weights of one GVP for the KS edge kernel (csrc/gvp_ws.inl vec_fma): Wh [vin, h] and Wu [h, vout] as plain
    fp32 [24][28] / [24][20] images (zero padded), then the to_feats_out bias padded to 256 and the gates bias padded to 16.
    xfirst: the kernel keeps the x_diff channel LAST, so Wh's rows are rotated (as in pack_gvp_small)."""
    Wh, Wu = Wh.detach().float().cpu(), Wu.detach().float().cpu()
    if xfirst:
        Wh = torch.cat([Wh[1:], Wh[:1]])
    ih = torch.zeros(24, _WH_LD_KS)
    ih[:Wh.shape[0], :Wh.shape[1]] = Wh
    iu = torch.zeros(24, _WU_LD_KS)
    iu[:Wu.shape[0], :Wu.shape[1]] = Wu
    b1 = torch.zeros(256)
    b1[:bf.numel()] = bf.detach().float().cpu()
    b2 = torch.zeros(16)
    b2[:bg.numel()] = bg.detach().float().cpu()
    return torch.cat([ih.reshape(-1), iu.reshape(-1), b1, b2])


def pack_gvp_small(Wh, Wu, bf, bg, xfirst: bool, split: bool) -> torch.Tensor:
    """Wh [vin, h] and Wu [h, vout] as mma.sync B fragments (pairs of consecutive K rows interleaved, tf32-rounded;
    with split=True followed by the tf32 residuals for the 3xTF32 mode), then the to_feats_out bias padded to 256 and
    the gates bias padded to 16.  xfirst: the kernel keeps the x_diff channel LAST, so Wh's rows are rotated."""
    Wh, Wu = Wh.detach().float().cpu(), Wu.detach().float().cpu()
    vin, hd = Wh.shape
    vout = Wu.shape[1]
    if xfirst:
        Wh = torch.cat([Wh[1:], Wh[:1]])
    ns = 2 if split else 1

    def frag(W, ld):
        K, N = W.shape
        full = torch.zeros(24, ld)
        full[:K, :N] = W
        return full.view(12, 2, ld).permute(0, 2, 1).contiguous().reshape(-1)     # [pair][n][2]

    out = []
    for W, ld in ((Wh, _WH_LD), (Wu, _WU_LD)):
        f = frag(W, ld)
        hi = _tf32_rna(f)
        out.append(hi)
        if split:
            out.append(_tf32_rna(f - hi))
    b1 = torch.zeros(256)
    b1[:bf.numel()] = bf.detach().float().cpu()
    b2 = torch.zeros(16)
    b2[:bg.numel()] = bg.detach().float().cpu()
    img = torch.cat(out + [b1, b2])
    assert img.numel() == ns * (_WH_SZ + _WU_SZ) + 272
    return img
