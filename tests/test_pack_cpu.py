"""CPU: the host-side weight packers for the tensor-core kernels (pack.py) -- layouts are what the
kernels' descriptors and fragment loads assume (csrc/tc.cuh, csrc/ws_common.cuh, csrc/gvp_ws.inl)."""
import torch

from keypoint_diffusion_b200 import pack


def _unpack_block(blob, NB, ks, split):
    """inverse of pack._tc_block for one <=256-row block: -> (hi, lo) [NB, ks*16] float tensors"""
    ns = 2 if split else 1
    x = blob.view(ks, ns, 2, NB // 8, 8, 8).float()                    # [ks][hi/lo][k-chunk][row group][row][8]
    out = []
    for p in range(ns):
        w = x[:, p].permute(2, 3, 0, 1, 4).reshape(NB, ks * 16)        # rows, then (ks, chunk, 8) columns
        out.append(w)
    return out


def test_pack_tc_weight_layout_and_split():
    g = torch.Generator().manual_seed(0)
    for (N, K) in [(16, 16), (40, 33), (256, 289), (257, 257), (520, 70)]:
        w = torch.randn(N, K, generator=g)
        ks = (K + 15) // 16
        for split in (False, True):
            blob = pack.pack_tc_weight(w, split)
            assert blob.dtype == torch.bfloat16
            off = 0
            for n0 in range(0, N, 256):
                n = min(256, N - n0)
                NB = (n + 15) // 16 * 16
                size = ks * (2 if split else 1) * 2 * (NB // 8) * 64
                parts = _unpack_block(blob[off:off + size], NB, ks, split)
                off += size
                ref = torch.zeros(NB, ks * 16)
                ref[:n, :K] = w[n0:n0 + n]
                hi = ref.to(torch.bfloat16).float()
                assert torch.equal(parts[0], hi)                         # hi plane = bf16(w), zero padded
                if split:
                    assert torch.equal(parts[1], (ref - hi).to(torch.bfloat16).float())
                    # hi + lo carries ~16 mantissa bits
                    assert (parts[0] + parts[1] - ref).abs().max() <= ref.abs().max() * 2.0 ** -16
            assert off == blob.numel()


def test_tf32_rounding_matches_cvt_rna():
    x = torch.tensor([1.0, 1.0 + 2.0 ** -11, 1.0 + 2.0 ** -10, -(1.0 + 3 * 2.0 ** -12), 0.0, 3.0e-5])
    y = pack._tf32_rna(x)
    assert torch.equal(y, torch.tensor([1.0, 1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10, -(1.0 + 2.0 ** -10), 0.0,
                                        float(torch.tensor(3.0e-5).view(torch.int32).add(0x1000).bitwise_and(~0x1FFF)
                                              .view(torch.float32))]))
    assert ((y.view(torch.int32) & 0x1FFF) == 0).all()                   # 13 low mantissa bits cleared


def test_pack_gvp_small_fragment_layout():
    """Wh / Wu staged as mma.sync m16n8k8 B fragments: element (k, n) at ((k // 2) * LD + n) * 2 + k % 2; the
    message GVP's x_diff row is rotated to the last input channel; biases follow, zero padded."""
    g = torch.Generator().manual_seed(1)
    vin, hd, vout = 17, 17, 16
    Wh, Wu = torch.randn(vin, hd, generator=g), torch.randn(hd, vout, generator=g)
    bf, bg = torch.randn(256, generator=g), torch.randn(vout, generator=g)
    for split in (False, True):
        img = pack.pack_gvp_small(Wh, Wu, bf, bg, xfirst=True, split=split)
        ns = 2 if split else 1
        assert img.numel() == ns * (pack._WH_SZ + pack._WU_SZ) + 272
        wh = img[:pack._WH_SZ].view(12, pack._WH_LD, 2)
        rot = torch.cat([Wh[1:], Wh[:1]])                                # our channel k <- reference row k + 1; last <- row 0
        for k in (0, 5, 16):
            for n in (0, 7, 16):
                assert wh[k // 2, n, k % 2] == pack._tf32_rna(rot[k, n].reshape(1))[0]
        assert wh[9:].abs().sum() == 0 and wh[:, hd:].abs().sum() == 0   # K and N padding are zeros
        wu = img[ns * pack._WH_SZ: ns * pack._WH_SZ + pack._WU_SZ].view(12, pack._WU_LD, 2)
        assert wu[8, 3, 0] == pack._tf32_rna(Wu[16, 3].reshape(1))[0]
        if split:
            lo = img[pack._WH_SZ:2 * pack._WH_SZ].view(12, pack._WH_LD, 2)
            k, n = 3, 4
            assert abs(float(wh[k // 2, n, k % 2] + lo[k // 2, n, k % 2] - rot[k, n])) <= abs(float(rot[k, n])) * 2.0 ** -20
        b = img[ns * (pack._WH_SZ + pack._WU_SZ):]
        assert torch.equal(b[:256], bf) and torch.equal(b[256:256 + vout], bg)


def test_pack_egnn_tc_entries():
    """one packed entry per tensor-core GEMM of the EGNN, in the order kpd_egnn_attach_tc reads them"""
    from oracle import params as P
    hidden, layers = 32, 2
    shapes = P.egnn_dynamics_shapes(10, 12, layers, hidden, True, True)
    sd = P.init_state_dict(shapes, seed=0)
    sd = {k[len("dynamics."):] if k.startswith("dynamics.") else k: v for k, v in sd.items()}
    blob, offs = pack.pack_egnn_tc(sd, hidden_nf=hidden, n_layers=layers, update_kp_feat=True, device="cpu", split=True)
    assert len(offs) == layers * (2 + 4 * 2 + 2 * 2)
    assert all(o % 128 == 0 for o in offs) and offs == sorted(offs)
    H, Hp = hidden + 1, 36
    ks = (H + 15) // 16
    # first entry: the ligand per-node first-layer weight, 8 slots x Hp rows, K = H
    first = offs[1] - offs[0]
    n_rows = 8 * Hp
    full_blocks, tail = divmod(n_rows, 256)
    expect = (full_blocks * 256 + (tail + 15) // 16 * 16) * ks * 16 * 2 * 2          # bf16 bytes, hi + lo
    assert first == (expect + 127) // 128 * 128


def _slab_bytes(n_rows, K, split=True):
    """Bytes of pack_tc_weight of an [n_rows, K] weight, padded to the 128-byte entry alignment."""
    ks = (K + 15) // 16
    rows = sum((min(256, n_rows - n0) + 15) // 16 * 16 for n0 in range(0, n_rows, 256))
    return (rows * ks * 16 * (2 if split else 1) * 2 + 127) // 128 * 128


def test_egnn_tensor_core_rule_and_pack_at_every_width():
    """hidden_nf 1..259: the tensor-core modes are attached exactly for 8 <= H <= 257 with H % 8 < 4 (nmain = H & ~3 a
    non-zero multiple of 8); hidden_nf 1 and 2 (nmain = 0) fall back to fp32.  At every such width pack_egnn_tc gives
    one entry per GEMM, the edge GEMMs nmain output rows padded to 16."""
    from oracle import params as P
    from keypoint_diffusion_b200 import ops
    accepted = []
    for hid in range(1, 260):
        H = hid + 1
        tc = ops.egnn_has_tc_tiles(hid)
        assert tc == (8 <= H <= 257 and H % 8 < 4), hid
        if not tc:
            continue
        accepted.append(hid)
        kp = hid % 2 == 0
        sd = P.init_state_dict(P.egnn_dynamics_shapes(3, 5, 1, hid, kp, False), seed=hid)
        sd = {k[len("dynamics."):]: v for k, v in sd.items()}
        blob, offs = pack.pack_egnn_tc(sd, hidden_nf=hid, n_layers=1, update_kp_feat=kp, device="cpu", split=True)
        n_et, n_upd = (4, 2) if kp else (2, 1)
        assert len(offs) == 2 + 2 * n_et + 2 * n_upd and all(o % 128 == 0 for o in offs), hid
        nmain, Hp = min(H, 256) // 4 * 4, (H + 3) // 4 * 4
        sizes = [b - a for a, b in zip(offs, offs[1:] + [2 * blob.numel()])]
        assert sizes[2:2 + 2 * n_et] == [_slab_bytes(nmain, H)] * (2 * n_et), hid
        assert sizes[2 + 2 * n_et:] == [_slab_bytes(H, 2 * Hp), _slab_bytes(H, H)] * n_upd, hid
    assert accepted[0] == 7 and accepted[-1] == 256 and 255 in accepted and 257 not in accepted
    assert 36 not in accepted and 1 not in accepted and 2 not in accepted


def test_gvp_tensor_core_rule_and_pack_at_every_width():
    """S = 4..256 step 4, V in {1, 16}, rbf_dim in {2, 32}: the tensor-core modes exactly at S % 16 == 0; there
    pack_gvp_tc gives three 128-byte-aligned entries per GVP, to_feats_out padded to 16 rows over K = hd + fin."""
    from oracle import params as P
    from keypoint_diffusion_b200 import ops
    for S in range(4, 257, 4):
        assert ops.gvp_has_tc_tiles(S) == (S % 16 == 0)
        if S % 16:
            continue
        for V in (1, 16):
            for rbf in (2, 32):
                sd = P.init_state_dict(P.gvp_dynamics_shapes(10, 12, V, 1, S, False, 1, 1, 1, rbf_dim=rbf), seed=S)
                sd = {k[len("dynamics."):]: v for k, v in sd.items()}
                blob, offs = pack.pack_gvp_tc(sd, n_convs=1, update_kp=False, n_message_gvps=1, n_update_gvps=1,
                                              n_noise_gvps=1, device="cpu", split=True)
                assert len(offs) == 3 * 4 and all(o % 128 == 0 for o in offs), (S, V, rbf)
                # GVP order: message ll, message kl, update lig, head; to_feats_out [fout, hd + fin]
                expect = [(S, V + 1 + S + rbf), (S, V + 1 + S + rbf), (S, V + S), (64, V + S)]
                for g, (fout, K) in enumerate(expect):
                    assert offs[3 * g + 1] - offs[3 * g] == _slab_bytes(fout, K), (S, V, rbf, g)
