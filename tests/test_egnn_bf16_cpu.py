"""CPU: the host side of the EGNN 'bf16' mode -- the precision is accepted by the module, and the plain-bf16 pack holds,
entry for entry, pack_tc_weight(w, split=False) of the same weights the bf16x3 pack splits."""
import pytest
import torch

from keypoint_diffusion_b200 import pack


def test_egnn_dynamics_accepts_bf16_and_rejects_unknown_modes():
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.dynamics import LigRecDynamics
    assert set(ops.EgnnModel.PRECISIONS) == {"fp32", "bf16", "bf16x3"}
    dyn = LigRecDynamics(10, 12, n_layers=1, hidden_nf=32)
    assert dyn.precision == "bf16x3"
    for mode in ("bf16", "fp32", "bf16x3", "bf16"):
        dyn.set_precision(mode)
        assert dyn.precision == mode
    for bad in ("fp16", "BF16", "tf32", ""):
        with pytest.raises(ValueError):
            dyn.set_precision(bad)
    assert dyn.precision == "bf16"


def test_pack_egnn_tc_plain_entries_match_pack_tc_weight():
    from oracle import params as P
    hidden, layers = 32, 2
    H, Hp = hidden + 1, 36
    nmain = min(H, 256) // 4 * 4
    sd = P.init_state_dict(P.egnn_dynamics_shapes(10, 12, layers, hidden, True, True), seed=0)
    sd = {k[len("dynamics."):] if k.startswith("dynamics.") else k: v for k, v in sd.items()}
    blob, offs = pack.pack_egnn_tc(sd, hidden_nf=hidden, n_layers=layers, update_kp_feat=True, device="cpu", split=False)
    _, offs2 = pack.pack_egnn_tc(sd, hidden_nf=hidden, n_layers=layers, update_kp_feat=True, device="cpu", split=True)
    assert len(offs) == len(offs2) == layers * (2 + 4 * 2 + 2 * 2)
    assert all(o % 128 == 0 for o in offs) and offs == sorted(offs)

    def entry(i, ref):
        b0 = offs[i] // 2
        got = blob[b0:b0 + ref.numel()]
        assert torch.equal(got.view(torch.int16), ref.view(torch.int16)), i
        end = offs[i + 1] // 2 if i + 1 < len(offs) else blob.numel()
        assert end - b0 == (ref.numel() + 63) // 64 * 64, i       # padded to 128 bytes, nothing else

    per_layer = 2 + 4 * 2 + 2 * 2
    for l in range(layers):
        q = f"egnn.conv_layers.{l}."
        i = l * per_layer + 2          # (entries 0, 1: the per-node first-layer weights of lig and kp)
        for et in ("ll", "kl", "lk", "kk"):
            for mlp in ("edge_mlp", "coord_mlp"):
                entry(i, pack.pack_tc_weight(sd[f"{q}{mlp}.{et}.2.weight"][:nmain], False))
                i += 1
        for nt in ("lig", "kp"):
            W1 = sd[f"{q}node_mlp.{nt}.0.weight"].float()
            entry(i, pack.pack_tc_weight(torch.cat([W1[:, :H], torch.zeros(H, Hp - H), W1[:, H:]], dim=1), False))
            entry(i + 1, pack.pack_tc_weight(sd[f"{q}node_mlp.{nt}.2.weight"], False))
            i += 2
    # the plain pack is the hi half of the split one: bf16(w) per k-step slab, no lo slab
    w = sd["egnn.conv_layers.0.edge_mlp.ll.2.weight"][:nmain]
    assert pack.pack_tc_weight(w, True).numel() == 2 * pack.pack_tc_weight(w, False).numel()
