"""Teacher-forced parity cases at the SHIPPED hyper-parameters of every shipped trained model.

One builder for all eight (trained_models/{egnn_20kp, gvp_20kp, egnn_40kp, gvp_40kp, egnn_all_atom, gvp_all_atom,
egnn_ca, gvp_ca}; the first five are the BASELINE.json configs): seeded
weights in the reference state_dict layout (oracle/params.py; the checkpoints are not in the reference tree), the
synthetic pocket kind SURVEY.md section 8d prescribes for the config, a handful of complexes of mixed ligand size so the
CPU oracle stays cheap.  The hyper-parameters come from tests/golden/shipped_configs.yml, an extract of the reference's
own trained_models/*/config.yml written by tests/golden/make_golden.py.
"""
from pathlib import Path

import torch
import yaml

GOLDEN = Path(__file__).resolve().parent / "golden"

# config name -> (pocket kind, pocket nodes, ligand sizes, pockets)
SHIPPED = {
    "egnn_20kp": ("keypoint", 20, [20, 8, 35, 20, 13, 27], 3),
    "gvp_20kp": ("keypoint", 20, [20, 8, 35, 20, 13, 27], 3),
    "egnn_40kp": ("keypoint", 40, [20, 8, 35, 60, 2, 27], 3),
    # >= 300 pocket atoms as keypoints (fixed encoder: rec_nf = 10 -> the 10 -> 20 -> 256 encoder MLP), ll radius 6
    "egnn_all_atom": ("all_atom", 336, [20, 33, 5], 2),
    # C-alpha pocket: 42 nodes >= 3.8 A apart, kk = rr radius 3.5 (empty), message_norm 'mean'
    "gvp_ca": ("ca", 42, [20, 1, 44, 9, 27], 2),
    "gvp_40kp": ("keypoint", 40, [20, 8, 35, 60, 2, 27], 3),
    # the only GVP model with hundreds of keypoints per complex: fixed encoder, kk := rr, message_norm 'mean'
    "gvp_all_atom": ("all_atom", 336, [20, 33, 1, 5], 2),
    "egnn_ca": ("ca", 42, [20, 1, 44, 9, 27], 2),
}


def shipped_configs():
    return yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))


def dynamics_kwargs(cfg):
    """(arch, ctor kwargs of the dynamics module, rec_nf) as model_setup.model_from_config derives them
    (reference model_setup.py:4-64)."""
    arch = cfg["diffusion"].get("architecture", "egnn")
    learned = cfg["diffusion"].get("rec_encoder_type", "learned") == "learned"
    cut = cfg["graph"]["graph_cutoffs"]
    if arch == "egnn":
        d = cfg["dynamics"]
        rec_nf = cfg["rec_encoder"]["out_n_node_feat"] if learned else len(cfg["dataset"]["rec_elements"])
        kw = dict(n_layers=d["n_layers"], hidden_nf=d["hidden_nf"], use_tanh=d["use_tanh"], message_norm=d["message_norm"],
                  update_kp_feat=d["update_kp_feat"], norm=d["norm"], ll_k=d["ll_k"], kl_k=d["kl_k"], graph_cutoffs=cut)
    else:
        d = cfg["dynamics_gvp"]
        rec_nf = cfg["rec_encoder_gvp"]["out_scalar_size"] if learned else len(cfg["dataset"]["rec_elements"])
        kw = dict(vector_size=d["vector_size"], n_convs=d["n_convs"], n_hidden_scalars=d["n_hidden_scalars"],
                  message_norm=d["message_norm"], update_kp=d["update_kp"], ll_k=d["ll_k"], kl_k=d["kl_k"],
                  n_message_gvps=d["n_message_gvps"], n_update_gvps=d["n_update_gvps"], n_noise_gvps=d["n_noise_gvps"],
                  graph_cutoffs=cut)
    return arch, kw, rec_nf


def seeded_state_dict(arch, kw, rec_nf, atom_nf=10, seed=3):
    from oracle import params as P
    if arch == "egnn":
        shapes = P.egnn_dynamics_shapes(atom_nf, rec_nf, kw["n_layers"], kw["hidden_nf"], kw["update_kp_feat"], kw["norm"])
        return P.init_state_dict(shapes, seed=seed, coord_gain=0.3)        # SURVEY N5: exercise the coordinate path
    shapes = P.gvp_dynamics_shapes(atom_nf, rec_nf, kw["vector_size"], kw["n_convs"], kw["n_hidden_scalars"], kw["update_kp"],
                                   kw["n_message_gvps"], kw["n_update_gvps"], kw["n_noise_gvps"])
    sd = P.init_state_dict(shapes, seed=seed + 1)
    for k in sd:
        if k.endswith(".Wh") or k.endswith(".Wu"):
            sd[k] = sd[k] * 2.0                     # keeps the vector channel O(0.1) on random weights
    return sd


def make_pockets(kind, n_nodes, rec_nf, vector_size, cut, n_pockets):
    from keypoint_diffusion_b200 import synthetic
    if kind == "keypoint":
        return [synthetic.keypoint_pocket(i, n_nodes, rec_nf, vector_size, cut["kk"]) for i in range(n_pockets)]
    if kind == "all_atom":
        pockets = [synthetic.all_atom_pocket(i, n_nodes, rec_nf, vector_size, cut["rr"]) for i in range(n_pockets)]
    else:
        pockets = [synthetic.ca_pocket(i, n_nodes, rec_nf, vector_size, cut["rr"]) for i in range(n_pockets)]
    for i, pk in enumerate(pockets):       # the fixed encoder gives v_0 = 0; non-zero vectors exercise the kp vector path too
        if vector_size:
            pk.kp_v = 0.1 * torch.randn(pk.n_kp, vector_size, 3, generator=torch.Generator().manual_seed(50 + i))
    return pockets


def assemble_inputs(pockets, n_lig, atom_nf, seed, with_v):
    """Flat inputs of a batch: complex i uses pockets[i % len(pockets)]."""
    from keypoint_diffusion_b200 import synthetic
    x_l, h_l = synthetic.ligand_noise_state(n_lig, atom_nf, seed)
    kx, kh, kv, ks, kd, kn, off = [], [], [], [], [], [], 0
    for i in range(len(n_lig)):
        pk = pockets[i % len(pockets)]
        kx.append(pk.kp_x); kh.append(pk.kp_h)
        if with_v:
            kv.append(pk.kp_v)
        ks.append(pk.kk_src + off); kd.append(pk.kk_dst + off)
        off += pk.n_kp
        kn.append(pk.n_kp)
    d = {"lig_n": torch.tensor(n_lig), "kp_n": torch.tensor(kn), "lig_x": x_l, "lig_h": h_l, "kp_x": torch.cat(kx),
         "kp_h": torch.cat(kh), "kk_src": torch.cat(ks), "kk_dst": torch.cat(kd)}
    if with_v:
        d["kp_v"] = torch.cat(kv)
    return d


def shipped_case(name, n_lig=None):
    """-> (arch, state_dict, ctor kwargs, rec_nf, flat inputs) for shipped config `name`."""
    kind, n_nodes, sizes, n_pockets = SHIPPED[name]
    cfg = shipped_configs()[name]
    arch, kw, rec_nf = dynamics_kwargs(cfg)
    sd = seeded_state_dict(arch, kw, rec_nf)
    vs = kw.get("vector_size", 0)
    pockets = make_pockets(kind, n_nodes, rec_nf, vs, kw["graph_cutoffs"], n_pockets)
    inputs = assemble_inputs(pockets, n_lig or sizes, 10, seed=5, with_v=bool(vs))
    return arch, sd, kw, rec_nf, inputs
