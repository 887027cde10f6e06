"""Batch helpers with the reference's names (reference utils.py:81-170), on the duck-typed
graph surface of hetero.HeteroBatch (or a real DGL heterograph), and the output decode that follows the
sampling path (SURVEY 8f rank 4: reference utils.py:11-21, test.py:199-209), with a multi-frame XYZ writer for the
trajectories of visualize=True."""
from typing import Dict, List, Tuple

import torch

from . import hetero


def get_batch_info(g) -> Tuple[dict, dict]:
    """reference utils.py:81-90"""
    return ({nt: g.batch_num_nodes(nt) for nt in g.ntypes},
            {et: g.batch_num_edges(et) for et in g.canonical_etypes})


def get_batch_idxs(g) -> Dict[str, torch.Tensor]:
    """reference utils.py:158-170: node -> complex index per node type."""
    ar = torch.arange(g.batch_size, device=g.device)
    return {nt: ar.repeat_interleave(g.batch_num_nodes(nt).to(g.device)) for nt in g.ntypes}


def get_edges_per_batch(edge_node_idxs: torch.Tensor, batch_size: int, node_batch_idxs: torch.Tensor):
    """reference utils.py:92-98 (edges grouped by complex)."""
    if edge_node_idxs.numel() == 0:
        return torch.zeros(batch_size, dtype=torch.long, device=edge_node_idxs.device)
    return torch.bincount(node_batch_idxs[edge_node_idxs], minlength=batch_size)


def copy_graph(g, n_copies: int, lig_atoms_per_copy: torch.Tensor = None, batched_graph=False) -> List:
    """reference utils.py:103-156: n_copies of a single-complex graph, optionally with a chosen
    number of (zero-filled) ligand atoms per copy."""
    out = []
    for i in range(n_copies):
        bnn = {nt: g.batch_num_nodes(nt).clone() for nt in g.ntypes}
        nd = {nt: {k: v.detach().clone() for k, v in g.nodes[nt].data.items()} for nt in g.ntypes}
        if lig_atoms_per_copy is not None:
            n = int(lig_atoms_per_copy[i])
            bnn["lig"] = torch.tensor([n], device=g.device)
            nd["lig"] = {k: torch.zeros((n,) + tuple(v.shape[1:]), dtype=v.dtype, device=g.device)
                         for k, v in g.nodes["lig"].data.items()}
        edges = {et: tuple(t.clone() for t in g.edges(form="uv", etype=et)) for et in g.canonical_etypes}
        bne = {et: g.batch_num_edges(et).clone() for et in g.canonical_etypes}
        out.append(hetero.HeteroBatch(bnn, nd, edges, bne))
    return out


def write_xyz_file(coords, atom_types, filename=None):
    """reference utils.py:11-21 (taken there from DiffSBDD): an XYZ block for one molecule; returns the text when
    ``filename`` is None, else writes it."""
    out = f"{len(coords)}\n\n"
    assert len(coords) == len(atom_types)
    for i in range(len(coords)):
        out += f"{atom_types[i]} {coords[i, 0]:.3f} {coords[i, 1]:.3f} {coords[i, 2]:.3f}\n"
    if filename is None:
        return out
    with open(filename, 'w') as f:
        f.write(out)


def decode_ligands(lig_pos: List[torch.Tensor], lig_feat: List[torch.Tensor], lig_elements: List[str],
                   atom_types: List[torch.Tensor] = None) -> List[Tuple]:
    """What the reference does with the sampler's output before molecule building (test.py:199-203): the atom type
    of every generated atom is the argmax over its feature channels, mapped through the dataset's ``lig_elements``
    (``dataset.lig_atom_idx_to_element``).  Returns one (positions [n,3], element symbols) pair per ligand; bond
    perception / sanitisation (OpenBabel, RDKit) stay with the caller."""
    out = []
    if atom_types is not None:        # already decoded on the device (sample_from_encoded_receptors(decode=True))
        for pos, idx in zip(lig_pos, atom_types):
            out.append((pos, [lig_elements[int(i)] for i in idx.tolist()]))
        return out
    for pos, feat in zip(lig_pos, lig_feat):
        idx = torch.argmax(feat, dim=1).tolist()
        out.append((pos, [lig_elements[i] for i in idx]))
    return out


def write_xyz_trajectory(frames: Dict[str, torch.Tensor], lig_elements: List[str], filename=None):
    """A multi-frame XYZ file of one ligand's trajectory (a dict of sample_from_encoded_receptors(visualize=True)): one
    write_xyz_file block per state frame, its atom types decoded from that frame's features as decode_ligands does.
    Returns the text when ``filename`` is None, else writes it."""
    pos, feat = frames['positions'].cpu(), frames['features'].cpu()
    out = "".join(write_xyz_file(p, elems) for p, elems in decode_ligands(list(pos), list(feat), lig_elements))
    if filename is None:
        return out
    with open(filename, 'w') as f:
        f.write(out)


def split_bounds(n_complexes: int, n_groups: int):
    """Boundaries of n_groups contiguous, near-equal groups of complexes: [b_0 = 0, ..., b_n = n_complexes].
    Used by KeypointDiffusion._sub_samplers (a batch sampled as concurrent sub-batches)."""
    n_groups = max(1, min(int(n_groups), int(n_complexes)))
    return [round(i * n_complexes / n_groups) for i in range(n_groups + 1)]
