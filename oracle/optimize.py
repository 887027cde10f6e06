"""Ligand optimisation by partial noising (oracle, CPU): the restatement the CUDA start path is held to.

SDEdit-style optimisation, DiffSBDD's "molecule optimisation", is an extension beyond the reference (DESIGN.md section
6.2 states it): a given ligand is noised forward to level t0 and the reverse loop runs from step t0-1 down to 0.  Only
the frame setup is new; the reverse steps are flat.sample_p_zs_given_zt (or, with a fragment, the inpainting step of
oracle/inpaint.py) and the frame restore is the plain loop's, op for op.

Test infrastructure only (see oracle/__init__.py): never imported by the product.
"""
import torch

from . import inpaint as I
from . import schedule as S
from .flat import FlatBatch, _segment_mean, remove_com, sample_p_zs_given_zt

# Draws come from noise_fn(step, u, kind, shape) with shape (N_l, 3+F), position channels first, as in oracle/inpaint.py:
# (-1, 0, 0) is the forward draw of the start (the plain loop's initial draw), (s, 0, 0) the posterior draw of step s.


def start_coefficients(gamma, t0):
    """(alpha_t0, sigma_t0) as 1-element fp32 tensors: sqrt(sigmoid(-gamma[t0])), sqrt(sigmoid(gamma[t0]))."""
    g = gamma[torch.full((1,), int(t0), dtype=torch.long)]
    return S.alpha(g), S.sigma(g)


def partial_noise(batch: FlatBatch, x_in, h_in, alpha_t0, sigma_t0, draw, lig_feat_norm_constant=1.0):
    """The start: c_b = mean of x_in per complex; keypoints -= c_b; z = alpha*(x_in - c_b, h_in / norm) + sigma*draw;
    then the ligand COM is removed from ligand and keypoints."""
    lig_b, kp_b = batch.batch_idx()
    dt = batch.kp_x.dtype
    x_in = x_in.to(dt)
    c = _segment_mean(x_in, lig_b, batch.B)
    batch.kp_x = batch.kp_x - c[kp_b]
    x0 = x_in - c[lig_b]
    h0 = h_in.to(dt) / lig_feat_norm_constant
    a, s = alpha_t0.to(dt), sigma_t0.to(dt)
    batch.lig_x = a * x0 + s * draw[:, :3].to(dt)
    batch.lig_h = a * h0 + s * draw[:, 3:].to(dt)
    return remove_com(batch, lig_b, kp_b, "ligand")


def sample_from_encoded_receptors(dyn_fn, gamma, T, batch: FlatBatch, x_in, h_in, t0, noise_fn, fragment=None,
                                  resamplings=1, lig_feat_norm_constant=1.0, n_steps=None, atom_nf=None):
    """The reverse loop from the start ligand (x_in [N_l,3] in the frame the loop returns ligands in, h_in [N_l,F] in the
    returned feature space) noised to level t0: steps t0-1 .. 0 of the plain loop, or of the inpainting loop with
    ``fragment = (mask, x_fix, h_fix)`` and ``resamplings`` passes per step; then the plain frame restore."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    init_kp_com = _segment_mean(batch.kp_x, kp_b, B)
    N_l = int(batch.lig_n.sum())
    shape = (N_l, 3 + atom_nf)
    a, s = start_coefficients(gamma, t0)
    batch = partial_noise(batch, x_in, h_in, a, s, noise_fn(-1, 0, 0, shape), lig_feat_norm_constant)
    steps = list(reversed(range(0, int(t0))))
    if n_steps is not None:
        steps = steps[:n_steps]
    dt = batch.kp_x.dtype
    for s_int in steps:
        if fragment is None:
            d = noise_fn(s_int, 0, 0, shape).to(dt)
            batch = sample_p_zs_given_zt(dyn_fn, gamma, T, s_int, batch, d[:, :3], d[:, 3:])
            continue
        mask, x_fix, h_fix = fragment
        for u in range(resamplings):
            post = noise_fn(s_int, u, 0, shape).to(dt)
            known = noise_fn(s_int, u, 1, shape).to(dt)
            batch = I.sample_p_zs_given_zt(dyn_fn, gamma, T, s_int, batch, mask.to(torch.bool), x_fix, h_fix,
                                           init_kp_com, post, known, lig_feat_norm_constant)
            if u < resamplings - 1:
                batch = I.renoise(gamma, T, s_int, batch, noise_fn(s_int, u, 2, shape).to(dt))
    batch = remove_com(batch, lig_b, kp_b, "receptor")
    batch.lig_x = batch.lig_x + init_kp_com[lig_b]
    batch.kp_x = batch.kp_x + init_kp_com[kp_b]
    batch.lig_h = batch.lig_h * lig_feat_norm_constant
    ptr = torch.zeros(B + 1, dtype=torch.long)
    ptr[1:] = torch.cumsum(batch.lig_n, 0)
    lig_pos = [batch.lig_x[ptr[i]:ptr[i + 1]].clone() for i in range(B)]
    lig_feat = [batch.lig_h[ptr[i]:ptr[i + 1]].clone() for i in range(B)]
    return lig_pos, lig_feat
