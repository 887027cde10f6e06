"""Fragment-conditioned sampling (oracle, CPU): the restatement the CUDA inpainting path is held to.

Inpainting with RePaint-style resampling is an extension beyond the reference, which has none (DESIGN.md section 6.1
states the algorithm); it follows DiffSBDD's inpainting sampler for the same class of model, with the keypoints in the
pocket's role.  Built on the plain loop of oracle/flat.py: frame setup, posterior arithmetic and COM removal are those
of flat.sample_from_encoded_receptors / flat.sample_p_zs_given_zt, op for op.

Test infrastructure only (see oracle/__init__.py): never imported by the product.
"""
import torch

from . import schedule as S
from .flat import FlatBatch, _segment_mean, remove_com

# The atoms of `mask` are pinned to (x_fix, h_fix) -- positions in the frame the loop returns ligands in, features in the returned
# feature space.  Draws come from noise_fn(step, u, kind, shape) with shape (N_l, 3+F), position channels first:
# kind 0 = posterior, 1 = known part, 2 = re-noise; (-1, 0, 0) is the initial draw.

def sample_p_zs_given_zt(dyn_fn, gamma, T, s_int, batch: FlatBatch, mask, x_fix, h_fix, init_kp_com,
                                 post_noise, known_noise, lig_feat_norm_constant=1.0):
    """One pass of reverse step s: posterior sample (as flat.sample_p_zs_given_zt), known part noised to level s, COM
    alignment of the known part (and the keypoints) to the generated part over the fixed atoms, merge, COM removal."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    dt = batch.lig_x.dtype
    s = torch.full((B,), s_int) / T
    t = (torch.full((B,), s_int) + 1) / T
    gamma_s = S.gamma_lookup(gamma, s, T)
    gamma_t = S.gamma_lookup(gamma, t, T)
    sigma2_ts, sigma_ts, alpha_ts = S.sigma_and_alpha_t_given_s(gamma_t, gamma_s)
    sigma_s, sigma_t = S.sigma(gamma_s), S.sigma(gamma_t)
    alpha_s = S.alpha(gamma_s)
    eps_h, eps_x = dyn_fn(batch, t)
    var_terms = sigma2_ts / alpha_ts / sigma_t
    a = alpha_ts[lig_b].view(-1, 1).to(dt)
    vt = var_terms[lig_b].view(-1, 1).to(dt)
    mu_pos = batch.lig_x / a - vt * eps_x
    mu_feat = batch.lig_h / a - vt * eps_h
    sig = (sigma_ts * sigma_s / sigma_t)[lig_b].view(-1, 1).to(dt)
    z_unk_x = mu_pos + sig * post_noise[:, :3]
    z_unk_h = mu_feat + sig * post_noise[:, 3:]
    # known part at level s, mapped into the current frame: p -> p - init_kp_com + kp_com_now
    kp_com = _segment_mean(batch.kp_x, kp_b, B)
    a_s = alpha_s[lig_b].view(-1, 1).to(dt)
    s_s = sigma_s[lig_b].view(-1, 1).to(dt)
    x0 = (x_fix.to(dt) - init_kp_com[lig_b]) + kp_com[lig_b]
    z_kn_x = a_s * x0 + s_s * known_noise[:, :3]
    z_kn_h = a_s * (h_fix.to(dt) / lig_feat_norm_constant) + s_s * known_noise[:, 3:]
    # align: dx = mean_M(z_unk_x) - mean_M(z_kn_x) per complex with a fixed atom
    fb = lig_b[mask]
    n_fix = torch.bincount(fb, minlength=B)
    cnt = n_fix.clamp(min=1).to(dt)[:, None]
    sum_u = torch.zeros(B, 3, dtype=dt).index_add_(0, fb, z_unk_x[mask])
    sum_k = torch.zeros(B, 3, dtype=dt).index_add_(0, fb, z_kn_x[mask])
    dx = sum_u / cnt - sum_k / cnt
    has = (n_fix > 0)[:, None]
    z_kn_x = z_kn_x + dx[lig_b]
    m = mask.view(-1, 1)
    batch.lig_x = torch.where(m, z_kn_x, z_unk_x)
    batch.lig_h = torch.where(m, z_kn_h, z_unk_h)
    batch.kp_x = torch.where(has[kp_b], batch.kp_x + dx[kp_b], batch.kp_x)
    return remove_com(batch, lig_b, kp_b, "ligand")


def renoise(gamma, T, s_int, batch: FlatBatch, noise):
    """z_t = alpha_t|s z_s + sigma_t|s e (positions and features), then the ligand COM removal."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    dt = batch.lig_x.dtype
    s = torch.full((B,), s_int) / T
    t = (torch.full((B,), s_int) + 1) / T
    _, sigma_ts, alpha_ts = S.sigma_and_alpha_t_given_s(S.gamma_lookup(gamma, t, T), S.gamma_lookup(gamma, s, T))
    a = alpha_ts[lig_b].view(-1, 1).to(dt)
    sg = sigma_ts[lig_b].view(-1, 1).to(dt)
    batch.lig_x = a * batch.lig_x + sg * noise[:, :3]
    batch.lig_h = a * batch.lig_h + sg * noise[:, 3:]
    return remove_com(batch, lig_b, kp_b, "ligand")


def sample_from_encoded_receptors(dyn_fn, gamma, T, batch: FlatBatch, init_lig_pos, noise_fn, mask, x_fix, h_fix,
                                  resamplings=1, lig_feat_norm_constant=1.0, n_steps=None, atom_nf=None):
    """flat.sample_from_encoded_receptors with the atoms of `mask` (bool [N_l]) pinned to (x_fix [N_l,3], h_fix [N_l,F])
    and `resamplings` passes per reverse step, re-noising to level t between passes.  Frame setup and restore are
    those of the plain loop."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    dt = batch.kp_x.dtype
    init_kp_com = _segment_mean(batch.kp_x, kp_b, B)
    assert init_lig_pos.shape == (B, 3)
    batch.kp_x = batch.kp_x - init_lig_pos.to(dt)[kp_b]
    N_l = int(batch.lig_n.sum())
    shape = (N_l, 3 + atom_nf)
    d = noise_fn(-1, 0, 0, shape).to(dt)
    batch.lig_x, batch.lig_h = d[:, :3], d[:, 3:]
    batch = remove_com(batch, lig_b, kp_b, "ligand")
    steps = list(reversed(range(0, T)))
    if n_steps is not None:
        steps = steps[:n_steps]
    mask = mask.to(torch.bool)
    for s_int in steps:
        for u in range(resamplings):
            post = noise_fn(s_int, u, 0, shape).to(dt)
            known = noise_fn(s_int, u, 1, shape).to(dt)
            batch = sample_p_zs_given_zt(dyn_fn, gamma, T, s_int, batch, mask, x_fix, h_fix, init_kp_com, post,
                                         known, lig_feat_norm_constant)
            if u < resamplings - 1:
                batch = renoise(gamma, T, s_int, batch, noise_fn(s_int, u, 2, shape).to(dt))
    batch = remove_com(batch, lig_b, kp_b, "receptor")
    batch.lig_x = batch.lig_x + init_kp_com[lig_b]
    batch.kp_x = batch.kp_x + init_kp_com[kp_b]
    batch.lig_h = batch.lig_h * lig_feat_norm_constant
    ptr = torch.zeros(B + 1, dtype=torch.long)
    ptr[1:] = torch.cumsum(batch.lig_n, 0)
    lig_pos = [batch.lig_x[ptr[i]:ptr[i + 1]].clone() for i in range(B)]
    lig_feat = [batch.lig_h[ptr[i]:ptr[i + 1]].clone() for i in range(B)]
    return lig_pos, lig_feat
