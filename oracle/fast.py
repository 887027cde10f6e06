"""Fewer-step sampling (oracle, CPU): the restatement the CUDA strided-ancestral and DDIM paths are held to.

Fewer-step sampling is an extension beyond the reference's sampling loop (DESIGN.md section 6.3 states it): the reverse
loop runs the steps tau_{k+1} -> tau_k of the grid tau_k = (k t_start) // n, k = n-1 .. 0, instead of every step.

* A strided ancestral step is the reference's own sample_p_zs_given_zt (ligand_diffuser.py:497-538) evaluated at
  (s, t) = (tau_k/T, tau_{k+1}/T), which it permits for any s < t: flat.sample_p_zs_given_zt with t = t_int instead
  of s+1, op for op.
* A DDIM(eta) step is written in its direct form, z_s = alpha_s x^ + sqrt(sigma_s^2 - c^2) eps^ + c xi with
  x^ = (z_t - sigma_t eps^) / alpha_t and c = eta sigma_t|s sigma_s / sigma_t, in the batch dtype -- not the product's
  closed form z/alpha_t|s - vt eps^ + sg xi.
* The loops (plain, from a start ligand, with a fragment) restate those of oracle/flat.py, oracle/optimize.py and
  oracle/inpaint.py on the grid; frame setup and restore are theirs.

Draws come from noise_fn(k, u, kind, shape) with shape (N_l, 3+F), position channels first, as in oracle/inpaint.py but
keyed by the row k of the grid: (-1, 0, 0) is the initial (or forward) draw, kind 0 = posterior, 1 = known part,
2 = re-noise.  Test infrastructure only (see oracle/__init__.py): never imported by the product.
"""
import torch

from . import schedule as S
from .flat import FlatBatch, _segment_mean, remove_com
from .optimize import partial_noise, start_coefficients


def grid(t_start, n):
    """tau_k = (k t_start) // n for k = 0..n."""
    return [k * int(t_start) // int(n) for k in range(int(n) + 1)]


def _levels(gamma, T, s_int, t_int, B):
    s = torch.full((B,), s_int) / T
    t = torch.full((B,), t_int) / T
    return t, S.gamma_lookup(gamma, s, T), S.gamma_lookup(gamma, t, T)


def posterior(dyn_fn, gamma, T, s_int, t_int, batch: FlatBatch, pos_noise, feat_noise, eta=None):
    """(z_s positions, z_s features) of the reverse step t_int -> s_int, before the ligand COM removal: the reference's
    ancestral step (eta=None), or the DDIM(eta) step in its direct form."""
    lig_b, _ = batch.batch_idx()
    dt = batch.lig_x.dtype
    t, gamma_s, gamma_t = _levels(gamma, T, s_int, t_int, batch.B)
    sigma2_ts, sigma_ts, alpha_ts = S.sigma_and_alpha_t_given_s(gamma_t, gamma_s)
    sigma_s, sigma_t = S.sigma(gamma_s), S.sigma(gamma_t)
    eps_h, eps_x = dyn_fn(batch, t)
    if eta is None:                                                                  # flat.sample_p_zs_given_zt
        var_terms = sigma2_ts / alpha_ts / sigma_t
        a = alpha_ts[lig_b].view(-1, 1).to(dt)
        vt = var_terms[lig_b].view(-1, 1).to(dt)
        mu_pos = batch.lig_x / a - vt * eps_x
        mu_feat = batch.lig_h / a - vt * eps_h
        sig = (sigma_ts * sigma_s / sigma_t)[lig_b].view(-1, 1).to(dt)
        return mu_pos + sig * pos_noise, mu_feat + sig * feat_noise

    def col(v):
        return v[lig_b].view(-1, 1).to(dt)
    a_s, s_s, a_t, s_t = col(S.alpha(gamma_s)), col(sigma_s), col(S.alpha(gamma_t)), col(sigma_t)
    c = float(eta) * torch.sqrt(col(sigma2_ts)) / s_t * s_s
    keep = torch.sqrt(s_s * s_s - c * c)
    x_hat = (batch.lig_x - s_t * eps_x) / a_t
    h_hat = (batch.lig_h - s_t * eps_h) / a_t
    return a_s * x_hat + keep * eps_x + c * pos_noise, a_s * h_hat + keep * eps_h + c * feat_noise


def sample_p_zs_given_zt(dyn_fn, gamma, T, s_int, batch: FlatBatch, pos_noise, feat_noise, t_int=None, eta=None):
    """flat.sample_p_zs_given_zt from level t_int (default s_int + 1) to s_int, ancestral or DDIM(eta)."""
    lig_b, kp_b = batch.batch_idx()
    t_int = s_int + 1 if t_int is None else int(t_int)
    batch.lig_x, batch.lig_h = posterior(dyn_fn, gamma, T, s_int, t_int, batch, pos_noise, feat_noise, eta)
    return remove_com(batch, lig_b, kp_b, "ligand")


def inpaint_step(dyn_fn, gamma, T, s_int, t_int, batch: FlatBatch, mask, x_fix, h_fix, init_kp_com, post_noise,
                 known_noise, lig_feat_norm_constant=1.0, eta=None):
    """One pass of the fragment-conditioned reverse step t_int -> s_int (inpaint.sample_p_zs_given_zt on the grid): the
    posterior sample, the known part noised to level s_int and aligned over the fixed atoms, merge, COM removal."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    dt = batch.lig_x.dtype
    z_unk_x, z_unk_h = posterior(dyn_fn, gamma, T, s_int, t_int, batch, post_noise[:, :3], post_noise[:, 3:], eta)
    _, gamma_s, _ = _levels(gamma, T, s_int, t_int, B)
    kp_com = _segment_mean(batch.kp_x, kp_b, B)
    a_s = S.alpha(gamma_s)[lig_b].view(-1, 1).to(dt)
    s_s = S.sigma(gamma_s)[lig_b].view(-1, 1).to(dt)
    x0 = (x_fix.to(dt) - init_kp_com[lig_b]) + kp_com[lig_b]
    z_kn_x = a_s * x0 + s_s * known_noise[:, :3]
    z_kn_h = a_s * (h_fix.to(dt) / lig_feat_norm_constant) + s_s * known_noise[:, 3:]
    fb = lig_b[mask]
    n_fix = torch.bincount(fb, minlength=B)
    cnt = n_fix.clamp(min=1).to(dt)[:, None]
    dx = (torch.zeros(B, 3, dtype=dt).index_add_(0, fb, z_unk_x[mask]) / cnt
          - torch.zeros(B, 3, dtype=dt).index_add_(0, fb, z_kn_x[mask]) / cnt)
    has = (n_fix > 0)[:, None]
    m = mask.view(-1, 1)
    batch.lig_x = torch.where(m, z_kn_x + dx[lig_b], z_unk_x)
    batch.lig_h = torch.where(m, z_kn_h, z_unk_h)
    batch.kp_x = torch.where(has[kp_b], batch.kp_x + dx[kp_b], batch.kp_x)
    return remove_com(batch, lig_b, kp_b, "ligand")


def renoise(gamma, T, s_int, t_int, batch: FlatBatch, noise):
    """From level s_int back to t_int: z_t = alpha_t|s z_s + sigma_t|s e, then the ligand COM removal."""
    lig_b, kp_b = batch.batch_idx()
    dt = batch.lig_x.dtype
    _, gamma_s, gamma_t = _levels(gamma, T, s_int, t_int, batch.B)
    _, sigma_ts, alpha_ts = S.sigma_and_alpha_t_given_s(gamma_t, gamma_s)
    a = alpha_ts[lig_b].view(-1, 1).to(dt)
    sg = sigma_ts[lig_b].view(-1, 1).to(dt)
    batch.lig_x = a * batch.lig_x + sg * noise[:, :3]
    batch.lig_h = a * batch.lig_h + sg * noise[:, 3:]
    return remove_com(batch, lig_b, kp_b, "ligand")


def sample_from_encoded_receptors(dyn_fn, gamma, T, batch: FlatBatch, noise_fn, n, eta=None, init_lig_pos=None,
                                  start=None, fragment=None, resamplings=1, lig_feat_norm_constant=1.0, atom_nf=None):
    """The reverse loop on the n-step grid over [0, t_start]: from pure noise with init_lig_pos (t_start = T, frame
    setup of flat.sample_from_encoded_receptors), or from ``start = (x_in, h_in, t0)`` (t_start = t0, the start of
    optimize.sample_from_encoded_receptors); plain steps, or with ``fragment = (mask, x_fix, h_fix)`` the inpainting
    step with ``resamplings`` passes; ancestral (eta=None) or DDIM(eta).  Then the plain frame restore."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    dt = batch.kp_x.dtype
    init_kp_com = _segment_mean(batch.kp_x, kp_b, B)
    N_l = int(batch.lig_n.sum())
    shape = (N_l, 3 + atom_nf)
    if start is None:
        t_start = T
        assert init_lig_pos.shape == (B, 3)
        batch.kp_x = batch.kp_x - init_lig_pos.to(dt)[kp_b]
        d = noise_fn(-1, 0, 0, shape).to(dt)
        batch.lig_x, batch.lig_h = d[:, :3], d[:, 3:]
        batch = remove_com(batch, lig_b, kp_b, "ligand")
    else:
        x_in, h_in, t_start = start
        a, s = start_coefficients(gamma, t_start)
        batch = partial_noise(batch, x_in, h_in, a, s, noise_fn(-1, 0, 0, shape), lig_feat_norm_constant)
        dt = batch.kp_x.dtype
    tau = grid(t_start, n)
    for k in reversed(range(int(n))):
        s_int, t_int = tau[k], tau[k + 1]
        if fragment is None:
            d = noise_fn(k, 0, 0, shape).to(dt)
            batch = sample_p_zs_given_zt(dyn_fn, gamma, T, s_int, batch, d[:, :3], d[:, 3:], t_int, eta)
            continue
        mask, x_fix, h_fix = fragment
        for u in range(resamplings):
            post = noise_fn(k, u, 0, shape).to(dt)
            known = noise_fn(k, u, 1, shape).to(dt)
            batch = inpaint_step(dyn_fn, gamma, T, s_int, t_int, batch, mask.to(torch.bool), x_fix, h_fix, init_kp_com,
                                 post, known, lig_feat_norm_constant, eta)
            if u < resamplings - 1:
                batch = renoise(gamma, T, s_int, t_int, batch, noise_fn(k, u, 2, shape).to(dt))
    batch = remove_com(batch, lig_b, kp_b, "receptor")
    batch.lig_x = batch.lig_x + init_kp_com[lig_b]
    batch.kp_x = batch.kp_x + init_kp_com[kp_b]
    batch.lig_h = batch.lig_h * lig_feat_norm_constant
    ptr = torch.zeros(B + 1, dtype=torch.long)
    ptr[1:] = torch.cumsum(batch.lig_n, 0)
    lig_pos = [batch.lig_x[ptr[i]:ptr[i + 1]].clone() for i in range(B)]
    lig_feat = [batch.lig_h[ptr[i]:ptr[i + 1]].clone() for i in range(B)]
    return lig_pos, lig_feat
