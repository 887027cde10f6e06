"""Predefined noise schedule + the per-step posterior coefficient table.

Mirrors PredefinedNoiseSchedule / polynomial_schedule / clip_noise_schedule of the reference
(models/ligand_diffuser.py:620-690); `gamma` stays a non-trainable nn.Parameter so that it
round-trips through the checkpoint (SURVEY N9).  The table [T,4] = (alpha_t|s, var_terms,
sigma, t) is what the CUDA step kernel reads; it restates models/ligand_diffuser.py:232-252 and
:505-527 on the host, once per model (the values are identical for every complex of a batch).
inpaint_table [T,4] = (alpha_s, sigma_s, alpha_t|s, sigma_t|s) is the second table that
fragment-conditioned sampling reads (DESIGN.md section 6.1); start_coefficients gives (alpha_t0, sigma_t0), the
forward noising of a start ligand in ligand optimisation (section 6.2).
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F


def _clip(alphas2, clip_value=0.001):
    alphas2 = np.concatenate([np.ones(1), alphas2], axis=0)
    step = np.clip(alphas2[1:] / alphas2[:-1], a_min=clip_value, a_max=1.0)
    return np.cumprod(step, axis=0)


def polynomial_schedule(timesteps: int, s=1e-4, power=3.0):
    steps = timesteps + 1
    x = np.linspace(0, steps, steps)
    alphas2 = _clip((1 - np.power(x / steps, power)) ** 2)
    return (1 - 2 * s) * alphas2 + s


def cosine_beta_schedule(timesteps, s=0.008, raise_to_power: float = 1):
    steps = timesteps + 2
    x = np.linspace(0, steps, steps)
    ac = np.cos(((x / steps) + s) / (1 + s) * np.pi * 0.5) ** 2
    ac = ac / ac[0]
    betas = np.clip(1 - (ac[1:] / ac[:-1]), a_min=0, a_max=0.999)
    ac = np.cumprod(1.0 - betas, axis=0)
    return np.power(ac, raise_to_power) if raise_to_power != 1 else ac


class PredefinedNoiseSchedule(nn.Module):
    def __init__(self, noise_schedule, timesteps, precision):
        super().__init__()
        self.timesteps = timesteps
        if noise_schedule == "cosine":
            alphas2 = cosine_beta_schedule(timesteps)
        elif "polynomial" in noise_schedule:
            parts = noise_schedule.split("_")
            assert len(parts) == 2
            alphas2 = polynomial_schedule(timesteps, s=precision, power=float(parts[1]))
        else:
            raise ValueError(noise_schedule)
        sigmas2 = 1 - alphas2
        gamma = -(np.log(alphas2) - np.log(sigmas2))
        self.gamma = nn.Parameter(torch.from_numpy(gamma).float(), requires_grad=False)

    def forward(self, t):
        t_int = torch.round(t * self.timesteps).long()
        return self.gamma[t_int]


def sigma(gamma):
    return torch.sqrt(torch.sigmoid(gamma))


def alpha(gamma):
    return torch.sqrt(torch.sigmoid(-gamma))


def sigma_and_alpha_t_given_s(gamma_t, gamma_s):
    sigma2_t_given_s = -torch.expm1(F.softplus(gamma_s) - F.softplus(gamma_t))
    alpha_t_given_s = torch.exp(0.5 * (F.logsigmoid(-gamma_t) - F.logsigmoid(-gamma_s)))
    return sigma2_t_given_s, torch.sqrt(sigma2_t_given_s), alpha_t_given_s


def coefficient_table(gamma: torch.Tensor, T: int) -> torch.Tensor:
    """fp32 [T,4] on the CPU; row s = (alpha_t|s, var_terms, sigma, t=(s+1)/T).

    Evaluated row by row on 1-element fp32 tensors with the same torch ops the reference applies
    per step (ligand_diffuser.py:405-408, :505-527).  (A vectorised evaluation over all T rows
    differs in the last bit because torch's SIMD and scalar transcendental paths round
    differently; the scalar path is what the oracle pins.)"""
    g = gamma.detach().float().cpu()
    rows = []
    for s_int in range(T):
        s = torch.full((1,), s_int) / T
        t = (torch.full((1,), s_int) + 1) / T
        gs = g[torch.round(s * T).long()]
        gt = g[torch.round(t * T).long()]
        s2, s1, a = sigma_and_alpha_t_given_s(gt, gs)
        sig_s, sig_t = sigma(gs), sigma(gt)
        rows.append(torch.stack([a[0], (s2 / a / sig_t)[0], (s1 * sig_s / sig_t)[0], t[0].float()]))
    return torch.stack(rows).contiguous()


def inpaint_table(gamma: torch.Tensor, T: int) -> torch.Tensor:
    """fp32 [T,4] on the CPU; row s = (alpha_s, sigma_s, alpha_t|s, sigma_t|s) with t = s+1: the known-part noising
    and the re-noise coefficients of fragment-conditioned sampling.  Evaluated like coefficient_table (scalar fp32 ops,
    row by row), so its alpha_t|s column equals coefficient_table's column 0 bit for bit."""
    g = gamma.detach().float().cpu()
    rows = []
    for s_int in range(T):
        s = torch.full((1,), s_int) / T
        t = (torch.full((1,), s_int) + 1) / T
        gs = g[torch.round(s * T).long()]
        gt = g[torch.round(t * T).long()]
        _, s1, a = sigma_and_alpha_t_given_s(gt, gs)
        rows.append(torch.stack([alpha(gs)[0], sigma(gs)[0], a[0], s1[0]]))
    return torch.stack(rows).contiguous()


def start_coefficients(gamma: torch.Tensor, t0: int):
    """(alpha_t0, sigma_t0) as Python floats holding fp32 values: the level a start ligand is noised to before the
    reverse loop runs from step t0 (ligand optimisation by partial noising).  Evaluated like coefficient_table, with the
    scalar fp32 ops on a 1-element tensor gamma[t0]."""
    g = gamma.detach().float().cpu()
    g0 = g[torch.full((1,), int(t0), dtype=torch.long)]
    return float(alpha(g0)[0]), float(sigma(g0)[0])
