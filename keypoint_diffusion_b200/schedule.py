"""Predefined noise schedule + the per-step posterior coefficient table.

Mirrors PredefinedNoiseSchedule / polynomial_schedule / clip_noise_schedule of the reference
(models/ligand_diffuser.py:620-690); `gamma` stays a non-trainable nn.Parameter so that it
round-trips through the checkpoint (SURVEY N9).  The table [T,4] = (alpha_t|s, var_terms,
sigma, t) is what the CUDA step kernel reads; it restates models/ligand_diffuser.py:232-252 and
:505-527 on the host, once per model (the values are identical for every complex of a batch).
inpaint_table [T,4] = (alpha_s, sigma_s, alpha_t|s, sigma_t|s) is the second table that
fragment-conditioned sampling reads (DESIGN.md section 6.1); start_coefficients gives (alpha_t0, sigma_t0), the
forward noising of a start ligand in ligand optimisation (section 6.2).  Both tables are the unit-step case of
coefficient_rows / inpaint_rows over a step grid (step_grid), which also give the strided ancestral and DDIM rows of
fewer-step sampling (section 6.3).  prediction_rows and frame_levels serve recorded trajectories (section 6.4);
multistep_rows the second-order DPM-Solver++(2M) steps (section 6.5).
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


def step_grid(t_start: int, n: int) -> list:
    """The n-step grid tau_k = (k t_start) // n, k = 0..n (DESIGN.md section 6.3): tau_0 = 0, tau_n = t_start, strictly
    increasing; row k of a grid table is the reverse step tau_{k+1} -> tau_k.  n = t_start is the unit grid."""
    t_start, n = int(t_start), int(n)
    if not 1 <= n <= t_start:
        raise ValueError(f"a step grid over [0, {t_start}] needs 1 <= n <= {t_start}, got n = {n}")
    return [k * t_start // n for k in range(n + 1)]


def _row_gammas(g, T, s_int, t_int):
    """(gamma_s, gamma_t, t) of the step t_int -> s_int as 1-element fp32 tensors, looked up as the reference does
    (ligand_diffuser.py:405-408, :688-690)."""
    s = torch.full((1,), s_int) / T
    t = torch.full((1,), t_int) / T
    return g[torch.round(s * T).long()], g[torch.round(t * T).long()], t


def _ddim_columns(gs, gt, eta: float):
    """(vt, sg) of a DDIM(eta) row, in fp64 from the fp32 gammas, rounded once to fp32 (DESIGN.md section 6.3):
    rho = sigma2_t|s / sigma_t^2, vt = (sigma_t / alpha_t|s) rho (1 + eta^2 - eta^2 rho) / (1 + sqrt((1-rho)(1-eta^2 rho))),
    sg = eta sqrt(rho) sigma_s."""
    gs, gt = gs.double(), gt.double()
    s2 = -torch.expm1(F.softplus(gs) - F.softplus(gt))
    a = torch.exp(0.5 * (F.logsigmoid(-gt) - F.logsigmoid(-gs)))
    sig2_t = torch.sigmoid(gt)
    rho = s2 / sig2_t
    e2 = float(eta) ** 2
    vt = torch.sqrt(sig2_t) / a * rho * (1 + e2 - e2 * rho) / (1 + torch.sqrt((1 - rho) * (1 - e2 * rho)))
    sg = float(eta) * torch.sqrt(rho) * torch.sqrt(torch.sigmoid(gs))
    return vt.float(), sg.float()


def coefficient_rows(gamma: torch.Tensor, T: int, grid, eta=None) -> torch.Tensor:
    """fp32 [n,4] on the CPU over a step grid (step_grid): row k = (alpha_t|s, var_terms, sigma, t = tau_{k+1}/T) of the
    reverse step tau_{k+1} -> tau_k, the reference's sample_p_zs_given_zt at (s, t) = (tau_k/T, tau_{k+1}/T).

    Evaluated row by row on 1-element fp32 tensors with the same torch ops the reference applies per step
    (ligand_diffuser.py:405-408, :505-527).  (A vectorised evaluation over all rows differs in the last bit because
    torch's SIMD and scalar transcendental paths round differently; the scalar path is what the oracle pins.)
    eta in [0, 1]: DDIM(eta) rows instead -- columns 0 and 3 as above, columns 1 and 2 from _ddim_columns."""
    g = gamma.detach().float().cpu()
    rows = []
    for s_int, t_int in zip(grid[:-1], grid[1:]):
        gs, gt, t = _row_gammas(g, T, s_int, t_int)
        s2, s1, a = sigma_and_alpha_t_given_s(gt, gs)
        sig_s, sig_t = sigma(gs), sigma(gt)
        vt, sg = (s2 / a / sig_t, s1 * sig_s / sig_t) if eta is None else _ddim_columns(gs, gt, eta)
        rows.append(torch.stack([a[0], vt[0], sg[0], t[0].float()]))
    return torch.stack(rows).contiguous()


def coefficient_table(gamma: torch.Tensor, T: int) -> torch.Tensor:
    """fp32 [T,4] on the CPU; row s = (alpha_t|s, var_terms, sigma, t=(s+1)/T): coefficient_rows over the unit grid."""
    return coefficient_rows(gamma, T, list(range(T + 1)))


def inpaint_rows(gamma: torch.Tensor, T: int, grid) -> torch.Tensor:
    """fp32 [n,4] on the CPU over a step grid; row k = (alpha_s, sigma_s, alpha_t|s, sigma_t|s) with (s, t) = (tau_k,
    tau_{k+1}): the known-part noising and the re-noise coefficients of fragment-conditioned sampling.  Evaluated like
    coefficient_rows (scalar fp32 ops, row by row), so its alpha_t|s column equals coefficient_rows' column 0 bit for bit."""
    g = gamma.detach().float().cpu()
    rows = []
    for s_int, t_int in zip(grid[:-1], grid[1:]):
        gs, gt, _ = _row_gammas(g, T, s_int, t_int)
        _, s1, a = sigma_and_alpha_t_given_s(gt, gs)
        rows.append(torch.stack([alpha(gs)[0], sigma(gs)[0], a[0], s1[0]]))
    return torch.stack(rows).contiguous()


def inpaint_table(gamma: torch.Tensor, T: int) -> torch.Tensor:
    """fp32 [T,4] on the CPU: inpaint_rows over the unit grid (row s: t = s+1)."""
    return inpaint_rows(gamma, T, list(range(T + 1)))


def prediction_rows(gamma: torch.Tensor, T: int, grid) -> torch.Tensor:
    """fp32 [n,2] on the CPU over a step grid; row k = (alpha_t, sigma_t) at t = tau_{k+1}, the level of the state row k
    starts from: what a recorded trajectory's clean-ligand estimate (z - sigma_t eps) / alpha_t divides by (DESIGN.md
    section 6.4).  Scalar fp32 ops like coefficient_rows, so row k equals start_coefficients(gamma, tau_{k+1}) bit for
    bit.  The same for every eta."""
    g = gamma.detach().float().cpu()
    rows = []
    for s_int, t_int in zip(grid[:-1], grid[1:]):
        _, gt, _ = _row_gammas(g, T, s_int, t_int)
        rows.append(torch.stack([alpha(gt)[0], sigma(gt)[0]]))
    return torch.stack(rows).contiguous()


def prediction_table(gamma: torch.Tensor, T: int) -> torch.Tensor:
    """fp32 [T,2] on the CPU: prediction_rows over the unit grid (row s: t = s+1)."""
    return prediction_rows(gamma, T, list(range(T + 1)))


SOLVERS = ("dpmpp_2m",)


def multistep_rows(gamma: torch.Tensor, T: int, grid) -> torch.Tensor:
    """fp32 [n,4] on the CPU over a step grid; row k = (c_k, alpha_t, sigma_t, 0) with t = tau_{k+1}: the second-order
    correction z_s += c_k (x^_k - x^_prev) of a DPM-Solver++(2M) run on top of the DDIM eta = 0 row k (DESIGN.md section
    6.5), and the level its clean-ligand estimate x^_k = (z - sigma_t eps) / alpha_t divides by.  Columns 1-2 are
    prediction_rows' bit for bit.  With h_k = (gamma[tau_{k+1}] - gamma[tau_k]) / 2, the log-SNR step of row k,
        c_k = alpha_{tau_k} (-expm1(-h_k)) h_k / (2 h_{k+1})
    evaluated in fp64 from the fp32 gammas and rounded once to fp32, like _ddim_columns.  c is 0 on the top row k = n-1
    (no history) and on row 0 (the large log-SNR jump into tau_0 = 0, where a second-order correction does harm)."""
    g = gamma.detach().float().cpu()
    n = len(grid) - 1
    gam, rows = [], []
    for s_int, t_int in zip(grid[:-1], grid[1:]):
        gs, gt, _ = _row_gammas(g, T, s_int, t_int)
        gam.append((float(gs[0]), float(gt[0])))
        rows.append([alpha(gt)[0], sigma(gt)[0]])
    out = torch.zeros(n, 4, dtype=torch.float32)
    for k in range(n):
        out[k, 1], out[k, 2] = rows[k]
        if 1 <= k <= n - 2:
            gs, gt = gam[k]
            h = 0.5 * (torch.tensor(gt, dtype=torch.float64) - torch.tensor(gs, dtype=torch.float64))
            h_prev = 0.5 * (torch.tensor(gam[k + 1][1], dtype=torch.float64) - torch.tensor(gam[k + 1][0],
                                                                                              dtype=torch.float64))
            a_s = torch.sqrt(torch.sigmoid(-torch.tensor(gs, dtype=torch.float64)))
            out[k, 0] = (a_s * -torch.expm1(-h) * h / (2 * h_prev)).float()
    return out.contiguous()


def frame_levels(grid, n: int, every: int) -> torch.Tensor:
    """long [ceil(n / every) + 1]: the diffusion level of every frame a run of n steps records with stride `every`, the
    run starting from row n-1 of a table over `grid`: frame j < m is the state before executed step j*every, at level
    tau_{n - j*every}; the last frame, the output, is at level 0."""
    m = -(-int(n) // int(every))
    return torch.tensor([grid[int(n) - j * int(every)] for j in range(m)] + [0], dtype=torch.long)


def start_coefficients(gamma: torch.Tensor, t0: int):
    """(alpha_t0, sigma_t0) as Python floats holding fp32 values: the level a start ligand is noised to before the
    reverse loop runs from step t0 (ligand optimisation by partial noising).  Evaluated like coefficient_table, with the
    scalar fp32 ops on a 1-element tensor gamma[t0]."""
    g = gamma.detach().float().cpu()
    g0 = g[torch.full((1,), int(t0), dtype=torch.long)]
    return float(alpha(g0)[0]), float(sigma(g0)[0])
