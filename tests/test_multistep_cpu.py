"""CPU: second-order multistep sampling (solver="dpmpp_2m", DESIGN.md section 6.5) -- the multistep rows against
prediction_rows and an independent fp64 evaluation, accuracy against the exact probability-flow ODE of Gaussian data,
the multistep reference the GPU tests hold the captured loop to (multistep_oracle below), the argument checks that must
fire before any device work, and the new C entry points."""
from pathlib import Path

import pytest
import torch

from helpers import flat_batch, load_golden, oracle_cfg
from oracle import fast as Q, flat, schedule as S
from oracle.optimize import partial_noise, start_coefficients


def multistep_oracle(dyn_fn, gamma, T, batch, noise_fn, n, init_lig_pos=None, start=None, lig_feat_norm_constant=1.0,
                     atom_nf=None, zero_c=False, on_step=None):
    """DPM-Solver++(2M) with data prediction on the n-step grid over [0, t_start], in its direct form and the batch
    dtype: with x^ = (z_t - sigma_t eps^) / alpha_t and h = lambda_s - lambda_t (lambda = log(alpha / sigma)),
        z_s = (sigma_s / sigma_t) z_t + alpha_s (1 - e^{-h}) D,   D = x^ + (h / 2 h_prev) (x^ - x^_prev),
    D = x^ on the first executed row and on row 0 (and everywhere with zero_c=True).  x^_prev is the previous executed
    row's estimate, its positions moved by every ligand-COM removal since.  Frame setup and restore are oracle/fast.py's
    (pure noise with init_lig_pos, or ``start = (x_in, h_in, t0)``); noise_fn(k, 0, 0, shape) is drawn for every row,
    as a DDIM eta = 0 run draws, and not used.  on_step(k, x^, h^, z positions, kp positions) is called with each
    row's estimate before its step (the recorded prediction frame).  Not the product's closed form."""
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    dt = batch.kp_x.dtype
    init_kp_com = flat._segment_mean(batch.kp_x, kp_b, B)
    N_l = int(batch.lig_n.sum())
    shape = (N_l, 3 + atom_nf)
    if start is None:
        t_start = T
        batch.kp_x = batch.kp_x - init_lig_pos.to(dt)[kp_b]
        d = noise_fn(-1, 0, 0, shape).to(dt)
        batch.lig_x, batch.lig_h = d[:, :3], d[:, 3:]
        batch = flat.remove_com(batch, lig_b, kp_b, "ligand")
    else:
        x_in, h_in, t_start = start
        a, s = start_coefficients(gamma, t_start)
        batch = partial_noise(batch, x_in, h_in, a, s, noise_fn(-1, 0, 0, shape).to(dt), lig_feat_norm_constant)
    tau = Q.grid(t_start, n)
    prev = None
    for k in reversed(range(int(n))):
        noise_fn(k, 0, 0, shape)
        t, gamma_s, gamma_t = Q._levels(gamma, T, tau[k], tau[k + 1], B)
        col = lambda v: v[lig_b].view(-1, 1).to(dt)
        a_s, s_s, a_t, s_t = col(S.alpha(gamma_s)), col(S.sigma(gamma_s)), col(S.alpha(gamma_t)), col(S.sigma(gamma_t))
        eps_h, eps_x = dyn_fn(batch, t)
        x_hat = (batch.lig_x - s_t * eps_x) / a_t
        h_hat = (batch.lig_h - s_t * eps_h) / a_t
        if on_step is not None:
            on_step(k, x_hat, h_hat, batch.lig_x, batch.kp_x)
        h = torch.log(a_s / s_s) - torch.log(a_t / s_t)
        if prev is None or k == 0 or zero_c:
            dx, dh = x_hat, h_hat
        else:
            w = h / (2 * prev[2])
            dx, dh = x_hat + w * (x_hat - prev[0]), h_hat + w * (h_hat - prev[1])
        gain = a_s * -torch.expm1(-h)
        batch.lig_x = (s_s / s_t) * batch.lig_x + gain * dx
        batch.lig_h = (s_s / s_t) * batch.lig_h + gain * dh
        com = flat._segment_mean(batch.lig_x, lig_b, B)
        batch = flat.remove_com(batch, lig_b, kp_b, "ligand")
        prev = (x_hat - com[lig_b], h_hat, h)
    batch = flat.remove_com(batch, lig_b, kp_b, "receptor")
    batch.lig_x = batch.lig_x + init_kp_com[lig_b]
    batch.kp_x = batch.kp_x + init_kp_com[kp_b]
    batch.lig_h = batch.lig_h * lig_feat_norm_constant
    ptr = torch.zeros(B + 1, dtype=torch.long)
    ptr[1:] = torch.cumsum(batch.lig_n, 0)
    return ([batch.lig_x[ptr[i]:ptr[i + 1]].clone() for i in range(B)],
            [batch.lig_h[ptr[i]:ptr[i + 1]].clone() for i in range(B)])


def _gamma(T=1000):
    """The polynomial_2 schedule of a default KeypointDiffusion (precision 1e-4)."""
    return S.gamma_table(T, 1e-4)


@pytest.mark.parametrize("t_start,n", [(1000, 1), (1000, 2), (1000, 3), (1000, 5), (1000, 20), (1000, 300),
                                       (1000, 1000), (7, 3), (40, 40)])
def test_multistep_rows(t_start, n):
    """c is 0 exactly on the top row and row 0; columns 1-2 are prediction_rows bit for bit, column 3 is 0; c is the
    fp64 formula alpha_{tau_k} (-expm1(-h_k)) h_k / (2 h_{k+1}), evaluated independently here, rounded to fp32."""
    from keypoint_diffusion_b200.schedule import multistep_rows, prediction_rows, step_grid
    T = 1000
    gamma = _gamma(T)
    tau = step_grid(t_start, n)
    rows = multistep_rows(gamma, T, tau)
    assert rows.shape == (n, 4) and rows.dtype == torch.float32 and rows.is_contiguous()
    assert float(rows[0, 0]) == 0.0 and float(rows[n - 1, 0]) == 0.0
    assert torch.equal(rows[:, 1:3], prediction_rows(gamma, T, tau))
    assert bool((rows[:, 3] == 0).all())
    g = gamma.double()
    lam = -g / 2
    for k in range(1, n - 1):
        h, h_prev = lam[tau[k]] - lam[tau[k + 1]], lam[tau[k + 1]] - lam[tau[k + 2]]
        want = torch.sqrt(torch.sigmoid(-g[tau[k]])) * -torch.expm1(-h) * h / (2 * h_prev)
        assert h > 0 and h_prev > 0
        assert abs(float(rows[k, 0]) - float(want)) <= 6e-8 * abs(float(want)), k
        assert float(rows[k, 0]) > 0


def _gaussian_run(rows, ms, tau, al, sg, m, v, z, second_order):
    """The kernel's closed form z/a - vt eps^ + c (x^_k - x^_prev) in fp64 with the fp32 rows and the ideal denoiser of
    x ~ N(m, v) per coordinate (as eps^); no COM removal (the toy has no frame)."""
    prev = None
    n = len(tau) - 1
    for k in reversed(range(n)):
        t = tau[k + 1]
        eps = (z - al[t] * (m + al[t] * v * (z - al[t] * m) / (al[t] ** 2 * v + sg[t] ** 2))) / sg[t]
        x_hat = (z - ms[k, 2] * eps) / ms[k, 1]         # as the kernel forms it, from eps^ and the fp32 row
        z_new = z / rows[k, 0] - rows[k, 1] * eps
        if second_order and prev is not None:
            z_new = z_new + ms[k, 0] * (x_hat - prev)
        prev, z = x_hat, z_new
    return z


def test_gaussian_data_beats_ddim():
    """Gaussian data x ~ N(m, v) per coordinate (256 coordinates, m ~ N(0, 1), v ~ U(0.05, 0.55)): the ideal denoiser is
    x^ = m + alpha v (z - alpha m) / (alpha^2 v + sigma^2) and the exact probability-flow map is affine,
    z_s = alpha_s m + sqrt(alpha_s^2 v + sigma_s^2) (z_t - alpha_t m) / sqrt(alpha_t^2 v + sigma_t^2).  From z_T the
    2M rows must end closer to the exact z_0 than the DDIM eta = 0 rows at every n, and at most 1/5 of DDIM's error from
    n = 20 on.  Measured max errors at tau_0 (DDIM, 2M, ratio):
        n = 5:  0.41, 0.23, 0.56      n = 10: 0.22, 0.073, 0.34     n = 20: 0.11, 0.0077, 0.069
        n = 40: 0.056, 0.0072, 0.13   n = 80: 0.028, 0.0037, 0.13
    No clean order-2 slope is asserted: at large n the first-order step across the final log-SNR jump (row 0) dominates."""
    from keypoint_diffusion_b200.schedule import coefficient_rows, multistep_rows, step_grid
    T = 1000
    gamma = _gamma(T)
    g64 = gamma.double()
    al, sg = torch.sqrt(torch.sigmoid(-g64)), torch.sqrt(torch.sigmoid(g64))
    gen = torch.Generator().manual_seed(0)
    m = torch.randn(256, generator=gen, dtype=torch.float64)
    v = 0.05 + 0.5 * torch.rand(256, generator=gen, dtype=torch.float64)
    z_T = al[T] * m + torch.sqrt(al[T] ** 2 * v + sg[T] ** 2) * torch.randn(256, generator=gen, dtype=torch.float64)
    exact = al[0] * m + torch.sqrt(al[0] ** 2 * v + sg[0] ** 2) * (z_T - al[T] * m) / torch.sqrt(al[T] ** 2 * v + sg[T] ** 2)
    for n in (5, 10, 20, 40, 80):
        tau = step_grid(T, n)
        rows = coefficient_rows(gamma, T, tau, eta=0.0).double()
        ms = multistep_rows(gamma, T, tau).double()
        e1 = float((_gaussian_run(rows, ms, tau, al, sg, m, v, z_T, False) - exact).abs().max())
        e2 = float((_gaussian_run(rows, ms, tau, al, sg, m, v, z_T, True) - exact).abs().max())
        print(f"n={n}: DDIM {e1:.3g}  2M {e2:.3g}  ratio {e2 / e1:.3g}")
        assert e2 < e1, n
        if n >= 20:
            assert e2 <= e1 / 5, n


def _loop_fixture(dtype=torch.float32):
    fx = load_golden("loop_egnn")
    kw, F = fx["kwargs"], fx["atom_nf"]
    cfg = oracle_cfg("egnn", kw, F, fx["rec_nf"])
    sd = {k: v.to(dtype) if v.is_floating_point() else v for k, v in fx["state_dict"].items()}
    dyn = lambda b, t: flat.egnn_forward(sd, cfg, b, t)
    return fx, dyn, F


@pytest.mark.parametrize("from_start", [False, True])
def test_oracle_with_zero_c_is_ddim_eta0(from_start):
    """On the golden loop fixture in fp64: the 2M loop with every correction dropped equals the DDIM eta = 0 grid loop
    of oracle/fast.py to fp64 rounding, from pure noise (n = 5 over [0, T]) and from a start ligand (n = 3 over [0, 7]);
    with the corrections it differs."""
    fx, dyn, F = _loop_fixture(torch.float64)
    T, gamma = fx["T"], fx["state_dict"]["gamma.gamma"]
    lig_n = fx["inputs"]["lig_n"]
    N_l = int(lig_n.sum())
    g = torch.Generator().manual_seed(3)
    draws = {}

    def fn(k, u, kind, shape):
        if (k, u, kind) not in draws:
            draws[(k, u, kind)] = torch.randn(N_l, 3 + F, generator=g, dtype=torch.float64)
        return draws[(k, u, kind)]
    lig_b = torch.arange(len(lig_n)).repeat_interleave(lig_n)
    x_in = fx["init_lig_pos"][lig_b].double() + torch.randn(N_l, 3, generator=g, dtype=torch.float64)
    h_in = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).double()
    n, kw = (3, dict(start=(x_in, h_in, 7))) if from_start else (5, dict(init_lig_pos=fx["init_lig_pos"].double()))
    b = lambda: flat_batch(fx["inputs"], torch.float64)
    ddim = Q.sample_from_encoded_receptors(dyn, gamma, T, b(), fn, n, eta=0.0, atom_nf=F, **kw)
    zero = multistep_oracle(dyn, gamma, T, b(), fn, n, atom_nf=F, zero_c=True, **kw)
    full = multistep_oracle(dyn, gamma, T, b(), fn, n, atom_nf=F, **kw)
    for i in (0, 1):
        a, z, f = torch.cat(ddim[i]), torch.cat(zero[i]), torch.cat(full[i])
        err = float((a - z).abs().max() / a.abs().max())
        assert err < 1e-12, (i, err)
        assert float((a - f).abs().max() / a.abs().max()) > 1e-6, i


def test_oracle_ignores_the_step_draws():
    """The 2M loop does not depend on its per-step draws (only on the initial one)."""
    fx, dyn, F = _loop_fixture()
    T, gamma = fx["T"], fx["state_dict"]["gamma.gamma"]
    N_l = int(fx["inputs"]["lig_n"].sum())
    outs = []
    for seed in (0, 1):
        g = torch.Generator().manual_seed(seed)
        d0 = torch.randn(N_l, 3 + F, generator=torch.Generator().manual_seed(9))
        fn = lambda k, u, kind, shape: d0 if k < 0 else torch.randn(shape, generator=g)
        outs.append(multistep_oracle(dyn, gamma, T, flat_batch(fx["inputs"]), fn, 5,
                                     init_lig_pos=fx["init_lig_pos"], atom_nf=F))
    assert torch.equal(torch.cat(outs[0][0]), torch.cat(outs[1][0]))
    assert torch.equal(torch.cat(outs[0][1]), torch.cat(outs[1][1]))


def _cpu_model():
    import os
    from shipped_cases import shipped_configs
    from keypoint_diffusion_b200 import model_from_config
    os.chdir(Path(__file__).resolve().parents[1])
    torch.manual_seed(0)
    return model_from_config(shipped_configs()["egnn_20kp"])


def test_solver_arguments_are_checked_before_any_device_work(monkeypatch):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    model = _cpu_model()
    F = model.n_lig_features

    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    monkeypatch.setattr(model, "_encode_all", no_device)
    graphs = [object(), object()]
    sizes = [[20, 20], [20]]
    lig = (torch.zeros(20, 3), torch.zeros(20, F))
    frag = (torch.zeros(3, 3), torch.zeros(3, F))
    bad = [dict(solver="dpmpp_3m"), dict(solver=""), dict(solver=True), dict(solver=2), dict(solver="DPMPP_2M"),
           dict(solver="dpmpp_2m", eta=0.0), dict(solver="dpmpp_2m", eta=1.0, timesteps=10),
           dict(solver="dpmpp_2m", capacity=False), dict(solver="dpmpp_2m", timesteps=0)]
    for kw in bad:
        with pytest.raises(ValueError, match="solver|timesteps"):
            model._sample(graphs, sizes, **kw)
        with pytest.raises(ValueError, match="solver|timesteps"):
            model.sample_given_pocket(object(), torch.tensor([20]), **kw)
    with pytest.raises(ValueError, match="fragment"):
        model._sample(graphs, sizes, fragments=[frag, None], solver="dpmpp_2m")
    with pytest.raises(ValueError, match="fragment"):
        model.sample_given_pocket(object(), torch.tensor([20]), fragment=frag, solver="dpmpp_2m", timesteps=10)
    with pytest.raises(ValueError, match="start_step"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=0, solver="dpmpp_2m")
    with pytest.raises(ValueError, match="timesteps"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=10, timesteps=11, solver="dpmpp_2m")

    pk = synthetic.keypoint_pocket(0, 20, 256, 0, 8.0)
    g = HeteroBatch.from_pockets([pk], [20, 12], F)
    for kw in bad:
        with pytest.raises(ValueError, match="solver|timesteps"):
            model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(2, 3), **kw)
    n = 32
    with pytest.raises(ValueError, match="fragment"):
        model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(2, 3), solver="dpmpp_2m",
                                            fixed_mask=torch.ones(n, dtype=torch.bool), fixed_pos=torch.zeros(n, 3),
                                            fixed_feat=torch.zeros(n, F))
    start = dict(start_pos=torch.zeros(n, 3), start_feat=torch.zeros(n, F))
    with pytest.raises(ValueError, match="start_step"):
        model.sample_from_encoded_receptors(g, start_step=0, solver="dpmpp_2m", **start)


def test_multistep_entry_points_are_exported():
    import ctypes
    from keypoint_diffusion_b200 import _lib
    header = (Path(__file__).resolve().parents[1] / "include" / "kpdiff_b200.h").read_text()
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in ("kpd_ddpm_multistep_step", "kpd_sampler_enable_multistep", "kpd_sampler_set_multistep"):
        assert f"int {name}(" in header
        assert name in _lib.EXPORTED and hasattr(lib, name)
