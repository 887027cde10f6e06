"""CPU: fewer-step sampling -- the step grid, the strided ancestral and DDIM tables against the unit tables, the
ancestral rows and an ideal denoiser, the oracle's grid loops against the plain ones, the argument checks that must
fire before any device work, and the new C entry point."""
from pathlib import Path

import pytest
import torch

from helpers import flat_batch, load_golden, oracle_cfg
from oracle import fast as Q, flat, inpaint as I, optimize as O, schedule as S


def _gamma(T=1000):
    return S.gamma_table(T, 1e-5)


@pytest.mark.parametrize("t_start,n", [(1000, 1000), (1000, 300), (1000, 1), (1000, 7), (1000, 999), (7, 3), (1, 1),
                                       (12, 5)])
def test_step_grid(t_start, n):
    from keypoint_diffusion_b200.schedule import step_grid
    tau = step_grid(t_start, n)
    assert len(tau) == n + 1 and tau[0] == 0 and tau[-1] == t_start
    assert all(a < b for a, b in zip(tau[:-1], tau[1:]))
    assert tau == [k * t_start // n for k in range(n + 1)] == Q.grid(t_start, n)
    if n == t_start:
        assert tau == list(range(t_start + 1))
    if (t_start, n) == (1000, 300):
        assert tau[:4] == [0, 3, 6, 10] and tau[299] == 996
        assert set(b - a for a, b in zip(tau[:-1], tau[1:])) == {3, 4}


@pytest.mark.parametrize("t_start,n", [(1000, 0), (1000, 1001), (5, 6), (0, 1)])
def test_step_grid_rejects_bad_counts(t_start, n):
    from keypoint_diffusion_b200.schedule import step_grid
    with pytest.raises(ValueError):
        step_grid(t_start, n)


def test_unit_grid_tables_are_the_step_tables():
    """n = T gives coefficient_table / inpaint_table (and the oracle's independent table) bit for bit; the grid over
    [0, t0] at n = t0 gives their first t0 rows."""
    from keypoint_diffusion_b200.schedule import (coefficient_rows, coefficient_table, inpaint_rows, inpaint_table,
                                                  step_grid)
    T = 1000
    gamma = _gamma(T)
    coef, coef2 = coefficient_table(gamma, T), inpaint_table(gamma, T)
    assert torch.equal(coefficient_rows(gamma, T, step_grid(T, T)), coef)
    assert torch.equal(inpaint_rows(gamma, T, step_grid(T, T)), coef2)
    assert torch.equal(coef, S.coefficient_table(gamma, T))
    for t0 in (1, 7, 300):
        assert torch.equal(coefficient_rows(gamma, T, step_grid(t0, t0)), coef[:t0])
        assert torch.equal(inpaint_rows(gamma, T, step_grid(t0, t0)), coef2[:t0])


def test_strided_rows_are_the_reference_step_at_s_t():
    """Row k of a strided grid is the reference's step at (s, t) = (tau_k, tau_{k+1}): the oracle's per-step
    coefficients restated independently, and the t column tau_{k+1} / T."""
    from keypoint_diffusion_b200.schedule import coefficient_rows, inpaint_rows, step_grid
    T = 1000
    gamma = _gamma(T)
    tau = step_grid(T, 300)
    rows, rows2 = coefficient_rows(gamma, T, tau), inpaint_rows(gamma, T, tau)
    assert rows.shape == (300, 4) and rows.dtype == torch.float32
    for k in (0, 1, 150, 299):
        gs, gt = gamma[tau[k]:tau[k] + 1], gamma[tau[k + 1]:tau[k + 1] + 1]
        s2, s1, a = S.sigma_and_alpha_t_given_s(gt, gs)
        want = torch.stack([a[0], (s2 / a / S.sigma(gt))[0], (s1 * S.sigma(gs) / S.sigma(gt))[0],
                            (torch.full((1,), tau[k + 1]) / T)[0]])
        assert torch.equal(rows[k], want), k
        assert torch.equal(rows2[k], torch.stack([S.alpha(gs)[0], S.sigma(gs)[0], a[0], s1[0]])), k


def _ancestral_fp64(gamma, tau):
    """(var_terms, sigma) of the ancestral rows, the reference's formulas evaluated in fp64 from the fp32 gammas."""
    g = gamma.double()
    rows = []
    for s, t in zip(tau[:-1], tau[1:]):
        gs, gt = g[s:s + 1], g[t:t + 1]
        s2, s1, a = S.sigma_and_alpha_t_given_s(gt, gs)
        rows.append(torch.stack([(s2 / a / S.sigma(gt))[0], (s1 * S.sigma(gs) / S.sigma(gt))[0]]))
    return torch.stack(rows)


@pytest.mark.parametrize("n", [1, 7, 300, 1000])
def test_ddim_rows_against_ancestral(n):
    """eta = 1: columns 0 and 3 are the ancestral row's bit for bit; columns 1 and 2 are the ancestral formulas rounded
    once to fp32 (within 1e-7 relative of their fp64 values), so they differ from the fp32 ancestral rows only by the
    rounding of those rows' scalar fp32 evaluation (up to 3.2e-5 relative at n = 1000, where expm1 takes the difference
    of two fp32 softplus values; within 1e-6 up to n = 50).  eta = 0: column 2 is 0."""
    from keypoint_diffusion_b200.schedule import coefficient_rows, step_grid
    T = 1000
    gamma = _gamma(T)
    tau = step_grid(T, n)
    anc = coefficient_rows(gamma, T, tau)
    rel = lambda a, b: float(((a.double() - b.double()).abs() / b.double().abs()).max())
    for eta in (1.0, 0.5, 0.0):
        dd = coefficient_rows(gamma, T, tau, eta=eta)
        assert torch.equal(dd[:, 0], anc[:, 0]) and torch.equal(dd[:, 3], anc[:, 3])
        assert bool((dd[:, 1] > 0).all()) and bool((dd[:, 2] >= 0).all())
        if eta == 1.0:
            assert rel(dd[:, 1:3], _ancestral_fp64(gamma, tau)) < 1e-7
            assert rel(dd[:, 1:3], anc[:, 1:3]) < (1e-6 if n <= 50 else 5e-5)
        if eta == 0.0:
            assert bool((dd[:, 2] == 0).all())


@pytest.mark.parametrize("n", [1, 7, 50, 1000])
def test_ddim_eta0_rows_follow_an_ideal_denoiser(n):
    """One-point data x*: with the ideal eps^ = (z - alpha_t x*) / sigma_t, the eta = 0 rows (fp32) applied through the
    step kernel's formula z/a - vt eps^ keep z_k = alpha_{tau_k} x* + sigma_{tau_k} e from z_n = alpha_T x* + sigma_T e
    within 1e-5 / min_k a_k.  Pins the sign and form of the DDIM vt column independently of the oracle.  The bound
    scales with 1 / alpha_t|s because the formula divides z by the fp32 column 0 (the ancestral value, whose scalar
    fp32 evaluation is off by up to ~5e-7 relative) and subtracts vt eps^ of the same size: at n = 1, 1/a = 316 and
    the error is 1.7e-5; at n = 7 it is 9.4e-5 with 1/a = 85; from n = 50 on it is below 6e-6."""
    from keypoint_diffusion_b200.schedule import coefficient_rows, step_grid
    T = 1000
    gamma = _gamma(T)
    tau = step_grid(T, n)
    rows = coefficient_rows(gamma, T, tau, eta=0.0).double()
    g = torch.Generator().manual_seed(0)
    x_star = torch.randn(64, generator=g, dtype=torch.float64)
    e = torch.randn(64, generator=g, dtype=torch.float64)
    g64 = gamma.double()
    al, sg = torch.sqrt(torch.sigmoid(-g64)), torch.sqrt(torch.sigmoid(g64))
    z = al[T] * x_star + sg[T] * e
    worst = 0.0
    for k in reversed(range(n)):
        t = tau[k + 1]
        eps = (z - al[t] * x_star) / sg[t]
        z = z / rows[k, 0] - rows[k, 1] * eps + rows[k, 2] * 0.0
        worst = max(worst, float((z - (al[tau[k]] * x_star + sg[tau[k]] * e)).abs().max()))
    assert worst < 1e-5 / float(rows[:, 0].min()), worst


def test_ddim_rows_match_the_oracle_direct_form():
    """The product's closed form z/a - vt eps^ + sg xi with the (fp32) DDIM rows against the oracle's direct form in
    fp64, for one strided step and a fixed eps^: equal up to the fp32 rounding of the rows."""
    from keypoint_diffusion_b200.schedule import coefficient_rows
    T = 1000
    gamma = _gamma(T)
    g = torch.Generator().manual_seed(1)
    lig_n, kp_n = torch.tensor([4, 6]), torch.tensor([3, 2])
    for s_int, t_int, eta in ((3, 17, 0.0), (400, 500, 0.3), (990, 1000, 1.0), (0, 1000, 0.0)):
        x = torch.randn(10, 3, generator=g, dtype=torch.float64)
        h = torch.randn(10, 5, generator=g, dtype=torch.float64)
        ex, eh = torch.randn_like(x), torch.randn_like(h)
        nx, nh = torch.randn_like(x), torch.randn_like(h)
        fb = flat.FlatBatch(lig_n=lig_n, kp_n=kp_n, kp_x=torch.zeros(5, 3, dtype=torch.float64),
                            kp_h=torch.zeros(5, 1), kk_src=torch.zeros(0, dtype=torch.long),
                            kk_dst=torch.zeros(0, dtype=torch.long), lig_x=x.clone(), lig_h=h.clone())
        ox, oh = Q.posterior(lambda b, t: (eh, ex), gamma, T, s_int, t_int, fb, nx, nh, eta=eta)
        a, vt, sg, _ = coefficient_rows(gamma, T, [s_int, t_int], eta=eta)[0].double()
        px, ph = x / a - vt * ex + sg * nx, h / a - vt * eh + sg * nh
        err = max(float((px - ox).abs().max() / ox.abs().max()), float((ph - oh).abs().max() / oh.abs().max()))
        assert err < 1e-6, (s_int, t_int, eta, err)


def _loop_fixture():
    fx = load_golden("loop_egnn")
    kw, F = fx["kwargs"], fx["atom_nf"]
    cfg = oracle_cfg("egnn", kw, F, fx["rec_nf"])
    dyn = lambda b, t: flat.egnn_forward(fx["state_dict"], cfg, b, t)
    return fx, dyn, F


def test_oracle_grid_loops_at_the_unit_grid_are_the_plain_loops():
    """n = t_start: the grid loop is flat's plain loop, optimize's loop from a start and inpaint's loop bit for bit."""
    fx, dyn, F = _loop_fixture()
    T, gamma = fx["T"], fx["state_dict"]["gamma.gamma"]
    lig_n = fx["inputs"]["lig_n"]
    N_l = int(lig_n.sum())
    g = torch.Generator().manual_seed(5)
    draws = {}

    def draw(k, u=0, kind=0):
        if (k, u, kind) not in draws:
            draws[(k, u, kind)] = torch.randn(N_l, 3 + F, generator=g)
        return draws[(k, u, kind)]

    fast_fn = lambda k, u, kind, shape: draw(k, u, kind)
    plain_fn = lambda s, kind, shape: draw(s)[:, :3] if kind == "x" else draw(s)[:, 3:]
    pos, feat = flat.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fx["init_lig_pos"],
                                                   plain_fn, atom_nf=F)
    qpos, qfeat = Q.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fast_fn, T,
                                                  init_lig_pos=fx["init_lig_pos"], atom_nf=F)
    assert torch.equal(torch.cat(pos), torch.cat(qpos)) and torch.equal(torch.cat(feat), torch.cat(qfeat))
    lig_b = torch.arange(len(lig_n)).repeat_interleave(lig_n)
    x_in = fx["init_lig_pos"][lig_b] + torch.randn(N_l, 3, generator=g)
    h_in = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).float()
    t0 = 7
    pos, feat = O.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), x_in, h_in, t0, fast_fn,
                                                atom_nf=F)
    qpos, qfeat = Q.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fast_fn, t0,
                                                  start=(x_in, h_in, t0), atom_nf=F)
    assert torch.equal(torch.cat(pos), torch.cat(qpos)) and torch.equal(torch.cat(feat), torch.cat(qfeat))
    mask = torch.zeros(N_l, dtype=torch.bool)
    mask[:3] = True
    pos, feat = I.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fx["init_lig_pos"], fast_fn,
                                                mask, x_in, h_in, resamplings=2, atom_nf=F)
    qpos, qfeat = Q.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fast_fn, T,
                                                  init_lig_pos=fx["init_lig_pos"], fragment=(mask, x_in, h_in),
                                                  resamplings=2, atom_nf=F)
    assert torch.equal(torch.cat(pos), torch.cat(qpos)) and torch.equal(torch.cat(feat), torch.cat(qfeat))


def test_oracle_ddim_eta0_loop_ignores_the_draws():
    """eta = 0: the oracle's DDIM loop does not depend on the per-step draws (only on the initial one)."""
    fx, dyn, F = _loop_fixture()
    T, gamma = fx["T"], fx["state_dict"]["gamma.gamma"]
    N_l = int(fx["inputs"]["lig_n"].sum())
    outs = []
    for seed in (0, 1):
        g = torch.Generator().manual_seed(seed)
        d0 = torch.randn(N_l, 3 + F, generator=torch.Generator().manual_seed(9))
        fn = lambda k, u, kind, shape: d0 if k < 0 else torch.randn(shape, generator=g)
        outs.append(Q.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fn, 5, eta=0.0,
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


def test_schedule_arguments_are_checked_before_any_device_work(monkeypatch):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    model = _cpu_model()
    F, T = model.n_lig_features, model.n_timesteps

    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    monkeypatch.setattr(model, "_encode_all", no_device)
    graphs = [object(), object()]
    sizes = [[20, 20], [20]]
    lig = (torch.zeros(20, 3), torch.zeros(20, F))
    bad = [dict(timesteps=0), dict(timesteps=T + 1), dict(timesteps=-3), dict(timesteps=2.0), dict(timesteps=True),
           dict(timesteps="50"), dict(eta=-0.1), dict(eta=1.5), dict(eta=float("nan")), dict(eta=float("inf")),
           dict(eta="0"), dict(eta=True), dict(timesteps=50, capacity=False), dict(eta=0.0, capacity=False)]
    for kw in bad:
        with pytest.raises(ValueError, match="timesteps|eta|capacity"):
            model._sample(graphs, sizes, **kw)
        with pytest.raises(ValueError, match="timesteps|eta|capacity"):
            model.sample_given_pocket(object(), torch.tensor([20]), **kw)
    # with start ligands the grid spans [0, t0]
    with pytest.raises(ValueError, match="timesteps"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=10, timesteps=11)
    with pytest.raises(ValueError, match="timesteps"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=0, timesteps=1)

    pk = synthetic.keypoint_pocket(0, 20, 256, 0, 8.0)
    g = HeteroBatch.from_pockets([pk], [20, 12], F)
    for kw in bad:
        with pytest.raises(ValueError, match="timesteps|eta|capacity"):
            model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(2, 3), **kw)
    start = dict(start_pos=torch.zeros(32, 3), start_feat=torch.zeros(32, F))
    with pytest.raises(ValueError, match="timesteps"):
        model.sample_from_encoded_receptors(g, start_step=30, timesteps=31, **start)
    with pytest.raises(ValueError, match="timesteps"):
        model.sample_from_encoded_receptors(g, start_step=0, timesteps=1, **start)
    # the per-step API: t must be above s
    for s, t in ((0.5, 0.5), (0.5, 0.4), (0.3, 1.2)):
        with pytest.raises(ValueError, match="s < t"):
            model.sample_p_zs_given_zt(torch.tensor([s]), torch.tensor([t]), object())


def test_schedule_entry_point_is_exported():
    import ctypes
    from keypoint_diffusion_b200 import _lib
    header = (Path(__file__).resolve().parents[1] / "include" / "kpdiff_b200.h").read_text()
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    assert "int kpd_sampler_set_schedule(" in header
    assert "kpd_sampler_set_schedule" in _lib.EXPORTED and hasattr(lib, "kpd_sampler_set_schedule")
