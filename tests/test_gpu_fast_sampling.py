"""GPU: fewer-step sampling (strided ancestral and DDIM steps on a step grid), held to the CPU restatement in
oracle/fast.py.

* the captured loop with a schedule and injected draws against the oracle's grid loop (<= 1e-3, the bar of the plain
  loop): plain, with fragments and from a start ligand; ancestral and DDIM steps;
* an explicit unit grid is the default run bit for bit (Philox and injected draws, from noise and from a start);
  at eta = 0 the per-step draws do not matter; one capture serves every schedule;
* the per-step API with a strided (s, t); full-size models, sub-batch agreement and the _sample /
  sample_given_pocket / sample_random_sizes drivers.
"""
import pytest
import torch

from helpers import flat_batch, rel_err
from test_gpu_inpaint import SIZES, _dense_model, _pockets, _slot
from test_gpu_optimize import _loop_case

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _rows(gamma, T, t_start, n, eta=None, dev=None):
    from keypoint_diffusion_b200.schedule import coefficient_rows, inpaint_rows, step_grid
    grid = step_grid(t_start, n)
    return (coefficient_rows(gamma, T, grid, eta).to(dev).contiguous(),
            inpaint_rows(gamma, T, grid).to(dev).contiguous())


def _draws(c, keys):
    draws = {k: torch.randn(c["N_l"], 3 + c["F"], generator=c["gen"]) for k in keys}
    noise = torch.stack([_slot(draws[k]) for k in keys]).to(_dev()).contiguous()
    return draws, noise


def _run(c, sampler, noise=None, seed=0):
    t_in = c["t_in"]
    init = c["fx"]["init_lig_pos"].to(_dev())
    x, h, _ = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), init, noise=noise, seed=seed)
    torch.cuda.synchronize()
    return x.clone(), h.clone()


@pytest.mark.parametrize("n,eta", [(5, None), (3, 0.0), (1, 0.5), (12, 1.0)])
@pytest.mark.parametrize("mode", ["fp32", "bf16x3"])
@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_loop_with_schedule_matches_oracle(arch, mode, n, eta):
    """The captured loop (steps_per_graph = 4) on the n-step grid with injected draws against the oracle's grid loop:
    n = 5 runs one replay and one eager step, 3 and 1 eager steps only, 12 three replays."""
    from oracle import fast as Q
    from keypoint_diffusion_b200 import ops
    c = _loop_case(arch, mode)
    dev, T, F = _dev(), c["T"], c["F"]
    keys = [(-1, 0, 0)] + [(k, 0, 0) for k in reversed(range(n))]
    draws, noise = _draws(c, keys)
    sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4)
    coef, _ = _rows(c["gamma"], T, T, n, eta, dev)
    sampler.set_schedule(coef)
    assert sampler.start_step == n and noise.shape[0] == sampler.noise_slots == n + 1
    x_lig, h_lig = _run(c, sampler, noise)
    pos, feat = Q.sample_from_encoded_receptors(c["dyn"], c["gamma"], T, flat_batch(c["fx"]["inputs"]),
                                                lambda k, u, kind, shape: draws[(k, u, kind)], n, eta=eta,
                                                init_lig_pos=c["fx"]["init_lig_pos"], atom_nf=F)
    ex, eh = rel_err(x_lig.cpu(), torch.cat(pos)), rel_err(h_lig.cpu(), torch.cat(feat))
    print(f"grid loop {arch} [{mode}] n={n} eta={eta}: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < 1e-3 and eh < 1e-3


def test_unit_grid_is_the_default_run():
    """An explicit schedule of every step (timesteps = t_start) gives the run without a schedule bit for bit, with
    Philox and with injected draws, from pure noise and from a start ligand at t0 = 7 (n = 7); restoring the default
    gives it again."""
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import start_coefficients
    c = _loop_case("gvp", "bf16x3")
    dev, T, F = _dev(), c["T"], c["F"]
    sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4)
    xs, hs = c["x_in"].to(dev), c["h_in"].to(dev)
    for t0 in (None, 7):
        t_start = T if t0 is None else t0
        if t0 is not None:
            sampler.set_start(t0, xs, hs, *start_coefficients(c["gamma"], t0))
        _, noise = _draws(c, list(range(t_start + 1)))
        outs = []
        for sched in (False, True, False):
            sampler.set_schedule(_rows(c["gamma"], T, t_start, t_start, None, dev)[0] if sched else None)
            outs.append((_run(c, sampler, seed=41), _run(c, sampler, noise=noise)))
        for a in outs[1:]:
            for (x0, h0), (x1, h1) in zip(outs[0], a):
                assert torch.equal(x0, x1) and torch.equal(h0, h1), t0


@pytest.mark.parametrize("eta", [None, 0.0])
@pytest.mark.parametrize("case", ["frag_r1", "frag_r2", "start", "start_frag_r2"])
def test_fragment_and_start_with_schedule_match_oracle(case, eta):
    """Fragments (r = 1, 2) on the 5-step grid over [0, T], and a start at t0 = 7 on the 3-step grid over [0, 7]
    (alone and with a fragment), ancestral and eta = 0, against the oracle's grid loop."""
    from oracle import fast as Q
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import start_coefficients
    c = _loop_case("gvp", "bf16x3")
    dev, T, F, N_l, lig_n = _dev(), c["T"], c["F"], c["N_l"], c["lig_n"].tolist()
    r = 2 if case.endswith("r2") else 1
    frag = case.startswith("frag") or case.endswith("frag_r2")
    t0 = 7 if case.startswith("start") else None
    t_start, n = (T, 5) if t0 is None else (t0, 3)
    mask = torch.zeros(N_l, dtype=torch.bool)
    mask[0:3] = True
    mask[lig_n[0] + lig_n[1]:lig_n[0] + lig_n[1] + 4] = True
    if frag:
        keys = [(-1, 0, 0)] + [(k, u, kind) for k in reversed(range(n)) for u in range(r)
                               for kind in range(3 if u < r - 1 else 2)]
    else:
        keys = [(-1, 0, 0)] + [(k, 0, 0) for k in reversed(range(n))]
    draws, noise = _draws(c, keys)
    coef, coef2 = _rows(c["gamma"], T, t_start, n, eta, dev)
    if frag:
        sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4,
                              resamplings=r, inpaint_coef=_rows(c["gamma"], T, T, T, None, dev)[1])
        sampler.set_fragment(mask.to(dev, torch.uint8), c["x_in"].to(dev), c["h_in"].to(dev))
        sampler.set_schedule(coef, coef2)
    else:
        sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4)
        sampler.set_schedule(coef)
    xs, hs = c["x_in"].to(dev), c["h_in"].to(dev)
    if t0 is not None:
        sampler.set_start(n, xs, hs, *start_coefficients(c["gamma"], t0))
    assert noise.shape[0] == sampler.noise_slots
    x_lig, h_lig = _run(c, sampler, noise)
    pos, feat = Q.sample_from_encoded_receptors(
        c["dyn"], c["gamma"], T, flat_batch(c["fx"]["inputs"]), lambda k, u, kind, shape: draws[(k, u, kind)], n,
        eta=eta, init_lig_pos=c["fx"]["init_lig_pos"], start=None if t0 is None else (c["x_in"], c["h_in"], t0),
        fragment=(mask, c["x_in"], c["h_in"]) if frag else None, resamplings=r, atom_nf=F)
    ex, eh = rel_err(x_lig.cpu(), torch.cat(pos)), rel_err(h_lig.cpu(), torch.cat(feat))
    print(f"grid loop {case} eta={eta}: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < 1e-3 and eh < 1e-3


def test_eta0_ignores_the_step_draws():
    """At eta = 0 the reverse steps are deterministic: new values in every per-step noise slot (slot 0, the initial
    draw, kept) leave the output bit-identical; an ancestral schedule does change."""
    from keypoint_diffusion_b200 import ops
    c = _loop_case("egnn", "bf16x3")
    dev, T, F = _dev(), c["T"], c["F"]
    n = 5
    sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4)
    _, noise = _draws(c, list(range(n + 1)))
    other = noise.clone()
    other[1:] = torch.randn(other[1:].shape, generator=c["gen"]).to(dev)
    for eta, same in ((0.0, True), (None, False)):
        sampler.set_schedule(_rows(c["gamma"], T, T, n, eta, dev)[0])
        (x0, h0), (x1, h1) = _run(c, sampler, noise), _run(c, sampler, other)
        assert (torch.equal(x0, x1) and torch.equal(h0, h1)) == same, eta


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_strided_per_step_api_matches_oracle(arch):
    """sample_p_zs_given_zt(s = 3/T, t = 5/T) takes the strided step (row (3, 5), Philox key 3) -- against the oracle's
    step fed the same denoiser output (<= 1e-6); unit steps still match the plain step."""
    from oracle import fast as Q
    from keypoint_diffusion_b200.utils import get_batch_idxs
    from test_gpu_cases import _module_case
    _, model, g_cpu = _module_case(arch)
    dev = _dev()
    T = model.n_timesteps
    gamma = model.gamma.gamma.detach().float().cpu()
    gen = torch.Generator().manual_seed(0)
    nx, nh = torch.randn(39, 3, generator=gen), torch.randn(39, 10, generator=gen)
    for s_int, t_int in ((3, 5), (700, 701), (0, T)):
        g = g_cpu.to(dev)
        s = torch.full((3,), s_int / T, device=dev)
        t = torch.full((3,), t_int / T, device=dev)
        eps_h, eps_x = model.dynamics(g, t, get_batch_idxs(g))
        inputs = {"lig_n": g_cpu.batch_num_nodes("lig"), "kp_n": g_cpu.batch_num_nodes("kp"),
                  "lig_x": g_cpu.nodes["lig"].data["x_0"], "lig_h": g_cpu.nodes["lig"].data["h_0"],
                  "kp_x": g_cpu.nodes["kp"].data["x_0"], "kp_h": g_cpu.nodes["kp"].data["h_0"],
                  "kk_src": g_cpu.edges(form="uv", etype="kk")[0], "kk_dst": g_cpu.edges(form="uv", etype="kk")[1]}
        fb = Q.sample_p_zs_given_zt(lambda b, tt: (eps_h.cpu(), eps_x.cpu()), gamma, T, s_int, flat_batch(inputs),
                                    nx, nh, t_int=t_int)
        model.sample_p_zs_given_zt(s, t, g, get_batch_idxs(g), noise=(nx.to(dev), nh.to(dev)))
        torch.cuda.synchronize()
        for got, want in ((g.nodes["lig"].data["x_0"], fb.lig_x), (g.nodes["lig"].data["h_0"], fb.lig_h),
                          (g.nodes["kp"].data["x_0"], fb.kp_x)):
            assert rel_err(got.cpu(), want) < 1e-6, (s_int, t_int)


def test_one_capture_serves_every_schedule():
    """One capacity sampler runs several (timesteps, eta) values, with sub-batches too, then the default again: no
    new capture, and the last default run equals the first bit for bit."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model("gvp", _dev())
    F = model.n_lig_features
    g = HeteroBatch.from_pockets(_pockets("gvp", cfg, 2), SIZES, F)
    kw = dict(init_lig_pos=torch.zeros(len(SIZES), 3), seed=3, steps_per_graph=10, return_device_tensors=True)
    x0, h0 = (t.clone() for t in model.sample_from_encoded_receptors(g, **kw))
    before = model.cold_captures
    for ts, eta in ((7, None), (25, 0.0), (40, 0.5), (None, 1.0), (1, None), (40, None)):
        x, h = model.sample_from_encoded_receptors(g, timesteps=ts, eta=eta, **kw)
        assert bool(torch.isfinite(x).all()) and bool(torch.isfinite(h).all()), (ts, eta)
        if ts == 40 and eta is None:        # the unit grid: the default run
            assert torch.equal(x, x0) and torch.equal(h, h0)
        else:
            assert not torch.equal(x, x0), (ts, eta)
    assert model.cold_captures == before
    x1, h1 = model.sample_from_encoded_receptors(g, **kw)
    assert torch.equal(x1, x0) and torch.equal(h1, h0)


def test_sub_batches_follow_the_undivided_schedule():
    """Full-size gvp_20kp at T = 1000, timesteps = 100: every sub-batch split follows the undivided run (<= 1e-5)."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model("gvp", _dev(), T=1000)
    F = model.n_lig_features
    g = HeteroBatch.from_pockets(_pockets("gvp", cfg, 2), SIZES, F)
    kw = dict(init_lig_pos=torch.zeros(len(SIZES), 3), seed=19, steps_per_graph=50, timesteps=100,
              return_device_tensors=True)
    x1, h1 = model.sample_from_encoded_receptors(g, sub_batches=1, **kw)
    for sub in (None, 3):
        xs, hs = model.sample_from_encoded_receptors(g, sub_batches=sub, **kw)
        ex, eh = rel_err(xs.cpu(), x1.cpu()), rel_err(hs.cpu(), h1.cpu())
        assert ex < 1e-5 and eh < 1e-5, (sub, ex, eh)


@pytest.mark.parametrize("arch", ["gvp", "egnn"])
def test_full_size_fewer_steps(arch):
    """Shipped 20-keypoint models at T = 1000, 50 steps, ancestral and eta = 0: finite ligands of the requested sizes."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model(arch, _dev(), T=1000)
    F = model.n_lig_features
    sizes = [20] * 32
    g = HeteroBatch.from_pockets(_pockets(arch, cfg, 1), sizes, F)
    for eta in (None, 0.0):
        pos, feat = model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(len(sizes), 3), seed=7,
                                                        steps_per_graph=50, timesteps=50, eta=eta)
        assert [p.shape for p in pos] == [(20, 3)] * 32 and [f.shape for f in feat] == [(20, F)] * 32
        assert all(bool(torch.isfinite(p).all()) for p in pos) and all(bool(torch.isfinite(f).all()) for f in feat)


def test_drivers_with_timesteps():
    """_sample, sample_given_pocket and sample_random_sizes pass timesteps / eta through: receptor-major results of the
    requested sizes, finite, and different from the full-step run with the same seed."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model("egnn", _dev())
    F = model.n_lig_features
    pks = _pockets("egnn", cfg, 2)
    enc = [HeteroBatch.from_pockets([pk], [1], F) for pk in pks]
    centers = [pk.kp_x.mean(0) for pk in pks]
    kw = dict(encoded=True, seed=5, steps_per_graph=10)
    p, f = model.sample_given_pocket(enc[0], torch.tensor([20, 12]), init_lig_pos=centers[:1], timesteps=9, **kw)
    p_full, _ = model.sample_given_pocket(enc[0], torch.tensor([20, 12]), init_lig_pos=centers[:1], **kw)
    assert [q.shape[0] for q in p] == [20, 12] and all(bool(torch.isfinite(q).all()) for q in p)
    assert not torch.equal(p[0], p_full[0])
    out = model._sample(enc, [[20, 20], [16]], init_lig_pos=centers, timesteps=13, eta=0.0, **kw)
    assert [[q.shape[0] for q in o["positions"]] for o in out] == [[20, 20], [16]]
    assert all(bool(torch.isfinite(q).all()) for o in out for q in o["positions"])
    out = model.sample_random_sizes(enc, n_replicates=3, init_lig_pos=centers, timesteps=4, **kw)
    assert [len(o["positions"]) for o in out] == [3, 3]
    assert all(bool(torch.isfinite(q).all()) and q.shape[1] == 3 for o in out for q in o["positions"])
