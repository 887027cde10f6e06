"""GPU: second-order multistep sampling (solver="dpmpp_2m"; DESIGN.md section 6.5), held to an op-by-op restatement of
one step and to the multistep reference test_multistep_cpu.multistep_oracle (DPM-Solver++(2M) in its direct form).

* one kpd_ddpm_multistep_step against the op-by-op fp32 restatement, bit for bit (state, keypoints, shifted history);
  on the run's first row an all-NaN history is never read;
* with every c = 0 a multistep sampler returns what the plain sampler returns on the DDIM eta = 0 rows, bit for bit;
* the captured loop against the reference (<= 1e-3, the bar of the loop): both denoisers, fp32 and bf16x3, from noise
  and from a start ligand; recording changes nothing and its prediction frames follow the reference;
* the capacity path: sub-batch agreement, the captures a multistep call adds, and the drivers.
"""
import pytest
import torch

from helpers import flat_batch, rel_err
from test_gpu_fast_sampling import _draws, _rows
from test_gpu_inpaint import SIZES, _dense_model, _pockets
from test_gpu_optimize import _loop_case
from test_multistep_cpu import multistep_oracle

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _ms_rows(gamma, T, t_start, n):
    from keypoint_diffusion_b200.schedule import multistep_rows, step_grid
    return multistep_rows(gamma, T, step_grid(t_start, n)).to(_dev()).contiguous()


def _step_case(seed):
    from oracle import schedule as S
    T, F = 1000, 10
    gamma = S.gamma_table(T, 1e-4)
    lig_n, kp_n = [5, 20, 1, 33], [4, 20, 7, 2]
    g = torch.Generator().manual_seed(seed)
    N_l, N_k = sum(lig_n), sum(kp_n)
    t = dict(x=torch.randn(N_l, 3, generator=g), h=torch.randn(N_l, F, generator=g),
             xk=torch.randn(N_k, 3, generator=g) * 5, ex=torch.randn(N_l, 3, generator=g),
             eh=torch.randn(N_l, F, generator=g), nx=torch.randn(N_l, 3, generator=g),
             nh=torch.randn(N_l, F, generator=g), hx=torch.randn(N_l, 3, generator=g),
             hh=torch.randn(N_l, F, generator=g))
    return T, F, gamma, lig_n, kp_n, t


def _restated_step(t, lig_n, kp_n, row, ms, correct):
    """The step op by op in fp32 on the CPU: every product, quotient, sum and difference rounded on its own, the COM a
    sequential sum in atom order; divisors as full tensors (no scalar-reciprocal path)."""
    a, vt, sg = (float(v) for v in row[:3])
    c, at, st = (float(v) for v in ms[:3])
    full = lambda v, like: torch.full_like(like, v)
    out = {}
    for key, e, nz, hist in (("x", "ex", "nx", "hx"), ("h", "eh", "nh", "hh")):
        z = t[key]
        zs = (z / full(a, z) - full(vt, z) * t[e]) + full(sg, z) * t[nz]
        xh = (z - full(st, z) * t[e]) / full(at, z)
        if correct:
            zs = zs + full(c, z) * (xh - t[hist])
        out[key], out[hist] = zs, xh
    xk = t["xk"].clone()
    l0 = k0 = 0
    for nl, nk in zip(lig_n, kp_n):
        com = torch.zeros(3, dtype=torch.float32)
        for j in range(nl):
            com = com + out["x"][l0 + j]
        com = com / torch.full((3,), float(nl))
        for key in ("x", "hx"):
            out[key][l0:l0 + nl] = out[key][l0:l0 + nl] - com
        xk[k0:k0 + nk] = xk[k0:k0 + nk] - com
        l0, k0 = l0 + nl, k0 + nk
    out["xk"] = xk
    return out


@pytest.mark.parametrize("n,s", [(20, 7), (20, 1), (5, 3)])
def test_multistep_step_matches_restatement(n, s):
    """One kpd_ddpm_multistep_step on a corrected row (first_row = n-1 != s), injected eps / noise / history, against
    the op-by-op restatement: positions, features, keypoints and the shifted history bit for bit."""
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import coefficient_rows, multistep_rows, step_grid
    dev = _dev()
    T, F, gamma, lig_n, kp_n, t = _step_case(s)
    grid = step_grid(T, n)
    coef, ms = coefficient_rows(gamma, T, grid, eta=0.0), multistep_rows(gamma, T, grid)
    assert float(ms[s, 0]) != 0.0
    want = _restated_step(t, lig_n, kp_n, coef[s], ms[s], True)
    batch = ops.DeviceBatch(lig_n, kp_n, dev)
    D = lambda k: t[k].to(dev).contiguous()
    x, h, xk, hx, hh = D("x"), D("h"), D("xk"), D("hx"), D("hh")
    step = torch.tensor([s], dtype=torch.int32, device=dev)
    ops.ddpm_multistep_step(batch, x, h, xk, D("ex"), D("eh"), coef.to(dev), ms.to(dev), step, n - 1, hx, hh,
                            D("nx"), D("nh"))
    torch.cuda.synchronize()
    for got, key in ((x, "x"), (h, "h"), (xk, "xk"), (hx, "hx"), (hh, "hh")):
        assert torch.equal(got.cpu(), want[key]), key


def test_first_row_does_not_read_the_history():
    """On the run's first row (s == first_row) a history of NaN gives finite outputs: the plain DDIM eta = 0 step, bit
    for bit, and the history then holds x^ (positions shifted by the COM)."""
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import coefficient_rows, multistep_rows, step_grid
    dev = _dev()
    n, s = 10, 9
    T, F, gamma, lig_n, kp_n, t = _step_case(4)
    grid = step_grid(T, n)
    coef, ms = coefficient_rows(gamma, T, grid, eta=0.0), multistep_rows(gamma, T, grid)
    ms[s, 0] = 0.5                      # a non-zero c must not matter either
    t["hx"].fill_(float("nan"))
    t["hh"].fill_(float("nan"))
    want = _restated_step(t, lig_n, kp_n, coef[s], ms[s], False)
    batch = ops.DeviceBatch(lig_n, kp_n, dev)
    D = lambda k: t[k].to(dev).contiguous()
    x, h, xk, hx, hh = D("x"), D("h"), D("xk"), D("hx"), D("hh")
    step = torch.tensor([s], dtype=torch.int32, device=dev)
    ops.ddpm_multistep_step(batch, x, h, xk, D("ex"), D("eh"), coef.to(dev), ms.to(dev), step, s, hx, hh,
                            D("nx"), D("nh"))
    torch.cuda.synchronize()
    for got, key in ((x, "x"), (h, "h"), (xk, "xk"), (hx, "hx"), (hh, "hh")):
        assert bool(torch.isfinite(got).all()), key
        assert torch.equal(got.cpu(), want[key]), key


def _sampler(c, multistep, record=False, steps_per_graph=4):
    from keypoint_diffusion_b200 import ops
    return ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], c["T"], c["F"],
                       steps_per_graph=steps_per_graph, multistep=multistep, record=record)


def _run(c, sampler, **kw):
    t_in = c["t_in"]
    out = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), c["fx"]["init_lig_pos"].to(_dev()), **kw)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_zero_c_is_the_ddim_eta0_run(arch):
    """ms_coef with c = 0 everywhere: the multistep sampler returns the plain sampler's outputs on the DDIM eta = 0 rows
    bit for bit, n = 5 and 11 at steps_per_graph = 4 (replayed and eager steps), Philox and injected draws, from noise
    and from a start ligand; the launches per step are the plain sampler's."""
    from keypoint_diffusion_b200.schedule import start_coefficients
    c = _loop_case(arch, "bf16x3")
    dev, T = _dev(), c["T"]
    plain, multi = _sampler(c, False), _sampler(c, True)
    xs, hs = c["x_in"].to(dev), c["h_in"].to(dev)
    for t_start, n in ((T, 5), (T, 11), (7, 5)):
        coef = _rows(c["gamma"], T, t_start, n, 0.0, dev)[0]
        ms = _ms_rows(c["gamma"], T, t_start, n)
        ms[:, 0] = 0.0
        for smp in (plain, multi):
            smp.set_schedule(coef)
            if t_start != T:
                smp.set_start(n, xs, hs, *start_coefficients(c["gamma"], t_start))
            else:
                smp.set_start(None)
        multi.set_multistep(ms)
        _, noise = _draws(c, list(range(n + 1)))
        for kw in (dict(seed=23), dict(noise=noise)):
            px, ph, pk = _run(c, plain, **kw)
            mx, mh, mk = _run(c, multi, **kw)
            assert torch.equal(px, mx) and torch.equal(ph, mh) and torch.equal(pk, mk), (t_start, n, kw.keys())
    assert multi.launches_per_step == plain.launches_per_step


CASES = [(arch, mode, start, n) for arch in ("egnn", "gvp") for mode in ("fp32", "bf16x3")
         for start, n in ((False, 5), (False, 12), (True, 5), (True, 7))]


@pytest.mark.parametrize("arch,mode,start,n", CASES)
def test_loop_matches_oracle(arch, mode, start, n):
    """The captured multistep loop (steps_per_graph = 4) with injected draws against multistep_oracle (<= 1e-3): from
    noise at n = 5 and n = T = 12 of the loop fixture, and from a start ligand at t0 = 7 with n = 5 and 7."""
    from keypoint_diffusion_b200.schedule import start_coefficients
    c = _loop_case(arch, mode)
    dev, T, F = _dev(), c["T"], c["F"]
    t_start = 7 if start else T
    keys = [(-1, 0, 0)] + [(k, 0, 0) for k in reversed(range(n))]
    draws, noise = _draws(c, keys)
    smp = _sampler(c, True)
    smp.set_schedule(_rows(c["gamma"], T, t_start, n, 0.0, dev)[0])
    smp.set_multistep(_ms_rows(c["gamma"], T, t_start, n))
    if start:
        smp.set_start(n, c["x_in"].to(dev), c["h_in"].to(dev), *start_coefficients(c["gamma"], t_start))
    assert noise.shape[0] == smp.noise_slots == n + 1
    x, h, _ = _run(c, smp, noise=noise)
    pos, feat = multistep_oracle(c["dyn"], c["gamma"], T, flat_batch(c["fx"]["inputs"]),
                                 lambda k, u, kind, shape: draws[(k, u, kind)], n,
                                 init_lig_pos=c["fx"]["init_lig_pos"],
                                 start=(c["x_in"], c["h_in"], t_start) if start else None, atom_nf=F)
    ex, eh = rel_err(x.cpu(), torch.cat(pos)), rel_err(h.cpu(), torch.cat(feat))
    print(f"2M loop {arch} [{mode}] start={start} n={n}: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < 1e-3 and eh < 1e-3


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_recording_a_multistep_run(arch):
    """A multistep sampler that also records returns the non-recording multistep sampler's outputs bit for bit, and its
    prediction frames (every step) follow the reference's x^ moved to the output frame (<= 1e-3)."""
    c = _loop_case(arch, "bf16x3")
    dev, T, F = _dev(), c["T"], c["F"]
    n = 6
    keys = [(-1, 0, 0)] + [(k, 0, 0) for k in reversed(range(n))]
    draws, noise = _draws(c, keys)
    coef = _rows(c["gamma"], T, T, n, 0.0, dev)[0]
    ms = _ms_rows(c["gamma"], T, T, n)
    plain, rec = _sampler(c, True), _sampler(c, True, record=True)
    for smp in (plain, rec):
        smp.set_schedule(coef)
        smp.set_multistep(ms)
    x0, h0, _ = _run(c, plain, noise=noise)
    x1, h1, _, fr = _run(c, rec, noise=noise, record_every=1, pred_coef=ms[:, 1:3].contiguous())
    assert torch.equal(x0, x1) and torch.equal(h0, h1)
    assert rec.launches_per_step == plain.launches_per_step + 1
    batch = flat_batch(c["fx"]["inputs"])
    lig_b, kp_b = batch.batch_idx()
    init_kp_com = torch.zeros(batch.B, 3).index_add_(0, kp_b, batch.kp_x) / batch.kp_n[:, None].float()
    want = {}

    def on_step(k, x_hat, h_hat, z, kp_x):
        kp_com = torch.zeros(batch.B, 3).index_add_(0, kp_b, kp_x) / batch.kp_n[:, None].float()
        want[k] = ((x_hat - kp_com[lig_b]) + init_kp_com[lig_b], h_hat)
    multistep_oracle(c["dyn"], c["gamma"], T, batch, lambda k, u, kind, shape: draws[(k, u, kind)], n,
                     init_lig_pos=c["fx"]["init_lig_pos"], atom_nf=F, on_step=on_step)
    errs = []
    for j in range(n):
        wx, wh = want[n - 1 - j]
        errs.append(max(rel_err(fr["pred_positions"][j].cpu(), wx), rel_err(fr["pred_features"][j].cpu(), wh)))
    print(f"2M prediction frames {arch}: max rel_err {max(errs):.2e}")
    assert max(errs) < 1e-3, errs


def test_sub_batches_and_captures():
    """Full-size gvp_20kp at T = 1000, 20 steps: 1 and 4 sub-batches agree (<= 1e-5); the first multistep call adds one
    capture per bucket and sub-batch, a call with another n adds none, and visualize=True changes no output."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model("gvp", _dev(), T=1000)
    F = model.n_lig_features
    g = HeteroBatch.from_pockets(_pockets("gvp", cfg, 2), SIZES, F)
    kw = dict(init_lig_pos=torch.zeros(len(SIZES), 3), seed=19, steps_per_graph=10, return_device_tensors=True)
    x1, h1 = (v.clone() for v in model.sample_from_encoded_receptors(g, sub_batches=1, timesteps=20, **kw))
    model.sample_from_encoded_receptors(g, sub_batches=4, timesteps=20, **kw)     # warms the plain samplers
    before = model.cold_captures
    ref = model.sample_from_encoded_receptors(g, sub_batches=1, timesteps=20, solver="dpmpp_2m", **kw)
    x_ref, h_ref = (v.clone() for v in ref)
    assert model.cold_captures == before + 1
    assert not torch.equal(x_ref, x1)
    xs, hs = model.sample_from_encoded_receptors(g, sub_batches=4, timesteps=20, solver="dpmpp_2m", **kw)
    assert model.cold_captures == before + 1 + 4
    ex, eh = rel_err(xs.cpu(), x_ref.cpu()), rel_err(hs.cpu(), h_ref.cpu())
    assert ex < 1e-5 and eh < 1e-5, (ex, eh)
    for n in (10, 25):
        x, h = model.sample_from_encoded_receptors(g, sub_batches=4, timesteps=n, solver="dpmpp_2m", **kw)
        assert bool(torch.isfinite(x).all()) and bool(torch.isfinite(h).all()), n
    assert model.cold_captures == before + 1 + 4
    xv, hv, frames = model.sample_from_encoded_receptors(g, sub_batches=1, timesteps=20, solver="dpmpp_2m",
                                                         visualize=True, frame_every=5, **kw)
    assert torch.equal(xv, x_ref) and torch.equal(hv, h_ref)
    assert len(frames) == len(SIZES) and frames[0]["pred_positions"].shape == (4, SIZES[0], 3)


def test_drivers_with_solver():
    """_sample, sample_given_pocket and sample_random_sizes pass solver through (with timesteps, and from a start
    ligand): results of the requested sizes, finite, and different from the DDIM eta = 0 run with the same seed."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model("egnn", _dev())
    F = model.n_lig_features
    pks = _pockets("egnn", cfg, 2)
    enc = [HeteroBatch.from_pockets([pk], [1], F) for pk in pks]
    centers = [pk.kp_x.mean(0) for pk in pks]
    kw = dict(encoded=True, seed=5, steps_per_graph=10)
    p, f = model.sample_given_pocket(enc[0], torch.tensor([20, 12]), init_lig_pos=centers[:1], timesteps=10,
                                     solver="dpmpp_2m", **kw)
    p_ddim, _ = model.sample_given_pocket(enc[0], torch.tensor([20, 12]), init_lig_pos=centers[:1], timesteps=10,
                                          eta=0.0, **kw)
    assert [q.shape[0] for q in p] == [20, 12] and all(bool(torch.isfinite(q).all()) for q in p)
    assert not torch.equal(p[0], p_ddim[0])
    out = model._sample(enc, [[20, 20], [16]], init_lig_pos=centers, solver="dpmpp_2m", **kw)
    assert [[q.shape[0] for q in o["positions"]] for o in out] == [[20, 20], [16]]
    assert all(bool(torch.isfinite(q).all()) for o in out for q in o["positions"])
    out = model.sample_random_sizes(enc, n_replicates=3, init_lig_pos=centers, timesteps=12, solver="dpmpp_2m", **kw)
    assert [len(o["positions"]) for o in out] == [3, 3]
    assert all(bool(torch.isfinite(q).all()) and q.shape[1] == 3 for o in out for q in o["positions"])
    lig = (torch.randn(14, 3) + centers[0], torch.nn.functional.one_hot(torch.randint(0, F, (14,)), F).float())
    p, f = model.sample_given_pocket(enc[0], torch.tensor([14, 14]), start_ligand=lig, start_step=30, timesteps=10,
                                     solver="dpmpp_2m", **kw)
    assert [q.shape for q in p] == [(14, 3)] * 2 and all(bool(torch.isfinite(q).all()) for q in p + f)
