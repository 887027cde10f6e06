"""GPU: ligand optimisation by partial noising (a run of the captured loop from a given ligand at step t0), held to the
CPU restatement in oracle/optimize.py.

* the start kernel (kpd_partial_noise) with injected draws against the oracle start (<= 1e-6), and its Philox draw is
  the plain loop's initial draw;
* the whole loop from a start with injected draws against the oracle (<= 1e-3, the bar of the plain loop), with and
  without a fragment; a zero start at n_steps = 0 is sigma_t0 times the plain start (Philox keying, atom offset);
* sub-batch agreement, full-size models at t0 = 0 and t0 = 300, no new capture for a new t0 or start ligand, and the
  _sample / sample_given_pocket / sample_sharded drivers.
"""
import pytest
import torch

from helpers import flat_batch, load_golden, oracle_cfg, rel_err
from test_gpu_inpaint import SIZES, _bound, _dense_model, _pockets, _slot

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def test_partial_noise_matches_oracle():
    from oracle import flat, optimize as O, schedule as S
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200._lib import check, lib, ptr
    dev = _dev()
    T, F = 1000, 10
    gamma = S.gamma_table(T, 1e-5)
    lig_n, kp_n = [5, 20, 1, 33, 7], [4, 20, 7, 2, 9]
    N_l, N_k = sum(lig_n), sum(kp_n)
    g = torch.Generator().manual_seed(4)
    x_in = torch.randn(N_l, 3, generator=g) * 3 + 2.0
    h_in = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).float() * 2.0
    xk = torch.randn(N_k, 3, generator=g) * 5
    d = torch.randn(N_l, 3 + F, generator=g)
    norm = 2.0
    batch = ops.DeviceBatch(lig_n, kp_n, dev)
    D = lambda t: t.to(dev).contiguous()
    for t0 in (0, 1, 500, 1000):
        a, s = O.start_coefficients(gamma, t0)
        fb = flat.FlatBatch(lig_n=torch.tensor(lig_n), kp_n=torch.tensor(kp_n), kp_x=xk.clone(),
                            kp_h=torch.zeros(N_k, 1), kk_src=torch.zeros(0, dtype=torch.long),
                            kk_dst=torch.zeros(0, dtype=torch.long))
        fb = O.partial_noise(fb, x_in, h_in, a, s, d, norm)
        dk = D(xk.clone())
        dx, dh = ops.partial_noise(batch, D(x_in), D(h_in), dk, float(a), float(s), norm, noise=D(_slot(d)))
        torch.cuda.synchronize()
        errs = [rel_err(dx.cpu(), fb.lig_x), rel_err(dh.cpu(), fb.lig_h), rel_err(dk.cpu(), fb.kp_x)]
        assert max(errs) < 1e-6, (t0, errs)
    # Philox: a zero start with sigma = 1 is exactly the plain loop's initial draw (kpd_randn_init) after the COM removal
    zx, zh = torch.zeros(N_l, 3, device=dev), torch.zeros(N_l, F, device=dev)
    dk = D(xk.clone())
    dx, dh = ops.partial_noise(batch, zx, zh, dk, 0.25, 1.0, noise=None, seed=77)
    rx, rh, rk = torch.empty(N_l, 3, device=dev), torch.empty(N_l, F, device=dev), D(xk.clone())
    check(lib.kpd_randn_init(ptr(rx), ptr(rh), N_l, F, 77, ops._stream()), "kpd_randn_init")
    ops.remove_com(batch, rx, rk, "ligand")
    torch.cuda.synchronize()
    assert torch.equal(dx, rx) and torch.equal(dh, rh) and torch.equal(dk, rk)


def _loop_case(arch, mode):
    from oracle import flat, schedule as S
    from keypoint_diffusion_b200 import ops
    from test_gpu_parity import build_model, device_inputs
    dev = _dev()
    fx = load_golden(f"loop_{arch}")
    kw, T, F = fx["kwargs"], fx["T"], fx["atom_nf"]
    model = build_model(arch, fx["state_dict"], kw, F, fx["rec_nf"], dev)
    model.set_precision(mode)
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    gamma = fx["state_dict"]["gamma.gamma"]
    coef = S.coefficient_table(gamma, T).to(dev).contiguous()
    lig_n = fx["inputs"]["lig_n"]
    N_l = int(lig_n.sum())
    g = torch.Generator().manual_seed(8)
    lig_b = torch.arange(len(lig_n)).repeat_interleave(lig_n)
    x_in = fx["init_lig_pos"][lig_b] + torch.randn(N_l, 3, generator=g) * 1.5
    h_in = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).float()
    cfg = oracle_cfg(arch, kw, F, fx["rec_nf"])
    fwd = flat.egnn_forward if arch == "egnn" else flat.gvp_forward
    dyn = lambda b, t: fwd(fx["state_dict"], cfg, b, t)
    return dict(fx=fx, T=T, F=F, model=model, batch=batch, kk=kk, t_in=t_in, gp=gp, gamma=gamma, coef=coef, N_l=N_l,
                x_in=x_in, h_in=h_in, dyn=dyn, lig_n=lig_n, gen=g)


@pytest.mark.parametrize("t0", [1, 7, "T"])
@pytest.mark.parametrize("mode", ["fp32", "bf16x3"])
@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_loop_from_start_matches_oracle(arch, mode, t0):
    """The captured loop from a start ligand with injected draws against oracle/optimize.py.  steps_per_graph = 4:
    t0 = 1 runs one eager step, 7 one replay and three eager steps, T = 12 three replays."""
    from oracle import optimize as O
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import start_coefficients
    c = _loop_case(arch, mode)
    dev, T, F, N_l = _dev(), c["T"], c["F"], c["N_l"]
    t0 = T if t0 == "T" else t0
    keys = [(-1, 0, 0)] + [(s, 0, 0) for s in reversed(range(t0))]
    draws = {k: torch.randn(N_l, 3 + F, generator=c["gen"]) for k in keys}
    noise = torch.stack([_slot(draws[k]) for k in keys]).to(dev).contiguous()
    sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4)
    xs, hs = c["x_in"].to(dev), c["h_in"].to(dev)
    sampler.set_start(t0, xs, hs, *start_coefficients(c["gamma"], t0))
    assert noise.shape[0] == sampler.noise_slots == t0 + 1
    t_in = c["t_in"]
    x_lig, h_lig, _ = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), torch.zeros(len(c["lig_n"]), 3, device=dev),
                                  noise=noise)
    torch.cuda.synchronize()
    pos, feat = O.sample_from_encoded_receptors(c["dyn"], c["gamma"], T, flat_batch(c["fx"]["inputs"]), c["x_in"],
                                                c["h_in"], t0, lambda s, u, k, shape: draws[(s, u, k)], atom_nf=F)
    ex, eh = rel_err(x_lig.cpu(), torch.cat(pos)), rel_err(h_lig.cpu(), torch.cat(feat))
    print(f"optimise loop {arch} [{mode}] t0={t0}: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < 1e-3 and eh < 1e-3


@pytest.mark.parametrize("r", [1, 2])
def test_loop_from_start_with_fragment_matches_oracle(r):
    """A start ligand whose first atoms stay pinned (the inpainting loop from t0), against the oracle."""
    from oracle import optimize as O
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import inpaint_table, start_coefficients
    c = _loop_case("gvp", "bf16x3")
    dev, T, F, N_l, lig_n = _dev(), c["T"], c["F"], c["N_l"], c["lig_n"].tolist()
    t0 = 7
    mask = torch.zeros(N_l, dtype=torch.bool)
    mask[0:3] = True                                          # complex 0: 3 of 5 atoms; complex 1: none
    mask[lig_n[0] + lig_n[1]:lig_n[0] + lig_n[1] + 4] = True   # complex 2: 4 of 9
    keys = [(-1, 0, 0)] + [(s, u, k) for s in reversed(range(t0)) for u in range(r) for k in range(3 if u < r - 1 else 2)]
    draws = {k: torch.randn(N_l, 3 + F, generator=c["gen"]) for k in keys}
    noise = torch.stack([_slot(draws[k]) for k in keys]).to(dev).contiguous()
    coef2 = inpaint_table(c["gamma"], T).to(dev)
    sampler = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], T, F, steps_per_graph=4, resamplings=r,
                          inpaint_coef=coef2)
    xs, hs = c["x_in"].to(dev), c["h_in"].to(dev)
    dm = mask.to(dev, torch.uint8)
    sampler.set_fragment(dm, xs, hs)
    sampler.set_start(t0, xs, hs, *start_coefficients(c["gamma"], t0))
    assert noise.shape[0] == sampler.noise_slots == 1 + t0 * (3 * r - 1)
    t_in = c["t_in"]
    x_lig, h_lig, _ = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), torch.zeros(len(lig_n), 3, device=dev),
                                  noise=noise)
    torch.cuda.synchronize()
    pos, feat = O.sample_from_encoded_receptors(c["dyn"], c["gamma"], T, flat_batch(c["fx"]["inputs"]), c["x_in"],
                                                c["h_in"], t0, lambda s, u, k, shape: draws[(s, u, k)],
                                                fragment=(mask, c["x_in"], c["h_in"]), resamplings=r, atom_nf=F)
    ex, eh = rel_err(x_lig.cpu(), torch.cat(pos)), rel_err(h_lig.cpu(), torch.cat(feat))
    print(f"optimise loop with fragment r={r}: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < 1e-3 and eh < 1e-3


def test_zero_start_is_sigma_times_the_plain_start():
    """The forward draw is the plain initial draw: a zero start ligand at n_steps = 0 returns sigma_t0 times what the
    plain loop returns at n_steps = 0 with init_lig_pos = 0 -- features bit for bit, positions up to the rounding of the
    COM shifts -- with a nonzero atom offset on both."""
    from oracle import schedule as S
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import start_coefficients
    c = _loop_case("gvp", "bf16x3")
    dev, F, N_l = _dev(), c["F"], c["N_l"]
    T = 1000
    gamma = S.gamma_table(T, 1e-5)
    coef = S.coefficient_table(gamma, T).to(dev).contiguous()
    smp = ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], coef, T, F, atom_offset=37)
    t_in = c["t_in"]
    init = torch.zeros(len(c["lig_n"]), 3, device=dev)
    run = lambda: smp.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), init, seed=5, n_steps=0)
    xp, hp, _ = (t.clone() for t in run())
    zx, zh = torch.zeros(N_l, 3, device=dev), torch.zeros(N_l, F, device=dev)
    for t0 in (500, T):
        a, s = start_coefficients(gamma, t0)
        smp.set_start(t0, zx, zh, a, s)
        xs, hs, _ = run()
        torch.cuda.synchronize()
        assert torch.equal(hs, s * hp), t0
        assert float((xs - s * xp).abs().max()) < 1e-5, t0
    smp.set_start(None)
    xq, hq, _ = run()
    assert torch.equal(xq, xp) and torch.equal(hq, hp)


def _start_ligands(pocket, F, sizes, seed=0):
    """Per-atom start rows for complexes of the given sizes: positions around the pocket's keypoint centroid, one-hot
    atom types."""
    g = torch.Generator().manual_seed(seed)
    n = sum(sizes)
    pos = pocket.kp_x.mean(0) + torch.randn(n, 3, generator=g) * 1.5
    feat = torch.nn.functional.one_hot(torch.randint(0, F, (n,), generator=g), F).float()
    return pos, feat


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_sub_batches_follow_the_undivided_start(arch):
    """With sub-batches every group follows the undivided trajectory from the start (atom offsets), including the eager
    remainder of t0 = 25 at steps_per_graph = 10."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model(arch, _dev())
    F = model.n_lig_features
    pks = _pockets(arch, cfg, 2)
    g = HeteroBatch.from_pockets(pks, SIZES, F)
    pos, feat = _start_ligands(pks[0], F, SIZES)
    kw = dict(start_pos=pos, start_feat=feat, start_step=25, seed=17, steps_per_graph=10, return_device_tensors=True)
    x1, h1 = model.sample_from_encoded_receptors(g, sub_batches=1, **kw)
    for sub in (None, 3):
        xs, hs = model.sample_from_encoded_receptors(g, sub_batches=sub, **kw)
        ex, eh = rel_err(xs.cpu(), x1.cpu()), rel_err(hs.cpu(), h1.cpu())
        assert ex < 1e-5 and eh < 1e-5, (sub, ex, eh)
    assert bool(torch.isfinite(x1).all()) and bool(torch.isfinite(h1).all())


@pytest.mark.parametrize("arch", ["gvp", "egnn"])
def test_full_size_start(arch):
    """Shipped 20-keypoint models at T = 1000: t0 = 300 gives finite ligands; t0 = 0 returns every coordinate within
    6 sigma_0 of its start (plus the (1 - alpha_0) shrink toward the start ligand's mean) and its atom types; another t0
    with other start ligands in the same capacity bucket captures nothing new."""
    from keypoint_diffusion_b200 import HeteroBatch
    from keypoint_diffusion_b200.schedule import alpha, sigma
    model, cfg = _dense_model(arch, _dev(), T=1000)
    F = model.n_lig_features
    pk = _pockets(arch, cfg, 1)[0]
    sizes = [20] * 32
    g = HeteroBatch.from_pockets([pk], sizes, F)
    pos, feat = _start_ligands(pk, F, sizes)
    kw = dict(seed=23, steps_per_graph=50)
    p300, f300 = model.sample_from_encoded_receptors(g, start_pos=pos, start_feat=feat, start_step=300, **kw)
    assert all(bool(torch.isfinite(p).all()) for p in p300) and all(bool(torch.isfinite(f).all()) for f in f300)
    assert [p.shape[0] for p in p300] == sizes
    before = model.cold_captures
    p0, _, types = model.sample_from_encoded_receptors(g, start_pos=pos, start_feat=feat, start_step=0, decode=True, **kw)
    g0 = model.gamma.gamma[0].float().cpu()
    a0, s0 = float(alpha(g0)), float(sigma(g0))
    c = pos.view(len(sizes), 20, 3).mean(1).repeat_interleave(20, 0)
    bound = 6 * s0 + (1 - a0) * float((pos - c).abs().max()) + 1e-5
    worst = float((torch.cat(p0) - pos).abs().max())
    print(f"{arch}: t0 = 0 returns the start within {worst:.2e} (bound {bound:.2e})")
    assert worst <= bound
    assert torch.equal(torch.cat(types).long(), feat.argmax(1))
    pos2, feat2 = _start_ligands(pk, F, sizes, seed=1)
    p137, _ = model.sample_from_encoded_receptors(g, start_pos=pos2, start_feat=feat2, start_step=137, **kw)
    assert model.cold_captures == before
    assert all(bool(torch.isfinite(p).all()) for p in p137)


def test_start_drivers():
    """sample_given_pocket(start_ligand=...), and _sample / sample_sharded with start ligands, fragments and a complexes
    subset: receptor-major results with the start ligands' atom counts, each complex started from its own receptor's
    ligand, pinned scaffold atoms within the bound of the fragment tests."""
    from keypoint_diffusion_b200 import HeteroBatch
    from keypoint_diffusion_b200.schedule import sigma
    model, cfg = _dense_model("egnn", _dev())
    F = model.n_lig_features
    pks = _pockets("egnn", cfg, 2)
    enc = [HeteroBatch.from_pockets([pk], [1], F) for pk in pks]
    lig0 = _start_ligands(pks[0], F, [20], seed=2)
    lig1 = _start_ligands(pks[1], F, [16], seed=3)
    kw = dict(encoded=True, seed=5, steps_per_graph=10)
    p, f = model.sample_given_pocket(enc[0], torch.tensor([20, 20, 20]), start_ligand=lig0, start_step=12, **kw)
    assert [q.shape[0] for q in p] == [20, 20, 20] and all(bool(torch.isfinite(q).all()) for q in p)
    # t0 = 0: each complex comes back at its own receptor's start ligand, whichever subset is sampled
    tol = 6 * float(sigma(model.gamma.gamma[0].float().cpu())) + 1e-3
    sizes = [[20, 20], [16]]
    pos, feat = model._sample(enc, sizes, start_ligands=[lig0, lig1], start_step=0, complexes=[2, 0], **kw)
    assert [q.shape[0] for q in pos] == [16, 20]
    assert float((pos[0] - lig1[0]).abs().max()) < tol and float((pos[1] - lig0[0]).abs().max()) < tol
    out = model.sample_sharded(enc, sizes, start_ligands=[lig0, lig1], start_step=0, **kw)
    assert [len(o["positions"]) for o in out] == [2, 1]
    for o, lig in zip(out, (lig0, lig1)):
        for q in o["positions"]:
            assert float((q - lig[0]).abs().max()) < tol
    # a scaffold of the first receptor's start ligand stays pinned while the rest is re-generated from t0
    m = 6
    out = model._sample(enc, sizes, start_ligands=[lig0, lig1], start_step=30,
                        fragments=[(lig0[0][:m], lig0[1][:m]), None], resamplings=2, **kw)
    assert [[q.shape[0] for q in o["positions"]] for o in out] == [[20, 20], [16]]
    allp = torch.cat(out[0]["positions"] + out[1]["positions"])
    for q in out[0]["positions"]:
        assert float((q[:m] - lig0[0][:m]).abs().max()) <= _bound(model, lig0[0][:m], allp)
    assert all(bool(torch.isfinite(q).all()) for q in out[1]["positions"])
