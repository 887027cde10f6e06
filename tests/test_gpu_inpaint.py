"""GPU: fragment-conditioned sampling (inpainting with resampling), held to the CPU restatement in oracle/inpaint.py.

* one step: kpd_ddpm_inpaint_step and kpd_renoise with injected draws against the oracle step (<= 1e-6), for complexes
  with no, some and all atoms fixed;
* without a fragment nothing changes: an all-false mask at resamplings = 1 gives the plain sampler's output bit for bit,
  and so do the fragment-free complexes of a batch that mixes both;
* the whole captured loop with injected draws against the oracle loop (<= 1e-3, the bar of the plain loop);
* full-size models: the fragment comes back (within a bound from the schedule's alpha_0 / sigma_0), decoded types,
  free atoms that differ, sub-batch agreement and no new capture for a new fragment; the _sample / sample_given_pocket
  drivers.
"""
import pytest
import torch

from helpers import flat_batch, load_golden, oracle_cfg, rel_err

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _slot(d):
    """[N, 3+F] draw -> the flat in-slot layout of the sampler (x channels [N,3] first, then features [N,F])."""
    return torch.cat([d[:, :3].reshape(-1), d[:, 3:].reshape(-1)])


def test_inpaint_step_and_renoise_match_oracle():
    from oracle import flat, inpaint as I, schedule as S
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import inpaint_table
    dev = _dev()
    T, F = 1000, 10
    gamma = S.gamma_table(T, 1e-5)
    coef = S.coefficient_table(gamma, T).to(dev).contiguous()
    coef2 = inpaint_table(gamma, T).to(dev)
    lig_n, kp_n = [5, 20, 1, 33, 7], [4, 20, 7, 2, 9]
    N_l, N_k, B = sum(lig_n), sum(kp_n), len(lig_n)
    off = [0]
    for n in lig_n:
        off.append(off[-1] + n)
    mask = torch.zeros(N_l, dtype=torch.bool)          # complex 0: none; 1: some; 2: all (1 atom); 3: some; 4: all
    mask[off[1]:off[1] + 6] = True
    mask[off[2]] = True
    mask[[off[3] + 3, off[3] + 10, off[3] + 11, off[3] + 30]] = True
    mask[off[4]:off[5]] = True
    g = torch.Generator().manual_seed(2)
    x, h, xk = torch.randn(N_l, 3, generator=g), torch.randn(N_l, F, generator=g), torch.randn(N_k, 3, generator=g) * 5
    ex, eh = torch.randn(N_l, 3, generator=g), torch.randn(N_l, F, generator=g)
    pn, kn, rn = (torch.randn(N_l, 3 + F, generator=g) for _ in range(3))
    x_fix = torch.randn(N_l, 3, generator=g) * 3 + 1.0
    h_fix = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).float() * 2.0
    init_kp_com = torch.randn(B, 3, generator=g) * 4
    norm = 2.0
    batch = ops.DeviceBatch(lig_n, kp_n, dev)
    D = lambda t: t.to(dev).contiguous()
    for s_int in (999, 500, 0):
        for u in (0, 1):
            fb = flat.FlatBatch(lig_n=torch.tensor(lig_n), kp_n=torch.tensor(kp_n), kp_x=xk.clone(),
                                kp_h=torch.zeros(N_k, 1), kk_src=torch.zeros(0, dtype=torch.long),
                                kk_dst=torch.zeros(0, dtype=torch.long), lig_x=x.clone(), lig_h=h.clone())
            fb = I.sample_p_zs_given_zt(lambda b, t: (eh, ex), gamma, T, s_int, fb, mask, x_fix, h_fix, init_kp_com, pn,
                                        kn, norm)
            dx, dh, dk = D(x.clone()), D(h.clone()), D(xk.clone())
            step = torch.tensor([s_int], dtype=torch.int32, device=dev)
            noise = D(torch.stack([_slot(pn), _slot(kn)]))
            ops.ddpm_inpaint_step(batch, dx, dh, dk, D(ex), D(eh), coef, coef2, step, u, D(mask), D(x_fix), D(h_fix),
                                  D(init_kp_com), norm, noise=noise)
            torch.cuda.synchronize()
            errs = [rel_err(dx.cpu(), fb.lig_x), rel_err(dh.cpu(), fb.lig_h), rel_err(dk.cpu(), fb.kp_x)]
            assert max(errs) < 1e-6, (s_int, u, errs)
            fb = I.renoise(gamma, T, s_int, fb, rn)
            ops.renoise(batch, dx, dh, dk, coef2, step, u, noise=D(_slot(rn)))
            torch.cuda.synchronize()
            errs = [rel_err(dx.cpu(), fb.lig_x), rel_err(dh.cpu(), fb.lig_h), rel_err(dk.cpu(), fb.kp_x)]
            assert max(errs) < 1e-6, (s_int, u, "renoise", errs)
    # Philox draws: pass 0 without a fixed atom is kpd_ddpm_step exactly; pass 1 draws other noise
    step = torch.tensor([700], dtype=torch.int32, device=dev)
    outs = []
    for u in (None, 0, 1):
        dx, dh, dk = D(x.clone()), D(h.clone()), D(xk.clone())
        if u is None:
            ops.ddpm_step(batch, dx, dh, dk, D(ex), D(eh), coef, step, seed=77)
        else:
            ops.ddpm_inpaint_step(batch, dx, dh, dk, D(ex), D(eh), coef, coef2, step, u, None, None, None,
                                  D(init_kp_com), seed=77)
        outs.append((dx.cpu(), dh.cpu(), dk.cpu()))
    assert all(torch.equal(a, b) for a, b in zip(outs[0], outs[1]))
    assert not torch.equal(outs[0][1], outs[2][1])


def _dense_model(arch, dev, T=40):
    """A bench-like model (shipped 20-keypoint hyper-parameters, seeded weights) with the ll graph held dense, as
    bench.py builds it: every edge count is then fixed by the sizes, so complexes share no tile-boundary rounding."""
    import os
    from pathlib import Path
    from shipped_cases import shipped_configs
    from keypoint_diffusion_b200 import model_from_config
    os.chdir(Path(__file__).resolve().parents[1])
    cfg = shipped_configs()["gvp_20kp" if arch == "gvp" else "egnn_20kp"]
    cfg["diffusion"]["n_timesteps"] = T
    cfg["graph"]["graph_cutoffs"]["ll"] = 1e5
    torch.manual_seed(0)
    return model_from_config(cfg).to(dev).eval(), cfg


def _pockets(arch, cfg, n):
    from keypoint_diffusion_b200 import synthetic
    vs = cfg["dynamics_gvp"]["vector_size"] if arch == "gvp" else 0
    width = cfg["rec_encoder_gvp"]["out_scalar_size"] if arch == "gvp" else cfg["rec_encoder"]["out_n_node_feat"]
    return [synthetic.keypoint_pocket(i, 20, width, vs, cfg["graph"]["graph_cutoffs"]["kk"]) for i in range(n)]


SIZES = [20, 8, 35, 20, 13, 27, 22, 19, 31, 16, 25, 9, 20, 20, 18, 23, 30, 12, 21, 17, 26, 14, 20, 28, 11, 24, 20, 19,
         33, 15, 22, 18]


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_without_fragment_nothing_changes(arch):
    from keypoint_diffusion_b200 import HeteroBatch
    dev = _dev()
    model, cfg = _dense_model(arch, dev)
    F = model.n_lig_features
    g = HeteroBatch.from_pockets(_pockets(arch, cfg, 2), SIZES, F)       # host graph: nothing is written back into it
    n = sum(SIZES)
    init = torch.zeros(len(SIZES), 3)
    kw = dict(init_lig_pos=init, seed=11, steps_per_graph=10, return_device_tensors=True)
    plain = {}
    for sub in (1, None):
        x0, h0 = model.sample_from_encoded_receptors(g, sub_batches=sub, **kw)
        plain[sub] = (x0.clone(), h0.clone())
        x1, h1 = model.sample_from_encoded_receptors(g, sub_batches=sub, fixed_mask=torch.zeros(n, dtype=torch.bool),
                                                     fixed_pos=torch.randn(n, 3), fixed_feat=torch.randn(n, F),
                                                     resamplings=1, **kw)
        assert torch.equal(x0, x1) and torch.equal(h0, h1), sub
    # a batch mixing complexes with and without a fragment: the fragment-free ones are untouched
    mask = torch.zeros(n, dtype=torch.bool)
    off = [0]
    for s in SIZES:
        off.append(off[-1] + s)
    with_frag = [1, 4, 5, 17, 30]
    for c in with_frag:
        mask[off[c]:off[c] + 6] = True
    free = torch.ones(n, dtype=torch.bool)
    for c in with_frag:
        free[off[c]:off[c + 1]] = False
    pos = torch.randn(n, 3) * 2
    feat = torch.nn.functional.one_hot(torch.randint(0, F, (n,)), F).float()
    x2, h2 = model.sample_from_encoded_receptors(g, sub_batches=1, fixed_mask=mask, fixed_pos=pos, fixed_feat=feat, **kw)
    free_d = free.to(dev)
    assert torch.equal(x2[free_d], plain[1][0][free_d]) and torch.equal(h2[free_d], plain[1][1][free_d])
    assert not torch.equal(x2[~free_d], plain[1][0][~free_d])


@pytest.mark.parametrize("r", [1, 3])
@pytest.mark.parametrize("mode", ["fp32", "bf16x3"])
@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_inpaint_loop_matches_oracle(arch, mode, r):
    """The captured inpainting loop with injected draws against oracle/inpaint.py (fragments on two of three
    complexes), at the bar of test_full_loop_matches_reference."""
    from oracle import flat, inpaint as I, schedule as S
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.schedule import inpaint_table
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
    coef2 = inpaint_table(gamma, T).to(dev)
    lig_n = fx["inputs"]["lig_n"].tolist()                     # [5, 2, 9]
    N_l = sum(lig_n)
    mask = torch.zeros(N_l, dtype=torch.bool)
    mask[0:3] = True                                          # complex 0: 3 of 5 atoms; complex 1: none
    mask[lig_n[0] + lig_n[1]:lig_n[0] + lig_n[1] + 4] = True   # complex 2: 4 of 9
    g = torch.Generator().manual_seed(5)
    lig_b = torch.arange(len(lig_n)).repeat_interleave(torch.tensor(lig_n))
    x_fix = fx["init_lig_pos"][lig_b] + torch.randn(N_l, 3, generator=g) * 1.5
    h_fix = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).float()
    keys = [(-1, 0, 0)] + [(s, u, k) for s in reversed(range(T)) for u in range(r) for k in range(3 if u < r - 1 else 2)]
    draws = {k: torch.randn(N_l, 3 + F, generator=g) for k in keys}
    noise = torch.stack([_slot(draws[k]) for k in keys]).to(dev).contiguous()
    sampler = ops.Sampler(model, batch, gp, kk, coef, T, F, steps_per_graph=4, resamplings=r, inpaint_coef=coef2)
    assert noise.shape[0] == sampler.noise_slots == 1 + T * (3 * r - 1)
    dm, dxf, dhf = mask.to(dev, torch.uint8), x_fix.to(dev), h_fix.to(dev)
    sampler.set_fragment(dm, dxf, dhf)
    x_lig, h_lig, _ = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), fx["init_lig_pos"].to(dev), noise=noise)
    torch.cuda.synchronize()
    cfg = oracle_cfg(arch, kw, F, fx["rec_nf"])
    fwd = flat.egnn_forward if arch == "egnn" else flat.gvp_forward
    pos, feat = I.sample_from_encoded_receptors(lambda b, t: fwd(fx["state_dict"], cfg, b, t), gamma, T,
                                                flat_batch(fx["inputs"]), fx["init_lig_pos"],
                                                lambda s, u, k, shape: draws[(s, u, k)], mask, x_fix, h_fix,
                                                resamplings=r, atom_nf=F)
    ex, eh = rel_err(x_lig.cpu(), torch.cat(pos)), rel_err(h_lig.cpu(), torch.cat(feat))
    print(f"inpaint loop {arch} [{mode}] r={r}: rel_err pos={ex:.2e} feat={eh:.2e} "
          f"launches/step={sampler.launches_per_step}")
    assert ex < 1e-3 and eh < 1e-3


def _fragment(pocket, F, m=8, seed=0, shift=0.0):
    """An m-atom fragment near the pocket's keypoint centroid, one-hot atom types."""
    g = torch.Generator().manual_seed(seed)
    pos = pocket.kp_x.mean(0) + torch.randn(m, 3, generator=g) * 1.5 + shift
    types = torch.arange(m) % F
    return pos, torch.nn.functional.one_hot(types, F).float(), types


def _bound(model, x_fix, lig_pos):
    """|returned - x_fix| <= (1 - alpha_0) * |x_fix - (init_kp_com - kp_com)| + sigma_0 * |e| at the fixed atoms: the
    last step writes alpha_0 x0 + sigma_0 e, and init_kp_com - kp_com is the ligand's place in the returned frame."""
    from keypoint_diffusion_b200.schedule import alpha, sigma
    g0 = model.gamma.gamma[0].float().cpu()
    a0, s0 = float(alpha(g0)), float(sigma(g0))
    return (1 - a0) * (float(x_fix.abs().max()) + 2 * float(lig_pos.abs().max()) + 10.0) + 6.0 * s0


@pytest.mark.parametrize("arch", ["gvp", "egnn"])
def test_fragment_full_size(arch):
    from keypoint_diffusion_b200 import HeteroBatch
    dev = _dev()
    model, cfg = _dense_model(arch, dev)
    F = model.n_lig_features
    pk = _pockets(arch, cfg, 1)[0]
    sizes = [20] * 32
    n, m, r = sum(sizes), 8, 2
    g = HeteroBatch.from_pockets([pk], sizes, F)
    init = torch.zeros(len(sizes), 3)

    def request(pos, feat):
        mask = torch.zeros(n, dtype=torch.bool)
        xf, hf = torch.zeros(n, 3), torch.zeros(n, F)
        for c in range(len(sizes)):
            mask[20 * c:20 * c + m] = True
            xf[20 * c:20 * c + m] = pos
            hf[20 * c:20 * c + m] = feat
        return dict(fixed_mask=mask, fixed_pos=xf, fixed_feat=hf, resamplings=r)

    pos, feat, types = _fragment(pk, F)
    kw = dict(init_lig_pos=init, seed=21, steps_per_graph=10)
    out_pos, out_feat, out_types = model.sample_from_encoded_receptors(g, sub_batches=1, decode=True, **request(pos, feat),
                                                                       **kw)
    bound = _bound(model, pos, torch.cat(out_pos))
    assert bound < 0.1, bound
    worst = max(float((p[:m] - pos).abs().max()) for p in out_pos)
    print(f"{arch}: fragment atoms within {worst:.2e} of the fragment (bound {bound:.2e})")
    assert worst <= bound
    for t in out_types:
        assert torch.equal(t[:m].long(), types)
    assert float((out_pos[0][m:] - out_pos[1][m:]).abs().max()) > 0.1       # free atoms of two ligands differ
    assert all(torch.isfinite(p).all() for p in out_pos)
    # the default sub-batch split draws the same noise (atom offsets); tiles differ, so not bitwise
    d_pos, d_feat = model.sample_from_encoded_receptors(g, **request(pos, feat), **kw)
    ex = rel_err(torch.cat(d_pos), torch.cat(out_pos))
    eh = rel_err(torch.cat(d_feat), torch.cat(out_feat))
    assert ex < 1e-5 and eh < 1e-5, (ex, eh)
    # another fragment in the same capacity bucket: the captured graphs are re-pointed, not captured again
    before = model.cold_captures
    pos2, feat2, _ = _fragment(pk, F, seed=1, shift=0.7)
    p2, _ = model.sample_from_encoded_receptors(g, sub_batches=1, **request(pos2, feat2), **kw)
    assert model.cold_captures == before
    assert max(float((p[:m] - pos2).abs().max()) for p in p2) <= _bound(model, pos2, torch.cat(p2))


def test_fragment_drivers():
    """sample_given_pocket(fragment=...) and _sample(fragments=[frag, None]): the first receptor's ligands start with
    the fragment, the second receptor's are those of a call without fragments."""
    from keypoint_diffusion_b200 import HeteroBatch
    dev = _dev()
    model, cfg = _dense_model("egnn", dev)
    F = model.n_lig_features
    pks = _pockets("egnn", cfg, 2)
    enc = [HeteroBatch.from_pockets([pk], [1], F) for pk in pks]
    pos, feat, _ = _fragment(pks[0], F, m=6)
    kw = dict(encoded=True, seed=5, steps_per_graph=10)
    p, _ = model.sample_given_pocket(enc[0], torch.tensor([20, 12, 15]), fragment=(pos, feat),
                                     init_lig_pos=[torch.zeros(3)], **kw)
    assert [q.shape[0] for q in p] == [20, 12, 15]
    for q in p:
        assert float((q[:6] - pos).abs().max()) <= _bound(model, pos, torch.cat(p))
    sizes = [[20, 14], [18, 10]]
    centers = [torch.zeros(3), torch.zeros(3)]
    out = model._sample(enc, sizes, init_lig_pos=centers, fragments=[(pos, feat), None], **kw)
    ref = model._sample(enc, sizes, init_lig_pos=centers, **kw)
    allp = torch.cat(out[0]["positions"] + out[1]["positions"])
    for q in out[0]["positions"]:
        assert float((q[:6] - pos).abs().max()) <= _bound(model, pos, allp)
    for q, q0, f, f0 in zip(out[1]["positions"], ref[1]["positions"], out[1]["features"], ref[1]["features"]):
        assert torch.equal(q, q0) and torch.equal(f, f0)
        assert float((q[:6] - pos).abs().max()) > 0.5                      # unconstrained
