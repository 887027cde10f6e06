"""CPU: fragment-conditioned sampling (inpainting) -- the oracle restatement against the plain loop, the second
coefficient table, and the argument checks that must fire before any device work."""
from pathlib import Path

import pytest
import torch

from helpers import flat_batch, load_golden, oracle_cfg
from oracle import flat, inpaint as I, schedule as S


def _draws(N_l, F, T, r, seed=7):
    """A dict (step, u, kind) -> [N_l, 3+F] of seeded draws covering the whole inpainting loop."""
    g = torch.Generator().manual_seed(seed)
    keys = [(-1, 0, 0)] + [(s, u, k) for s in reversed(range(T)) for u in range(r) for k in range(3 if u < r - 1 else 2)]
    return {k: torch.randn(N_l, 3 + F, generator=g) for k in keys}


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_oracle_inpainting_without_fixed_atoms_is_the_plain_loop(arch):
    """All-false mask, r = 1, the same draws: the inpainting loop is the plain loop, bit for bit."""
    fx = load_golden(f"loop_{arch}")
    cfg = oracle_cfg(arch, fx["kwargs"], fx["atom_nf"], fx["rec_nf"])
    sd, T, F = fx["state_dict"], fx["T"], fx["atom_nf"]
    gamma = sd["gamma.gamma"]
    fwd = flat.egnn_forward if arch == "egnn" else flat.gvp_forward
    dyn = lambda b, t: fwd(sd, cfg, b, t)
    N_l = int(fx["inputs"]["lig_n"].sum())
    d = _draws(N_l, F, T, 1)
    plain_noise = lambda step, kind, shape: d[(step, 0, 0)][:, :3] if kind == "x" else d[(step, 0, 0)][:, 3:]
    pos, feat = flat.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fx["init_lig_pos"],
                                                   plain_noise, atom_nf=F)
    mask = torch.zeros(N_l, dtype=torch.bool)
    ipos, ifeat = I.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fx["init_lig_pos"],
                                                  lambda step, u, kind, shape: d[(step, u, kind)], mask,
                                                  torch.randn(N_l, 3), torch.randn(N_l, F), resamplings=1, atom_nf=F)
    for a, b in zip(pos + feat, ipos + ifeat):
        assert torch.equal(a, b)


def test_inpaint_table_rows():
    """inpaint_table row s = (alpha_s, sigma_s, alpha_t|s, sigma_t|s); its alpha_t|s column is coefficient_table's
    column 0, bit for bit."""
    from keypoint_diffusion_b200.schedule import coefficient_table, inpaint_table
    T = 1000
    gamma = S.gamma_table(T, 1e-5)
    tab, coef = inpaint_table(gamma, T), coefficient_table(gamma, T)
    assert tab.shape == (T, 4) and tab.dtype == torch.float32
    assert torch.equal(tab[:, 2], coef[:, 0])
    for s_int in (0, 1, 500, 998, 999):
        gs, gt = gamma[s_int:s_int + 1], gamma[s_int + 1:s_int + 2]
        _, sig_ts, a_ts = S.sigma_and_alpha_t_given_s(gt, gs)
        want = torch.stack([S.alpha(gs)[0], S.sigma(gs)[0], a_ts[0], sig_ts[0]])
        assert torch.equal(tab[s_int], want), s_int
    assert bool((tab > 0).all()) and bool((tab[:, :3] <= 1).all())


def _cpu_model():
    import os
    from shipped_cases import shipped_configs
    from keypoint_diffusion_b200 import model_from_config
    os.chdir(Path(__file__).resolve().parents[1])
    torch.manual_seed(0)
    return model_from_config(shipped_configs()["egnn_20kp"])


def test_fragment_arguments_are_checked_before_any_device_work(monkeypatch):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    model = _cpu_model()
    F = model.n_lig_features

    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    monkeypatch.setattr(model, "_encode_all", no_device)
    frag = (torch.zeros(8, 3), torch.zeros(8, F))
    graphs = [object(), object()]
    with pytest.raises(ValueError, match="below"):
        model._sample(graphs, [[20, 7], [20]], fragments=[frag, None])
    with pytest.raises(ValueError, match="positions"):
        model._sample(graphs, [[20], [20]], fragments=[(torch.zeros(8, 4), torch.zeros(8, F)), None])
    with pytest.raises(ValueError, match="features"):
        model._sample(graphs, [[20], [20]], fragments=[(torch.zeros(8, 3), torch.zeros(8, F + 1)), None])
    with pytest.raises(ValueError, match="resamplings"):
        model._sample(graphs, [[20], [20]], fragments=[frag, None], resamplings=0)
    with pytest.raises(ValueError, match="resamplings"):
        model._sample(graphs, [[20], [20]], fragments=[None, None], resamplings=3)
    with pytest.raises(ValueError, match="resamplings"):
        model._sample(graphs, [[20], [20]], resamplings=2)
    with pytest.raises(ValueError, match="below"):
        model.sample_given_pocket(object(), torch.tensor([5]), fragment=frag)

    pk = synthetic.keypoint_pocket(0, 20, 256, 0, 8.0)
    g = HeteroBatch.from_pockets([pk], [20, 12], F)
    n = 32
    mask = torch.zeros(n, dtype=torch.bool)
    mask[:8] = True
    ok = dict(fixed_mask=mask, fixed_pos=torch.zeros(n, 3), fixed_feat=torch.zeros(n, F))
    init = torch.zeros(2, 3)
    with pytest.raises(ValueError, match="fixed_pos"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, **dict(ok, fixed_pos=torch.zeros(n, 2)))
    with pytest.raises(ValueError, match="fixed_feat"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, **dict(ok, fixed_feat=torch.zeros(n, 3)))
    with pytest.raises(ValueError, match="fixed_mask"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, **dict(ok, fixed_mask=mask[:10]))
    with pytest.raises(ValueError, match="resamplings"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, resamplings=0, **ok)
    with pytest.raises(ValueError, match="fixed atom"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, resamplings=2,
                                            **dict(ok, fixed_mask=torch.zeros(n, dtype=torch.bool)))
    with pytest.raises(ValueError, match="resamplings"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, resamplings=2)
    with pytest.raises(ValueError, match="capacity"):
        model.sample_from_encoded_receptors(g, init_lig_pos=init, capacity=False, **ok)
