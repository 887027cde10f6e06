"""CPU: ligand optimisation by partial noising -- the oracle's start against its closed form, the start coefficients,
the argument checks that must fire before any device work, and the new C entry points."""
from pathlib import Path

import pytest
import torch

from helpers import flat_batch, load_golden
from oracle import optimize as O, schedule as S


def test_oracle_at_t0_zero_is_the_closed_form():
    """t0 = 0 runs no reverse step: the output is alpha_0 (x_in - c_b) + c_b + sigma_0 e, with c_b the start ligand's
    mean per complex and e the forward draw; features alpha_0 h_in + sigma_0 e_h."""
    fx = load_golden("loop_egnn")
    F = fx["atom_nf"]
    gamma = fx["state_dict"]["gamma.gamma"]
    lig_n = fx["inputs"]["lig_n"]
    N_l = int(lig_n.sum())
    g = torch.Generator().manual_seed(3)
    lig_b = torch.arange(len(lig_n)).repeat_interleave(lig_n)
    x_in = fx["init_lig_pos"][lig_b] + torch.randn(N_l, 3, generator=g) * 1.5
    h_in = torch.nn.functional.one_hot(torch.randint(0, F, (N_l,), generator=g), F).float()
    d = torch.randn(N_l, 3 + F, generator=g)

    def no_denoiser(b, t):
        raise AssertionError("t0 = 0 runs no reverse step")

    pos, feat = O.sample_from_encoded_receptors(no_denoiser, gamma, fx["T"], flat_batch(fx["inputs"]), x_in, h_in, 0,
                                                lambda s, u, k, shape: d, atom_nf=F)
    a0, s0 = float(S.alpha(gamma[:1])), float(S.sigma(gamma[:1]))
    c = torch.zeros(len(lig_n), 3).index_add_(0, lig_b, x_in) / lig_n[:, None].float()
    want_x = a0 * (x_in - c[lig_b]) + c[lig_b] + s0 * d[:, :3]
    want_h = a0 * h_in + s0 * d[:, 3:]
    assert float((torch.cat(pos) - want_x).abs().max()) < 1e-5
    assert float((torch.cat(feat) - want_h).abs().max()) < 1e-6
    assert float((torch.cat(pos) - x_in).abs().max()) < 6 * s0 * float(d.abs().max()) + 1e-4


@pytest.mark.parametrize("t0", [0, 1, 500, 1000])
def test_start_coefficients_are_the_scalar_fp32_ops(t0):
    from keypoint_diffusion_b200.schedule import start_coefficients
    gamma = S.gamma_table(1000, 1e-5)
    a, s = start_coefficients(gamma, t0)
    g = gamma[t0:t0 + 1]
    assert a == float(S.alpha(g)[0]) and s == float(S.sigma(g)[0])
    oa, os_ = O.start_coefficients(gamma, t0)
    assert a == float(oa[0]) and s == float(os_[0])
    assert torch.tensor(a, dtype=torch.float32).item() == a        # fp32 values, passed to the kernel exactly


def _cpu_model():
    import os
    from shipped_cases import shipped_configs
    from keypoint_diffusion_b200 import model_from_config
    os.chdir(Path(__file__).resolve().parents[1])
    torch.manual_seed(0)
    return model_from_config(shipped_configs()["egnn_20kp"])


def test_start_arguments_are_checked_before_any_device_work(monkeypatch):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    model = _cpu_model()
    F, T = model.n_lig_features, model.n_timesteps

    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    monkeypatch.setattr(model, "_encode_all", no_device)
    lig = (torch.zeros(20, 3), torch.zeros(20, F))
    graphs = [object(), object()]
    sizes = [[20, 20], [20]]
    with pytest.raises(ValueError, match="start_step"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=T + 1)
    with pytest.raises(ValueError, match="start_step"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=-1)
    with pytest.raises(ValueError, match="start_step"):
        model._sample(graphs, sizes, start_ligands=[lig, lig])
    with pytest.raises(ValueError, match="start ligands"):
        model._sample(graphs, sizes, start_step=10)
    with pytest.raises(ValueError, match="no start ligand"):
        model._sample(graphs, sizes, start_ligands=[lig, None], start_step=10)
    with pytest.raises(ValueError, match="one entry per receptor"):
        model._sample(graphs, sizes, start_ligands=[lig], start_step=10)
    with pytest.raises(ValueError, match="differs"):
        model._sample(graphs, [[20, 19], [20]], start_ligands=[lig, lig], start_step=10)
    with pytest.raises(ValueError, match="positions"):
        model._sample(graphs, sizes, start_ligands=[(torch.zeros(20, 2), torch.zeros(20, F)), lig], start_step=10)
    with pytest.raises(ValueError, match="features"):
        model._sample(graphs, sizes, start_ligands=[(torch.zeros(20, 3), torch.zeros(20, F + 1)), lig], start_step=10)
    with pytest.raises(ValueError, match="init_lig_pos"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=10, init_lig_pos=[torch.zeros(3)] * 2)
    with pytest.raises(ValueError, match="use_ref_lig_com"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=10, use_ref_lig_com=True)
    with pytest.raises(ValueError, match="capacity"):
        model._sample(graphs, sizes, start_ligands=[lig, lig], start_step=10, capacity=False)
    with pytest.raises(ValueError, match="differs"):
        model.sample_given_pocket(object(), torch.tensor([20, 5]), start_ligand=lig, start_step=10)
    with pytest.raises(ValueError, match="start ligands"):
        model.sample_given_pocket(object(), torch.tensor([20]), start_step=10)
    # a start ligand with a fragment: the fragment size rule and the start rule both apply
    with pytest.raises(ValueError, match="differs"):
        model._sample(graphs, [[20, 24], [20]], start_ligands=[lig, lig], start_step=10,
                      fragments=[(torch.zeros(8, 3), torch.zeros(8, F)), None])

    pk = synthetic.keypoint_pocket(0, 20, 256, 0, 8.0)
    g = HeteroBatch.from_pockets([pk], [20, 12], F)
    n = 32
    ok = dict(start_pos=torch.zeros(n, 3), start_feat=torch.zeros(n, F), start_step=100)
    with pytest.raises(ValueError, match="start_pos"):
        model.sample_from_encoded_receptors(g, **dict(ok, start_pos=torch.zeros(n, 2)))
    with pytest.raises(ValueError, match="start_pos"):
        model.sample_from_encoded_receptors(g, **dict(ok, start_pos=torch.zeros(n - 1, 3)))
    with pytest.raises(ValueError, match="start_feat"):
        model.sample_from_encoded_receptors(g, **dict(ok, start_feat=torch.zeros(n, F - 1)))
    with pytest.raises(ValueError, match="start_step"):
        model.sample_from_encoded_receptors(g, **dict(ok, start_step=None))
    with pytest.raises(ValueError, match="start_step"):
        model.sample_from_encoded_receptors(g, **dict(ok, start_step=T + 5))
    with pytest.raises(ValueError, match="start_step"):
        model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(2, 3), start_step=5)
    with pytest.raises(ValueError, match="start_pos and start_feat"):
        model.sample_from_encoded_receptors(g, **dict(ok, start_feat=None))
    with pytest.raises(ValueError, match="init_lig_pos"):
        model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(2, 3), **ok)
    with pytest.raises(ValueError, match="capacity"):
        model.sample_from_encoded_receptors(g, capacity=False, **ok)


def test_start_entry_points_are_exported():
    import ctypes
    from keypoint_diffusion_b200 import _lib
    header = (Path(__file__).resolve().parents[1] / "include" / "kpdiff_b200.h").read_text()
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for sym in ("kpd_partial_noise", "kpd_sampler_set_start"):
        assert f"int {sym}(" in header
        assert sym in _lib.EXPORTED and hasattr(lib, sym)
