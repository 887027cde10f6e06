"""CPU: recorded trajectories (visualize=True) -- the prediction rows against start_coefficients, frame counts and
levels, the argument checks that must fire before any device work, the multi-frame XYZ writer, the new C entry points,
and the recording reference the GPU tests hold the captured loop to (recorded_oracle below)."""
from pathlib import Path

import pytest
import torch

from helpers import flat_batch, load_golden, oracle_cfg
from oracle import fast as Q, flat, schedule as S


def recorded_oracle(dyn, gamma, T, inputs, noise_fn, n, every, init_lig_pos=None, start=None, fragment=None,
                    resamplings=1, eta=None, lig_feat_norm_constant=1.0, atom_nf=None):
    """oracle/fast.py's grid loop (same arguments) with the trajectory of DESIGN.md section 6.4 recorded around it:
    ``dyn`` is wrapped so that the first denoiser pass of executed step i (i % every == 0) records the state it is given,
    moved to the output frame with the final restore's ops, and the clean-ligand estimate (z - sigma_t eps) / alpha_t
    at that pass's level t.  Returns (lig_pos, lig_feat, frames) with frames = {'positions' [m+1,N,3], 'features'
    [m+1,N,F], 'pred_positions' [m,N,3], 'pred_features' [m,N,F]}; the last state frame is the returned ligands."""
    batch = flat_batch(inputs)
    lig_b, kp_b = batch.batch_idx()
    B = batch.B
    init_kp_com = flat._segment_mean(batch.kp_x, kp_b, B)[lig_b]
    passes = resamplings if fragment is not None else 1
    calls = [0]
    rec = {"positions": [], "features": [], "pred_positions": [], "pred_features": []}

    def recording_dyn(b, t):
        eps_h, eps_x = dyn(b, t)
        i, u = divmod(calls[0], passes)
        calls[0] += 1
        if u == 0 and i % every == 0:
            kp_com = flat._segment_mean(b.kp_x, kp_b, B)[lig_b]
            g_t = S.gamma_lookup(gamma, t, T)
            a = S.alpha(g_t)[lig_b].view(-1, 1).to(b.lig_x.dtype)
            s = S.sigma(g_t)[lig_b].view(-1, 1).to(b.lig_x.dtype)
            rec["positions"].append((b.lig_x - kp_com) + init_kp_com)
            rec["features"].append(b.lig_h * lig_feat_norm_constant)
            rec["pred_positions"].append(((b.lig_x - s * eps_x) / a - kp_com) + init_kp_com)
            rec["pred_features"].append((b.lig_h - s * eps_h) / a * lig_feat_norm_constant)
        return eps_h, eps_x

    pos, feat = Q.sample_from_encoded_receptors(recording_dyn, gamma, T, batch, noise_fn, n, eta=eta,
                                                init_lig_pos=init_lig_pos, start=start, fragment=fragment,
                                                resamplings=resamplings, lig_feat_norm_constant=lig_feat_norm_constant,
                                                atom_nf=atom_nf)
    rec["positions"].append(torch.cat(pos))
    rec["features"].append(torch.cat(feat))
    F = feat[0].shape[1]
    N = int(batch.lig_n.sum())
    empty = {"positions": (0, N, 3), "features": (0, N, F), "pred_positions": (0, N, 3), "pred_features": (0, N, F)}
    frames = {k: torch.stack(v) if v else torch.zeros(empty[k]) for k, v in rec.items()}
    return pos, feat, frames


def _gamma(T=1000):
    return S.gamma_table(T, 1e-5)


@pytest.mark.parametrize("t_start,n", [(1000, 1000), (7, 7), (1000, 300), (7, 3), (1000, 1)])
def test_prediction_rows_are_start_coefficients(t_start, n):
    """Row k of prediction_rows over a grid is start_coefficients(gamma, tau_{k+1}) bit for bit (the unit grid and
    strided grids from T and from a start t0); prediction_table is the unit grid; no eta anywhere."""
    from keypoint_diffusion_b200.schedule import prediction_rows, prediction_table, start_coefficients, step_grid
    T = 1000
    gamma = _gamma(T)
    tau = step_grid(t_start, n)
    rows = prediction_rows(gamma, T, tau)
    assert rows.shape == (n, 2) and rows.dtype == torch.float32 and rows.is_contiguous()
    for k in range(n):
        assert tuple(rows[k].tolist()) == start_coefficients(gamma, tau[k + 1]), k
    if n == t_start:
        assert torch.equal(rows, prediction_table(gamma, T)[:n])


@pytest.mark.parametrize("every", [1, 3, 50])
@pytest.mark.parametrize("n", [0, 1, 7, 1000])
def test_frame_counts_and_levels(n, every):
    """m = ceil(n / every) state frames before steps 0, every, 2 every, ... plus the output: levels tau_{n - j every}
    (the start level first), then 0; on the unit grid of a plain run, on a strided grid and from a start t0."""
    from keypoint_diffusion_b200.schedule import frame_levels, step_grid
    m = -(-n // every)
    unit = list(range(1001))
    lv = frame_levels(unit, n, every)
    assert lv.dtype == torch.long and lv.shape == (m + 1,)
    assert lv.tolist() == [n - j * every for j in range(m)] + [0]
    if n:
        assert int(lv[0]) == n and int(lv[m - 1]) == n - (m - 1) * every >= 1
        tau = step_grid(1000, n)                    # n strided steps over [0, T]
        lv = frame_levels(tau, n, every)
        assert lv.tolist() == [tau[n - j * every] for j in range(m)] + [0] and int(lv[0]) == 1000
        assert all(a > b for a, b in zip(lv.tolist()[:-1], lv.tolist()[1:]))


def _cpu_model():
    import os
    from shipped_cases import shipped_configs
    from keypoint_diffusion_b200 import model_from_config
    os.chdir(Path(__file__).resolve().parents[1])
    torch.manual_seed(0)
    return model_from_config(shipped_configs()["egnn_20kp"])


def test_visualize_arguments_are_checked_before_any_device_work(monkeypatch):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    model = _cpu_model()
    F = model.n_lig_features

    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    monkeypatch.setattr(model, "_encode_all", no_device)
    graphs = [object(), object()]
    sizes = [[20, 20], [20]]
    bad = [dict(frame_every=2), dict(visualize=False, frame_every=1), dict(visualize=True, frame_every=0),
           dict(visualize=True, frame_every=-3), dict(visualize=True, frame_every=2.0),
           dict(visualize=True, frame_every=True), dict(visualize=True, frame_every="5"),
           dict(visualize=True, capacity=False), dict(visualize=True, frame_every=4, capacity=False)]
    for kw in bad:
        with pytest.raises(ValueError, match="frame_every|visualize"):
            model._sample(graphs, sizes, **kw)
        with pytest.raises(ValueError, match="frame_every|visualize"):
            model.sample_given_pocket(object(), torch.tensor([20]), **kw)
    with pytest.raises(ValueError, match="sample_sharded"):
        model.sample_sharded(graphs, sizes, visualize=True)
    with pytest.raises(ValueError, match="sample_sharded"):
        model._sample(graphs, sizes, complexes=[0, 2], visualize=True)
    pk = synthetic.keypoint_pocket(0, 20, 256, 0, 8.0)
    g = HeteroBatch.from_pockets([pk], [20, 12], F)
    for kw in bad:
        with pytest.raises(ValueError, match="frame_every|visualize"):
            model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(2, 3), **kw)


def test_write_xyz_trajectory_format(tmp_path):
    """One write_xyz_file block per state frame, atom types from that frame's argmax (lowest index on ties)."""
    from keypoint_diffusion_b200.utils import write_xyz_file, write_xyz_trajectory
    elements = ["C", "N", "O"]
    pos = torch.tensor([[[0.0, 1.0, 2.0], [3.0, 4.0, 5.0]],
                        [[-1.25, 0.5, 0.0004], [10.0, -2.0, 3.3333]]])
    feat = torch.tensor([[[0.1, 0.9, 0.0], [1.0, 1.0, 0.0]],
                         [[0.0, 0.0, 2.0], [-1.0, -3.0, -2.0]]])
    frames = {"t": torch.tensor([5, 0]), "positions": pos, "features": feat,
              "pred_positions": pos[:1], "pred_features": feat[:1]}
    text = write_xyz_trajectory(frames, elements)
    want = ("2\n\nN 0.000 1.000 2.000\nC 3.000 4.000 5.000\n"
            "2\n\nO -1.250 0.500 0.000\nC 10.000 -2.000 3.333\n")
    assert text == want
    assert text == write_xyz_file(pos[0], ["N", "C"]) + write_xyz_file(pos[1], ["O", "C"])
    out = tmp_path / "traj.xyz"
    assert write_xyz_trajectory(frames, elements, str(out)) is None
    assert out.read_text() == want


def _loop_fixture(arch="egnn"):
    fx = load_golden(f"loop_{arch}")
    kw, F = fx["kwargs"], fx["atom_nf"]
    cfg = oracle_cfg(arch, kw, F, fx["rec_nf"])
    fwd = flat.egnn_forward if arch == "egnn" else flat.gvp_forward
    dyn = lambda b, t: fwd(fx["state_dict"], cfg, b, t)
    return fx, dyn, F


@pytest.mark.parametrize("every", [1, 3, 5])
def test_recorded_oracle_frames_are_truncated_runs(every):
    """The recording reference at the unit grid: the last state frame is the returned ligands, state frame j is
    oracle/flat.py's loop stopped after j*every steps (same draws, same restore) bit for bit, and recording leaves the
    output unchanged."""
    fx, dyn, F = _loop_fixture()
    T, gamma = fx["T"], fx["state_dict"]["gamma.gamma"]
    N_l = int(fx["inputs"]["lig_n"].sum())
    g = torch.Generator().manual_seed(3)
    draws = {k: torch.randn(N_l, 3 + F, generator=g) for k in range(-1, T)}
    fast_fn = lambda k, u, kind, shape: draws[k]
    plain_fn = lambda s, kind, shape: draws[s][:, :3] if kind == "x" else draws[s][:, 3:]
    pos, feat, fr = recorded_oracle(dyn, gamma, T, fx["inputs"], fast_fn, T, every,
                                    init_lig_pos=fx["init_lig_pos"], atom_nf=F)
    m = -(-T // every)
    assert fr["positions"].shape == (m + 1, N_l, 3) and fr["features"].shape == (m + 1, N_l, F)
    assert fr["pred_positions"].shape == (m, N_l, 3) and fr["pred_features"].shape == (m, N_l, F)
    assert torch.equal(fr["positions"][m], torch.cat(pos)) and torch.equal(fr["features"][m], torch.cat(feat))
    qpos, qfeat = Q.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fast_fn, T,
                                                  init_lig_pos=fx["init_lig_pos"], atom_nf=F)
    assert torch.equal(torch.cat(qpos), torch.cat(pos)) and torch.equal(torch.cat(qfeat), torch.cat(feat))
    for j in range(m):
        p, f = flat.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(fx["inputs"]), fx["init_lig_pos"],
                                                  plain_fn, n_steps=j * every, atom_nf=F)
        assert torch.equal(fr["positions"][j], torch.cat(p)) and torch.equal(fr["features"][j], torch.cat(f)), j


def test_recording_entry_points_are_exported():
    import ctypes
    from keypoint_diffusion_b200 import _lib
    header = (Path(__file__).resolve().parents[1] / "include" / "kpdiff_b200.h").read_text()
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in ("kpd_sampler_enable_recording", "kpd_sampler_set_recording"):
        assert f"int {name}(" in header
        assert name in _lib.EXPORTED and hasattr(lib, name)
