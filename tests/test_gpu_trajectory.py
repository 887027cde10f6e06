"""GPU: recorded trajectories (visualize=True; DESIGN.md section 6.4), held to the recording reference of
test_trajectory_cpu.recorded_oracle (oracle/fast.py's grid loop with the frames taken around its denoiser calls).

* recording changes nothing: a recording sampler's outputs equal a plain one's bit for bit, with Philox and injected
  draws, plain and inpainting, and its captured step holds exactly one more launch;
* state frame j is the loop's own state: the output of a plain run stopped after j*k steps, bit for bit (replays and an
  eager tail); prediction frame 0 is the formula applied to the GPU denoiser's eps on the same state (<= 1e-6);
* state and prediction frames against the recording reference with injected draws (<= 1e-3, the bar of the loop):
  plain, fragment, start, DDIM and a start on a strided grid;
* the capacity path: sub-batch agreement, no filler atoms, no new capture for new strides, schedules and starts, and
  the _sample / sample_given_pocket / sample_random_sizes structure.
"""
import pytest
import torch

from helpers import rel_err
from test_gpu_fast_sampling import _draws, _rows
from test_gpu_inpaint import SIZES, _dense_model, _pockets
from test_gpu_optimize import _loop_case
from test_trajectory_cpu import recorded_oracle

pytestmark = pytest.mark.gpu

KEYS = ("positions", "features", "pred_positions", "pred_features")


def _dev():
    return torch.device("cuda:0")


def _pred(c, grid=None):
    from keypoint_diffusion_b200.schedule import prediction_rows
    grid = list(range(c["T"] + 1)) if grid is None else grid
    return prediction_rows(c["gamma"], c["T"], grid).to(_dev()).contiguous()


def _run(c, sampler, **kw):
    t_in = c["t_in"]
    init = c["fx"]["init_lig_pos"].to(_dev())
    out = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), init, **kw)
    torch.cuda.synchronize()
    return out


def _sampler(c, record, resamplings=0, norm=1.0):
    from keypoint_diffusion_b200 import ops
    inp = _rows(c["gamma"], c["T"], c["T"], c["T"], None, _dev())[1] if resamplings else None
    return ops.Sampler(c["model"], c["batch"], c["gp"], c["kk"], c["coef"], c["T"], c["F"], steps_per_graph=4,
                       resamplings=resamplings, inpaint_coef=inp, record=record, lig_feat_norm_constant=norm)


def _mask(c):
    lig_n = c["lig_n"].tolist()
    mask = torch.zeros(c["N_l"], dtype=torch.bool)
    mask[0:3] = True
    mask[lig_n[0] + lig_n[1]:lig_n[0] + lig_n[1] + 4] = True
    return mask


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_recording_changes_nothing(arch):
    """Outputs of a recording sampler (every step recorded, or every 5th, or recording off) equal the plain sampler's
    bit for bit, with Philox and with injected draws, for the plain loop and the inpainting loop (r = 2); the recording
    sampler's captured step holds exactly one more launch."""
    c = _loop_case(arch, "bf16x3")
    dev, T = _dev(), c["T"]
    pred = _pred(c)
    for r in (0, 2):
        plain, rec = _sampler(c, False, r), _sampler(c, True, r)
        if r:
            for s in (plain, rec):
                s.set_fragment(_mask(c).to(dev, torch.uint8), c["x_in"].to(dev), c["h_in"].to(dev))
        n_slots = plain.noise_slots
        noise = torch.randn(n_slots, c["N_l"] * (3 + c["F"]), generator=c["gen"]).to(dev)
        for kw in (dict(seed=5), dict(noise=noise)):
            want = _run(c, plain, **kw)
            for every in (1, 5, None):
                got = _run(c, rec, record_every=every, pred_coef=pred, **kw)
                assert all(torch.equal(a, b) for a, b in zip(want, got[:3])), (r, every, kw.keys())
                if every is not None:
                    fr = got[3]
                    assert torch.equal(fr["positions"][-1], want[0]) and torch.equal(fr["features"][-1], want[1])
                    assert fr["positions"].shape[0] == -(-T // every) + 1
        assert rec.launches_per_step == plain.launches_per_step + 1, (r, rec.launches_per_step, plain.launches_per_step)


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_frames_are_the_loops_own_states(arch):
    """steps_per_graph = 4, n = 10 executed steps (two replays and an eager tail of two), k = 3: state frame j equals
    the output of a plain run with n_steps = 3j bit for bit; the last frame equals the output."""
    c = _loop_case(arch, "bf16x3")
    plain, rec = _sampler(c, False), _sampler(c, True)
    n, k = 10, 3
    x, h, _, fr = _run(c, rec, seed=9, n_steps=n, record_every=k, pred_coef=_pred(c))
    m = -(-n // k)
    assert fr["positions"].shape == (m + 1, c["N_l"], 3) and fr["pred_features"].shape == (m, c["N_l"], c["F"])
    assert torch.equal(fr["positions"][m], x) and torch.equal(fr["features"][m], h)
    for j in range(m):
        px, ph, _ = _run(c, plain, seed=9, n_steps=j * k)
        assert torch.equal(fr["positions"][j], px) and torch.equal(fr["features"][j], ph), j
    px, ph, _ = _run(c, plain, seed=9, n_steps=n)
    assert torch.equal(px, x) and torch.equal(ph, h)


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_prediction_frame_matches_the_formula(arch):
    """Prediction frame 0 against (z - sigma_t eps) / alpha_t moved to the output frame, eps from the GPU denoiser on
    the loop's initial state (rebuilt from injected slot 0 with the library's own COM removal), t = 1 (<= 1e-6)."""
    from keypoint_diffusion_b200 import ops
    c = _loop_case(arch, "bf16x3")
    dev, T, F, N_l = _dev(), c["T"], c["F"], c["N_l"]
    rec = _sampler(c, True)
    noise = torch.randn(rec.noise_slots, N_l * (3 + F), generator=c["gen"]).to(dev)
    pred = _pred(c)
    _, _, _, fr = _run(c, rec, noise=noise, n_steps=1, record_every=1, pred_coef=pred)
    b, t_in = c["batch"], c["t_in"]
    kp_b = torch.arange(b.B, device=dev).repeat_interleave(torch.tensor(b.kp_n, device=dev))
    lig_b = torch.arange(b.B, device=dev).repeat_interleave(torch.tensor(b.lig_n, device=dev))
    init = c["fx"]["init_lig_pos"].to(dev)
    x_kp = (t_in["kp_x"] - init[kp_b]).contiguous()
    x = noise[0, :N_l * 3].view(N_l, 3).clone()
    h = noise[0, N_l * 3:].view(N_l, F).clone()
    ops.remove_com(b, x, x_kp, "ligand")
    graphs = ops.LigandGraphs(b, c["gp"], rec.has_lk).build(x, x_kp)
    t = torch.ones(1, device=dev)
    args = (t_in["kp_v"],) if arch == "gvp" else ()
    eps_h, eps_x = c["model"].forward(b, graphs, c["kk"] if rec.has_lk else None, h, x, t_in["kp_h"], x_kp, *args, t)
    torch.cuda.synchronize()
    a, s = (float(v) for v in pred[T - 1])
    d = lambda v: v.double().cpu()
    kp_com = torch.zeros(b.B, 3, dtype=torch.float64).index_add_(0, kp_b.cpu(), d(x_kp)) / torch.tensor(
        b.kp_n, dtype=torch.float64)[:, None]
    init_com = torch.zeros(b.B, 3, dtype=torch.float64).index_add_(0, kp_b.cpu(), d(t_in["kp_x"])) / torch.tensor(
        b.kp_n, dtype=torch.float64)[:, None]
    lb = lig_b.cpu()
    want_x = (d(x) - s * d(eps_x)) / a - kp_com[lb] + init_com[lb]
    want_h = (d(h) - s * d(eps_h)) / a
    ex, eh = rel_err(fr["pred_positions"][0].cpu(), want_x), rel_err(fr["pred_features"][0].cpu(), want_h)
    print(f"prediction frame 0 {arch}: rel_err x={ex:.2e} h={eh:.2e}")
    assert ex < 1e-6 and eh < 1e-6


CASES = [("plain", "egnn", "fp32"), ("plain", "egnn", "bf16x3"), ("plain", "gvp", "fp32"), ("plain", "gvp", "bf16x3"),
         ("frag_r2", "gvp", "bf16x3"), ("start7", "egnn", "bf16x3"), ("ddim5", "gvp", "bf16x3"),
         ("start7_grid3", "gvp", "bf16x3")]


@pytest.mark.parametrize("case,arch,mode", CASES)
def test_frames_match_the_recording_oracle(case, arch, mode):
    """State and prediction frames of the captured loop (steps_per_graph = 4) with injected draws against the recording
    reference (<= 1e-3 relative each): the plain loop at k = 1 (both architectures, fp32 and bf16x3), a fragment with
    r = 2, a start at t0 = 7, 5 DDIM steps at eta = 0 with lig_feat_norm_constant = 4, and a start at t0 = 7 on the
    3-step grid over [0, 7], at k = 2."""
    from keypoint_diffusion_b200.schedule import start_coefficients, step_grid
    c = _loop_case(arch, mode)
    dev, T, F = _dev(), c["T"], c["F"]
    r = 2 if case == "frag_r2" else 0
    t0 = 7 if case.startswith("start") else None
    n, eta, grid = T, None, None
    if case == "start7":
        n = 7
    elif case == "ddim5":
        n, eta, grid = 5, 0.0, step_grid(T, 5)
    elif case == "start7_grid3":
        n, grid = 3, step_grid(7, 3)
    every = 1 if case == "plain" else 2
    norm = 4.0 if case == "ddim5" else 1.0
    if r:
        keys = [(-1, 0, 0)] + [(k, u, kind) for k in reversed(range(n)) for u in range(r)
                               for kind in range(3 if u < r - 1 else 2)]
    else:
        keys = [(-1, 0, 0)] + [(k, 0, 0) for k in reversed(range(n))]
    draws, noise = _draws(c, keys)
    sampler = _sampler(c, True, r, norm)
    mask = _mask(c)
    xs, hs = c["x_in"].to(dev), c["h_in"].to(dev)
    if r:
        sampler.set_fragment(mask.to(dev, torch.uint8), xs, hs)
    if grid is not None:
        sampler.set_schedule(_rows(c["gamma"], T, grid[-1], n, eta, dev)[0])
    if t0 is not None:
        sampler.set_start(n, xs, hs, *start_coefficients(c["gamma"], t0))
    assert noise.shape[0] == sampler.noise_slots
    x, h, _, fr = _run(c, sampler, noise=noise, record_every=every, pred_coef=_pred(c, grid))
    pos, feat, want = recorded_oracle(
        c["dyn"], c["gamma"], T, c["fx"]["inputs"], lambda k, u, kind, shape: draws[(k, u, kind)], n, every,
        init_lig_pos=c["fx"]["init_lig_pos"], start=None if t0 is None else (c["x_in"], c["h_in"], t0),
        fragment=(mask, c["x_in"], c["h_in"]) if r else None, resamplings=max(r, 1), eta=eta,
        lig_feat_norm_constant=norm, atom_nf=F)
    m = -(-n // every)
    errs = {}
    for key in KEYS:
        assert fr[key].shape == want[key].shape and want[key].shape[0] == (m + 1 if key in KEYS[:2] else m), key
        errs[key] = max(rel_err(fr[key][j].cpu(), want[key][j]) for j in range(want[key].shape[0]))
    print(f"recorded frames {case} {arch} [{mode}]: " + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) < 1e-3, errs


def test_capacity_path_frames():
    """The drop-in call with visualize=True: sub-batched frames follow the undivided call (<= 1e-5), every complex's
    frames hold its own atoms only (no filler rows) and end at its returned ligand, recording leaves the ligands
    unchanged, and new strides, schedules and starts capture nothing after the first recording call."""
    from keypoint_diffusion_b200 import HeteroBatch
    model, cfg = _dense_model("gvp", _dev())
    T, F = model.n_timesteps, model.n_lig_features
    g = HeteroBatch.from_pockets(_pockets("gvp", cfg, 2), SIZES, F)
    kw = dict(init_lig_pos=torch.zeros(len(SIZES), 3), seed=13, steps_per_graph=10, return_device_tensors=True)
    x0, h0 = (t.clone() for t in model.sample_from_encoded_receptors(g, sub_batches=1, **kw))
    x1, h1, fr1 = model.sample_from_encoded_receptors(g, sub_batches=1, visualize=True, frame_every=3, **kw)
    assert torch.equal(x0, x1) and torch.equal(h0, h1)
    m = -(-T // 3)
    off = 0
    for i, (n_at, fr) in enumerate(zip(SIZES, fr1)):
        assert fr["t"].tolist() == [T - 3 * j for j in range(m)] + [0]
        assert fr["positions"].shape == (m + 1, n_at, 3) and fr["features"].shape == (m + 1, n_at, F)
        assert fr["pred_positions"].shape == (m, n_at, 3) and fr["pred_features"].shape == (m, n_at, F)
        assert torch.equal(fr["positions"][m], x1[off:off + n_at]) and torch.equal(fr["features"][m], h1[off:off + n_at])
        off += n_at
    xs, hs, frs = model.sample_from_encoded_receptors(g, sub_batches=None, visualize=True, frame_every=3, **kw)
    assert model.default_sub_batches(len(SIZES)) > 1
    assert rel_err(xs.cpu(), x1.cpu()) < 1e-5 and rel_err(hs.cpu(), h1.cpu()) < 1e-5
    for key in KEYS:
        a = torch.cat([f[key] for f in frs], dim=1).cpu()
        b = torch.cat([f[key] for f in fr1], dim=1).cpu()
        assert max(rel_err(a[j], b[j]) for j in range(a.shape[0])) < 1e-5, key
    # one capture serves every stride, schedule and start of the recording loop
    before = model.cold_captures
    n_lig = sum(SIZES)
    start = dict(start_pos=x1.cpu(), start_feat=h1.cpu(), start_step=9)
    for extra, n_run, every in ((dict(), T, 1), (dict(frame_every=7), T, 7), (dict(timesteps=10, frame_every=2), 10, 2),
                                (dict(timesteps=5, eta=0.0), 5, 1), (dict(start, frame_every=4), 9, 4),
                                (dict(start, timesteps=3), 3, 1), (dict(start_pos=x1.cpu(), start_feat=h1.cpu(),
                                                                        start_step=0), 0, 1)):
        call = dict(kw, **extra)
        if "start_pos" in extra:
            call.pop("init_lig_pos")
        x, h, fr = model.sample_from_encoded_receptors(g, sub_batches=1, visualize=True, **call)
        m = -(-n_run // every)
        assert len(fr) == len(SIZES) and fr[0]["positions"].shape == (m + 1, SIZES[0], 3), extra.keys()
        assert fr[0]["t"][-1] == 0 and len(fr[0]["t"]) == m + 1
        assert bool(torch.isfinite(torch.cat([f["pred_positions"] for f in fr], dim=1)).all())
        assert torch.equal(torch.cat([f["positions"][-1] for f in fr]), x)
    assert model.cold_captures == before
    assert n_lig == x.shape[0]


def test_drivers_with_visualize():
    """_sample, sample_given_pocket and sample_random_sizes with visualize=True: the documented structure, on the CPU,
    with every trajectory ending at its ligand."""
    from keypoint_diffusion_b200 import HeteroBatch
    from keypoint_diffusion_b200.schedule import step_grid
    model, cfg = _dense_model("egnn", _dev())
    T, F = model.n_timesteps, model.n_lig_features
    pks = _pockets("egnn", cfg, 2)
    enc = [HeteroBatch.from_pockets([pk], [1], F) for pk in pks]
    centers = [pk.kp_x.mean(0) for pk in pks]
    kw = dict(encoded=True, seed=5, steps_per_graph=10)

    def check(pos, feat, frames, every, n=T):
        m = -(-n // every)
        tau = step_grid(T, n)
        assert len(frames) == len(pos)
        for p, f, fr in zip(pos, feat, frames):
            assert set(fr) == {"t", "positions", "features", "pred_positions", "pred_features"}
            assert all(v.device.type == "cpu" for v in fr.values())
            assert fr["t"].tolist() == [tau[n - every * j] for j in range(m)] + [0]
            assert fr["positions"].shape == (m + 1, p.shape[0], 3) and fr["features"].shape == (m + 1, p.shape[0], F)
            assert fr["pred_positions"].shape == (m, p.shape[0], 3) and fr["pred_features"].shape == (m, p.shape[0], F)
            assert torch.equal(fr["positions"][-1], p) and torch.equal(fr["features"][-1], f)

    p, f, frames = model.sample_given_pocket(enc[0], torch.tensor([20, 12]), init_lig_pos=centers[:1], visualize=True,
                                             frame_every=4, **kw)
    assert [q.shape[0] for q in p] == [20, 12]
    check(p, f, frames, 4)
    p_plain, _ = model.sample_given_pocket(enc[0], torch.tensor([20, 12]), init_lig_pos=centers[:1], **kw)
    assert all(torch.equal(a, b) for a, b in zip(p, p_plain))
    out = model._sample(enc, [[20, 20], [16]], init_lig_pos=centers, visualize=True, timesteps=13, **kw)
    assert [[q.shape[0] for q in o["positions"]] for o in out] == [[20, 20], [16]]
    for o in out:
        check(o["positions"], o["features"], o["frames"], 1, n=13)
    out = model.sample_random_sizes(enc, n_replicates=3, init_lig_pos=centers, visualize=True, frame_every=10, **kw)
    assert [len(o["frames"]) for o in out] == [3, 3]
    for o in out:
        check(o["positions"], o["features"], o["frames"], 10)
