"""GPU: the plain-bf16 tensor-core mode of the EGNN denoiser ('bf16': tcgen05 with bf16 operands and fp32 accumulation
in the edge kernel -- one M = 64 MMA per k-step on 64-edge tiles -- and one-MUFU activations).

Operands are rounded to bf16 (8-bit mantissa), so the bar is max|a-b|/max|b| < 3e-2 of the output scale -- the bar the
GVP bf16 mode is held to, stated separately from the 1e-4 parity bar of the fp32 and bf16x3 modes.  Every test prints
the errors it measured.  Edge sets are exact in every mode (graph construction does not depend on the precision)."""
import pytest
import torch

from helpers import GOLDEN, edge_set, err_report, flat_batch, fmt_err, load_golden, oracle_cfg, oracle_forward, rel_err
from shipped_cases import SHIPPED, shipped_case

pytestmark = pytest.mark.gpu
TOL_BF16 = 3e-2


def _dev():
    return torch.device("cuda:0")


@pytest.mark.parametrize("name", ["egnn_small_kp", "egnn_small_nokp"])
def test_egnn_bf16_mode_small(name):
    """Golden fixtures (the reference's own fp32 outputs) at every stored t."""
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    fx = load_golden(name)
    kw = fx["kwargs"]
    model = build_model("egnn", fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    assert model.tc_blob2 is not None
    model.set_precision("bf16")
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, bool(kw.get("update_kp_feat", False))).build(t_in["lig_x"], t_in["kp_x"])
    cfg = oracle_cfg("egnn", kw, fx["atom_nf"], fx["rec_nf"])
    for tkey, out in fx["outputs"].items():
        h, x = run_forward("egnn", model, batch, graphs, kk, t_in, float(tkey), dev)
        torch.cuda.synchronize()
        fb = flat_batch(fx["inputs"])
        ref_h, ref_x = oracle_forward("egnn", fx["state_dict"], cfg, fb, torch.full((fb.B,), float(tkey)))
        eh, ex = rel_err(h.cpu(), out["eps_h"]), rel_err(x.cpu(), out["eps_x"])
        oh, ox = rel_err(h.cpu(), ref_h), rel_err(x.cpu(), ref_x)
        print(f"{name} bf16 t={tkey}: vs golden eps_h={eh:.2e} eps_x={ex:.2e} | vs oracle eps_h={oh:.2e} eps_x={ox:.2e}")
        assert max(eh, ex, oh, ox) < TOL_BF16


def test_egnn_bf16_mode_full_size():
    import yaml
    from test_gpu_parity import _full_size_case, build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    sd, kw, rec_nf, inputs = _full_size_case("egnn", cfgs)
    cfg = oracle_cfg("egnn", kw, 10, rec_nf)
    model = build_model("egnn", sd, kw, 10, rec_nf, dev)
    model.set_precision("bf16")
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
    for tval in (0.001, 0.5, 1.0):
        fb = flat_batch(inputs)
        ref_h, ref_x = oracle_forward("egnn", sd, cfg, fb, torch.full((fb.B,), tval))
        eps_h, eps_x = run_forward("egnn", model, batch, graphs, kk, t_in, tval, dev)
        torch.cuda.synchronize()
        eh, ex = rel_err(eps_h.cpu(), ref_h), rel_err(eps_x.cpu(), ref_x)
        print(f"egnn full size bf16 t={tval}: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
        assert eh < TOL_BF16 and ex < TOL_BF16


@pytest.mark.parametrize("name", sorted(n for n in SHIPPED if n.startswith("egnn")))
def test_egnn_bf16_shipped_config_vs_oracle(name):
    """Every shipped EGNN width (H = 257: the compile-time-width edge kernel) against the CPU oracle."""
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    arch, sd, kw, rec_nf, inputs = shipped_case(name)
    cfg = oracle_cfg(arch, kw, 10, rec_nf)
    model = build_model(arch, sd, kw, 10, rec_nf, dev)
    assert model.tc_blob2 is not None, "every shipped width must run on the tensor cores"
    model.set_precision("bf16")
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
    with_lk = bool(kw.get("update_kp_feat", False))
    graphs = ops.LigandGraphs(batch, gp, with_lk).build(t_in["lig_x"], t_in["kp_x"])
    for tval in (0.001, 0.5, 1.0):
        fb = flat_batch(inputs)
        ref_h, ref_x, edges, _ = oracle_forward(arch, sd, cfg, fb, torch.full((fb.B,), tval), return_edges=True)
        eps_h, eps_x = run_forward(arch, model, batch, graphs, kk, t_in, tval, dev)
        torch.cuda.synchronize()
        for et in ("ll", "kl") + (("lk",) if with_lk else ()):
            assert edge_set(getattr(graphs, et).edges()) == edge_set(torch.stack(edges[et])), (name, et)
        rh, rx = err_report(eps_h.cpu(), ref_h), err_report(eps_x.cpu(), ref_x)
        print(f"{name} [bf16] t={tval}: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)}")
        assert rh["norm"] < TOL_BF16 and rx["norm"] < TOL_BF16, (name, tval, rh, rx)


def test_egnn_bf16_all_atom_rows_span_many_tiles():
    """A ligand atom with ~300 kl edges: its CSR row spans more than three 64-edge tiles, so the segmented reduction's
    per-tile partial slots (first / last segment of a tile) are exercised in the bf16 layout; run-time hidden width (33)."""
    from test_gpu_cases import _inputs, _run_both
    from oracle import params as P
    from keypoint_diffusion_b200 import synthetic
    kw = dict(n_layers=2, hidden_nf=32, use_tanh=True, message_norm=0.0, update_kp_feat=True, norm=True, ll_k=0, kl_k=5,
              graph_cutoffs={"ll": 6, "kl": 6, "kk": 8, "rr": 3.5})
    sd = P.init_state_dict(P.egnn_dynamics_shapes(10, 10, 2, 32, True, True), seed=11, coord_gain=0.3)
    pockets = [synthetic.all_atom_pocket(i, 300, 10, 0, 3.5) for i in range(2)]
    inputs = _inputs(pockets, [20, 5, 1, 33], 10, seed=3, with_v=False)
    (eh, ex, graphs, _), = _run_both("egnn", sd, kw, 10, 10, inputs, mode="bf16")
    rp = graphs.kl.rowptr.cpu()
    deg = int((rp[1:] - rp[:-1]).max())
    assert deg > 3 * 64, "test should exercise rows spanning more than three tiles"
    print(f"all-atom egnn [bf16]: max kl in-degree {deg}, rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
    assert eh < TOL_BF16 and ex < TOL_BF16


def test_egnn_bf16_e3_properties_and_determinism_at_baseline_size():
    """100 ligands of 20 atoms: eps_h invariant and eps_x equivariant under a rotation plus shift within the bf16 bar;
    two identical launches agree bit for bit."""
    from test_gpu_properties import _baseline_case, _forward, _rotation
    dev = _dev()
    model, gp, inputs, device_inputs = _baseline_case("egnn", 100, dev)
    model.set_precision("bf16")
    h0, x0, e0 = _forward("egnn", model, gp, inputs, device_inputs, dev)
    h0b, x0b, _ = _forward("egnn", model, gp, inputs, device_inputs, dev)
    assert torch.equal(h0, h0b) and torch.equal(x0, x0b), "two identical launches must agree bit for bit"
    R = _rotation(5)
    shift = torch.tensor([3.0, -2.0, 1.5], dtype=torch.float64)
    moved = dict(inputs)
    moved["lig_x"] = (inputs["lig_x"].double() @ R.t() + shift).float()
    moved["kp_x"] = (inputs["kp_x"].double() @ R.t() + shift).float()
    h1, x1, e1 = _forward("egnn", model, gp, moved, device_inputs, dev)
    assert e0 == e1
    eh = rel_err(h1.cpu(), h0.cpu())
    ex = rel_err(x1.cpu(), (x0.cpu().double() @ R.t()))
    print(f"egnn [bf16] equivariance at 100 ligands: invariance of eps_h {eh:.2e}, equivariance of eps_x {ex:.2e}")
    assert eh < TOL_BF16 and ex < TOL_BF16


def _loop_sampler(model, fx, dev, use_graph=True):
    """The injected-noise loop of the loop_egnn golden through the captured sampler."""
    from oracle import schedule as S
    from test_gpu_parity import device_inputs
    from keypoint_diffusion_b200 import ops
    kw, T, F = fx["kwargs"], fx["T"], fx["atom_nf"]
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    coef = S.coefficient_table(fx["state_dict"]["gamma.gamma"], T).to(dev).contiguous()
    torch.manual_seed(fx["noise_seed"])
    slots = []
    for _ in range(T + 1):
        nx = torch.randn(batch.n_lig, 3)
        nh = torch.randn(batch.n_lig, F)
        slots.append(torch.cat([nx.reshape(-1), nh.reshape(-1)]))
    noise = torch.stack(slots).to(dev).contiguous()
    sampler = ops.Sampler(model, batch, gp, kk, coef, T, F, steps_per_graph=4, use_cuda_graph=use_graph)
    x_lig, h_lig, _ = sampler.run(t_in["kp_x"], t_in["kp_h"], None, fx["init_lig_pos"].to(dev), noise=noise)
    torch.cuda.synchronize()
    return x_lig.cpu(), h_lig.cpu()


def test_egnn_bf16_full_loop_matches_reference():
    from test_gpu_parity import build_model
    dev = _dev()
    fx = load_golden("loop_egnn")
    model = build_model("egnn", fx["state_dict"], fx["kwargs"], fx["atom_nf"], fx["rec_nf"], dev)
    model.set_precision("bf16")
    x, h = _loop_sampler(model, fx, dev)
    ex, eh = rel_err(x, torch.cat(fx["positions"])), rel_err(h, torch.cat(fx["features"]))
    print(f"loop egnn [bf16] captured: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < TOL_BF16 and eh < TOL_BF16


def test_egnn_bf16_seeded_sampling_is_reproducible():
    from test_gpu_cases import _module_case
    _, model, g = _module_case("egnn")
    model.dynamics.set_precision("bf16")
    model.n_timesteps = 1000
    init = torch.zeros(3, 3)
    pos, feat = model.sample_from_encoded_receptors(g, init_lig_pos=init, seed=5, steps_per_graph=25)
    assert model.dynamics.device_model(torch.device("cuda:0")).precision == "bf16"
    pos2, feat2 = model.sample_from_encoded_receptors(g, init_lig_pos=init, seed=5, steps_per_graph=25)
    assert all(torch.isfinite(p).all() for p in pos)
    assert all(torch.equal(a, b) for a, b in zip(pos, pos2)) and all(torch.equal(a, b) for a, b in zip(feat, feat2))
    print(f"egnn [bf16] seeded sampling: {len(pos)} ligands, bit-identical on a second run")


def test_egnn_no_leakage_from_bf16_into_bf16x3():
    """A model that ran in bf16 and was switched back to bf16x3 computes exactly what a model that never saw bf16 does:
    one forward call, and one captured sampling run."""
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    fx = load_golden("egnn_small_kp")
    kw = fx["kwargs"]
    fresh = build_model("egnn", fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    fresh.set_precision("bf16x3")
    switched = build_model("egnn", fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, bool(kw.get("update_kp_feat", False))).build(t_in["lig_x"], t_in["kp_x"])
    switched.set_precision("bf16")
    h16, _ = run_forward("egnn", switched, batch, graphs, kk, t_in, 0.5, dev)
    h16 = h16.clone()
    switched.set_precision("bf16x3")
    ha, xa = run_forward("egnn", fresh, batch, graphs, kk, t_in, 0.5, dev)
    hb, xb = run_forward("egnn", switched, batch, graphs, kk, t_in, 0.5, dev)
    torch.cuda.synchronize()
    d16 = rel_err(h16.cpu(), ha.cpu())
    assert d16 > 0, "the bf16 mode should differ from bf16x3 in the last bits at least"
    assert torch.equal(ha, hb) and torch.equal(xa, xb)

    lp = load_golden("loop_egnn")
    fresh = build_model("egnn", lp["state_dict"], lp["kwargs"], lp["atom_nf"], lp["rec_nf"], dev)
    fresh.set_precision("bf16x3")
    switched = build_model("egnn", lp["state_dict"], lp["kwargs"], lp["atom_nf"], lp["rec_nf"], dev)
    switched.set_precision("bf16")
    _loop_sampler(switched, lp, dev)
    switched.set_precision("bf16x3")
    xa, ha = _loop_sampler(fresh, lp, dev)
    xb, hb = _loop_sampler(switched, lp, dev)
    assert torch.equal(xa, xb) and torch.equal(ha, hb)
    print(f"egnn bf16 -> bf16x3: forward and captured loop bit-identical to a fresh bf16x3 model "
          f"(the bf16 forward differs from bf16x3 by {d16:.2e})")
