"""GPU: the GVP denoiser at the batch layouts and shapes the sampler runs, against an fp64 restatement of the oracle.

  A. oracle parity on both sides of the 32-complex switch (gvp.cu: 32-row node / head tiles below 32 complexes, 64-row
     tiles from 32 on), at B = 31, 32, 100, in fp32, bf16x3 and bf16; complexes 0..30 of B = 32 against B = 31;
  B. destination rows that span three or more edge tiles (all-atom pocket, kl radius graph);
  C. a per-complex time vector, through GvpModel.forward and through the drop-in dynamics(g, t, batch_idxs);
  D. the plain-bf16 mode on the shipped configs, and a bf16 -> bf16x3 switch that leaves nothing behind;
  E. the headline sampling layout: 100 ligands in 4 groups, capacity buckets of 32 complexes vs the exact layout;
  F. graph construction past 1024 complexes (the carry between the 1024-wide chunks of the per-complex scan).

The reference is oracle/flat.py in fp64, on the edge lists the oracle builds from the fp32 coordinates (so a distance
within rounding of a cutoff cannot make the two sides disagree on the graph).  Bars: fp32 and bf16x3 -- max|a-b|/max|b|
and rms-relative <= 1e-4, per-channel <= 5e-4 (helpers.err_report); bf16 -- max|a-b|/max|b| <= 3e-2; edge sets exact.
Every test prints the errors it measured."""
import functools

import pytest
import torch
import yaml

from helpers import GOLDEN, edge_set, err_report, flat_batch, fmt_err, load_golden, oracle_cfg, oracle_forward, rel_err
from shipped_cases import SHIPPED, shipped_case

pytestmark = pytest.mark.gpu
TOL, TOL_CHAN, TOL_BF16 = 1e-4, 5e-4, 3e-2
MODES = ["fp32", "bf16x3", "bf16"]


def _dev():
    return torch.device("cuda:0")


def _assert_bars(mode, rh, rx, ctx):
    for r in (rh, rx):
        if mode == "bf16":
            assert r["norm"] < TOL_BF16, (ctx, mode, rh, rx)
        else:
            assert r["norm"] < TOL and r["rms"] < TOL and r["chan"] < TOL_CHAN, (ctx, mode, rh, rx)


def _with_lk(kw):
    return bool(kw.get("update_kp_feat", kw.get("update_kp", False)))


def _reference(arch, sd, cfg, inputs, t, with_lk):
    """(eps_h, eps_x, edges) of the oracle in fp64; the graph is built from the fp32 coordinates the device sees."""
    from oracle import flat
    fb = flat_batch(inputs)
    lig_b, kp_b = fb.batch_idx()
    edges = flat.build_lig_edges(fb.lig_x, fb.kp_x, lig_b, kp_b, fb.B, cfg.graph_cutoffs, cfg.ll_k, cfg.kl_k, with_lk)
    h, x = oracle_forward(arch, sd, cfg, flat_batch(inputs, torch.float64), t.double(), edges=edges)
    return h, x, edges[0]


def _device_run(arch, model, inputs, kw, t):
    """One forward on the device; t: [1] (shared) or [B] (per complex) CPU tensor.  -> (eps_h, eps_x, graphs)."""
    from test_gpu_parity import device_inputs
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    with_lk = _with_lk(kw)
    graphs = ops.LigandGraphs(batch, gp, with_lk).build(t_in["lig_x"], t_in["kp_x"])
    args = [t_in["lig_h"], t_in["lig_x"], t_in["kp_h"], t_in["kp_x"]] + ([t_in["kp_v"]] if arch == "gvp" else [])
    eps_h, eps_x = model.forward(batch, graphs, kk if with_lk else None, *args, t.float().to(dev))
    torch.cuda.synchronize()
    return eps_h.cpu(), eps_x.cpu(), graphs, batch


def _check_edges(graphs, edges, with_lk, ctx):
    for et in ("ll", "kl") + (("lk",) if with_lk else ()):
        assert edge_set(getattr(graphs, et).edges()) == edge_set(torch.stack(edges[et])), (ctx, et)


def _model(arch, sd, kw, rec_nf, mode):
    from test_gpu_parity import build_model
    model = build_model(arch, sd, kw, 10, rec_nf, _dev())
    if mode != "fp32":
        assert model.tc_blob2 is not None, "this case should run on the tensor cores"
        model.set_precision(mode)
    return model


def _prefix(inputs, n):
    """The first n complexes of a batch (flat inputs; kk edges grouped by complex)."""
    ln, kn = inputs["lig_n"], inputs["kp_n"]
    L, K = int(ln[:n].sum()), int(kn[:n].sum())
    m = inputs["kk_dst"] < K
    out = {"lig_n": ln[:n], "kp_n": kn[:n], "lig_x": inputs["lig_x"][:L], "lig_h": inputs["lig_h"][:L],
           "kp_x": inputs["kp_x"][:K], "kp_h": inputs["kp_h"][:K], "kk_src": inputs["kk_src"][m],
           "kk_dst": inputs["kk_dst"][m]}
    if "kp_v" in inputs:
        out["kp_v"] = inputs["kp_v"][:K]
    return out


# --------------------------------------------------------------------------- A. the 32-complex switch

@functools.lru_cache(maxsize=None)
def _baseline_case(arch, B):
    """Full-size 20-keypoint model (shipped hyper-parameters, seeded weights), one pocket, B ligands of mixed size."""
    from test_gpu_parity import _full_size_case
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    sizes = [(20, 8, 35, 20, 13, 27, 17, 24)[i % 8] for i in range(B)]
    return _full_size_case(arch, cfgs, n_lig=sizes, n_pockets=1)


@functools.lru_cache(maxsize=None)
def _baseline_reference(arch, B, tval):
    sd, kw, rec_nf, inputs = _baseline_case(arch, max(B, 32))
    inputs = _prefix(inputs, B)
    cfg = oracle_cfg(arch, kw, 10, rec_nf)
    return _reference(arch, sd, cfg, inputs, torch.full((B,), tval), True)


@pytest.mark.parametrize("arch,mode", [("gvp", "fp32"), ("gvp", "bf16x3"), ("gvp", "bf16"), ("egnn", "bf16")])
def test_oracle_parity_across_the_32_complex_node_tile_switch(arch, mode):
    """B = 31 runs the 32-row GVP node / head kernels, B = 32 and 100 the 64-row ones.  B = 31 is the first 31 complexes
    of the B = 32 batch, so their rows must agree (same per-row arithmetic, other tiles)."""
    sd, kw, rec_nf, _ = _baseline_case(arch, 32)
    model = _model(arch, sd, kw, rec_nf, mode)
    seen_B = set()
    for B in (31, 32, 100):
        _, _, _, full = _baseline_case(arch, max(B, 32))
        inputs = _prefix(full, B)
        for tval in (0.001, 0.5, 1.0):
            ref_h, ref_x, edges = _baseline_reference(arch, B, tval)
            eps_h, eps_x, graphs, batch = _device_run(arch, model, inputs, kw, torch.full((1,), tval))
            seen_B.add(batch.B)
            _check_edges(graphs, edges, True, (arch, B))
            rh, rx = err_report(eps_h, ref_h), err_report(eps_x, ref_x)
            print(f"{arch} [{mode}] B={B} t={tval}: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)}")
            _assert_bars(mode, rh, rx, (arch, B, tval))
    assert min(seen_B) < 32 <= max(seen_B), "both node-tile sizes must run"
    _, _, _, full = _baseline_case(arch, 32)
    n31 = int(full["lig_n"][:31].sum())
    for tval in (0.001, 0.5, 1.0):
        h31, x31, _, _ = _device_run(arch, model, _prefix(full, 31), kw, torch.full((1,), tval))
        h32, x32, _, _ = _device_run(arch, model, full, kw, torch.full((1,), tval))
        dh, dx = rel_err(h32[:n31], h31), rel_err(x32[:n31], x31)
        print(f"{arch} [{mode}] t={tval}: complexes 0..30 of B=32 vs B=31: eps_h {dh:.2e} eps_x {dx:.2e}")
        assert dh < 2e-5 and dx < 2e-5, (tval, dh, dx)


# --------------------------------------------------------------------------- B. rows spanning many edge tiles

# (n_hidden_scalars, rbf_dim, message_norm) -> edge tile of each mode: fp32 SIMT 64 rows; bf16 128; bf16x3 the 128-row
# KS kernel, except at S = 256, rbf_dim = 32 where its tile does not fit in shared memory and the stacked 64-row
# kernel runs (gvp.cu: kpd_gvp_attach_tc).  Shipped width S = 256: at S = 64 the vector output of this case is ~5x worse
# conditioned in every mode, and bf16 lands at 3.3e-2.
MANY_TILE_CASES = {"S256_mean": (256, 16, "mean", {"fp32": 64, "bf16": 128, "bf16x3": 128}),
                   "S256_rbf32_zero": (256, 32, 0, {"fp32": 64, "bf16": 128, "bf16x3": 64})}


@functools.lru_cache(maxsize=None)
def _many_tile_case(name):
    """Two 600-atom all-atom pockets (keypoints := atoms, non-zero vectors), a kl radius graph of 7 A around ligand
    atoms near the pocket centre (hundreds of kl edges into one atom), ligands of 20, 1, 33 and 12 atoms."""
    from oracle import params as P
    from keypoint_diffusion_b200 import synthetic
    from test_gpu_cases import _inputs
    S, rbf_dim, norm, _ = MANY_TILE_CASES[name]
    kw = dict(vector_size=16, n_convs=2, n_hidden_scalars=S, message_norm=norm, update_kp=True, ll_k=0, kl_k=0,
              n_message_gvps=3, n_update_gvps=2, n_noise_gvps=4, rbf_dim=rbf_dim,
              graph_cutoffs={"ll": 6, "kl": 7, "kk": 8, "rr": 3.5})
    sd = P.init_state_dict(P.gvp_dynamics_shapes(10, 10, 16, 2, S, True, 3, 2, 4, rbf_dim=rbf_dim), seed=14)
    for k in sd:
        if k.endswith(".Wh") or k.endswith(".Wu"):
            sd[k] = sd[k] * 2.0
    pockets = [synthetic.all_atom_pocket(i, 600, 10, 16, 3.5) for i in range(2)]
    for i, pk in enumerate(pockets):
        pk.kp_v = 0.1 * torch.randn(pk.n_kp, 16, 3, generator=torch.Generator().manual_seed(60 + i))
    inputs = _inputs(pockets, [20, 1, 33, 12], 10, seed=7, with_v=True)
    cfg = oracle_cfg("gvp", kw, 10, 10)
    ref = _reference("gvp", sd, cfg, inputs, torch.full((4,), 0.3), True)
    return sd, kw, inputs, ref


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", sorted(MANY_TILE_CASES))
def test_gvp_rows_span_many_edge_tiles(name, mode):
    sd, kw, inputs, (ref_h, ref_x, edges) = _many_tile_case(name)
    tile = MANY_TILE_CASES[name][3][mode]
    model = _model("gvp", sd, kw, 10, mode)
    eps_h, eps_x, graphs, _ = _device_run("gvp", model, inputs, kw, torch.full((1,), 0.3))
    _check_edges(graphs, edges, True, name)
    rp = graphs.kl.rowptr.cpu().long()
    deg = int((rp[1:] - rp[:-1]).max())
    assert int(inputs["lig_n"].min()) == 1
    assert deg > 2 * tile, f"a kl row must span three or more {tile}-edge tiles (max in-degree {deg})"
    rh, rx = err_report(eps_h, ref_h), err_report(eps_x, ref_x)
    print(f"gvp many-tile {name} [{mode}] max kl in-degree {deg} (edge tile {tile}): eps_h {fmt_err(rh)} | "
          f"eps_x {fmt_err(rx)}")
    _assert_bars(mode, rh, rx, name)


# --------------------------------------------------------------------------- C. per-complex t

@pytest.mark.parametrize("mode", MODES)
def test_gvp_per_complex_time(mode):
    """A [B] vector of distinct t through GvpModel.forward: the SIMT time concatenation and the per-complex gather of
    the fused tensor-core encoder."""
    from test_gpu_parity import _full_size_case
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    sd, kw, rec_nf, inputs = _full_size_case("gvp", cfgs)
    t = torch.tensor([0.001, 0.2, 0.35, 0.5, 0.75, 1.0])
    assert t.numel() == int(inputs["lig_n"].numel()) and len(set(t.tolist())) == t.numel()
    ref_h, ref_x, edges = _reference("gvp", sd, oracle_cfg("gvp", kw, 10, rec_nf), inputs, t, True)
    model = _model("gvp", sd, kw, rec_nf, mode)
    eps_h, eps_x, graphs, _ = _device_run("gvp", model, inputs, kw, t)
    _check_edges(graphs, edges, True, "per-complex t")
    rh, rx = err_report(eps_h, ref_h), err_report(eps_x, ref_x)
    print(f"gvp per-complex t [{mode}]: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)}")
    _assert_bars(mode, rh, rx, "per-complex t")
    # and t does reach each complex: the shared-t result differs from the per-complex one
    h_one, _, _, _ = _device_run("gvp", model, inputs, kw, t[:1])
    assert not torch.equal(h_one, eps_h)


@pytest.mark.parametrize("mode", MODES)
def test_gvp_dynamics_module_per_complex_time(mode):
    """dynamics(g, t, batch_idxs) of the drop-in LigRecDynamicsGVP with a distinct t per complex."""
    from test_gpu_cases import _module_case
    from keypoint_diffusion_b200.utils import get_batch_idxs
    cfg, model, g_cpu = _module_case("gvp")
    model.dynamics.set_precision(mode)
    g = g_cpu.to(_dev())
    t = torch.tensor([0.1, 0.55, 0.9])
    assert t.numel() == g.batch_size and len(set(t.tolist())) == t.numel()
    eps_h, eps_x = model.dynamics(g, t.to(_dev()), get_batch_idxs(g))
    torch.cuda.synchronize()
    assert model.dynamics.device_model(_dev()).precision == mode
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    kw = dict(cfg["dynamics_gvp"])
    kw["graph_cutoffs"] = cfg["graph"]["graph_cutoffs"]
    ocfg = oracle_cfg("gvp", kw, 10, 128)
    ks, kd = g_cpu.edges(form="uv", etype="kk")
    inputs = {"lig_n": g_cpu.batch_num_nodes("lig"), "kp_n": g_cpu.batch_num_nodes("kp"),
              "lig_x": g_cpu.nodes["lig"].data["x_0"], "lig_h": g_cpu.nodes["lig"].data["h_0"],
              "kp_x": g_cpu.nodes["kp"].data["x_0"], "kp_h": g_cpu.nodes["kp"].data["h_0"],
              "kp_v": g_cpu.nodes["kp"].data["v_0"], "kk_src": ks, "kk_dst": kd}
    ref_h, ref_x, _ = _reference("gvp", sd, ocfg, inputs, t, True)
    rh, rx = err_report(eps_h.cpu(), ref_h), err_report(eps_x.cpu(), ref_x)
    print(f"gvp dynamics module per-complex t [{mode}]: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)}")
    _assert_bars(mode, rh, rx, "module per-complex t")


# --------------------------------------------------------------------------- D. plain bf16 at the shipped configs

@pytest.mark.parametrize("name", sorted(n for n in SHIPPED if n.startswith("gvp")))
def test_gvp_bf16_shipped_config_vs_oracle(name):
    arch, sd, kw, rec_nf, inputs = shipped_case(name)
    cfg = oracle_cfg(arch, kw, 10, rec_nf)
    model = _model(arch, sd, kw, rec_nf, "bf16")
    for tval in (0.001, 0.5, 1.0):
        ref_h, ref_x, edges = _reference(arch, sd, cfg, inputs, torch.full((int(inputs["lig_n"].numel()),), tval),
                                         _with_lk(kw))
        eps_h, eps_x, graphs, _ = _device_run(arch, model, inputs, kw, torch.full((1,), tval))
        _check_edges(graphs, edges, _with_lk(kw), name)
        rh, rx = err_report(eps_h, ref_h), err_report(eps_x, ref_x)
        print(f"{name} [bf16] t={tval}: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)}")
        _assert_bars("bf16", rh, rx, (name, tval))


def test_gvp_bf16_full_loop_matches_reference():
    from test_gpu_egnn_bf16 import _loop_sampler
    from test_gpu_parity import build_model
    dev = _dev()
    fx = load_golden("loop_gvp")
    model = build_model("gvp", fx["state_dict"], fx["kwargs"], fx["atom_nf"], fx["rec_nf"], dev)
    model.set_precision("bf16")
    x, h = _loop_sampler(model, fx, dev)
    ex, eh = rel_err(x, torch.cat(fx["positions"])), rel_err(h, torch.cat(fx["features"]))
    print(f"loop gvp [bf16] captured: rel_err pos={ex:.2e} feat={eh:.2e}")
    assert ex < TOL_BF16 and eh < TOL_BF16


def test_gvp_no_leakage_from_bf16_into_bf16x3():
    """A GVP model that ran in bf16 and was switched back to bf16x3 computes exactly what a model that never ran bf16
    does: one forward (at 32 complexes: the 64-row node tiles) and one captured sampling run."""
    from test_gpu_egnn_bf16 import _loop_sampler
    from test_gpu_parity import build_model
    dev = _dev()
    sd, kw, rec_nf, inputs = _baseline_case("gvp", 32)
    fresh = _model("gvp", sd, kw, rec_nf, "bf16x3")
    switched = _model("gvp", sd, kw, rec_nf, "bf16")
    h16, _, _, _ = _device_run("gvp", switched, inputs, kw, torch.full((1,), 0.5))
    switched.set_precision("bf16x3")
    ha, xa, _, _ = _device_run("gvp", fresh, inputs, kw, torch.full((1,), 0.5))
    hb, xb, _, _ = _device_run("gvp", switched, inputs, kw, torch.full((1,), 0.5))
    d16 = rel_err(h16, ha)
    assert d16 > 0, "the bf16 mode should differ from bf16x3 in the last bits at least"
    assert torch.equal(ha, hb) and torch.equal(xa, xb)

    lp = load_golden("loop_gvp")
    fresh = build_model("gvp", lp["state_dict"], lp["kwargs"], lp["atom_nf"], lp["rec_nf"], dev)
    fresh.set_precision("bf16x3")
    switched = build_model("gvp", lp["state_dict"], lp["kwargs"], lp["atom_nf"], lp["rec_nf"], dev)
    switched.set_precision("bf16")
    _loop_sampler(switched, lp, dev)
    switched.set_precision("bf16x3")
    xa, ha = _loop_sampler(fresh, lp, dev)
    xb, hb = _loop_sampler(switched, lp, dev)
    assert torch.equal(xa, xb) and torch.equal(ha, hb)
    print(f"gvp bf16 -> bf16x3: forward and captured loop bit-identical to a fresh bf16x3 model "
          f"(the bf16 forward differs from bf16x3 by {d16:.2e})")


# --------------------------------------------------------------------------- E. the headline sampling layout

@pytest.mark.parametrize("mode", ["bf16x3", "bf16"])
def test_gvp_headline_layout_capacity_equals_exact(mode):
    """100 ligands in 4 concurrent groups of 25 complexes: capacity=True pads each group to a bucket of 32 complexes
    (64-row node / head tiles), capacity=False captures the exact 25-complex layout (32-row tiles).  The two layouts
    differ in the association of fp32 partial sums in the edge tile that straddles the real / filler boundary (~1 ulp);
    in bf16 such a difference can move an operand by one bf16 rounding step, which 40 steps carry to ~2.4e-5."""
    from test_gpu_sample_api import _bench_like_model
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    dev = _dev()
    model, cfg = _bench_like_model("gvp", dev, T=40)
    model.dynamics.set_precision(mode)
    pk = synthetic.keypoint_pocket(0, 20, cfg["rec_encoder_gvp"]["out_scalar_size"], cfg["dynamics_gvp"]["vector_size"],
                                   cfg["graph"]["graph_cutoffs"]["kk"])
    sizes = [(20, 14, 27, 20, 9, 31, 18, 22)[i % 8] for i in range(100)]
    g = HeteroBatch.from_pockets([pk], sizes, 10).to(dev)
    init = torch.zeros(100, 3, device=dev)
    out = {}
    for capacity in (True, False):
        x, h = model.sample_from_encoded_receptors(g, init_lig_pos=init, seed=7, steps_per_graph=10, sub_batches=4,
                                                   return_device_tensors=True, capacity=capacity)
        torch.cuda.synchronize()
        out[capacity] = (x.cpu(), h.cpu())
    cap_B = {k[2][0] for k in model._samplers if k[0] == "cap"}
    assert cap_B == {32}, f"the capacity plan of a 25-complex group should be 32 complexes, got {cap_B}"
    assert model.dynamics.device_model(dev).precision == mode
    (xc, hc), (xe, he) = out[True], out[False]
    assert torch.isfinite(xc).all() and torch.isfinite(hc).all()
    ex, eh = rel_err(xc, xe), rel_err(hc, he)
    print(f"headline layout [gvp {mode}]: capacity (B=32 buckets) vs exact (B=25): rel_err pos {ex:.2e} feat {eh:.2e}")
    tol = 1e-4 if mode == "bf16" else 1e-5
    assert ex < tol and eh < tol


# --------------------------------------------------------------------------- F. graph build past 1024 complexes

@pytest.mark.parametrize("ll_k,kl_k", [(0, 7), (4, 0)])
@pytest.mark.parametrize("B", [1023, 1024, 1025, 2100])
def test_graph_build_beyond_1024_complexes(B, ll_k, kl_k):
    from oracle import flat
    from test_gpu_properties import _ragged_case
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    g = torch.Generator().manual_seed(B + ll_k)
    sizes_l = torch.randint(1, 13, (B,), generator=g).tolist()
    sizes_k = torch.randint(1, 25, (B,), generator=g).tolist()
    cutoffs = {"ll": 5.0, "kl": 6.0}
    lig_x, kp_x = _ragged_case(B + kl_k, sizes_l, sizes_k, 0.5)
    batch = ops.DeviceBatch(sizes_l, sizes_k, dev)
    assert batch.B == B
    gp = ops.GraphParams.from_module(ll_k, kl_k, cutoffs)
    graphs = ops.LigandGraphs(batch, gp, True).build(lig_x.to(dev), kp_x.to(dev))
    torch.cuda.synchronize()
    lig_b = torch.repeat_interleave(torch.arange(B), torch.tensor(sizes_l))
    kp_b = torch.repeat_interleave(torch.arange(B), torch.tensor(sizes_k))
    edges, counts = flat.build_lig_edges(lig_x, kp_x, lig_b, kp_b, B, cutoffs, ll_k, kl_k, True)
    n_e = {}
    for et in ("ll", "kl", "lk"):
        csr = getattr(graphs, et)
        got = csr.edges()
        assert edge_set(got) == edge_set(torch.stack(edges[et])), et
        d = got[1]
        assert torch.all(d[1:] >= d[:-1]), et
        rp = csr.rowptr.cpu().long()
        assert int(rp[-1]) == got.shape[1]
        assert torch.equal(torch.bincount(d, minlength=csr.n_dst), rp[1:] - rp[:-1]), et
        n_e[et] = got.shape[1]
    assert torch.equal(graphs.counts_ll.cpu().long(), counts["ll"].long())
    assert torch.equal(graphs.counts_kl.cpu().long(), counts["kl"].long())
    kl = graphs.kl.edges()
    assert torch.equal(kp_b[kl[0]], lig_b[kl[1]])
    ll = graphs.ll.edges()
    assert torch.equal(lig_b[ll[0]], lig_b[ll[1]])
    print(f"graph build B={B} ll_k={ll_k} kl_k={kl_k}: {sum(sizes_l)} ligand atoms, {sum(sizes_k)} keypoints, "
          f"edges {n_e}: exact")
