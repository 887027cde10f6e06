"""GPU parity, edge cases and the drop-in module API (through the C ABI) against the CPU oracle:
destination rows spanning many 64-edge tiles (all-atom pockets), empty edge types, single-atom
ligands (fewer than k neighbours), the 'intended' EGNN normalisation flag, per-complex t, the
module-level API contract (g left unchanged, in-place step, CPU lists out)."""
import pytest
import torch

from helpers import edge_set, flat_batch, oracle_cfg, oracle_forward, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _dev():
    return torch.device("cuda:0")


def _inputs(pockets, n_lig, atom_nf, seed, with_v):
    from keypoint_diffusion_b200 import synthetic
    x_l, h_l = synthetic.ligand_noise_state(n_lig, atom_nf, seed)
    kx, kh, kv, ks, kd, kn, off = [], [], [], [], [], [], 0
    for i in range(len(n_lig)):
        pk = pockets[i % len(pockets)]
        kx.append(pk.kp_x); kh.append(pk.kp_h)
        if with_v:
            kv.append(pk.kp_v)
        ks.append(pk.kk_src + off); kd.append(pk.kk_dst + off)
        off += pk.n_kp
        kn.append(pk.n_kp)
    d = {"lig_n": torch.tensor(n_lig), "kp_n": torch.tensor(kn), "lig_x": x_l, "lig_h": h_l, "kp_x": torch.cat(kx),
         "kp_h": torch.cat(kh), "kk_src": torch.cat(ks), "kk_dst": torch.cat(kd)}
    if with_v:
        d["kp_v"] = torch.cat(kv)
    return d


MODES = ["fp32", "bf16x3"]      # SIMT kernels / tcgen05 kernels with split bf16 operands: same 1e-4 bar
TOL_BY_MODE = {"fp32": TOL, "bf16x3": TOL, "bf16": 3e-2}     # plain bf16 operands: 3e-2 of the output scale


def _run_both(arch, sd, kw, atom_nf, rec_nf, inputs, tvals=(0.3,), per_complex_t=False, z_effective=False, mode="fp32"):
    from test_gpu_parity import build_model, device_inputs
    from keypoint_diffusion_b200 import ops
    dev = _dev()
    cfg = oracle_cfg(arch, kw, atom_nf, rec_nf)
    if arch == "egnn":
        cfg.z_effective = z_effective
        sdd = {k[len("dynamics."):]: v for k, v in sd.items()}
        model = ops.EgnnModel(sdd, atom_nf=atom_nf, rec_nf=rec_nf, hidden_nf=kw["hidden_nf"], n_layers=kw["n_layers"],
                              use_tanh=kw["use_tanh"], update_kp_feat=kw["update_kp_feat"], norm=kw["norm"],
                              message_norm=kw["message_norm"], device=dev, z_effective=z_effective)
    else:
        model = build_model(arch, sd, kw, atom_nf, rec_nf, dev)
    if mode != "fp32":
        assert model.tc_blob2 is not None, "this case should be able to run on the tensor cores"
        model.set_precision(mode)
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    with_lk = bool(kw.get("update_kp_feat", kw.get("update_kp", False)))
    graphs = ops.LigandGraphs(batch, gp, with_lk).build(t_in["lig_x"], t_in["kp_x"])
    out = []
    for tv in tvals:
        fb = flat_batch(inputs)
        t = torch.full((fb.B,), tv)
        if per_complex_t:
            t = t + 0.05 * torch.arange(fb.B)
        ref_h, ref_x, edges, counts = oracle_forward(arch, sd, cfg, fb, t, return_edges=True)
        td = t.to(dev) if per_complex_t else t[:1].to(dev)
        args = [t_in["lig_h"], t_in["lig_x"], t_in["kp_h"], t_in["kp_x"]]
        if arch == "gvp":
            args.append(t_in["kp_v"])
        eps_h, eps_x = model.forward(batch, graphs, kk if with_lk else None, *args, td)
        torch.cuda.synchronize()
        for et in ("ll", "kl") + (("lk",) if with_lk else ()):
            got = getattr(graphs, et).edges()
            assert edge_set(got) == edge_set(torch.stack(edges[et])), et
        out.append((rel_err(eps_h.cpu(), ref_h), rel_err(eps_x.cpu(), ref_x), graphs, edges))
    return out


@pytest.mark.parametrize("mode", MODES)
def test_egnn_all_atom_rows_span_many_tiles(mode):
    """~300 pocket atoms as keypoints (fixed encoder): a ligand atom receives hundreds of kl edges, so
    its CSR row spans several 64-edge tiles and the per-tile partial slots are summed in tile order;
    includes a single-atom ligand (no ll edges, fewer than k candidates)."""
    from oracle import params as P
    from keypoint_diffusion_b200 import synthetic
    kw = dict(n_layers=2, hidden_nf=32, use_tanh=True, message_norm=0.0, update_kp_feat=True, norm=True, ll_k=0, kl_k=5,
              graph_cutoffs={"ll": 6, "kl": 6, "kk": 8, "rr": 3.5})
    sd = P.init_state_dict(P.egnn_dynamics_shapes(10, 10, 2, 32, True, True), seed=11, coord_gain=0.3)
    pockets = [synthetic.all_atom_pocket(i, 300, 10, 0, 3.5) for i in range(2)]
    inputs = _inputs(pockets, [20, 5, 1, 33], 10, seed=3, with_v=False)
    (eh, ex, graphs, edges), = _run_both("egnn", sd, kw, 10, 10, inputs, mode=mode)
    rp = graphs.kl.rowptr.cpu()
    assert int((rp[1:] - rp[:-1]).max()) > 3 * 64, "test should exercise rows spanning > 3 tiles"
    print(f"all-atom egnn [{mode}]: max kl in-degree {int((rp[1:] - rp[:-1]).max())}, rel_err {eh:.2e} {ex:.2e}")
    assert eh < TOL and ex < TOL


@pytest.mark.parametrize("mode", MODES + ["bf16"])
@pytest.mark.parametrize("norm", ["mean", 0, 10.0])
def test_gvp_ca_like_empty_kk_and_norm_modes(norm, mode):
    """C-alpha style pocket: 42 nodes >= 3.8 A apart, kk = radius 3.5 graph => (almost) no kk edges, so
    keypoints with zero in-degree and an empty edge type are exercised in all three norm modes."""
    from oracle import params as P
    from keypoint_diffusion_b200 import synthetic
    kw = dict(vector_size=16, n_convs=3, n_hidden_scalars=64, message_norm=norm, update_kp=True, ll_k=0, kl_k=7,
              n_message_gvps=3, n_update_gvps=2, n_noise_gvps=4, graph_cutoffs={"ll": 6, "kl": 6, "kk": 8, "rr": 3.5})
    sd = P.init_state_dict(P.gvp_dynamics_shapes(10, 10, 16, 3, 64, True, 3, 2, 4), seed=12)
    for k in sd:
        if k.endswith(".Wh") or k.endswith(".Wu"):
            sd[k] = sd[k] * 2.0
    pockets = [synthetic.ca_pocket(i, 42, 10, 16, 3.5) for i in range(2)]
    for pk in pockets:
        pk.kp_v = 0.1 * torch.randn(pk.n_kp, 16, 3, generator=torch.Generator().manual_seed(5))
    inputs = _inputs(pockets, [20, 1, 44, 9], 10, seed=4, with_v=True)
    assert inputs["kk_src"].numel() < 8
    (eh, ex, _, _), = _run_both("gvp", sd, kw, 10, 10, inputs, mode=mode)
    print(f"gvp ca-like norm={norm} [{mode}]: rel_err {eh:.2e} {ex:.2e}")
    assert eh < TOL_BY_MODE[mode] and ex < TOL_BY_MODE[mode]


@pytest.mark.parametrize("mode", MODES + ["bf16"])
@pytest.mark.parametrize("message_norm", [0.0, 3.0])
def test_egnn_intended_normalisation_flag(message_norm, mode):
    """z_effective=True divides h_neigh / x_neigh by z (what the reference's comments intend, DESIGN N11)."""
    from oracle import params as P
    from keypoint_diffusion_b200 import synthetic
    kw = dict(n_layers=3, hidden_nf=48, use_tanh=True, message_norm=message_norm, update_kp_feat=True, norm=True,
              ll_k=0, kl_k=5, graph_cutoffs={"ll": 5, "kl": 8, "kk": 8})
    sd = P.init_state_dict(P.egnn_dynamics_shapes(10, 24, 3, 48, True, True), seed=13, coord_gain=0.3)
    pockets = [synthetic.keypoint_pocket(i, 20, 24, 0, 8.0) for i in range(3)]
    inputs = _inputs(pockets, [20, 8, 35], 10, seed=6, with_v=False)
    tol = TOL_BY_MODE[mode]
    res = _run_both("egnn", sd, kw, 10, 24, inputs, z_effective=True, per_complex_t=True, mode=mode)
    for eh, ex, _, _ in res:
        print(f"egnn z_effective message_norm={message_norm} [{mode}] per-complex t: rel_err {eh:.2e} {ex:.2e}")
        assert eh < tol and ex < tol
    # and the flag matters: the default (as-executed) result differs
    res0 = _run_both("egnn", sd, kw, 10, 24, inputs, z_effective=False, mode=mode)
    assert res0[0][0] < tol


def _module_case(arch):
    import yaml
    from helpers import GOLDEN
    from keypoint_diffusion_b200 import HeteroBatch, model_from_config, synthetic
    import os
    from pathlib import Path
    os.chdir(Path(__file__).resolve().parents[1])
    cfg = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))[f"{arch}_20kp"]
    torch.manual_seed(3)
    model = model_from_config(cfg).to(_dev()).eval()
    vs = cfg["dynamics_gvp"]["vector_size"] if arch == "gvp" else 0
    pockets = [synthetic.keypoint_pocket(i, 20, 128, vs, 8.0) for i in range(2)]
    g = HeteroBatch.from_pockets(pockets, [12, 20, 7], 10)
    x_l, h_l = synthetic.ligand_noise_state([12, 20, 7], 10, seed=8)
    g.nodes["lig"].data["x_0"], g.nodes["lig"].data["h_0"] = x_l, h_l
    return cfg, model, g


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_module_api_contract(arch):
    """dynamics(g, t, batch_idxs) through the drop-in module: matches the oracle on the module's own
    state_dict, leaves g unchanged; sample_p_zs_given_zt mutates g in place like the reference."""
    from oracle import flat, schedule as OS
    from keypoint_diffusion_b200.utils import get_batch_idxs
    cfg, model, g_cpu = _module_case(arch)
    dev = _dev()
    g = g_cpu.to(dev)
    before = {nt: {k: v.clone() for k, v in g.nodes[nt].data.items()} for nt in ("lig", "kp")}
    t = torch.full((3,), 0.4, device=dev)
    eps_h, eps_x = model.dynamics(g, t, get_batch_idxs(g))
    torch.cuda.synchronize()
    for nt in before:
        for k, v in before[nt].items():
            assert torch.equal(g.nodes[nt].data[k], v), "dynamics.forward must leave g unchanged"
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    d = cfg["dynamics"] if arch == "egnn" else cfg["dynamics_gvp"]
    kw = {k: v for k, v in d.items()}
    kw["graph_cutoffs"] = cfg["graph"]["graph_cutoffs"]
    ocfg = oracle_cfg(arch, kw, 10, 128)
    inputs = {"lig_n": g_cpu.batch_num_nodes("lig"), "kp_n": g_cpu.batch_num_nodes("kp"),
              "lig_x": g_cpu.nodes["lig"].data["x_0"], "lig_h": g_cpu.nodes["lig"].data["h_0"],
              "kp_x": g_cpu.nodes["kp"].data["x_0"], "kp_h": g_cpu.nodes["kp"].data["h_0"],
              "kk_src": g_cpu.edges(form="uv", etype="kk")[0], "kk_dst": g_cpu.edges(form="uv", etype="kk")[1]}
    if arch == "gvp":
        inputs["kp_v"] = g_cpu.nodes["kp"].data["v_0"]
    fb = flat_batch(inputs)
    ref_h, ref_x = oracle_forward(arch, sd, ocfg, fb, torch.full((3,), 0.4))
    assert rel_err(eps_h.cpu(), ref_h) < TOL
    # eps_x of the EGNN is ~1e-3 with the reference's gain=0.001 coordinate init: compare on the scale of x
    assert float((eps_x.cpu() - ref_x).abs().max()) < TOL * max(float(ref_x.abs().max()), 1.0)
    # one reverse step with injected noise, in place
    T = model.n_timesteps
    gen = torch.Generator().manual_seed(0)
    nx, nh = torch.randn(39, 3, generator=gen), torch.randn(39, 10, generator=gen)
    s_int = 700
    fwd = flat.egnn_forward if arch == "egnn" else flat.gvp_forward
    fb = flat_batch(inputs)
    fb = flat.sample_p_zs_given_zt(lambda b, tt: fwd(sd, ocfg, b, tt), OS.gamma_table(T, 1e-5), T, s_int, fb, nx, nh)
    s = torch.full((3,), s_int / T, device=dev)
    tt = torch.full((3,), (s_int + 1) / T, device=dev)
    g2 = model.sample_p_zs_given_zt(s, tt, g, get_batch_idxs(g), noise=(nx.to(dev), nh.to(dev)))
    torch.cuda.synchronize()
    assert g2 is g
    assert rel_err(g.nodes["lig"].data["x_0"].cpu(), fb.lig_x) < TOL
    assert rel_err(g.nodes["lig"].data["h_0"].cpu(), fb.lig_h) < TOL
    assert rel_err(g.nodes["kp"].data["x_0"].cpu(), fb.kp_x) < TOL


def test_sample_from_encoded_receptors_api():
    """Host graph in, per-ligand CPU tensors out; seeded Philox sampling is reproducible and finite;
    _sample regroups per receptor; init_lig_pos is required without rec nodes (SURVEY N7)."""
    cfg, model, g_cpu = _module_case("gvp")
    model.n_timesteps = 1000
    init = torch.zeros(3, 3)
    pos, feat = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init, seed=5, steps_per_graph=25)
    assert [p.shape for p in pos] == [(12, 3), (20, 3), (7, 3)] and [f.shape for f in feat] == [(12, 10), (20, 10), (7, 10)]
    assert all(p.device.type == "cpu" and torch.isfinite(p).all() for p in pos)
    pos2, feat2 = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init, seed=5, steps_per_graph=25)
    assert all(torch.equal(a, b) for a, b in zip(pos, pos2)) and all(torch.equal(a, b) for a, b in zip(feat, feat2))
    pos3, _ = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init, seed=6, steps_per_graph=25)
    assert not torch.equal(pos[0], pos3[0])
    # the batch sampled as concurrent sub-batches (own CUDA graphs / streams): the noise is keyed by the global atom
    # index, so each complex follows the same trajectory; only the tile boundaries of the reductions move
    pos4, feat4 = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init, seed=5, steps_per_graph=25, sub_batches=3)
    pos5, feat5 = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init, seed=5, steps_per_graph=25, sub_batches=2)
    assert [p.shape for p in pos4] == [p.shape for p in pos]
    for a, b, c in zip(pos, pos4, pos5):
        assert torch.isfinite(b).all() and torch.isfinite(c).all()
    with pytest.raises(ValueError):
        model.sample_from_encoded_receptors(g_cpu, init_lig_pos=None)
    with pytest.raises(AssertionError):
        model.sample_from_encoded_receptors(g_cpu, init_lig_pos=torch.zeros(2, 3))
    from keypoint_diffusion_b200 import hetero
    singles = hetero.unbatch(g_cpu)[:2]
    samples = model._sample(singles, [[10, 11, 12], [8]], diff_batch_size=3, encoded=True,
                            init_lig_pos=[torch.zeros(3), torch.ones(3)])
    assert [len(s["positions"]) for s in samples] == [3, 1]
    assert [p.shape[0] for p in samples[0]["positions"]] == [10, 11, 12] and samples[1]["features"][0].shape == (8, 10)


def test_fixed_encoder_path():
    """rec_encoder_type='fixed' (all-atom / C-alpha models): keypoints := receptor atoms, kk := rr."""
    import yaml
    import os
    from pathlib import Path
    from helpers import GOLDEN
    from keypoint_diffusion_b200 import HeteroBatch, model_from_config, synthetic
    os.chdir(Path(__file__).resolve().parents[1])
    cfg = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))["egnn_all_atom"]
    torch.manual_seed(1)
    model = model_from_config(cfg).to(_dev()).eval()
    pk = synthetic.all_atom_pocket(0, 120, 10, 0, 3.5)
    B = 2
    g = HeteroBatch({"kp": torch.zeros(B, dtype=torch.long), "lig": torch.tensor([9, 14]), "rec": torch.tensor([120] * B)},
                    {"rec": {"x_0": pk.kp_x.repeat(B, 1), "h_0": pk.kp_h.repeat(B, 1)},
                     "lig": {"x_0": torch.zeros(23, 3), "h_0": torch.zeros(23, 10)},
                     "kp": {"x_0": torch.zeros(0, 3), "h_0": torch.zeros(0, 10)}},
                    {("rec", "rr", "rec"): (torch.cat([pk.kk_src, pk.kk_src + 120]), torch.cat([pk.kk_dst, pk.kk_dst + 120]))},
                    {("rec", "rr", "rec"): torch.tensor([pk.kk_src.numel()] * B)})
    enc = model.encode_receptors(g)
    assert enc.num_nodes("kp") == 240 and enc.num_nodes("rec") == 0 and enc.num_edges("kk") == 2 * pk.kk_src.numel()
    model.n_timesteps = 1000
    pos, feat = model.sample_from_encoded_receptors(enc, init_lig_pos=torch.zeros(B, 3), seed=2)
    assert [p.shape for p in pos] == [(9, 3), (14, 3)] and all(torch.isfinite(p).all() for p in pos)


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_raw_pocket_to_ligands_with_learned_encoder(arch):
    """SURVEY 8f rows 1-3: raw pocket atoms -> build_initial_complex_graph -> learned receptor encoder -> sampler, through
    sample_given_pocket / _sample as a user of the reference calls them (no init_lig_pos: the pocket centroid is used)."""
    import yaml
    import os
    from pathlib import Path
    from helpers import GOLDEN
    from keypoint_diffusion_b200 import hetero, model_from_config, synthetic
    os.chdir(Path(__file__).resolve().parents[1])
    cfg = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))[f"{arch}_20kp"]
    torch.manual_seed(4)
    model = model_from_config(cfg).to(_dev()).eval()
    cut = cfg["graph"]["graph_cutoffs"]
    raws = []
    for i, n in enumerate((150, 211)):
        x, h, res = synthetic.raw_pocket(i, n, 10)
        raws.append(hetero.build_initial_complex_graph(x, h, res, cfg["graph"]["n_keypoints"], cut))
    with torch.no_grad():
        enc = model.encode_receptors(hetero.batch(raws).to(_dev()))
        one = model.encode_receptors(raws[1].to(_dev()))
    assert enc.num_nodes("kp") == 40 and enc.nodes["kp"].data["h_0"].shape == (40, 128)
    assert torch.isfinite(enc.nodes["kp"].data["x_0"]).all() and torch.isfinite(enc.nodes["kp"].data["h_0"]).all()
    if arch == "gvp":
        assert enc.nodes["kp"].data["v_0"].shape == (40, 16, 3)
    # encoding the pockets one at a time gives the same keypoints as encoding the batch
    assert rel_err(one.nodes["kp"].data["x_0"].cpu(), enc.nodes["kp"].data["x_0"][20:].cpu()) < 1e-4
    assert rel_err(one.nodes["kp"].data["h_0"].cpu(), enc.nodes["kp"].data["h_0"][20:].cpu()) < 1e-4
    torch.manual_seed(11)
    samples = model._sample(raws, [[9, 14], [12]], rec_enc_batch_size=1, diff_batch_size=2)
    assert [len(s["positions"]) for s in samples] == [2, 1]
    assert [p.shape for p in samples[0]["positions"]] == [(9, 3), (14, 3)] and samples[1]["features"][0].shape == (12, 10)
    assert all(torch.isfinite(p).all() for s in samples for p in s["positions"])
    pos, feat = model.sample_given_pocket(raws[0], torch.tensor([7, 8]))
    assert [p.shape for p in pos] == [(7, 3), (8, 3)] and [f.shape for f in feat] == [(7, 10), (8, 10)]


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_sub_batch_sampling_draws_the_same_noise(arch):
    """A batch cut into concurrently sampled groups (KeypointDiffusion._sub_samplers: own CUDA graph and stream per
    group, Philox counter offset by the group's first atom) follows the trajectory of the undivided batch."""
    cfg, model, g_cpu = _module_case(arch)
    dev = _dev()
    g = g_cpu.to(dev)
    kp = g.nodes["kp"].data
    kx, kh, kv = kp["x_0"].float().contiguous(), kp["h_0"].float().contiguous(), kp.get("v_0")
    init = torch.tensor([[0.5, 0.0, -1.0], [0.0, 2.0, 0.0], [1.0, 1.0, 1.0]], device=dev)
    whole = model._sampler(g, 5, True)
    xw, hw, kw_ = whole.run(kx, kh, kv, init, seed=9, n_steps=10)
    torch.cuda.synchronize()
    subs = model._sub_samplers(g, 3, 5, True)
    assert len(subs) == 3
    for smp, (a, b), (k0, k1), (l0, l1), st in subs:
        with torch.cuda.stream(st):
            xs, hs, ks = smp.run(kx[k0:k1], kh[k0:k1], kv[k0:k1] if kv is not None else None, init[a:b], seed=9, n_steps=10)
        st.synchronize()
        ex, eh = rel_err(xs.cpu(), xw[l0:l1].cpu()), rel_err(hs.cpu(), hw[l0:l1].cpu())
        ek = rel_err(ks.cpu(), kw_[k0:k1].cpu())
        assert ex < 1e-5 and eh < 1e-5 and ek < 1e-5, (a, b, ex, eh, ek)
    # and through the public call: same shapes, finite, reproducible
    p1, f1 = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init.cpu(), seed=3, steps_per_graph=50, sub_batches=2)
    p2, f2 = model.sample_from_encoded_receptors(g_cpu, init_lig_pos=init.cpu(), seed=3, steps_per_graph=50, sub_batches=2)
    assert all(torch.equal(a, b) for a, b in zip(p1, p2)) and all(torch.equal(a, b) for a, b in zip(f1, f2))
    assert [p.shape[0] for p in p1] == [12, 20, 7] and all(torch.isfinite(p).all() for p in p1)


def test_captured_loop_graph_convs_match_serial_convs(monkeypatch):
    """The captured reverse-diffusion loop (CUDA graph replay) with the GVP convs as a multi-stream dependency graph
    against the same loop with serial convs (KPD_GVP_SERIAL=1 at model creation): identical state after 10 steps."""
    dev = _dev()
    init = torch.tensor([[0.5, 0.0, -1.0], [0.0, 2.0, 0.0], [1.0, 1.0, 1.0]], device=dev)
    outs = []
    for serial in ("0", "1"):
        monkeypatch.setenv("KPD_GVP_SERIAL", serial)
        cfg, model, g_cpu = _module_case("gvp")
        g = g_cpu.to(dev)
        kp = g.nodes["kp"].data
        smp = model._sampler(g, 5, True)
        x, h, k = smp.run(kp["x_0"].float().contiguous(), kp["h_0"].float().contiguous(), kp["v_0"].float().contiguous(),
                          init, seed=11, n_steps=10)
        torch.cuda.synchronize()
        outs.append((x.clone(), h.clone(), k.clone(), smp.launches_per_step))
    assert outs[0][3] > outs[1][3], "the dependency-graph path launches one kernel per edge / node type"
    for a, b in zip(outs[0][:3], outs[1][:3]):
        assert torch.isfinite(a).all() and torch.equal(a, b)
