"""GPU parity tests: the CUDA path (through the C ABI, keypoint_diffusion_b200.ops) against
the golden fixtures (outputs of the reference's own forward code) and the CPU oracle.

Tolerances
  * graph edge sets: exact;
  * denoiser outputs (fp32 mode): max|a-b| / max|b| <= 1e-4  (north_star's per-step bar);
  * one posterior step with injected noise: <= 1e-6 (op-by-op identical arithmetic).
"""
import json

import pytest
import torch

from helpers import (DENOISER_FIXTURES, GOLDEN, edge_set, flat_batch, load_golden, oracle_cfg, oracle_forward,
                     rel_err)

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _dev():
    return torch.device("cuda:0")


def _ops():
    from keypoint_diffusion_b200 import ops
    return ops


def _strip(sd, prefix="dynamics."):
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


def build_model(kind, sd, kw, atom_nf, rec_nf, dev):
    ops = _ops()
    sd = _strip(sd)
    if kind == "egnn":
        return ops.EgnnModel(sd, atom_nf=atom_nf, rec_nf=rec_nf, hidden_nf=kw.get("hidden_nf", 255),
                             n_layers=kw.get("n_layers", 4), use_tanh=kw.get("use_tanh", False),
                             update_kp_feat=kw.get("update_kp_feat", False), norm=kw.get("norm", False),
                             message_norm=kw.get("message_norm", 1), device=dev)
    return ops.GvpModel(sd, n_lig_scalars=atom_nf, n_kp_scalars=rec_nf, vector_size=kw.get("vector_size", 16),
                        n_convs=kw.get("n_convs", 4), n_hidden_scalars=kw.get("n_hidden_scalars", 128),
                        update_kp=kw.get("update_kp", False), n_message_gvps=kw.get("n_message_gvps", 3),
                        n_update_gvps=kw.get("n_update_gvps", 2), n_noise_gvps=kw.get("n_noise_gvps", 3),
                        message_norm=kw.get("message_norm", 1), rbf_dim=kw.get("rbf_dim", 16), device=dev)


def device_inputs(inputs, dev):
    ops = _ops()
    batch = ops.DeviceBatch(inputs["lig_n"].tolist(), inputs["kp_n"].tolist(), dev)
    kk = ops.Csr.from_edges(inputs["kk_src"], inputs["kk_dst"], batch.n_kp, dev)
    t = {k: v.to(dev).float().contiguous() for k, v in inputs.items() if k in ("lig_x", "lig_h", "kp_x", "kp_h", "kp_v")}
    return batch, kk, t


def run_forward(kind, model, batch, graphs, kk, t_in, tval, dev):
    t = torch.full((1,), float(tval), device=dev)
    has_lk = graphs.lk is not None
    if kind == "egnn":
        return model.forward(batch, graphs, kk if has_lk else None, t_in["lig_h"], t_in["lig_x"], t_in["kp_h"],
                             t_in["kp_x"], t)
    return model.forward(batch, graphs, kk if has_lk else None, t_in["lig_h"], t_in["lig_x"], t_in["kp_h"],
                         t_in["kp_x"], t_in["kp_v"], t)


def test_library_loaded_and_device():
    from keypoint_diffusion_b200 import _lib
    assert _lib.lib.kpd_version() >= 100
    cc = torch.cuda.get_device_capability(0)
    assert cc[0] >= 10, f"expected a Blackwell GPU, got sm_{cc[0]}{cc[1]}"


def test_linear_matches_torch():
    ops = _ops()
    dev = _dev()
    g = torch.Generator().manual_seed(0)
    for (M, K, N, act) in [(70, 33, 132, 1), (257, 257, 2080, 0), (5, 10, 64, 1), (1000, 514, 260, 1)]:
        x = torch.randn(M, K, generator=g)
        w = torch.randn(N, K, generator=g) / K ** 0.5
        b = torch.randn(N, generator=g)
        r = torch.randn(M, N, generator=g)
        ref = x.double() @ w.double().t() + b.double()
        if act:
            ref = torch.nn.functional.silu(ref)
        ref = ref + r.double()
        Np = (N + 3) // 4 * 4
        wt = torch.zeros(K, Np)
        wt[:, :N] = w.t()
        y = ops.linear(x.to(dev), wt.to(dev), b.to(dev), r.to(dev), act, n_out=N)
        assert rel_err(y.cpu(), ref) < 2e-6, (M, K, N)


@pytest.mark.parametrize("name", DENOISER_FIXTURES)
def test_graph_build_exact(name):
    """ll / kl / lk edge sets are bit-exact against what the reference code built."""
    ops = _ops()
    dev = _dev()
    fx = load_golden(name)
    kw = fx["kwargs"]
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    with_lk = bool(kw.get("update_kp_feat", kw.get("update_kp", False)))
    graphs = ops.LigandGraphs(batch, gp, with_lk).build(t_in["lig_x"], t_in["kp_x"])
    torch.cuda.synchronize()
    got = {"ll": graphs.ll.edges(), "kl": graphs.kl.edges()}
    if with_lk:
        got["lk"] = graphs.lk.edges()
    for et, ei in fx["edges"].items():
        if et not in got:
            assert ei.shape[1] == 0
            continue
        assert edge_set(got[et]) == edge_set(ei), et
        # CSR invariants: dst sorted, rowptr consistent
        d = got[et][1]
        assert torch.all(d[1:] >= d[:-1])
    csr = graphs.ll
    rp = csr.rowptr.cpu().long()
    assert torch.equal(torch.bincount(got["ll"][1], minlength=batch.n_lig), rp[1:] - rp[:-1])
    # per-complex counts (utils.get_edges_per_batch)
    lb = batch.lig_batch.cpu().long()
    assert torch.equal(graphs.counts_ll.cpu().long(), torch.bincount(lb[got["ll"][1]], minlength=batch.B))
    assert torch.equal(graphs.counts_kl.cpu().long(), torch.bincount(lb[got["kl"][1]], minlength=batch.B))


@pytest.mark.parametrize("name", DENOISER_FIXTURES)
def test_denoiser_matches_golden(name):
    """eps_h / eps_x against the outputs of the reference's own forward code (small models)."""
    ops = _ops()
    dev = _dev()
    fx = load_golden(name)
    kw = fx["kwargs"]
    model = build_model(fx["kind"], fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    with_lk = bool(kw.get("update_kp_feat", kw.get("update_kp", False)))
    graphs = ops.LigandGraphs(batch, gp, with_lk).build(t_in["lig_x"], t_in["kp_x"])
    for t_str, out in fx["outputs"].items():
        eps_h, eps_x = run_forward(fx["kind"], model, batch, graphs, kk, t_in, float(t_str), dev)
        torch.cuda.synchronize()
        eh, ex = rel_err(eps_h.cpu(), out["eps_h"]), rel_err(eps_x.cpu(), out["eps_x"])
        print(f"{name} t={t_str}: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
        assert eh < TOL and ex < TOL, (name, t_str, eh, ex)


def _full_size_case(arch, cfgs, n_lig=None, n_pockets=3, rbf_dim=16):
    """Shipped hyper-parameters (20-keypoint models), seeded weights, 6 complexes of mixed size.  rbf_dim: width of the
    GVP model's edge-distance RBF embedding (16 as shipped)."""
    from oracle import params as P
    from keypoint_diffusion_b200 import synthetic
    cfg = cfgs[f"{arch}_20kp"]
    n_lig = n_lig or [20, 8, 35, 20, 13, 27]
    if arch == "egnn":
        d = cfg["dynamics"]
        rec_nf = cfg["rec_encoder"]["out_n_node_feat"]
        shapes = P.egnn_dynamics_shapes(10, rec_nf, d["n_layers"], d["hidden_nf"], d["update_kp_feat"], d["norm"])
        sd = P.init_state_dict(shapes, seed=3, coord_gain=0.3)
        kw = dict(n_layers=d["n_layers"], hidden_nf=d["hidden_nf"], use_tanh=d["use_tanh"],
                  message_norm=d["message_norm"], update_kp_feat=d["update_kp_feat"], norm=d["norm"],
                  ll_k=d["ll_k"], kl_k=d["kl_k"], graph_cutoffs=cfg["graph"]["graph_cutoffs"])
        vs = 0
    else:
        d = cfg["dynamics_gvp"]
        rec_nf = cfg["rec_encoder_gvp"]["out_scalar_size"]
        shapes = P.gvp_dynamics_shapes(10, rec_nf, d["vector_size"], d["n_convs"], d["n_hidden_scalars"], d["update_kp"],
                                       d["n_message_gvps"], d["n_update_gvps"], d["n_noise_gvps"], rbf_dim=rbf_dim)
        sd = P.init_state_dict(shapes, seed=4)
        for k in sd:
            if k.endswith(".Wh") or k.endswith(".Wu"):
                sd[k] = sd[k] * 2.0
        kw = dict(vector_size=d["vector_size"], n_convs=d["n_convs"], n_hidden_scalars=d["n_hidden_scalars"],
                  message_norm=d["message_norm"], update_kp=d["update_kp"], ll_k=d["ll_k"], kl_k=d["kl_k"],
                  n_message_gvps=d["n_message_gvps"], n_update_gvps=d["n_update_gvps"],
                  n_noise_gvps=d["n_noise_gvps"], graph_cutoffs=cfg["graph"]["graph_cutoffs"], rbf_dim=rbf_dim)
        vs = d["vector_size"]
    pockets = [synthetic.keypoint_pocket(i, 20, rec_nf, vs, cfg["graph"]["graph_cutoffs"]["kk"]) for i in range(n_pockets)]
    x_l, h_l = synthetic.ligand_noise_state(n_lig, 10, seed=5)
    kp_x, kp_h, kp_v, ks, kd, off = [], [], [], [], [], 0
    for i in range(len(n_lig)):
        pk = pockets[i % n_pockets]
        kp_x.append(pk.kp_x); kp_h.append(pk.kp_h)
        if vs:
            kp_v.append(pk.kp_v)
        ks.append(pk.kk_src + off); kd.append(pk.kk_dst + off)
        off += pk.n_kp
    inputs = {"lig_n": torch.tensor(n_lig), "kp_n": torch.tensor([20] * len(n_lig)), "lig_x": x_l, "lig_h": h_l,
              "kp_x": torch.cat(kp_x), "kp_h": torch.cat(kp_h), "kk_src": torch.cat(ks), "kk_dst": torch.cat(kd)}
    if vs:
        inputs["kp_v"] = torch.cat(kp_v)
    return sd, kw, rec_nf, inputs


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
def test_denoiser_full_size_vs_oracle(arch):
    """Shipped-size model (H=257 / S=256,V=16, 6 layers): CUDA vs the CPU oracle, same seeded
    weights and inputs, teacher-forced at several t."""
    import yaml
    ops = _ops()
    dev = _dev()
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    sd, kw, rec_nf, inputs = _full_size_case(arch, cfgs)
    cfg = oracle_cfg(arch, kw, 10, rec_nf)
    model = build_model(arch, sd, kw, 10, rec_nf, dev)
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
    for tval in (0.001, 0.5, 1.0):
        fb = flat_batch(inputs)
        t = torch.full((fb.B,), tval)
        ref_h, ref_x, edges, _ = oracle_forward(arch, sd, cfg, fb, t, return_edges=True)
        eps_h, eps_x = run_forward(arch, model, batch, graphs, kk, t_in, tval, dev)
        torch.cuda.synchronize()
        assert edge_set(graphs.ll.edges()) == edge_set(torch.stack(edges["ll"]))
        assert edge_set(graphs.kl.edges()) == edge_set(torch.stack(edges["kl"]))
        assert edge_set(graphs.lk.edges()) == edge_set(torch.stack(edges["lk"]))
        eh, ex = rel_err(eps_h.cpu(), ref_h), rel_err(eps_x.cpu(), ref_x)
        print(f"{arch} full size t={tval}: rel_err eps_h={eh:.2e} eps_x={ex:.2e} "
              f"|eps_h|={float(ref_h.abs().max()):.3f} |eps_x|={float(ref_x.abs().max()):.3f}")
        assert eh < TOL and ex < TOL


def test_ddpm_step_matches_oracle():
    from oracle import flat, schedule as S
    ops = _ops()
    dev = _dev()
    T = 1000
    gamma = S.gamma_table(T, 1e-5)
    coef = S.coefficient_table(gamma, T).to(dev).contiguous()
    lig_n, kp_n = [5, 20, 1, 33], [4, 20, 7, 2]
    g = torch.Generator().manual_seed(1)
    N_l, N_k, F = sum(lig_n), sum(kp_n), 10
    x, h, xk = torch.randn(N_l, 3, generator=g), torch.randn(N_l, F, generator=g), torch.randn(N_k, 3, generator=g) * 5
    ex, eh = torch.randn(N_l, 3, generator=g), torch.randn(N_l, F, generator=g)
    nx, nh = torch.randn(N_l, 3, generator=g), torch.randn(N_l, F, generator=g)
    batch = ops.DeviceBatch(lig_n, kp_n, dev)
    for s_int in (999, 500, 0):
        fb = flat.FlatBatch(lig_n=torch.tensor(lig_n), kp_n=torch.tensor(kp_n), kp_x=xk.clone(), kp_h=torch.zeros(N_k, 1),
                            kk_src=torch.zeros(0, dtype=torch.long), kk_dst=torch.zeros(0, dtype=torch.long),
                            lig_x=x.clone(), lig_h=h.clone())
        fb = flat.sample_p_zs_given_zt(lambda b, t: (eh, ex), gamma, T, s_int, fb, nx, nh)
        dx, dh, dk = x.to(dev).clone(), h.to(dev).clone(), xk.to(dev).clone()
        step = torch.tensor([s_int], dtype=torch.int32, device=dev)
        ops.ddpm_step(batch, dx, dh, dk, ex.to(dev), eh.to(dev), coef, step, nx.to(dev), nh.to(dev))
        torch.cuda.synchronize()
        assert rel_err(dx.cpu(), fb.lig_x) < 1e-6
        assert rel_err(dh.cpu(), fb.lig_h) < 1e-6
        assert rel_err(dk.cpu(), fb.kp_x) < 1e-6


def test_philox_noise_is_standard_normal():
    ops = _ops()
    dev = _dev()
    from keypoint_diffusion_b200._lib import lib, ptr, check
    import ctypes as C
    n, F = 200000, 10
    x = torch.empty(n, 3, device=dev)
    h = torch.empty(n, F, device=dev)
    check(lib.kpd_randn_init(ptr(x), ptr(h), n, F, 1234, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    z = torch.cat([x.reshape(-1), h.reshape(-1)]).cpu().double()
    assert abs(float(z.mean())) < 5e-3 and abs(float(z.std()) - 1.0) < 5e-3
    assert abs(float((z ** 4).mean()) - 3.0) < 0.05
    c = torch.corrcoef(torch.stack([x[:, 0], x[:, 1], h[:, 0], h[:, 9]]).cpu().double())
    assert float((c - torch.eye(4)).abs().max()) < 0.01
    x2 = torch.empty_like(x); h2 = torch.empty_like(h)
    check(lib.kpd_randn_init(ptr(x2), ptr(h2), n, F, 1234, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(x, x2) and torch.equal(h, h2)        # counter-based: reproducible


@pytest.mark.parametrize("arch", ["egnn", "gvp"])
@pytest.mark.parametrize("use_graph", [False, True])
def test_full_loop_matches_reference(arch, use_graph):
    """The whole reverse-diffusion loop (frame setup, T steps, frame restore) with injected noise
    against KeypointDiffusion.sample_from_encoded_receptors run by the reference code."""
    from oracle import schedule as S
    ops = _ops()
    dev = _dev()
    fx = load_golden(f"loop_{arch}")
    kw, T, F = fx["kwargs"], fx["T"], fx["atom_nf"]
    model = build_model(arch, fx["state_dict"], kw, F, fx["rec_nf"], dev)
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    coef = S.coefficient_table(fx["state_dict"]["gamma.gamma"], T).to(dev).contiguous()
    # the reference draws x then h from the global generator at init and at every step
    torch.manual_seed(fx["noise_seed"])
    N_l = batch.n_lig
    slots = []
    for _ in range(T + 1):
        nx = torch.randn(N_l, 3)
        nh = torch.randn(N_l, F)
        slots.append(torch.cat([nx.reshape(-1), nh.reshape(-1)]))
    noise = torch.stack(slots).to(dev).contiguous()
    sampler = ops.Sampler(model, batch, gp, kk, coef, T, F, steps_per_graph=4, use_cuda_graph=use_graph)
    x_lig, h_lig, _ = sampler.run(t_in["kp_x"], t_in["kp_h"], t_in.get("kp_v"), fx["init_lig_pos"].to(dev), noise=noise)
    torch.cuda.synchronize()
    pos = torch.cat(fx["positions"])
    feat = torch.cat(fx["features"])
    ex, eh = rel_err(x_lig.cpu(), pos), rel_err(h_lig.cpu(), feat)
    print(f"loop {arch} graph={use_graph}: rel_err pos={ex:.2e} feat={eh:.2e} launches/step={sampler.launches_per_step}")
    assert ex < 1e-3 and eh < 1e-3
