"""GPU: the tcgen05 building block (bf16 operands, fp32 accumulation in TMEM) against torch."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("M,K,N,act", [(128, 16, 16, 0), (128, 64, 256, 0), (300, 272, 256, 1), (77, 289, 256, 1),
                                       (2000, 257, 64, 0), (129, 129, 240, 1), (300, 257, 514, 1), (200, 64, 2056, 0)])
def test_tc_linear_matches_bf16_reference(M, K, N, act):
    from keypoint_diffusion_b200 import ops, pack
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    r = torch.randn(M, N, generator=g)
    # reference on the bf16-rounded operands, accumulated in fp64
    xr, wr = x.to(torch.bfloat16).double(), w.to(torch.bfloat16).double()
    ref = xr @ wr.t() + b.double()
    if act:
        ref = torch.nn.functional.silu(ref)
    ref = ref + r.double()
    y = ops.tc_linear(x.to(dev), pack.pack_tc_weight(w).to(dev), N, b.to(dev), r.to(dev), act)
    torch.cuda.synchronize()
    err = rel_err(y.cpu(), ref)
    print(f"tc_linear M={M} K={K} N={N}: rel_err vs bf16-operand reference {err:.2e}; "
          f"vs fp32 {rel_err(y.cpu(), (x.double() @ w.double().t() + b.double()) if not act else ref):.2e}")
    assert err < 2e-5


@pytest.mark.parametrize("M,K,N,act", [(128, 16, 16, 0), (64, 64, 256, 0), (300, 272, 256, 1), (77, 257, 257, 1),
                                       (2000, 257, 64, 0), (129, 514, 257, 1), (200, 257, 2080, 0)])
def test_tc_linear_bf16x3_matches_fp32(M, K, N, act):
    """bf16x3: split (hi, lo) operands, all four products on the tensor cores -> fp32-grade results."""
    from keypoint_diffusion_b200 import ops, pack
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(M + K + N)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    r = torch.randn(M, N, generator=g)
    ref = x.double() @ w.double().t() + b.double()
    if act:
        ref = torch.nn.functional.silu(ref)
    ref = ref + r.double()
    y = ops.tc_linear(x.to(dev), pack.pack_tc_weight(w, split=True).to(dev), N, b.to(dev), r.to(dev), act, nsplit=2)
    torch.cuda.synchronize()
    err = rel_err(y.cpu(), ref)
    print(f"tc_linear bf16x3 M={M} K={K} N={N}: rel_err vs fp64 {err:.2e}")
    assert err < 2e-5


@pytest.mark.parametrize("name", ["gvp_small_sum", "gvp_small_mean", "gvp_small_zero"])
def test_gvp_bf16_mode_small(name):
    """bf16 tensor-core mode of the GVP denoiser vs the golden fp32 outputs of the reference code:
    operands are rounded to bf16 (8-bit mantissa), so the bar is 3e-2 of the output scale, stated
    separately from the 1e-4 fp32 bar."""
    from helpers import load_golden
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    fx = load_golden(name)
    kw = fx["kwargs"]
    model = build_model("gvp", fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
    out = fx["outputs"]["0.5"]
    h32, x32 = run_forward("gvp", model, batch, graphs, kk, t_in, 0.5, dev)
    model.set_precision("bf16")
    h16, x16 = run_forward("gvp", model, batch, graphs, kk, t_in, 0.5, dev)
    torch.cuda.synchronize()
    eh, ex = rel_err(h16.cpu(), out["eps_h"]), rel_err(x16.cpu(), out["eps_x"])
    print(f"{name} bf16 mode: rel_err eps_h={eh:.2e} eps_x={ex:.2e} (fp32 mode {rel_err(h32.cpu(), out['eps_h']):.1e})")
    assert eh < 3e-2 and ex < 3e-2


def test_gvp_bf16_mode_full_size():
    import yaml
    from helpers import GOLDEN, flat_batch, oracle_cfg, oracle_forward
    from test_gpu_parity import _full_size_case, build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    sd, kw, rec_nf, inputs = _full_size_case("gvp", cfgs)
    cfg = oracle_cfg("gvp", kw, 10, rec_nf)
    model = build_model("gvp", sd, kw, 10, rec_nf, dev)
    model.set_precision("bf16")
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
    fb = flat_batch(inputs)
    ref_h, ref_x = oracle_forward("gvp", sd, cfg, fb, torch.full((fb.B,), 0.5))
    eps_h, eps_x = run_forward("gvp", model, batch, graphs, kk, t_in, 0.5, dev)
    torch.cuda.synchronize()
    eh, ex = rel_err(eps_h.cpu(), ref_h), rel_err(eps_x.cpu(), ref_x)
    print(f"gvp full size bf16 mode: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
    assert eh < 3e-2 and ex < 3e-2


# ---------------------------------------------------------------------------------------------
# bf16x3: split (hi, lo) bf16 operands, three MMAs per product, fp32 accumulation -- the tensor-core
# parity mode.  Bar = the north star's 1e-4 (relative to the output scale), same as the fp32 SIMT mode.
TOL_X3 = 1e-4


@pytest.mark.parametrize("name", ["gvp_small_sum", "gvp_small_mean", "gvp_small_zero"])
def test_gvp_bf16x3_mode_small(name):
    from helpers import load_golden
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    fx = load_golden(name)
    kw = fx["kwargs"]
    model = build_model("gvp", fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    if model.tc_blob2 is None:
        pytest.skip("n_hidden_scalars not a multiple of 16: no tensor-core mode for this fixture")
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
    model.set_precision("bf16x3")
    for tkey, out in fx["outputs"].items():
        h, x = run_forward("gvp", model, batch, graphs, kk, t_in, float(tkey), dev)
        torch.cuda.synchronize()
        eh, ex = rel_err(h.cpu(), out["eps_h"]), rel_err(x.cpu(), out["eps_x"])
        print(f"{name} bf16x3 t={tkey}: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
        assert eh < TOL_X3 and ex < TOL_X3


def test_gvp_bf16x3_mode_full_size():
    """Shipped-size GVP model (S = 256, V = 16) in the bf16x3 mode against the oracle, for both edge kernels the mode
    selects from.  A message GVP's first input row is S + rbf_dim + V + 1 columns wide: at rbf_dim = 16 that is
    289 -> 38 k-chunks, and the KS edge tile needs 232,176 B, inside the 232,448 B (227 KB) a block may have, so the
    KS kernel runs.  At rbf_dim = 32, 305 columns -> 40 k-chunks, the KS tile would need 240,368 B > 232,448 B: this
    case runs the stacked (STACK) bf16x3 edge kernel."""
    import yaml
    from helpers import GOLDEN, flat_batch, oracle_cfg, oracle_forward
    from test_gpu_parity import _full_size_case, build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    for rbf_dim in (16, 32):
        sd, kw, rec_nf, inputs = _full_size_case("gvp", cfgs, rbf_dim=rbf_dim)
        cfg = oracle_cfg("gvp", kw, 10, rec_nf)
        model = build_model("gvp", sd, kw, 10, rec_nf, dev)
        model.set_precision("bf16x3")
        batch, kk, t_in = device_inputs(inputs, dev)
        gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
        graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
        for tval in (0.001, 0.5, 1.0):
            fb = flat_batch(inputs)
            ref_h, ref_x = oracle_forward("gvp", sd, cfg, fb, torch.full((fb.B,), tval))
            eps_h, eps_x = run_forward("gvp", model, batch, graphs, kk, t_in, tval, dev)
            torch.cuda.synchronize()
            eh, ex = rel_err(eps_h.cpu(), ref_h), rel_err(eps_x.cpu(), ref_x)
            print(f"gvp full size bf16x3 rbf_dim={rbf_dim} t={tval}: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
            assert eh < TOL_X3 and ex < TOL_X3, (rbf_dim, tval, eh, ex)


@pytest.mark.parametrize("name", ["egnn_small_kp", "egnn_small_nokp"])
def test_egnn_bf16x3_mode_small(name):
    """EGNN on the tensor cores (split bf16 operands) vs the golden fp32 outputs of the reference code."""
    from helpers import load_golden
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    fx = load_golden(name)
    kw = fx["kwargs"]
    model = build_model("egnn", fx["state_dict"], kw, fx["atom_nf"], fx["rec_nf"], dev)
    assert model.tc_blob2 is not None
    batch, kk, t_in = device_inputs(fx["inputs"], dev)
    gp = ops.GraphParams.from_module(kw.get("ll_k", 0), kw.get("kl_k", 0), kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, bool(kw.get("update_kp_feat", False))).build(t_in["lig_x"], t_in["kp_x"])
    model.set_precision("bf16x3")
    for tkey, out in fx["outputs"].items():
        h, x = run_forward("egnn", model, batch, graphs, kk, t_in, float(tkey), dev)
        torch.cuda.synchronize()
        eh, ex = rel_err(h.cpu(), out["eps_h"]), rel_err(x.cpu(), out["eps_x"])
        print(f"{name} bf16x3 t={tkey}: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
        assert eh < TOL_X3 and ex < TOL_X3


def test_egnn_bf16x3_mode_full_size():
    import yaml
    from helpers import GOLDEN, flat_batch, oracle_cfg, oracle_forward
    from test_gpu_parity import _full_size_case, build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    cfgs = yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))
    sd, kw, rec_nf, inputs = _full_size_case("egnn", cfgs)
    cfg = oracle_cfg("egnn", kw, 10, rec_nf)
    model = build_model("egnn", sd, kw, 10, rec_nf, dev)
    model.set_precision("bf16x3")
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
    graphs = ops.LigandGraphs(batch, gp, True).build(t_in["lig_x"], t_in["kp_x"])
    for tval in (0.001, 0.5, 1.0):
        fb = flat_batch(inputs)
        ref_h, ref_x = oracle_forward("egnn", sd, cfg, fb, torch.full((fb.B,), tval))
        eps_h, eps_x = run_forward("egnn", model, batch, graphs, kk, t_in, tval, dev)
        torch.cuda.synchronize()
        eh, ex = rel_err(eps_h.cpu(), ref_h), rel_err(eps_x.cpu(), ref_x)
        print(f"egnn full size bf16x3 t={tval}: rel_err eps_h={eh:.2e} eps_x={ex:.2e}")
        assert eh < TOL_X3 and ex < TOL_X3
