"""GPU parity at the SHIPPED width of every shipped trained model, in both parity-grade modes.

For each of tests/shipped_cases.py:SHIPPED (all eight trained_models/*): the CUDA denoiser (through the C
ABI) against the CPU oracle on the same seeded weights and inputs, teacher-forced at several t, in the fp32 SIMT mode
and the bf16x3 tensor-core mode; the ll / kl / lk edge sets compared exactly.  Bars (stated here): edge sets exact;
eps_h, eps_x max|a-b|/max|b| <= 1e-4 (north_star), RMS-relative <= 1e-4, per-channel max-relative <= 5e-4.
"""
import pytest
import torch

from helpers import edge_set, err_report, flat_batch, fmt_err, oracle_cfg, oracle_forward
from shipped_cases import SHIPPED, shipped_case

pytestmark = pytest.mark.gpu
TOL, TOL_CHAN = 1e-4, 5e-4


@pytest.mark.parametrize("mode", ["fp32", "bf16x3"])
@pytest.mark.parametrize("name", sorted(SHIPPED))
def test_shipped_config_denoiser_vs_oracle(name, mode):
    from test_gpu_parity import build_model, device_inputs, run_forward
    from keypoint_diffusion_b200 import ops
    dev = torch.device("cuda:0")
    arch, sd, kw, rec_nf, inputs = shipped_case(name)
    cfg = oracle_cfg(arch, kw, 10, rec_nf)
    model = build_model(arch, sd, kw, 10, rec_nf, dev)
    if mode != "fp32":
        assert model.tc_blob2 is not None, "every shipped width must run on the tensor cores"
        model.set_precision(mode)
    batch, kk, t_in = device_inputs(inputs, dev)
    gp = ops.GraphParams.from_module(kw["ll_k"], kw["kl_k"], kw["graph_cutoffs"])
    with_lk = bool(kw.get("update_kp_feat", kw.get("update_kp", False)))
    graphs = ops.LigandGraphs(batch, gp, with_lk).build(t_in["lig_x"], t_in["kp_x"])
    for tval in (0.001, 0.5, 1.0):
        fb = flat_batch(inputs)
        ref_h, ref_x, edges, _ = oracle_forward(arch, sd, cfg, fb, torch.full((fb.B,), tval), return_edges=True)
        eps_h, eps_x = run_forward(arch, model, batch, graphs, kk, t_in, tval, dev)
        torch.cuda.synchronize()
        for et in ("ll", "kl") + (("lk",) if with_lk else ()):
            assert edge_set(getattr(graphs, et).edges()) == edge_set(torch.stack(edges[et])), (name, et)
        rh, rx = err_report(eps_h.cpu(), ref_h), err_report(eps_x.cpu(), ref_x)
        n_e = {et: int(edges[et][0].numel()) for et in edges}
        print(f"{name} [{mode}] t={tval}: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)} | edges {n_e} kk {int(inputs['kk_src'].numel())}")
        for r in (rh, rx):
            assert r["norm"] < TOL and r["rms"] < TOL and r["chan"] < TOL_CHAN, (name, mode, tval, rh, rx)
