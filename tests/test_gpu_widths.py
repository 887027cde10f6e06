"""GPU: both denoisers against the fp64 oracle at every width class their tensor-core kernels accept, not only the
shipped ones.

The kernels take their widths at run time (csrc/gvp.cu kpd_gvp_create / kpd_gvp_attach_tc, csrc/egnn.cu
kpd_egnn_create / kpd_egnn_attach_tc): GVP scalar width S (multiples of 4 up to 256; tensor cores when S % 16 == 0),
vector width V in 1..16, rbf_dim in 2..32, 1..4 GVPs per chain; EGNN H = hidden_nf + 1 with nmain = min(H, 256) & ~3
columns on the tensor cores and nlo = H - nmain <= 3 beside them.  The cases below pin the width-dependent code paths:

  1. GVP width sweep (fp32, bf16x3, bf16): partial column groups, vector blocks on either side of hd = 16, single-GVP and
     four-GVP chains, the head's 64 output columns at S < 64, odd V and rbf_dim, feature counts other than 10; two
     cases also at B = 40 (64-row node / head tiles; B = 4 runs the 32-row ones);
  2. EGNN width sweep (fp32, bf16x3, bf16): nlo = 0..3, nmain < 16 and nmain % 16 == 8, the run-time-width edge kernel
     at H = 256 (the LigRecDynamics default); two fp32-only widths through the drop-in module;
  3. kl rows spanning more than three edge tiles at non-shipped widths (the per-tile partial slots are S + 3V and
     Hp + 4 floats wide);
  4. hidden pre-activations far past -45 (the ex2 clamp of sigmoid2_acc, the rcp(inf) limit of sigmoid_acc);
  5. the captured sampling loop with injected noise and decode_atom_types at other feature counts;
  6. which widths build, and which attach the tensor-core modes.

bf16x3 GVP edge kernel: KS (128-row tiles, hi / lo planes) when its tile fits in 227 KB of shared memory, which is
kch = 2 * ceil(max(S + rbf_dim + V + 1, 64 + V) / 16) <= 38; the 64-row STACK kernel otherwise.  Every case here runs
KS; STACK is reached only at S = 256, V = 16, rbf_dim = 32, which test_gpu_tensorcore.test_gvp_bf16x3_mode_full_size
and test_gpu_gvp_layouts.test_gvp_rows_span_many_edge_tiles cover.

Reference: oracle/flat.py in fp64 on the edge lists the oracle builds from the fp32 coordinates; edge sets exact.  Bars
as in the rest of the suite: fp32 and bf16x3 -- max|a-b|/max|b| and rms-relative < 1e-4, per-channel < 5e-4
(helpers.err_report); bf16 -- max|a-b|/max|b| < 3e-2.  Each case also prints its floor, the error of the fp32 oracle
against the fp64 one, which must be <= 1e-5 (a case that misses a bar with a low floor is a kernel error, not an
ill-conditioned case), and max|eps_x| must be at least a tenth of max|eps_h| (the vector and coordinate paths carry
signal).  Every test prints the errors it measured."""
import functools
import warnings

import pytest
import torch

from helpers import err_report, flat_batch, fmt_err, oracle_cfg, oracle_forward, rel_err
from shipped_cases import assemble_inputs
from test_gpu_gvp_layouts import _assert_bars, _check_edges, _device_run

pytestmark = pytest.mark.gpu
FLOOR = 1e-5
X_OVER_H = 0.1
MODES = ["fp32", "bf16x3", "bf16"]
TVALS = (0.001, 0.5, 1.0)
CUT = {"ll": 5.0, "kl": 8.0, "kk": 8.0, "rr": 3.5}
CUT_ALL_ATOM = {"ll": 6.0, "kl": 8.0, "kk": 8.0, "rr": 3.5}
SIZES = [9, 1, 14, 6]
SEED_B40 = 17       # V = 1 at B = 40: input seeds 15, 16, 18 leave an atom whose fp32 eps_x floor is 1e-5..7e-5


def _dev():
    return torch.device("cuda:0")


# name -> (S, V, rbf_dim, (message, update, noise) GVPs, F = ligand features, C = keypoint features)
GVP_CASES = {
    "S16_V1": (16, 1, 2, (1, 1, 1), 1, 3),          # smallest of everything; head writes 64 > S columns; kch = 10
    "S48_V7": (48, 7, 17, (2, 1, 2), 5, 13),        # partial column group (NBf = 48); message hd = 8; odd rbf_dim
    "S64_V8": (64, 8, 31, (4, 4, 4), 13, 10),       # message hd = 9: second vector block holds one channel; MAXG chains
    "S128_V16": (128, 16, 16, (3, 2, 3), 10, 128),  # the LigRecDynamicsGVP defaults
    "S240_V15": (240, 15, 32, (1, 2, 1), 16, 7),    # message hd = 16 (hd > 16 false at its edge); one-GVP chains, wide
    "S96_V9": (96, 9, 16, (3, 2, 3), 7, 12),        # odd V, vin = 10; partial-slot width S + 3V not a multiple of 4
}
GVP_B40 = ("S16_V1", "S240_V15")
# Wh / Wu gain per case (2 elsewhere, as shipped_cases): at these widths x2 leaves max|eps_x| at 2..10 % of max|eps_h|
GVP_WSCALE = {"S64_V8": 3.0, "S128_V16": 3.0, "S96_V9": 3.0}

# hidden_nf -> (atom_nf, rec_nf); H = hidden_nf + 1, nmain = min(H, 256) & ~3, nlo = H - nmain
EGNN_CASES = {
    7: (1, 3),          # H 8: nmain 8 < 16, N padded to 16
    31: (7, 13),        # H 32: no leftover column
    33: (13, 128),      # H 34: nlo 2
    34: (1, 13),        # H 35: nlo 3, the maximum
    39: (7, 128),       # H 40: nmain % 16 == 8 (N = 48)
    66: (13, 3),        # H 67: nmain 64, nlo 3
    127: (1, 128),      # H 128
    255: (7, 3),        # H 256: the LigRecDynamics default, run-time-width edge kernel (HS = 0)
}


def gvp_kch(S, V, rbf_dim):
    """k-chunks of the widest GVP row (csrc/gvp.cu kpd_gvp_create)."""
    wmax = max(S + rbf_dim + V + 1, 64 + V)
    return 2 * ((wmax + 15) // 16)


def gvp_edge_kernel(S, V, rbf_dim, mode):
    """(kernel, edge tile rows) of the GVP edge kernel a mode runs (csrc/gvp.cu kpd_gvp_create / kpd_gvp_attach_tc)."""
    if mode == "fp32":
        return "SIMT", 64
    if mode == "bf16":
        return "bf16", 128
    return ("KS", 128) if gvp_kch(S, V, rbf_dim) <= 38 else ("STACK", 64)


def _egnn_cols(hidden_nf):
    H = hidden_nf + 1
    nmain = min(H, 256) // 4 * 4
    return H, nmain, H - nmain


# --------------------------------------------------------------------------- cases

def _gvp_kw(S, V, rbf_dim, chains, cut=CUT, message_norm=1):
    m, u, n = chains
    return dict(vector_size=V, n_convs=2, n_hidden_scalars=S, message_norm=message_norm, update_kp=True, ll_k=0,
                kl_k=0, n_message_gvps=m, n_update_gvps=u, n_noise_gvps=n, rbf_dim=rbf_dim, graph_cutoffs=cut)


def _gvp_sd(F, C, S, V, rbf_dim, chains, seed, wscale=2.0):
    from oracle import params as P
    sd = P.init_state_dict(P.gvp_dynamics_shapes(F, C, V, 2, S, True, *chains, rbf_dim=rbf_dim), seed=seed)
    for k in sd:
        if k.endswith(".Wh") or k.endswith(".Wu"):
            sd[k] = sd[k] * wscale              # keeps the vector channel carrying signal on random weights
    return sd


def _egnn_kw(hidden_nf, update_kp_feat, cut=CUT):
    return dict(n_layers=2, hidden_nf=hidden_nf, use_tanh=update_kp_feat, message_norm=1, update_kp_feat=update_kp_feat,
                norm=True, ll_k=0, kl_k=0, graph_cutoffs=cut)


def _egnn_sd(F, C, hidden_nf, update_kp_feat, seed):
    from oracle import params as P
    return P.init_state_dict(P.egnn_dynamics_shapes(F, C, 2, hidden_nf, update_kp_feat, True), seed=seed,
                             coord_gain=0.3)


def _keypoint_inputs(F, C, V, sizes, seed):
    from keypoint_diffusion_b200 import synthetic
    pockets = [synthetic.keypoint_pocket(i, 20, C, V, CUT["kk"]) for i in range(3)]     # kp_v = 0.1 N(0, 1) when V > 0
    return assemble_inputs(pockets, sizes, F, seed=seed, with_v=V > 0)


def _all_atom_inputs(F, C, V, seed):
    """Two 600-atom all-atom pockets (keypoints := atoms; hundreds of kl edges into one ligand atom within 8 A),
    ligands of 20, 1, 33 and 12 atoms."""
    from keypoint_diffusion_b200 import synthetic
    pockets = [synthetic.all_atom_pocket(i, 600, C, V, 3.5) for i in range(2)]
    if V:
        for i, pk in enumerate(pockets):
            pk.kp_v = 0.1 * torch.randn(pk.n_kp, V, 3, generator=torch.Generator().manual_seed(60 + i))
    return assemble_inputs(pockets, [20, 1, 33, 12], F, seed=seed, with_v=V > 0)


def _saturate(sd, prefixes, bias_names):
    """Add -80 / +60 / 0 to every third column of the named biases: those pre-activations sit far past +-45."""
    sd = dict(sd)
    for k in list(sd):
        if any(k.startswith(p) for p in prefixes) and any(k.endswith(b) for b in bias_names):
            c = torch.zeros_like(sd[k])
            c[0::3], c[1::3] = -80.0, 60.0
            sd[k] = sd[k] + c
    return sd


GVP_SAT_PREFIX = "dynamics.noise_predictor.conv_layers.0.edge_message_fns."
EGNN_SAT_PREFIX = "dynamics.egnn.conv_layers.0.edge_mlp."


@functools.lru_cache(maxsize=None)
def _case(key):
    """key -> (arch, state_dict, ctor kwargs, F, C, flat inputs, with_lk)."""
    kind = key[0]
    if kind == "gvp":                                       # ("gvp", name, B)
        S, V, rbf, chains, F, C = GVP_CASES[key[1]]
        sizes = [(9, 1, 14, 6, 11, 3, 20, 7)[i % 8] for i in range(key[2])]
        seed = 5 if key[2] == 4 else SEED_B40
        return ("gvp", _gvp_sd(F, C, S, V, rbf, chains, seed=21, wscale=GVP_WSCALE.get(key[1], 2.0)),
                _gvp_kw(S, V, rbf, chains), F, C, _keypoint_inputs(F, C, V, sizes, seed=seed), True)
    if kind == "egnn":                                      # ("egnn", hidden_nf, update_kp_feat)
        hid, kp = key[1], key[2]
        F, C = EGNN_CASES[hid]
        return ("egnn", _egnn_sd(F, C, hid, kp, seed=22), _egnn_kw(hid, kp), F, C,
                _keypoint_inputs(F, C, 0, SIZES, seed=6), kp)
    if kind == "gvp_many":                                  # ("gvp_many", name)
        S, V, rbf, chains, F, C = GVP_CASES[key[1]]
        return ("gvp", _gvp_sd(F, C, S, V, rbf, chains, seed=23), _gvp_kw(S, V, rbf, chains, CUT_ALL_ATOM, "mean"), F,
                C, _all_atom_inputs(F, C, V, seed=7), True)
    if kind == "egnn_many":                                 # ("egnn_many", hidden_nf)
        hid = key[1]
        F, C = EGNN_CASES[hid]
        return ("egnn", _egnn_sd(F, C, hid, True, seed=24), _egnn_kw(hid, True, CUT_ALL_ATOM), F, C,
                _all_atom_inputs(F, C, 0, seed=8), True)
    if kind == "gvp_sat":                                   # ("gvp_sat", name)
        arch, sd, kw, F, C, inputs, lk = _case(("gvp", key[1], 4))
        sd = _saturate(sd, [GVP_SAT_PREFIX], [".0.to_feats_out.0.bias", ".0.scalar_to_vector_gates.bias"])
        return arch, sd, kw, F, C, inputs, lk
    if kind == "egnn_sat":                                  # ("egnn_sat", hidden_nf)
        arch, sd, kw, F, C, inputs, lk = _case(("egnn", key[1], True))
        return arch, _saturate(sd, [EGNN_SAT_PREFIX], [".0.bias"]), kw, F, C, inputs, lk
    raise KeyError(key)


def _sat_layer(arch, name):
    """The Linear layers _saturate shifted, as the oracle names them."""
    if arch == "gvp":
        return name.startswith(GVP_SAT_PREFIX) and (name.endswith(".0.to_feats_out.0") or
                                                    name.endswith(".0.scalar_to_vector_gates"))
    return name.startswith(EGNN_SAT_PREFIX) and name.endswith(".0")


@functools.lru_cache(maxsize=None)
def _ref(key, tval):
    """The fp64 oracle, its edge lists (built from the fp32 coordinates), the fp32 oracle's error against it (the
    floor of the case) and, for the saturated cases, the fraction of the shifted layers' pre-activations below -45."""
    from oracle import flat
    arch, sd, kw, F, C, inputs, with_lk = _case(key)
    cfg = oracle_cfg(arch, kw, F, C)
    fb = flat_batch(inputs)
    lig_b, kp_b = fb.batch_idx()
    edges = flat.build_lig_edges(fb.lig_x, fb.kp_x, lig_b, kp_b, fb.B, cfg.graph_cutoffs, cfg.ll_k, cfg.kl_k, with_lk)
    t = torch.full((fb.B,), tval)
    pre = []
    lin = flat._lin

    def recording_lin(sd_, name, x):
        y = lin(sd_, name, x)
        if _sat_layer(arch, name):
            pre.append(y.detach().reshape(-1))
        return y

    flat._lin = recording_lin
    try:
        h64, x64 = oracle_forward(arch, sd, cfg, flat_batch(inputs, torch.float64), t.double(), edges=edges)
    finally:
        flat._lin = lin
    h32, x32 = oracle_forward(arch, sd, cfg, fb, t, edges=edges)
    fh, fx = err_report(h32, h64), err_report(x32, x64)
    floor = max(fh["norm"], fh["rms"], fx["norm"], fx["rms"])
    below = float((torch.cat(pre) < -45).double().mean()) if pre else 0.0
    return {"h": h64, "x": x64, "edges": edges[0], "floor": floor, "below45": below}


def _model(key, mode):
    from test_gpu_parity import build_model
    arch, sd, kw, F, C, _, _ = _case(key)
    model = build_model(arch, sd, kw, F, C, _dev())
    if mode != "fp32":
        assert model.tc_blob2 is not None, f"{key} should run on the tensor cores"
        model.set_precision(mode)
    return model


def _check(key, mode, label, tvals=TVALS):
    """Device forward at each t against the fp64 oracle; asserts the bars, the floor, edge sets and signal in eps_x."""
    arch, sd, kw, F, C, inputs, with_lk = _case(key)
    model = _model(key, mode)
    worst = {"h": 0.0, "x": 0.0}
    for tval in tvals:
        r = _ref(key, tval)
        eps_h, eps_x, graphs, batch = _device_run(arch, model, inputs, kw, torch.full((1,), tval))
        _check_edges(graphs, r["edges"], with_lk, label)
        assert torch.isfinite(eps_h).all() and torch.isfinite(eps_x).all(), (label, mode, tval)
        rh, rx = err_report(eps_h, r["h"]), err_report(eps_x, r["x"])
        hmax, xmax = float(r["h"].abs().max()), float(r["x"].abs().max())
        print(f"{label} [{mode}] t={tval}: eps_h {fmt_err(rh)} | eps_x {fmt_err(rx)} | fp32-oracle floor "
              f"{r['floor']:.1e} | max|eps_h| {hmax:.3g} max|eps_x| {xmax:.3g}")
        assert r["floor"] <= FLOOR, f"{label} t={tval} is ill-conditioned (fp32 oracle vs fp64 {r['floor']:.1e})"
        assert xmax >= X_OVER_H * hmax, f"{label}: the coordinate path carries too little signal ({xmax} vs {hmax})"
        _assert_bars(mode, rh, rx, (label, tval))
        worst["h"], worst["x"] = max(worst["h"], rh["norm"]), max(worst["x"], rx["norm"])
    return graphs, batch, worst


# --------------------------------------------------------------------------- 1. GVP width sweep

@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,B", [(n, 4) for n in GVP_CASES] + [(n, 40) for n in GVP_B40])
def test_gvp_width_sweep_vs_oracle(name, B, mode):
    S, V, rbf, chains, F, C = GVP_CASES[name]
    kernel, tile = gvp_edge_kernel(S, V, rbf, mode)
    if mode == "bf16x3":
        assert kernel == "KS", f"{name}: kch {gvp_kch(S, V, rbf)} should select the KS edge kernel"
    _, batch, worst = _check(("gvp", name, B), mode, f"gvp {name} rbf={rbf} chains={chains} F={F} C={C} B={B}")
    assert batch.B == B
    print(f"gvp {name} B={B} [{mode}]: edge kernel {kernel} ({tile}-row tiles, kch {gvp_kch(S, V, rbf)}), "
          f"node / head tiles {32 if B < 32 else 64} rows; worst norm eps_h {worst['h']:.2e} eps_x {worst['x']:.2e}")


def test_gvp_width_cases_reach_what_they_claim():
    """The case table covers the width classes it names (no device work)."""
    hd = {n: c[1] + 1 for n, c in GVP_CASES.items()}           # message GVP 0: hd = max(vin = V + 1, vout = V)
    assert {n for n, h in hd.items() if h == 8} and {n for n, h in hd.items() if h == 9}
    assert {n for n, h in hd.items() if h == 16} and {n for n, h in hd.items() if h == 17}
    assert any(c[0] < 64 for c in GVP_CASES.values()) and any(c[0] % 32 for c in GVP_CASES.values())
    assert any((c[0] + 3 * c[1]) % 4 for c in GVP_CASES.values())
    assert {1, 4} <= {k for c in GVP_CASES.values() for k in c[3]}
    assert any(c[2] % 2 for c in GVP_CASES.values()) and any(c[1] % 2 for c in GVP_CASES.values())
    assert all(c[4] != 10 for n, c in GVP_CASES.items() if n != "S128_V16")
    assert all(gvp_edge_kernel(*GVP_CASES[n][:3], "bf16x3")[0] == "KS" for n in GVP_CASES)
    assert gvp_edge_kernel(256, 16, 32, "bf16x3")[0] == "STACK" and gvp_edge_kernel(256, 16, 16, "bf16x3")[0] == "KS"
    assert gvp_kch(16, 1, 2) == 10
    nlo = {_egnn_cols(h)[2] for h in EGNN_CASES}
    assert nlo == {0, 2, 3} and any(_egnn_cols(h)[1] < 16 for h in EGNN_CASES)
    assert any(_egnn_cols(h)[1] % 16 == 8 for h in EGNN_CASES) and 255 in EGNN_CASES


# --------------------------------------------------------------------------- 2. EGNN width sweep

@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("update_kp_feat", [True, False])
@pytest.mark.parametrize("hidden_nf", sorted(EGNN_CASES))
def test_egnn_width_sweep_vs_oracle(hidden_nf, update_kp_feat, mode):
    H, nmain, nlo = _egnn_cols(hidden_nf)
    F, C = EGNN_CASES[hidden_nf]
    _, _, worst = _check(("egnn", hidden_nf, update_kp_feat), mode,
                         f"egnn hidden_nf={hidden_nf} (H {H}, nmain {nmain}, nlo {nlo}) kp={update_kp_feat} F={F} C={C}")
    kernel = "SIMT" if mode == "fp32" else ("HS=257" if H == 257 else "run-time width (HS=0)")
    print(f"egnn hidden_nf={hidden_nf} kp={update_kp_feat} [{mode}]: edge kernel {kernel}; worst norm eps_h "
          f"{worst['h']:.2e} eps_x {worst['x']:.2e}")


@pytest.mark.parametrize("hidden_nf", [36, 257])
def test_egnn_fp32_only_width_warns_once_and_matches_oracle(hidden_nf):
    """hidden_nf 36 (nmain 36, not a multiple of 8) and 257 (H 258 > 257) have no tensor-core tiles: a drop-in module
    asked for bf16x3 says so once with a RuntimeWarning and runs the fp32 SIMT kernels."""
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    from keypoint_diffusion_b200.dynamics import LigRecDynamics
    from oracle import flat
    dev = _dev()
    F, C = 7, 13
    kw = _egnn_kw(hidden_nf, True)
    sd = _egnn_sd(F, C, hidden_nf, True, seed=25)
    dyn = LigRecDynamics(F, C, n_layers=2, hidden_nf=hidden_nf, use_tanh=True, graph_cutoffs=CUT, update_kp_feat=True,
                         norm=True)
    dyn.load_state_dict({k[len("dynamics."):]: v for k, v in sd.items()})
    dyn = dyn.to(dev).eval()
    dyn.set_precision("bf16x3")
    pockets = [synthetic.keypoint_pocket(i, 20, C, 0, CUT["kk"]) for i in range(3)]
    g_cpu = HeteroBatch.from_pockets(pockets, SIZES, F)
    x_l, h_l = synthetic.ligand_noise_state(SIZES, F, seed=9)
    g_cpu.nodes["lig"].data["x_0"], g_cpu.nodes["lig"].data["h_0"] = x_l, h_l
    g = g_cpu.to(dev)
    ks, kd = g_cpu.edges(form="uv", etype="kk")
    inputs = {"lig_n": g_cpu.batch_num_nodes("lig"), "kp_n": g_cpu.batch_num_nodes("kp"), "lig_x": x_l, "lig_h": h_l,
              "kp_x": g_cpu.nodes["kp"].data["x_0"], "kp_h": g_cpu.nodes["kp"].data["h_0"], "kk_src": ks, "kk_dst": kd}
    cfg = oracle_cfg("egnn", kw, F, C)
    fb = flat_batch(inputs)
    lig_b, kp_b = fb.batch_idx()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        for tval in TVALS:
            eps_h, eps_x = dyn(g, torch.full((len(SIZES),), tval, device=dev))
            torch.cuda.synchronize()
            edges = flat.build_lig_edges(fb.lig_x, fb.kp_x, lig_b, kp_b, fb.B, CUT, 0, 0, True)
            t = torch.full((fb.B,), tval, dtype=torch.float64)
            ref_h, ref_x = oracle_forward("egnn", sd, cfg, flat_batch(inputs, torch.float64), t, edges=edges)
            rh, rx = err_report(eps_h.cpu(), ref_h), err_report(eps_x.cpu(), ref_x)
            print(f"egnn fp32-only hidden_nf={hidden_nf} [bf16x3 requested] t={tval}: eps_h {fmt_err(rh)} | "
                  f"eps_x {fmt_err(rx)}")
            _assert_bars("fp32", rh, rx, (hidden_nf, tval))
    runtime = [w for w in caught if issubclass(w.category, RuntimeWarning)]
    assert len(runtime) == 1 and "no tensor-core tiles" in str(runtime[0].message), [str(w.message) for w in caught]
    model = dyn.device_model(dev)
    assert model.tc_blob2 is None and model.precision == "fp32" and dyn.precision == "bf16x3"


# --------------------------------------------------------------------------- 3. rows spanning several edge tiles

@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("key", [("gvp_many", "S48_V7"), ("egnn_many", 31), ("egnn_many", 34)],
                         ids=["gvp_S48_V7", "egnn_nlo0", "egnn_nlo3"])
def test_rows_span_many_edge_tiles_at_other_widths(key, mode):
    if key[0] == "gvp_many":
        S, V, rbf, _, _, _ = GVP_CASES[key[1]]
        kernel, tile = gvp_edge_kernel(S, V, rbf, mode)
        label = f"gvp many-tile {key[1]} (partial slot S + 3V = {S + 3 * V} floats)"
    else:
        H, nmain, nlo = _egnn_cols(key[1])
        kernel, tile = ("SIMT" if mode == "fp32" else "run-time width (HS=0)"), 64
        label = f"egnn many-tile hidden_nf={key[1]} (nlo {nlo}, partial slot Hp + 4 = {(H + 3) // 4 * 4 + 4} floats)"
    graphs, _, _ = _check(key, mode, label, tvals=(0.3,))
    rp = graphs.kl.rowptr.cpu().long()
    deg = int((rp[1:] - rp[:-1]).max())
    print(f"{label} [{mode}]: edge kernel {kernel}, max kl in-degree {deg} (edge tile {tile})")
    assert deg > 3 * tile, f"a kl row must span more than three {tile}-edge tiles (max in-degree {deg})"


# --------------------------------------------------------------------------- 4. saturated activations

@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("key", [("gvp_sat", "S48_V7"), ("egnn_sat", 34)], ids=["gvp_S48_V7", "egnn_hidden34"])
def test_saturated_pre_activations(key, mode):
    """Large constants on the biases of the first message GVP (to_feats_out and gates) / the first edge-MLP layer put a
    third of those pre-activations near -80 and a third near +60: SiLU and the sigmoid gates at their limits."""
    below = min(_ref(key, tval)["below45"] for tval in TVALS)
    print(f"{key} [{mode}]: fraction of the shifted layers' pre-activations below -45 (oracle): {below:.2f}")
    assert below >= 0.10
    _check(key, mode, f"saturated {key[0]} {key[1]}")


# --------------------------------------------------------------------------- 5. sampling loop and decode at other F

@pytest.mark.parametrize("mode", ["fp32", "bf16x3"])
@pytest.mark.parametrize("key", [("gvp", "S48_V7", 4), ("egnn", 39, True)], ids=["gvp_F5", "egnn_F7"])
def test_full_loop_at_other_feature_counts(key, mode):
    """The captured loop with injected noise (T = 12, 4 steps per graph) against oracle.flat.sample_from_encoded_receptors
    in fp64: the (3 + F)-channel posterior step and its noise layout at F = 5 and 7."""
    from oracle import flat, schedule as S
    from test_gpu_egnn_bf16 import _loop_sampler
    arch, sd, kw, F, C, inputs, with_lk = _case(key)
    T, seed = 12, 1234
    gamma = S.gamma_table(T, 1e-5)
    init = torch.randn(len(SIZES), 3, generator=torch.Generator().manual_seed(3))
    fx = {"kwargs": kw, "T": T, "atom_nf": F, "inputs": inputs, "state_dict": {"gamma.gamma": gamma},
          "noise_seed": seed, "init_lig_pos": init}
    x_dev, h_dev = _loop_sampler(_model(key, mode), fx, _dev())

    torch.manual_seed(seed)                 # the slots _loop_sampler drew: x then h per slot, init first, then s = T-1..0
    N = int(inputs["lig_n"].sum())
    slots = [(torch.randn(N, 3), torch.randn(N, F)) for _ in range(T + 1)]
    cfg = oracle_cfg(arch, kw, F, C)

    def noise_fn(step, kind, shape):
        nx, nh = slots[0 if step == -1 else T - step]
        return nx if kind == "x" else nh

    def dyn(b, t):
        lig_b, kp_b = b.batch_idx()
        edges = flat.build_lig_edges(b.lig_x.float(), b.kp_x.float(), lig_b, kp_b, b.B, cfg.graph_cutoffs, cfg.ll_k,
                                     cfg.kl_k, with_lk)
        return oracle_forward(arch, sd, cfg, b, t.double(), edges=edges)

    pos, feat = flat.sample_from_encoded_receptors(dyn, gamma, T, flat_batch(inputs, torch.float64), init.double(),
                                                   noise_fn, atom_nf=F)
    ex, eh = rel_err(x_dev, torch.cat(pos)), rel_err(h_dev, torch.cat(feat))
    print(f"loop {arch} F={F} [{mode}] T={T}: rel_err pos {ex:.2e} feat {eh:.2e}")
    assert ex < 1e-3 and eh < 1e-3


@pytest.mark.parametrize("F", [1, 5, 13])
def test_decode_atom_types_at_other_feature_counts(F):
    from keypoint_diffusion_b200 import ops
    g = torch.Generator().manual_seed(F)
    h = torch.randn(997, F, generator=g)
    h[:300] = torch.round(h[:300] * 2) / 2                  # coarse values: many exact ties
    h[300:310] = 0.0                                        # all channels tied
    h[310:320] = -1.5
    if F > 1:
        h[320:330, F - 1] = h[320:330, 0] = 9.0             # tie between the first and the last channel
        h[330:340, 1:] = 4.0                                # tie on every channel but the first
        h[330:340, 0] = 3.0
    hmax = h.max(1, keepdim=True).values
    ref = torch.where(h == hmax, torch.arange(F), F).min(1).values       # lowest index among the maxima
    got = ops.decode_atom_types(h.to(_dev())).cpu().long()
    n_tied = int(((h == hmax).sum(1) > 1).sum())
    print(f"decode_atom_types F={F}: {h.shape[0]} rows, {n_tied} with tied maxima: "
          f"{int((got != ref).sum())} mismatches")
    assert (F == 1 or n_tied >= 20) and torch.equal(got, ref)


# --------------------------------------------------------------------------- 6. which widths build

def test_egnn_every_hidden_width_builds():
    """hidden_nf 1..259: every width builds; the tensor-core modes attach exactly when nmain >= 8, nmain % 8 == 0 and
    H <= 257; only nlo > 3 (hidden_nf 259) is refused, by the library."""
    from oracle import params as P
    from keypoint_diffusion_b200 import ops
    from test_gpu_parity import _strip
    dev = _dev()
    n_tc = 0
    for hid in range(1, 260):
        H, nmain, nlo = _egnn_cols(hid)
        sd = _strip(P.init_state_dict(P.egnn_dynamics_shapes(10, 12, 1, hid, False, False), seed=hid))
        kw = dict(atom_nf=10, rec_nf=12, hidden_nf=hid, n_layers=1, use_tanh=False, update_kp_feat=False, norm=False,
                  message_norm=1, device=dev)
        if nlo > 3:
            with pytest.raises(RuntimeError, match="leftover columns"):
                ops.EgnnModel(sd, **kw)
            continue
        model = ops.EgnnModel(sd, **kw)
        tc = nmain >= 8 and nmain % 8 == 0 and H <= 257
        assert (model.tc_blob2 is not None) == tc, hid
        if tc:
            model.set_precision("bf16x3")
            n_tc += 1
        else:
            with pytest.raises(RuntimeError):
                model.set_precision("bf16x3")
        del model
    print(f"egnn hidden_nf 1..259: {n_tc} widths attach the tensor-core modes, hidden_nf 259 refused")


def test_gvp_every_scalar_width_builds():
    """S = 4..256 step 4, V in {1, 16}, rbf_dim in {2, 32}: construction never raises; the tensor-core modes attach
    exactly when S % 16 == 0."""
    from oracle import params as P
    from keypoint_diffusion_b200 import ops
    from test_gpu_parity import _strip
    dev = _dev()
    for S in range(4, 257, 4):
        for V in (1, 16):
            for rbf in (2, 32):
                sd = _strip(P.init_state_dict(P.gvp_dynamics_shapes(10, 12, V, 1, S, False, 1, 1, 1, rbf_dim=rbf),
                                              seed=S))
                model = ops.GvpModel(sd, n_lig_scalars=10, n_kp_scalars=12, vector_size=V, n_convs=1,
                                     n_hidden_scalars=S, update_kp=False, n_message_gvps=1, n_update_gvps=1,
                                     n_noise_gvps=1, message_norm=1, rbf_dim=rbf, device=dev)
                assert (model.tc_blob2 is not None) == (S % 16 == 0), (S, V, rbf)
                for mode in ("bf16", "bf16x3"):
                    if S % 16 == 0:
                        model.set_precision(mode)
                    else:
                        with pytest.raises(RuntimeError):
                            model.set_precision(mode)
                del model
    print("gvp S 4..256 x V {1, 16} x rbf_dim {2, 32}: all build; tensor-core modes exactly at S % 16 == 0")
