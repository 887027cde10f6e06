"""CPU: the drop-in modules' constructor / state_dict contract and host-side logic, and that the
C-ABI library loads and exports every symbol include/kpdiff_b200.h declares (no compute)."""
import ctypes
import json
import re
from pathlib import Path

import pytest
import torch
import yaml

from helpers import GOLDEN

ROOT = Path(__file__).resolve().parents[1]


def _cfgs():
    return yaml.safe_load(open(GOLDEN / "shipped_configs.yml"))


@pytest.mark.parametrize("name", ["egnn_20kp", "egnn_40kp", "egnn_all_atom", "egnn_ca", "gvp_20kp", "gvp_40kp",
                                  "gvp_all_atom", "gvp_ca"])
def test_state_dict_layout_matches_reference(name, monkeypatch):
    """model_from_config(cfg).state_dict() has exactly the reference's keys and shapes, so
    trained_models/*/model.pt loads with strict=True."""
    from keypoint_diffusion_b200 import model_from_config
    monkeypatch.chdir(ROOT)                      # dataset.location is relative, as in the reference
    inv = json.load(open(GOLDEN / "state_dict_shapes.json"))[name]
    model = model_from_config(_cfgs()[name])
    mine = {k: list(v.shape) for k, v in model.state_dict().items()}
    assert mine == inv
    # round trip through a checkpoint-shaped dict
    sd = {k: torch.randn(v) if v != [0] else torch.empty(0) for k, v in inv.items()}
    model.load_state_dict(sd, strict=True)
    assert torch.equal(model.state_dict()["gamma.gamma"], sd["gamma.gamma"])


def test_constructor_errors_match_reference(monkeypatch):
    from keypoint_diffusion_b200 import KeypointDiffusion, LigRecDynamicsGVP
    monkeypatch.chdir(ROOT)
    d = Path("data/bindingmoad_processed")
    with pytest.raises(ValueError):
        KeypointDiffusion(10, 128, d, architecture="transformer")
    with pytest.raises(ValueError):
        KeypointDiffusion(10, 128, d, rec_encoder_type="other", rec_encoder_config={"k_closest": 3})
    with pytest.raises(ValueError):
        KeypointDiffusion(10, 128, Path("/nonexistent"))
    with pytest.raises(NotImplementedError):
        LigRecDynamicsGVP(10, 128, no_cg=True)
    with pytest.raises(NotImplementedError):      # SURVEY A8: dead and broken in the reference, no shipped config enables it
        KeypointDiffusion(10, 128, d, use_fake_atoms=True)


def test_no_cpu_fallback(monkeypatch):
    """CPU tensors are refused loudly instead of being computed some other way."""
    from keypoint_diffusion_b200 import HeteroBatch, LigRecDynamics, synthetic
    dyn = LigRecDynamics(10, 16, n_layers=1, hidden_nf=15, graph_cutoffs={"ll": 5, "kl": 8}, kl_k=3)
    g = HeteroBatch.from_pockets([synthetic.keypoint_pocket(0, 5, 16)], [4], 10)
    with pytest.raises(RuntimeError, match="CUDA"):
        dyn(g, torch.tensor([0.5]), None)


def test_library_exports_every_declared_symbol():
    from keypoint_diffusion_b200 import _lib
    header = (ROOT / "include" / "kpdiff_b200.h").read_text()
    declared = set(re.findall(r"\b(kpd_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for sym in sorted(declared):
        assert hasattr(lib, sym), f"{sym} declared in include/kpdiff_b200.h but not exported"
    assert declared == set(_lib.EXPORTED)


def test_hetero_batch_roundtrip():
    from keypoint_diffusion_b200 import HeteroBatch, hetero, synthetic, utils
    pk = [synthetic.keypoint_pocket(i, 6, 12, 4) for i in range(2)]
    g = HeteroBatch.from_pockets(pk, [5, 2, 9], 10)
    assert g.batch_size == 3 and g.num_nodes("lig") == 16 and g.num_nodes("kp") == 18
    bi = utils.get_batch_idxs(g)
    assert bi["lig"].tolist() == [0] * 5 + [1] * 2 + [2] * 9
    parts = hetero.unbatch(g)
    assert [p.num_nodes("lig") for p in parts] == [5, 2, 9]
    g2 = hetero.batch(parts)
    assert torch.equal(g2.nodes["kp"].data["x_0"], g.nodes["kp"].data["x_0"])
    assert torch.equal(g2.edges(form="uv", etype="kk")[1], g.edges(form="uv", etype="kk")[1])
    copies = utils.copy_graph(parts[0], 3, torch.tensor([4, 6, 8]))
    assert [c.num_nodes("lig") for c in copies] == [4, 6, 8]
    with g.local_scope():
        g.nodes["lig"].data["h_0"] = torch.ones(16, 10)
    assert float(g.nodes["lig"].data["h_0"].abs().sum()) == 0.0


def test_ligand_size_distribution():
    from keypoint_diffusion_b200 import LigandSizeDistribution
    d = LigandSizeDistribution(ROOT / "data" / "bindingmoad_processed")
    torch.manual_seed(0)
    s = d.sample(torch.tensor([336, 5, 9999]), 50)
    assert s.shape == (3, 50) and int(s.min()) >= 2 and int(s.max()) <= 60


def test_edge_capacity_and_packer_offsets():
    from keypoint_diffusion_b200 import ops, pack
    b = object.__new__(ops.DeviceBatch)
    b.lig_n, b.kp_n = [20, 3, 60], [20, 20, 40]
    gp = ops.GraphParams(ll_k=0, ll_r=5, kl_k=5)
    assert ops.DeviceBatch.edge_capacity(b, gp) == (20 * 19 + 3 * 2 + 60 * 59, 20 * 5 + 20 * 3 + 40 * 5)
    gp = ops.GraphParams(ll_k=4, kl_k=0, kl_r=8)
    assert ops.DeviceBatch.edge_capacity(b, gp) == (20 * 4 + 3 * 2 + 60 * 4, 20 * 20 + 20 * 3 + 40 * 60)


def test_output_decode_matches_reference_format():
    """argmax -> element symbols and the XYZ text block of reference utils.py:11-21 / test.py:199-203."""
    from keypoint_diffusion_b200.utils import decode_ligands, write_xyz_file
    elements = ["C", "N", "O", "S", "P", "F", "Cl", "Br", "I", "B"]
    pos = [torch.tensor([[0.0, 1.0, 2.0], [1.23456, -2.0, 3.5]]), torch.zeros(1, 3)]
    feat = [torch.tensor([[0.1, 0.9] + [0.0] * 8, [0.0] * 6 + [2.0] + [0.0] * 3]), torch.eye(10)[2:3]]
    dec = decode_ligands(pos, feat, elements)
    assert [d[1] for d in dec] == [["N", "Cl"], ["O"]]
    txt = write_xyz_file(dec[0][0], dec[0][1])
    assert txt == "2\n\nN 0.000 1.000 2.000\nCl 1.235 -2.000 3.500\n"


def test_sub_batch_partition_and_default_count(monkeypatch):
    """Host logic of the concurrent sub-batch sampling: contiguous near-equal groups that cover the batch exactly;
    default group count per architecture, never fewer than 16 complexes per group; KPD_SUB_BATCHES overrides."""
    from keypoint_diffusion_b200 import model_from_config
    from keypoint_diffusion_b200.utils import split_bounds
    import os
    for B in (1, 2, 3, 16, 33, 100, 1024):
        for n in (1, 2, 3, 4, 7):
            b = split_bounds(B, n)
            assert b[0] == 0 and b[-1] == B and all(y > x for x, y in zip(b[:-1], b[1:]))
            sizes = [y - x for x, y in zip(b[:-1], b[1:])]
            assert len(sizes) == min(n, B) and max(sizes) - min(sizes) <= 1
    os.chdir(ROOT)
    monkeypatch.delenv("KPD_SUB_BATCHES", raising=False)
    cfgs = _cfgs()
    gvp, egnn = model_from_config(cfgs["gvp_20kp"]), model_from_config(cfgs["egnn_20kp"])
    assert [gvp.default_sub_batches(B) for B in (1, 10, 31, 32, 64, 100, 4096)] == [1, 1, 1, 2, 4, 4, 4]
    assert [egnn.default_sub_batches(B) for B in (10, 32, 100, 800)] == [1, 2, 2, 2]
    monkeypatch.setenv("KPD_SUB_BATCHES", "3")
    assert gvp.default_sub_batches(100) == 3 and gvp.default_sub_batches(2) == 2


def test_expand_complexes_equals_copy_graph_then_batch():
    """Device-side batch assembly (hetero.expand_complexes) builds exactly the batch the reference's host loop builds
    (utils.copy_graph per receptor + dgl.batch per diffusion batch, ligand_diffuser.py:292-313)."""
    from keypoint_diffusion_b200 import HeteroBatch, hetero, synthetic, utils
    pk = [synthetic.keypoint_pocket(i, 6 + i, 12, 4) for i in range(3)]
    encs = [HeteroBatch.from_pockets([p], [1], 10) for p in pk]
    enc = hetero.batch(encs)
    pocket_idx, n_lig = torch.tensor([0, 0, 2, 1, 2]), torch.tensor([5, 3, 7, 4, 6])
    g = hetero.expand_complexes(enc, pocket_idx, n_lig, 10)
    copies = []
    for c in range(5):
        copies.extend(utils.copy_graph(encs[int(pocket_idx[c])], 1, torch.tensor([int(n_lig[c])])))
    r = hetero.batch(copies)
    for k in ("x_0", "h_0", "v_0"):
        assert torch.equal(g.nodes["kp"].data[k], r.nodes["kp"].data[k]), k
    assert torch.equal(torch.stack(g.edges(form="uv", etype="kk")), torch.stack(r.edges(form="uv", etype="kk")))
    for nt in ("kp", "lig"):
        assert torch.equal(g.batch_num_nodes(nt), r.batch_num_nodes(nt))
    assert torch.equal(g.batch_num_edges("kk"), r.batch_num_edges("kk"))
    assert torch.equal(g.nodes["lig"].data["h_0"], r.nodes["lig"].data["h_0"])        # zero-filled (utils.py:142-144)
    assert g.batch_size == 5 and g.num_nodes("rec") == 0


def test_capacity_plan_properties():
    """plan_capacity: real complexes first and unchanged, fillers inside the per-complex maxima, totals and edge
    capacities cover the padded layout, and freshly drawn ligand sizes land in a handful of buckets."""
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.n_nodes_dist import LigandSizeDistribution
    from keypoint_diffusion_b200.utils import split_bounds
    g = torch.Generator().manual_seed(0)
    for gp in (ops.GraphParams(ll_r=6.0, kl_k=7), ops.GraphParams(ll_k=4, kl_k=0, kl_r=8.0), ops.GraphParams(ll_r=5.0, kl_k=5)):
        for trial in range(40):
            B = int(torch.randint(1, 70, (1,), generator=g))
            lig = torch.randint(1, 61, (B,), generator=g).tolist()
            kp = torch.randint(1, 50, (B,), generator=g).tolist() if trial % 2 else [20] * B
            n_kk = int(torch.randint(0, 400 * B, (1,), generator=g))
            p = ops.plan_capacity(lig, kp, n_kk, gp)
            Bc, N, K, ml, mk, cll, ckl, ckk = p.key
            assert list(p.lig_n[:B]) == lig and list(p.kp_n[:B]) == kp and p.n_real == B
            assert len(p.lig_n) == len(p.kp_n) == Bc and sum(p.lig_n) == N and sum(p.kp_n) == K
            assert Bc > B and min(p.lig_n) >= 1 and min(p.kp_n) >= 1 and max(p.lig_n) <= ml and max(p.kp_n) <= mk
            ll_lim = gp.ll_k if gp.ll_k > 0 else gp.ll_cap
            kl_lim = gp.kl_k if gp.kl_k > 0 else gp.kl_cap
            assert cll >= sum(n * min(n - 1, ll_lim) for n in p.lig_n)
            assert ckl >= sum(k * min(n, kl_lim) for n, k in zip(p.lig_n, p.kp_n))
            assert ckk >= max(n_kk, 1)
            assert N <= 1.34 * sum(lig) + 72 and K <= 1.34 * sum(kp) + 72            # bounded filler work
            assert ops.plan_capacity(lig, kp, n_kk, gp).key == p.key
    # the reference's real entry point draws new sizes per call (ligand_diffuser.py:490-495): few distinct buckets
    dist = LigandSizeDistribution(ROOT / "data" / "bindingmoad_processed")
    torch.manual_seed(1)
    gp = ops.GraphParams(ll_r=6.0, kl_k=7)
    keys, waste = set(), []
    for _ in range(60):
        sizes = dist.sample(torch.tensor([336]), 100)[0].tolist()
        bd = split_bounds(100, 4)
        for a, b in zip(bd[:-1], bd[1:]):
            p = ops.plan_capacity(sizes[a:b], [20] * (b - a), 322 * (b - a), gp)
            keys.add(p.key)
            waste.append((p.key[1] + p.key[2]) / (p.n_lig_real + p.n_kp_real) - 1.0)
    assert len(keys) <= 8, sorted(keys)
    assert sum(waste) / len(waste) < 0.10


def test_capacity_plan_batch_rounding_feeds_the_node_tile_rule():
    """kpd_gvp_forward runs the GVP node / head kernels on full 64-row tiles for calls of >= 32 complexes (csrc/gvp.cu:
    the GPU is kept full by the call's sibling sub-batches then) and on 32-row tiles below.  It sees the CAPACITY of the
    bucket, so the rule rests on how plan_capacity rounds the batch: up to 22 real complexes (a single group, the GPU
    not full) stay below 32, groups of 25 of the 100-ligand headline reach it."""
    from keypoint_diffusion_b200 import ops
    from keypoint_diffusion_b200.utils import split_bounds
    gp = ops.GraphParams(ll_r=6.0, kl_k=7)
    for B in range(1, 23):
        assert ops.plan_capacity([20] * B, [20] * B, 322 * B, gp).key[0] < 32, B
    for B in range(23, 70):
        assert ops.plan_capacity([20] * B, [20] * B, 322 * B, gp).key[0] >= 32, B
    bd = split_bounds(100, 4)
    assert all(ops.plan_capacity([20] * (b - a), [20] * (b - a), 322 * (b - a), gp).key[0] >= 32 for a, b in zip(bd[:-1], bd[1:]))


def test_reference_arm_weights_equal_product_arm():
    """bench.py --impl reference rebuilds the seeded weights without importing the product package (no .so in that
    process); they must be the weights the product arm's model_from_config draws."""
    import os
    import bench
    from keypoint_diffusion_b200 import model_from_config
    for name in ("gvp_20kp", "egnn_all_atom"):
        cfg = bench.load_config(name)
        os.chdir(ROOT)
        torch.manual_seed(0)
        model = model_from_config(cfg)
        sd, arch, kw, rec_nf = bench.reference_state_dict(cfg)
        msd = {k: v for k, v in model.state_dict().items() if k.startswith("dynamics.")}
        assert set(sd) == set(msd) and rec_nf == model.n_kp_feat
        assert all(torch.equal(sd[k], msd[k]) for k in sd)


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the ligands of the last timed step as float32 arrays in the order the call returns them;
    above the size limit, the same seeded sample of atom rows every time, with its row indices."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(0)
    x, h = torch.randn(60, 3, generator=g), torch.randn(60, 10, generator=g)
    bench.dump_outputs(tmp_path / "weak", ([x[:40], x[40:]], [h[:40], h[40:]], [[20, 20], [20]]), strong=False)
    assert sorted(p.name for p in (tmp_path / "weak").iterdir()) == ["features.npy", "positions.npy"]
    pos, feat = np.load(tmp_path / "weak" / "positions.npy"), np.load(tmp_path / "weak" / "features.npy")
    assert pos.dtype == feat.dtype == np.float32 and np.array_equal(pos, x.numpy()) and np.array_equal(feat, h.numpy())
    samples = [{"positions": [x[:20], x[20:40]], "features": [h[:20], h[20:40]]},
               {"positions": [x[40:].double()], "features": [h[40:].double()]}]
    def size(run):
        return sum(p.stat().st_size for p in (tmp_path / run).iterdir())

    limit = 3 * bench.NPY_HEADER_BYTES + 25 * (13 * 4 + 8)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, samples, strong=True)
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 25 and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    pos = np.load(tmp_path / "a" / "positions.npy")
    assert pos.dtype == np.float32 and np.array_equal(pos, x.numpy()[rows.astype(np.int64)])
    assert size("a") <= limit
    # data that alone fills the limit is sampled too: the files, .npy headers included, stay within it
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 60 * 13 * 4)
    bench.dump_outputs(tmp_path / "c", samples, strong=True)
    assert (tmp_path / "c" / "rows.npy").exists() and size("c") <= 60 * 13 * 4


def test_bench_dump_dir_is_relative_to_the_callers_cwd(tmp_path, monkeypatch):
    """A relative --dump-outputs DIR is where the caller ran bench.py from, although build_model() changes into the
    repository root before the dump is written."""
    import bench
    monkeypatch.chdir(tmp_path)
    args = bench.parse_args(["--dump-outputs", "out"])
    monkeypatch.chdir(ROOT)
    bench.dump_outputs(args.dump_outputs, ([torch.zeros(2, 3)], [torch.zeros(2, 10)], [[2]]), strong=False)
    assert (tmp_path / "out" / "positions.npy").is_file() and not (ROOT / "out").exists()


def test_reference_arm_does_not_load_the_product_library():
    """The CPU arm must not dlopen libkpdiff_b200.so (the judge checks which .so files that process loaded)."""
    import subprocess
    import sys
    code = ("import sys, json; sys.argv=['bench.py','--impl','reference','--steps','1','--warmup','0','--cpu-steps','1',"
            "'--workload','egnn_20kp_c1']; import runpy; runpy.run_path('bench.py', run_name='__main__');"
            "maps=open('/proc/self/maps').read(); assert 'libkpdiff_b200' not in maps, 'product library loaded';"
            "assert not any(m.startswith('keypoint_diffusion_b200') for m in sys.modules), 'product package imported'")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
