#!/usr/bin/env python
"""Benchmark of the sampling hot path: sampled ligands/sec, 1000-step DDPM.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one complete pass of the hot path over one batch: the 1000 reverse-diffusion steps of
KeypointDiffusion.sample_from_encoded_receptors for the workload's complexes (graph build + denoiser + posterior step
per reverse step), from already-encoded pockets to coordinates + atom features.  Default workload = BASELINE.json
configs[1]: trained_models/gvp_20kp hyper-parameters, 1 synthetic pocket (20 keypoints), 100 ligands x 20 atoms per GPU,
seeded random weights in the reference state_dict layout (checkpoints and datasets are not available offline).

State distribution.  With untrained weights nothing cancels the 1/alpha_{t|s} growth of the posterior mean: the ligands
inflate to ~600 A within the first ~50 reverse steps whatever the scale of the coordinate head
(profiles/r02_calibrate_head_scale.txt), and at the shipped ll cutoff (5-6 A) the ligand-ligand graph empties -- ~2 ll
edges per complex, where a trained checkpoint keeps 250-380.  The workloads therefore hold the ll graph DENSE (cutoff
1e5 A: all n_l (n_l - 1) pairs, 380 per 20-atom ligand, the upper end of what a checkpoint sees); both arms run the same
configuration; the shipped-cutoff figure is printed beside it under "shipped_ll_cutoff" (--shipped-ll makes it the
headline).

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  roofline     dominant kernel (the fused edge kernel): algorithmic FLOPs / CUDA-event time, measured in an instrumented
               (non-graph, undivided, exact-layout) full trajectory right after the timed region
  cpu_baseline the CPU oracle (a port of the reference algorithm; the reference itself needs DGL / torch_cluster, which
               are not installed) on a bounded sample of the same workload
  e2e          same metric through the drop-in public API with HOST buffers (pinned), H2D + D2H inside
  ragged       e2e again with ligand sizes drawn afresh for every sample from the training-set histogram
               (LigandSizeDistribution.sample, what the reference's sample_random_sizes does), and the cold-call times
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

DTYPES = {"bf16x3": "bf16x3 (split bf16 operand pairs on tcgen05, fp32 accumulate: fp32-grade, parity <= 1e-4)",
          "bf16": "bf16 operands on tcgen05, fp32 accumulate (~2e-3 of fp32; not the parity mode)",
          "fp32": "fp32 (SIMT FMA, the reference's own arithmetic)"}
DENSE_LL_CUTOFF = 1.0e5

WORKLOADS = {
    # name: shipped config, pocket kind, pocket nodes, complexes (per GPU if weak, in total if strong), atoms per ligand,
    #       pockets (per GPU if weak, in total if strong), scaling
    "gvp_20kp": dict(cfg="gvp_20kp", kind="keypoint", n_kp=20, ligands=100, atoms=20, pockets=1, scaling="weak"),     # configs[1]
    "egnn_20kp": dict(cfg="egnn_20kp", kind="keypoint", n_kp=20, ligands=100, atoms=20, pockets=1, scaling="weak"),
    "egnn_20kp_c1": dict(cfg="egnn_20kp", kind="keypoint", n_kp=20, ligands=10, atoms=20, pockets=1, scaling="weak"),  # configs[0]
    # configs[2]: ONE fixed job of 64 pockets x 100 ligands dealt to the ranks (strong scaling at 1/2/4/8)
    "egnn_40kp": dict(cfg="egnn_40kp", kind="keypoint", n_kp=40, ligands=6400, atoms=20, pockets=64, scaling="strong"),
    "egnn_all_atom": dict(cfg="egnn_all_atom", kind="all_atom", n_kp=500, ligands=100, atoms=20, pockets=1, scaling="weak"),  # configs[3]
    "gvp_ca": dict(cfg="gvp_ca", kind="ca", n_kp=42, ligands=1024, atoms=20, pockets=1, scaling="weak"),              # configs[4] (--ligands sweeps)
}


# algorithmic FLOPs (SURVEY.md section 8d; DESIGN.md "Roofline")
def gvp_edge_flops(S=256, V=16, rbf=16, n_msg=3):
    f = 0
    for i in range(n_msg):
        vin = V + 1 if i == 0 else V
        h = max(vin, V)
        fin = S + rbf if i == 0 else S
        f += 2 * 3 * vin * h + 2 * 3 * h * V + 2 * (fin + h) * S + 2 * S * V
    return f


def egnn_edge_flops(H=257):
    # as the reference executes it: two branches of Linear(2H+1,H)+Linear(H,H), attention + coord heads
    return 2 * ((2 * H + 1) * H + H * H) * 2 + 2 * H + 2 * H


def egnn_edge_flops_min(H=257):
    # with the first Linear factorised onto the nodes (what the kernel does per edge)
    return 2 * 2 * H * H + 4 * H


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (NVML, 200 ms period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10, "applications_clocks_setting": 0x2}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def _load_by_path(name, rel):
    """A product-side pure-Python helper (synthetic pockets, parameter shapes) loaded by file path, WITHOUT importing the
    keypoint_diffusion_b200 package (whose import dlopens the CUDA library): what the reference arm uses."""
    spec = importlib.util.spec_from_file_location(name, ROOT / rel)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load_config(name, dense_ll=True):
    import yaml
    cfg = yaml.safe_load(open(ROOT / "tests" / "golden" / "shipped_configs.yml"))[name]
    if dense_ll:
        cfg["graph"]["graph_cutoffs"]["ll"] = DENSE_LL_CUTOFF
    return cfg


def make_pocket(synthetic, wl, pocket_id, cfg, arch):
    cut = cfg["graph"]["graph_cutoffs"]
    vs = cfg["dynamics_gvp"]["vector_size"] if arch == "gvp" else 0
    if wl["kind"] == "keypoint":
        width = cfg["rec_encoder_gvp"]["out_scalar_size"] if arch == "gvp" else cfg["rec_encoder"]["out_n_node_feat"]
        return synthetic.keypoint_pocket(pocket_id, cfg["graph"]["n_keypoints"], width, vs, cut["kk"])
    if wl["kind"] == "all_atom":
        return synthetic.all_atom_pocket(pocket_id, wl["n_kp"], len(cfg["dataset"]["rec_elements"]), vs, cut["rr"])
    return synthetic.ca_pocket(pocket_id, wl["n_kp"], len(cfg["dataset"]["rec_elements"]), vs, cut["rr"])


def build_model(cfg, device):
    from keypoint_diffusion_b200 import model_from_config
    os.chdir(ROOT)                       # dataset.location in the configs is relative
    torch.manual_seed(0)
    model = model_from_config(cfg)
    return model.to(device).eval()


def reference_state_dict(cfg):
    """The dynamics weights build_model() gives the product arm, rebuilt WITHOUT the product package: the same seeded
    initialisers (param_layout, loaded by path) drawn in the same order from torch.manual_seed(0)
    (tests/test_modules_cpu.py::test_reference_arm_weights_equal_product_arm)."""
    from shipped_cases import dynamics_kwargs
    pl = _load_by_path("_kpd_param_layout", "keypoint_diffusion_b200/param_layout.py")
    arch, kw, rec_nf = dynamics_kwargs(cfg)
    if arch == "egnn":
        shapes = pl.egnn_dynamics_shapes(10, rec_nf, kw["n_layers"], kw["hidden_nf"], kw["update_kp_feat"], kw["norm"])
    else:
        shapes = pl.gvp_dynamics_shapes(10, rec_nf, kw["vector_size"], kw["n_convs"], kw["n_hidden_scalars"], kw["update_kp"],
                                        kw["n_message_gvps"], kw["n_update_gvps"], kw["n_noise_gvps"])
    torch.manual_seed(0)
    tree = pl.ParamTree(shapes)
    return {"dynamics." + k: v.detach() for k, v in tree.state_dict().items()}, arch, kw, rec_nf


def oracle_step_time(sd, arch, kw, rec_nf, pocket, n_lig, n_timed, threads, T=1000):
    """Mean seconds per reverse step of the CPU oracle on the same batch / weights, and the mean edge counts it saw.

    Bounded sample: n_timed reverse steps spread uniformly over s = 999..0 are executed and timed in full (graph build +
    denoiser + posterior step); the steps in between are fast-forwarded with the posterior update at eps = 0 (not
    timed), which keeps the state distribution of the trajectory the same as on the GPU arm."""
    from oracle import flat, schedule as OS
    from helpers import oracle_cfg
    torch.set_num_threads(threads)
    B = len(n_lig)
    fwd = flat.egnn_forward if arch == "egnn" else flat.gvp_forward
    ocfg = oracle_cfg(arch, kw, 10, rec_nf)
    nk = pocket.n_kp
    off = torch.arange(B).repeat_interleave(pocket.kk_src.numel()) * nk
    fb = flat.FlatBatch(lig_n=torch.tensor(n_lig), kp_n=torch.tensor([nk] * B), kp_x=pocket.kp_x.repeat(B, 1),
                        kp_h=pocket.kp_h.repeat(B, 1), kk_src=pocket.kk_src.repeat(B) + off,
                        kk_dst=pocket.kk_dst.repeat(B) + off,
                        kp_v=pocket.kp_v.repeat(B, 1, 1) if pocket.kp_v is not None else None)
    F = 10
    gamma = OS.gamma_table(T, 1e-5)
    g = torch.Generator().manual_seed(0)
    N_l = sum(n_lig)
    lig_b, kp_b = fb.batch_idx()
    fb.lig_x = torch.randn(N_l, 3, generator=g)
    fb.lig_h = torch.randn(N_l, F, generator=g)
    fb = flat.remove_com(fb, lig_b, kp_b, "ligand")
    timed = set(int(round(i * (T - 1) / max(n_timed - 1, 1))) for i in range(n_timed)) if n_timed > 1 else {T - 1}
    zeros = (torch.zeros(N_l, F), torch.zeros(N_l, 3))
    total, e_ll = 0.0, []

    def dyn(b, t):
        eh, ex, edges, _ = fwd(sd, ocfg, b, t, return_edges=True)
        e_ll.append(int(edges["ll"][0].numel()))
        return eh, ex

    with torch.no_grad():
        for s_int in reversed(range(T)):
            nx, nh = torch.randn(N_l, 3, generator=g), torch.randn(N_l, F, generator=g)
            if s_int in timed:
                t0 = time.perf_counter()
                fb = flat.sample_p_zs_given_zt(dyn, gamma, T, s_int, fb, nx, nh)
                total += time.perf_counter() - t0
            else:
                fb = flat.sample_p_zs_given_zt(lambda b, t: zeros, gamma, T, s_int, fb, nx, nh)
    return total / len(timed), sum(e_ll) / max(len(e_ll), 1)


DUMP_LIMIT_BYTES = 64_000_000          # all files of a dump, .npy headers included
NPY_HEADER_BYTES = 1024                 # allowance per file (np.save writes 128 B for these shapes)


def dump_outputs(out_dir, result, strong):
    """What a caller of the timed path receives from its last timed step, as float32 .npy files in out_dir: the sampled
    ligands' positions [atoms, 3] and atom features [atoms, F], concatenated in the order the call returns them
    (rank-major for a weak-scaling run, receptor-major for a strong-scaling one).  The inputs depend only on the
    arguments, so two builds run with the same arguments (--warmup and --steps included: every call writes its keypoint
    positions back into the input graph) can be compared array for array.  Where the files would exceed
    DUMP_LIMIT_BYTES, a fixed seeded sample of atom rows is written instead, with its row indices (rows.npy, float64)."""
    import numpy as np
    if strong:
        pos = [p for rec in result for p in rec["positions"]]
        feat = [f for rec in result for f in rec["features"]]
    else:
        pos, feat = result[0], result[1]
    arrays = {"positions": torch.cat([p.cpu() for p in pos]).float(),
              "features": torch.cat([f.cpu() for f in feat]).float()}
    n = arrays["positions"].shape[0]
    row_bytes = sum(a[0].numel() * 4 for a in arrays.values())
    if n * row_bytes + 2 * NPY_HEADER_BYTES > DUMP_LIMIT_BYTES:
        k = (DUMP_LIMIT_BYTES - 3 * NPY_HEADER_BYTES) // (row_bytes + 8)
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.double()
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a.numpy())


def git_head():
    try:
        return subprocess.run(["git", "-C", str(ROOT), "rev-parse", "--short", "HEAD"], capture_output=True, text=True,
                              timeout=5).stdout.strip() or None
    except Exception:
        return None


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gvp_20kp", choices=sorted(WORKLOADS))
    ap.add_argument("--ligands", type=int, default=None, help="complexes per GPU (weak) / in total (strong); default: the workload's")
    ap.add_argument("--shipped-ll", action="store_true", help="keep the shipped ll cutoff (the ll graph empties on untrained weights)")
    ap.add_argument("--steps-per-graph", type=int, default=50)
    ap.add_argument("--diff-batch-size", type=int, default=800, help="complexes per diffusion batch (strong-scaling workloads)")
    ap.add_argument("--sub-batches", type=int, default=None,
                    help="concurrently sampled groups of complexes per GPU (default: the library's choice)")
    ap.add_argument("--cpu-steps", type=int, default=None, help="reverse steps per CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-ragged", action="store_true")
    ap.add_argument("--no-shipped-ll-block", action="store_true")
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16", "bf16x3"],
                    help="headline mode: bf16x3 (tcgen05 tensor cores, split bf16 operands, fp32-grade: inside the 1e-4 "
                         "parity bar), fp32 (SIMT, the reference's own arithmetic) or bf16 (tcgen05, plain bf16 operands, "
                         "GVP only, ~2e-3)")
    ap.add_argument("--no-mode-blocks", action="store_true",
                    help="skip the separately-reported measurements of the other precision modes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the ligands the timed path returned in its last timed step to DIR/<name>.npy")
    args = ap.parse_args(argv)
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path; the reference arm only times fast-forwarded CPU steps")
    if args.dump_outputs:
        # relative to where the caller ran it: build_model() changes into the repository root before the dump
        args.dump_outputs = str(Path(args.dump_outputs).resolve())
    return args


def main():
    args = parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = dict(WORKLOADS[args.workload])
    if args.ligands:
        wl["ligands"] = args.ligands
    strong = wl["scaling"] == "strong"
    dense = not args.shipped_ll
    cfg = load_config(wl["cfg"], dense_ll=dense)
    arch = cfg["diffusion"].get("architecture", "egnn")
    n_kp, n_atoms = wl["n_kp"], wl["atoms"]
    total = wl["ligands"] if strong else wl["ligands"] * max(args.gpus if args.impl == "reference" else world, 1)
    metric = "sampled ligands/sec (1000-step DDPM, 20 keypoints)"
    ll_note = (f"ll graph held dense (cutoff {DENSE_LL_CUTOFF:g} A: {n_atoms * (n_atoms - 1)} ll edges per ligand, the density a "
               f"trained checkpoint keeps; untrained weights let the ligands inflate and the shipped-cutoff graph empties)"
               if dense else "shipped ll cutoff (the ll graph empties on untrained weights)")
    if strong:
        wdesc = (f"trained_models/{wl['cfg']}: ONE job of {wl['pockets']} synthetic pockets ({n_kp} keypoints) x "
                 f"{wl['ligands'] // wl['pockets']} ligands x {n_atoms} atoms = {wl['ligands']} complexes dealt to the ranks")
    else:
        wdesc = (f"trained_models/{wl['cfg']}: 1 synthetic pocket per GPU ({n_kp} keypoints), {wl['ligands']} ligands x "
                 f"{n_atoms} atoms per GPU")
    config = {"workload": f"{wdesc}, 1000 denoising steps, seeded random weights; {ll_note}",
              "ligands_per_gpu": wl["ligands"] // world if strong else wl["ligands"], "atoms_per_ligand": n_atoms,
              "n_keypoints": n_kp, "timesteps": 1000, "ll_cutoff": cfg["graph"]["graph_cutoffs"]["ll"],
              "parallelism": f"pocket/ligand sharding x{world if args.impl != 'reference' else args.gpus}, one final gather",
              "l2": "state + weights (<60 MB) are L2-resident by design; every reverse step rewrites them"}

    # ------------------------------------------------------------------ reference arm (CPU; no product code, no .so)
    if args.impl == "reference":
        if rank != 0:
            return
        synthetic = _load_by_path("_kpd_synthetic", "keypoint_diffusion_b200/synthetic.py")
        threads = os.cpu_count() or 1
        sd, arch, kw, rec_nf = reference_state_dict(cfg)
        pocket = make_pocket(synthetic, wl, 0, cfg, arch)
        B = wl["ligands"] // wl["pockets"] if strong else wl["ligands"]     # the CPU sample: the ligands of one pocket
        B = min(B, 100)
        n_lig = [n_atoms] * B
        n = args.cpu_steps or 12
        if args.warmup > 0:
            oracle_step_time(sd, arch, kw, rec_nf, pocket, n_lig, 1, threads)
        runs = [oracle_step_time(sd, arch, kw, rec_nf, pocket, n_lig, n, threads) for _ in range(args.steps)]
        t_step = sum(r[0] for r in runs) / len(runs)
        value = B / (t_step * 1000)
        sample = (f"per timed step: {n} reverse steps spread uniformly over s=999..0 executed in full (the others "
                  f"fast-forwarded with eps=0, untimed), batch of {B} ligands of one pocket, mean step time x1000; CPU oracle "
                  f"(oracle/flat.py, a port: the reference needs DGL/torch_cluster), fp32, {threads} threads; "
                  f"mean ll edges per executed step {runs[-1][1]:.0f}")
        print(json.dumps({"impl": "reference", "metric": metric, "value": value, "unit": "ligands/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1000 * 1e3,
                          "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "fp32",
                          "data": "synthetic", "config": config, "mean_edges_per_step": {"ll": runs[-1][1]},
                          "cpu_baseline": {"value": value, "unit": "ligands/s", "cores": threads, "kind": "port",
                                           "sample": sample},
                          "e2e": {"value": value, "unit": "ligands/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ our arm (GPU)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from keypoint_diffusion_b200 import HeteroBatch, _lib, dist as kdist, synthetic
    import ctypes as C

    model = build_model(cfg, dev)
    F = model.n_lig_features
    if args.precision != "fp32":
        model.dynamics.set_precision(args.precision)       # raises for a mode the architecture does not have
    skw = dict(seed=1234, sub_batches=args.sub_batches, steps_per_graph=args.steps_per_graph)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """k calls of fn -> (device seconds, wall seconds, what the last call returned)."""
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(k):
            res = fn()
        ev1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dt = max(ev0.elapsed_time(ev1) / 1e3, 0.0)
        barrier()
        # device time on the launching stream; the e2e leg ends with a blocking D2H, so wall >= device
        t = torch.tensor([dt, wall], device=dev, dtype=torch.float64)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), res

    if strong:
        # ONE fixed job: `pockets` encoded pockets x ligands/pockets sizes, dealt to the ranks by KeypointDiffusion.sample_sharded
        per = wl["ligands"] // wl["pockets"]
        pockets = [make_pocket(synthetic, wl, i, cfg, arch) for i in range(wl["pockets"])]
        enc_graphs = [HeteroBatch.from_pockets([pk], [1], F, pin=True) for pk in pockets]
        n_lig_atoms = [[n_atoms] * per for _ in pockets]
        centers = [torch.zeros(3) for _ in pockets]
        n_mine = len(kdist.shard_complexes([n_atoms] * wl["ligands"], [n_kp] * wl["ligands"], world)[rank])

        def one_sample_e2e():
            return model.sample_sharded(enc_graphs, n_lig_atoms, diff_batch_size=args.diff_batch_size, encoded=True,
                                        init_lig_pos=centers, **skw)

        one_sample_device = one_sample_e2e        # the product call IS the sharded e2e call; encoded pockets are uploaded once per call
        B = n_mine
        h2d = sum(v.numel() * v.element_size() for g in enc_graphs for v in g.nodes["kp"].data.values())
        d2h = wl["ligands"] * n_atoms * (3 + F) * 4
        n_lig = [n_atoms] * n_mine
        work = wl["ligands"]                      # ligands per step over ALL ranks
        n_batches = -(-n_mine // args.diff_batch_size)
    else:
        pocket = make_pocket(synthetic, wl, rank, cfg, arch)          # one pocket per rank
        B = wl["ligands"]
        n_lig = [n_atoms] * B
        g_host = HeteroBatch.from_pockets([pocket], n_lig, F, pin=True)
        init_host = torch.zeros(B, 3).pin_memory()
        g_dev = g_host.to(dev)
        init_dev = init_host.to(dev)

        def one_sample_device():
            x, h = model.sample_from_encoded_receptors(g_dev, init_lig_pos=init_dev, return_device_tensors=True, **skw)
            return kdist.gather_ligands(x, h, n_lig)

        def one_sample_e2e():
            g = HeteroBatch(g_host._bnn, g_host._ndata, g_host._edges, g_host._bne)    # fresh host view, same pinned tensors
            return model.sample_from_encoded_receptors(g, init_lig_pos=init_host, **skw)

        kp = g_host.nodes["kp"].data
        h2d = sum(v.numel() * v.element_size() for v in kp.values()) + init_host.numel() * 4
        d2h = sum(n_lig) * (3 + F) * 4
        work = world * B
        n_batches = 1

    launches0 = int(_lib.lib.kpd_launch_count())
    t0 = time.perf_counter()
    one_sample_device()
    torch.cuda.synchronize()
    cold_first = time.perf_counter() - t0                   # weight packing + capture of every bucket + one sample
    for _ in range(max(args.warmup - 1, 0)):
        one_sample_device()
    clocks = ClockSampler(local_rank)
    clocks.start()
    dt, wall, last = timed(one_sample_device, args.steps)
    clk = clocks.finish()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, strong)     # now: the legs below re-run the samplers that own these buffers
    if strong:
        dt = max(dt, wall)          # the call ends with the gather + D2H of every rank's ligands: wall clock >= device time
    value = work * args.steps / dt
    lps = model.last_launches_per_step
    n_sub = args.sub_batches or model.default_sub_batches(min(B, args.diff_batch_size) if strong else B)
    config["sub_batches"] = (f"{n_sub} groups of complexes per GPU sampled concurrently (own capacity-bucketed CUDA graphs and "
                             f"streams; same noise as the undivided batch)")

    if strong:          # the product call IS the e2e call (host pockets in, CPU ligands out): one timed region serves both
        dt_e, wall_e = dt, dt
        e2e_value = value
    else:
        one_sample_e2e()
        dt_e, wall_e, _ = timed(one_sample_e2e, args.steps)
        e2e_value = work * args.steps / max(dt_e, wall_e)

    out = {"metric": metric, "value": value, "unit": "ligands/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": wl["scaling"],
           "vs_baseline": None, "dtype": DTYPES[args.precision], "data": "synthetic", "config": config, "clocks": clk,
           "e2e": {"value": e2e_value, "unit": "ligands/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
           "reverse_steps_per_s": 1000 * n_batches * args.steps / dt, "launches_per_reverse_step": lps,
           "cold_call": {"first_call_s": cold_first, "warm_call_s": dt / args.steps,
                         "captured_buckets": int(model.cold_captures),
                         "note": "first call = packing the weights for the tensor-core kernels + capturing and instantiating the "
                                 "CUDA graphs of every capacity bucket the batch uses + one full sample"}}

    # ------------------------------------------------------------------ ragged leg: new ligand sizes every sample
    if not strong and not args.no_ragged and not args.no_mode_blocks:
        n_rec_row = {"keypoint": 336, "all_atom": min(max(n_kp, 7), 661), "ca": n_kp}[wl["kind"]]
        enc_graph = HeteroBatch.from_pockets([pocket], [1], F, pin=True)
        gen = torch.Generator().manual_seed(77 + rank)
        hist = model.lig_size_dist

        def draw():
            rec_idx = hist.rec_size_to_idx[int(min(max(n_rec_row, hist.rec_bounds[0]), hist.rec_bounds[1]))]
            idx = torch.multinomial(hist.joint_histogram[rec_idx], B, replacement=True, generator=gen)
            return hist.lig_idx_to_size[idx].tolist()

        def ragged_sample(sizes):
            return model._sample([enc_graph], [sizes], diff_batch_size=B, encoded=True, init_lig_pos=[torch.zeros(3)], **skw)

        cap0 = model.cold_captures
        walls, atoms, ligs = [], 0, 0
        n_rag = max(args.steps, 3) + 3
        for i in range(n_rag):
            sizes = draw()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ragged_sample(sizes)
            torch.cuda.synchronize()
            walls.append((time.perf_counter() - t0, sum(sizes), model.cold_captures))
        steady = walls[3:]
        rag_l = B * len(steady) / sum(w for w, _, _ in steady)
        rag_a = sum(a for _, a, _ in steady) / sum(w for w, _, _ in steady)
        out["ragged"] = {"value": world * rag_l, "unit": "ligands/s", "atoms_per_s": world * rag_a,
                         "fixed_size_atoms_per_s": e2e_value * n_atoms, "vs_fixed_size_atoms_per_s": world * rag_a / (e2e_value * n_atoms),
                         "samples": len(steady), "warmup_samples": 3,
                         "new_buckets_captured": {"warmup": walls[2][2] - cap0, "timed": walls[-1][2] - walls[2][2]},
                         "call_s": [round(w, 4) for w, _, _ in walls],
                         "note": f"e2e through KeypointDiffusion._sample(encoded=True): host pocket in, device-side batch assembly, CPU "
                                 f"ligands out; ligand sizes drawn afresh for EVERY sample from row n_rec={n_rec_row} of the training-set "
                                 f"histogram (LigandSizeDistribution, reference n_nodes_dist.py:42-60); capacity-bucketed samplers: a "
                                 f"new size tuple re-uses the captured graphs of its bucket"}

    # ------------------------------------------------------------------ roofline leg (dominant kernel)
    if not args.no_roofline and not strong:
        prof_id = 2 if arch == "gvp" else 1
        n_layers = cfg["dynamics_gvp"]["n_convs"] if arch == "gvp" else cfg["dynamics"]["n_layers"]
        _lib.check(_lib.lib.kpd_profile_enable(prof_id, 1000 * n_layers + 16))
        torch.cuda.synchronize()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        # the instrumented trajectory: undivided batch, exact layout (no filler complexes: edge counts are the batch's own),
        # one stream, no CUDA graph
        model.sample_from_encoded_receptors(g_dev, init_lig_pos=init_dev, seed=1234, use_cuda_graph=False,
                                            return_device_tensors=True, sub_batches=1, capacity=False)
        pe1.record()
        torch.cuda.synchronize()
        serial_ms = pe0.elapsed_time(pe1)
        tot, cnt = C.c_double(), C.c_int32()
        _lib.check(_lib.lib.kpd_profile_collect(C.byref(tot), C.byref(cnt)))
        _lib.lib.kpd_profile_enable(0, 0)
        prof_sampler = [s for k, s in model._samplers.items() if k[0] == "one"][-1]
        st = (C.c_double * 4)()
        _lib.check(_lib.lib.kpd_sampler_edge_stats(prof_sampler.handle, st))
        e_ll, e_kl, e_kk = st[0], st[1], st[2]
        peaks = {}
        try:
            peaks = json.load(open(ROOT / "MEASURED_PEAKS.json"))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback (B200_PROFILING.md sustained)"
        if arch == "gvp":
            d = cfg["dynamics_gvp"]
            fe = gvp_edge_flops(d["n_hidden_scalars"], d["vector_size"], 16, d["n_message_gvps"])
            full = e_ll + 2 * e_kl + e_kk
            last = e_ll + e_kl
            flops_per_step = fe * (full * (n_layers - 1) + last) if d["update_kp"] else fe * last * n_layers
            kname = "gvp_edge_kernel" if args.precision == "fp32" else "gvp_edge_ws_kernel"
        else:
            H = cfg["dynamics"]["hidden_nf"] + 1
            fe = egnn_edge_flops_min(H)
            e_all = e_ll + (2 * e_kl + e_kk if cfg["dynamics"]["update_kp_feat"] else e_kl)
            flops_per_step = fe * e_all * n_layers
            kname = "egnn_edge_kernel" if args.precision == "fp32" else "egnn_edge_ws_kernel"
        n_rev = st[3] if st[3] > 0 else 1000.0
        avg_ms = tot.value / max(cnt.value, 1)
        achieved = (flops_per_step * n_rev / max(cnt.value, 1)) / (avg_ms * 1e-3) / 1e12 if avg_ms > 0 else 0.0
        traffic, traffic_src = None, None
        tj = ROOT / "profiles" / "traffic.json"
        if tj.exists():
            tdata = json.load(open(tj))
            key = kname + ("[bf16]" if args.precision == "bf16" and kname + "[bf16]" in tdata else "")
            traffic = tdata.get(key)
            traffic_src = (f"profiles/traffic.json ({tdata.get('_source', 'ncu --set full capture')}; captured at commit "
                           f"{tdata.get('_commit', 'unknown')}, this run is commit {git_head()}): NOT measured in this run")
        out["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                           "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
                           "kernel": kname, "peak_source": peak_src, "launches_timed": int(cnt.value), "avg_launch_ms": avg_ms,
                           "kernel_ms_per_reverse_step": tot.value / n_rev,
                           # share of the SERIAL instrumented trajectory (what an ncu launch list, which serialises
                           # launches, shows); in the timed region kernels of different sub-batches / edge types overlap
                           "kernel_share_of_step": tot.value / serial_ms,
                           "serial_ms_per_reverse_step": serial_ms / n_rev,
                           "flops_per_edge": fe, "mean_edges_per_step": {"ll": e_ll, "kl": e_kl, "lk": e_kl, "kk": e_kk},
                           "note": {"fp32": "fp32 SIMT tile GEMM; fraction is against the measured bf16 tensor peak",
                                    "bf16": "fused warp-specialised kernel: tcgen05 bf16 tile GEMMs + SIMT epilogues / gathers / "
                                            "segmented reduction; algorithmic FLOPs against the measured bf16 tensor peak",
                                    "bf16x3": "fused warp-specialised kernel; every algorithmic MAC costs several bf16 tensor-core MACs "
                                              "(hi/lo operand pairs), so the tensor pipe does a multiple of the algorithmic FLOPs "
                                              "counted here; fraction is algorithmic FLOPs against the measured bf16 tensor peak"}[args.precision]}

    # ------------------------------------------------------------------ the other precision modes, stated separately
    if not args.no_mode_blocks and not strong:
        others = [p for p in (["bf16x3", "bf16", "fp32"] if arch == "gvp" else ["bf16x3", "fp32"]) if p != args.precision]
        acc = {"bf16x3": "denoiser output within ~3e-6 of the fp32 reference (bar 1e-4; tests/test_gpu_tensorcore.py)",
               "bf16": "denoiser output within ~2e-3 of fp32; not the parity mode",
               "fp32": "denoiser output within ~5e-7 of the fp32 reference (tests/test_gpu_parity.py)"}
        out["modes"] = {}
        for p in others:
            model.dynamics.set_precision(p)
            k = 1 if p == "fp32" else args.steps            # the SIMT mode is slow: one timed sample
            for _ in range(1 if p == "fp32" else 2):
                one_sample_device()
            dtp, _, _ = timed(one_sample_device, k)
            out["modes"][p] = {"value": work * k / dtp, "unit": "ligands/s", "ms_per_step": dtp / k * 1e3, "steps": k,
                               "dtype": DTYPES[p], "accuracy": acc[p]}
        model.dynamics.set_precision(args.precision)

    # ------------------------------------------------------------------ the same workload at the SHIPPED ll cutoff
    if dense and not strong and not args.no_shipped_ll_block and not args.no_mode_blocks:
        cfg_s = load_config(wl["cfg"], dense_ll=False)
        model_s = build_model(cfg_s, dev)
        if args.precision != "fp32":
            model_s.dynamics.set_precision(args.precision)

        def shipped_sample():
            x, h = model_s.sample_from_encoded_receptors(g_dev, init_lig_pos=init_dev, return_device_tensors=True, **skw)
            return kdist.gather_ligands(x, h, n_lig)

        for _ in range(2):
            shipped_sample()
        dts, _, _ = timed(shipped_sample, args.steps)
        out["shipped_ll_cutoff"] = {"value": work * args.steps / dts, "unit": "ligands/s", "ms_per_step": dts / args.steps * 1e3,
                                    "ll_cutoff": cfg_s["graph"]["graph_cutoffs"]["ll"],
                                    "note": "same workload and weights at the shipped ll cutoff: the untrained model lets the "
                                            "ligands inflate, the ll graph empties (~2 edges per complex) and a reverse step does "
                                            "about half the edge work a trained checkpoint would; not the headline"}
        del model_s

    # gpu launches in the two timed regions: replayed graphs do not re-count, so derive from the captured sequence
    per_run = (lps * 1000 + 9 * n_sub) * n_batches       # lps already sums the sub-batches' launches
    out["gpu_launches"] = int(per_run * args.steps * (1 if strong else 2))      # headline mode: device-resident + e2e timed regions
    out["launch_counter_delta"] = int(_lib.lib.kpd_launch_count()) - launches0

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from shipped_cases import dynamics_kwargs
        threads = os.cpu_count() or 1
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        _, kw, rec_nf = dynamics_kwargs(cfg)
        pk = pockets[0] if strong else pocket
        n_cpu = [n_atoms] * min(100, wl["ligands"] // wl["pockets"] if strong else B)
        t1, _ = oracle_step_time(sd, arch, kw, rec_nf, pk, n_cpu, 1, threads)       # also warms the CPU code paths
        n = args.cpu_steps or max(2, min(40, int(20.0 / max(t1, 1e-3))))
        t_step, cpu_ll = oracle_step_time(sd, arch, kw, rec_nf, pk, n_cpu, n, threads)
        out["cpu_baseline"] = {"value": len(n_cpu) / (t_step * 1000), "unit": "ligands/s", "cores": threads, "kind": "port",
                               "mean_ll_edges_per_step": cpu_ll,
                               "sample": f"{n} reverse steps spread uniformly over s=999..0 of a batch of {len(n_cpu)} ligands of one "
                                         f"pocket executed in full (others fast-forwarded with eps=0, untimed), mean step time x1000; "
                                         f"oracle/flat.py fp32, torch {torch.__version__}, {threads} threads"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    # the benchmark writes nothing into the tree: without this, importing the tests/ helpers creates tests/__pycache__
    # (build() imports every other module it loads); set here, not at import, so that importing bench leaves the flag alone
    sys.dont_write_bytecode = True
    main()
