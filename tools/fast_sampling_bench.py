"""Throughput of fewer-step sampling on the headline workloads.

For gvp_20kp and egnn_20kp as bench.py builds them (one synthetic 20-keypoint pocket, 100 ligands x 20 atoms, dense ll
graph, seeded random weights, bf16x3) it times full KeypointDiffusion.sample_from_encoded_receptors calls: the plain
1000-step call, the same call with timesteps = 25, 50, 100, 250, 500 and 1000 (strided ancestral steps), and with
timesteps = 100 at eta = 0 (DDIM).  steps_per_graph is 50, so every timesteps value except 25 runs whole graph replays;
25 is below steps_per_graph and runs every step as eager launches.  A least-squares line through the all-replay points
gives a fixed cost per call and a cost per captured step; the 25-step call, less that fixed cost, gives the cost per
eager step.  Device time on the launching stream (CUDA events), warm capacity buckets, outputs left on the device.
Prints one JSON line per workload (and writes them to --out), with cold_captures (capacity buckets captured over all
variants) and the card's name and power limit read in the same run.

    python tools/fast_sampling_bench.py --out profiles/r06_fast_sampling_bench.jsonl

--solvers times the second-order solver instead (DESIGN.md section 6.5): DDIM eta = 0 (ddim0_n) and DPM-Solver++(2M)
(2m_n) calls at timesteps = 10, 20, 25, 50 and 100 with steps_per_graph 50, and at 10 and 20 with steps_per_graph = n
(suffix _spg), the two solvers alternating in one loop.  It also reports, for information only, the RMS distance of each
call's positions to a 1000-step DDIM eta = 0 call from the same seed (seeded random weights: not a sample-quality claim).

    python tools/fast_sampling_bench.py --solvers --out profiles/r09_multistep_bench.jsonl
"""
import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import bench  # noqa: E402
from inpaint_bench import card  # noqa: E402

TIMESTEPS = (25, 50, 100, 250, 500, 1000)
STEPS_PER_GRAPH = 50


def run_workload(name, steps, warmup):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    wl = bench.WORKLOADS[name]
    dev = torch.device("cuda:0")
    cfg = bench.load_config(wl["cfg"], dense_ll=True)
    arch = cfg["diffusion"].get("architecture", "egnn")
    model = bench.build_model(cfg, dev)
    model.dynamics.set_precision("bf16x3")
    F = model.n_lig_features
    pocket = bench.make_pocket(synthetic, wl, 0, cfg, arch)
    B, n_at = wl["ligands"], wl["atoms"]
    g = HeteroBatch.from_pockets([pocket], [n_at] * B, F, pin=True)   # host graph: inputs identical for every call
    init = torch.zeros(B, 3).pin_memory()
    variants = {"plain": {}}
    for n in TIMESTEPS:
        variants[f"n_{n}"] = dict(timesteps=n)
    variants["ddim0_100"] = dict(timesteps=100, eta=0.0)
    res = {"workload": f"{name}: {B} ligands x {n_at} atoms, 1 pocket ({wl['n_kp']} keypoints), dense ll, bf16x3, "
                       f"seeded random weights, steps_per_graph {STEPS_PER_GRAPH}; plain = 1000 steps, n_k = k strided "
                       f"ancestral steps, ddim0_100 = 100 DDIM steps at eta 0", "ligands_per_s": {}, "ms_per_call": {},
           "speedup_vs_plain": {}}
    ms = {}
    for tag, kw in variants.items():
        call = lambda: model.sample_from_encoded_receptors(g, init_lig_pos=init, seed=1234, return_device_tensors=True,
                                                           steps_per_graph=STEPS_PER_GRAPH, **kw)
        for _ in range(warmup):
            call()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            call()
        ev1.record()
        torch.cuda.synchronize()
        ms[tag] = ev0.elapsed_time(ev1) / steps
        res["ligands_per_s"][tag] = round(B / (ms[tag] / 1e3), 2)
        res["ms_per_call"][tag] = round(ms[tag], 2)
    for tag in variants:
        res["speedup_vs_plain"][tag] = round(ms["plain"] / ms[tag], 3)
    pts = [(n, ms[f"n_{n}"]) for n in TIMESTEPS if n % STEPS_PER_GRAPH == 0]
    xs = torch.tensor([float(n) for n, _ in pts], dtype=torch.float64)
    ys = torch.tensor([v for _, v in pts], dtype=torch.float64)
    per_step = float(((xs - xs.mean()) * (ys - ys.mean())).sum() / ((xs - xs.mean()) ** 2).sum())
    fixed = float(ys.mean()) - per_step * float(xs.mean())
    resid = float((ys - (fixed + per_step * xs)).abs().max())
    eager = (ms["n_25"] - fixed) / 25
    res["fit"] = {"points": [n for n, _ in pts], "fixed_ms_per_call": round(fixed, 3),
                  "captured_ms_per_step": round(per_step, 4), "max_residual_ms": round(resid, 3),
                  "eager_ms_per_step": round(eager, 4), "eager_over_captured": round(eager / per_step, 3)}
    res["cold_captures"] = model.cold_captures
    return res


SOLVER_STEPS = (10, 20, 25, 50, 100)


def _timed(call, steps, warmup):
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        call()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps


def run_solver_sweep(name, steps, warmup):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    wl = bench.WORKLOADS[name]
    dev = torch.device("cuda:0")
    cfg = bench.load_config(wl["cfg"], dense_ll=True)
    arch = cfg["diffusion"].get("architecture", "egnn")
    model = bench.build_model(cfg, dev)
    model.dynamics.set_precision("bf16x3")
    F = model.n_lig_features
    pocket = bench.make_pocket(synthetic, wl, 0, cfg, arch)
    B, n_at = wl["ligands"], wl["atoms"]
    g = HeteroBatch.from_pockets([pocket], [n_at] * B, F, pin=True)
    init = torch.zeros(B, 3).pin_memory()
    variants = {}
    for n in SOLVER_STEPS:
        variants[f"ddim0_{n}"] = dict(timesteps=n, eta=0.0, steps_per_graph=STEPS_PER_GRAPH)
        variants[f"2m_{n}"] = dict(timesteps=n, solver="dpmpp_2m", steps_per_graph=STEPS_PER_GRAPH)
    for n in (10, 20):
        variants[f"ddim0_{n}_spg"] = dict(timesteps=n, eta=0.0, steps_per_graph=n)
        variants[f"2m_{n}_spg"] = dict(timesteps=n, solver="dpmpp_2m", steps_per_graph=n)

    def call(kw):
        return model.sample_from_encoded_receptors(g, init_lig_pos=init, seed=1234, return_device_tensors=True, **kw)
    ref, _ = call(dict(timesteps=1000, eta=0.0, steps_per_graph=STEPS_PER_GRAPH))
    ref = ref.clone()
    res = {"workload": f"{name}: {B} ligands x {n_at} atoms, 1 pocket ({wl['n_kp']} keypoints), dense ll, bf16x3, "
                       f"seeded random weights; ddim0_n = n DDIM eta 0 steps, 2m_n = n DPM-Solver++(2M) steps, "
                       f"steps_per_graph {STEPS_PER_GRAPH} (_spg: steps_per_graph = n)", "ms_per_call": {},
           "ligands_per_s": {}, "pos_rms_to_ddim1000": {}}
    for tag, kw in variants.items():
        ms = _timed(lambda: call(kw), steps, warmup)
        x, _ = call(kw)
        res["ms_per_call"][tag] = round(ms, 2)
        res["ligands_per_s"][tag] = round(B / (ms / 1e3), 2)
        res["pos_rms_to_ddim1000"][tag] = round(float((x - ref).pow(2).sum(1).mean().sqrt()), 4)
    res["cold_captures"] = model.cold_captures
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", nargs="+", default=["gvp_20kp", "egnn_20kp"], choices=["gvp_20kp", "egnn_20kp"])
    ap.add_argument("--steps", type=int, default=5, help="timed calls per variant")
    ap.add_argument("--warmup", type=int, default=1, help="untimed calls per variant (the first one captures)")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--solvers", action="store_true", help="time DDIM eta = 0 against DPM-Solver++(2M) instead")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 1:
        ap.error("--steps and --warmup must be >= 1 (the warm-up call captures the graphs)")
    if args.out:        # relative to where the caller ran it: build_model() changes into the repository root
        args.out = str(Path(args.out).resolve())
    if not torch.cuda.is_available():
        raise SystemExit("fast_sampling_bench.py needs a CUDA device")
    lines = []
    for name in args.workloads:
        r = (run_solver_sweep if args.solvers else run_workload)(name, args.steps, args.warmup)
        r.update(card())
        r["steps"], r["warmup"] = args.steps, args.warmup
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
