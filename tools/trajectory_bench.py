"""Cost of recording trajectories (visualize=True) on the headline workloads.

For gvp_20kp and egnn_20kp as bench.py builds them (one synthetic 20-keypoint pocket, 100 ligands x 20 atoms, dense ll
graph, seeded random weights, bf16x3, 1000 steps, steps_per_graph 50) it times full
KeypointDiffusion.sample_from_encoded_receptors calls in three variants: plain, visualize with frame_every = 1 and
visualize with frame_every = 10.  Two numbers per variant:

* device ms per call: CUDA events on the launching stream, outputs (and frames) left on the device;
* wall ms per call: host clock around calls that return CPU tensors, frames included, ending in a synchronise.

The variants alternate over --rounds rounds of --steps calls each; the median round is reported, with the overhead
against plain and the bytes of frames a call writes.  Prints one JSON line per workload (and writes them to --out), with
the card's name and power limit read in the same run.

    python tools/trajectory_bench.py --out profiles/r08_trajectory_bench.jsonl
"""
import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import bench  # noqa: E402
from inpaint_bench import card  # noqa: E402

STEPS_PER_GRAPH = 50
VARIANTS = {"plain": {}, "visualize_k1": dict(visualize=True), "visualize_k10": dict(visualize=True, frame_every=10)}


def run_workload(name, steps, warmup, rounds):
    from keypoint_diffusion_b200 import HeteroBatch, synthetic
    wl = bench.WORKLOADS[name]
    dev = torch.device("cuda:0")
    cfg = bench.load_config(wl["cfg"], dense_ll=True)
    arch = cfg["diffusion"].get("architecture", "egnn")
    model = bench.build_model(cfg, dev)
    model.dynamics.set_precision("bf16x3")
    F, T = model.n_lig_features, model.n_timesteps
    pocket = bench.make_pocket(synthetic, wl, 0, cfg, arch)
    B, n_at = wl["ligands"], wl["atoms"]
    g = HeteroBatch.from_pockets([pocket], [n_at] * B, F, pin=True)   # host graph: inputs identical for every call

    def call(kw, device):
        return model.sample_from_encoded_receptors(g, init_lig_pos=torch.zeros(B, 3), seed=1234,
                                                   return_device_tensors=device, steps_per_graph=STEPS_PER_GRAPH, **kw)

    for kw in VARIANTS.values():
        for _ in range(warmup):
            call(kw, True)
    torch.cuda.synchronize()
    dev_ms = {tag: [] for tag in VARIANTS}
    wall_ms = {tag: [] for tag in VARIANTS}
    for _ in range(rounds):
        for tag, kw in VARIANTS.items():
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(steps):
                call(kw, True)
            ev1.record()
            torch.cuda.synchronize()
            dev_ms[tag].append(ev0.elapsed_time(ev1) / steps)
            t0 = time.perf_counter()
            for _ in range(steps):
                call(kw, False)
            torch.cuda.synchronize()
            wall_ms[tag].append((time.perf_counter() - t0) * 1e3 / steps)
    res = {"workload": f"{name}: {B} ligands x {n_at} atoms, 1 pocket ({wl['n_kp']} keypoints), dense ll, bf16x3, "
                       f"seeded random weights, {T} steps, steps_per_graph {STEPS_PER_GRAPH}; visualize_kK records "
                       f"every K-th step", "device_ms_per_call": {}, "wall_ms_per_call_host_copy": {},
           "device_overhead_vs_plain": {}, "wall_overhead_vs_plain": {}, "frame_bytes_per_call": {},
           "device_ms_rounds": dev_ms, "wall_ms_rounds": wall_ms}
    med = {tag: statistics.median(v) for tag, v in dev_ms.items()}
    medw = {tag: statistics.median(v) for tag, v in wall_ms.items()}
    for tag, kw in VARIANTS.items():
        res["device_ms_per_call"][tag] = round(med[tag], 2)
        res["wall_ms_per_call_host_copy"][tag] = round(medw[tag], 2)
        res["device_overhead_vs_plain"][tag] = round(med[tag] / med["plain"] - 1, 4)
        res["wall_overhead_vs_plain"][tag] = round(medw[tag] / medw["plain"] - 1, 4)
        m = -(-T // kw.get("frame_every", 1))         # m state frames, the output and m prediction frames
        res["frame_bytes_per_call"][tag] = (2 * m + 1) * B * n_at * (3 + F) * 4 if kw else 0
    res["launches_per_step"] = {tag: None for tag in VARIANTS}
    for tag, kw in VARIANTS.items():
        call(kw, True)
        res["launches_per_step"][tag] = model.last_launches_per_step
    res["cold_captures"] = model.cold_captures
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", nargs="+", default=["gvp_20kp", "egnn_20kp"], choices=["gvp_20kp", "egnn_20kp"])
    ap.add_argument("--steps", type=int, default=2, help="timed calls per variant and round")
    ap.add_argument("--warmup", type=int, default=1, help="untimed calls per variant (the first one captures)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the variants")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 1 or args.rounds < 1:
        ap.error("--steps, --warmup and --rounds must be >= 1 (the warm-up call captures the graphs)")
    if args.out:        # relative to where the caller ran it: build_model() changes into the repository root
        args.out = str(Path(args.out).resolve())
    if not torch.cuda.is_available():
        raise SystemExit("trajectory_bench.py needs a CUDA device")
    lines = []
    for name in args.workloads:
        r = run_workload(name, args.steps, args.warmup, args.rounds)
        r.update(card())
        r["steps"], r["warmup"], r["rounds"] = args.steps, args.warmup, args.rounds
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
