"""Throughput of fragment-conditioned sampling (inpainting) on the headline workloads.

For gvp_20kp and egnn_20kp as bench.py builds them (one synthetic 20-keypoint pocket, 100 ligands x 20 atoms, dense ll
graph, seeded random weights, bf16x3) it times full 1000-step KeypointDiffusion.sample_from_encoded_receptors calls
for: the plain loop, an 8-atom fragment pinned in every ligand with resamplings = 1, and the same with resamplings = 5.
Device time on the launching stream (CUDA events), warm capacity buckets, outputs left on the device.  Prints one JSON
line per workload (and writes them to --out), with the card's name and power limit read in the same run.

    python tools/inpaint_bench.py --out inpaint_bench.jsonl
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True).stdout.strip().splitlines()[0]
        name, limit = [v.strip() for v in q.split(",")]
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        name, limit = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": limit}


def run_workload(name, steps, warmup, m=8):
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
    n = B * n_at
    gen = torch.Generator().manual_seed(0)
    frag_pos = pocket.kp_x.mean(0) + torch.randn(m, 3, generator=gen) * 1.5
    frag_feat = torch.nn.functional.one_hot(torch.arange(m) % F, F).float()
    mask = torch.zeros(n, dtype=torch.bool)
    pos, feat = torch.zeros(n, 3), torch.zeros(n, F)
    for c in range(B):
        mask[c * n_at:c * n_at + m] = True
        pos[c * n_at:c * n_at + m] = frag_pos
        feat[c * n_at:c * n_at + m] = frag_feat
    variants = {"plain": {}, "fragment8_r1": dict(fixed_mask=mask, fixed_pos=pos, fixed_feat=feat, resamplings=1),
                "fragment8_r5": dict(fixed_mask=mask, fixed_pos=pos, fixed_feat=feat, resamplings=5)}
    res = {"workload": f"{name}: {B} ligands x {n_at} atoms, 1 pocket ({wl['n_kp']} keypoints), 1000 steps, dense ll, "
                       f"bf16x3, seeded random weights; fragment = first {m} atoms of every ligand", "ligands_per_s": {},
           "ms_per_call": {}, "launches_per_step": {}}
    for tag, kw in variants.items():
        call = lambda: model.sample_from_encoded_receptors(g, init_lig_pos=init, seed=1234, return_device_tensors=True,
                                                           **kw)
        for _ in range(warmup):
            call()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            call()
        ev1.record()
        torch.cuda.synchronize()
        sec = ev0.elapsed_time(ev1) / 1e3 / steps
        res["ligands_per_s"][tag] = round(B / sec, 2)
        res["ms_per_call"][tag] = round(sec * 1e3, 1)
        res["launches_per_step"][tag] = model.last_launches_per_step
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", nargs="+", default=["gvp_20kp", "egnn_20kp"], choices=["gvp_20kp", "egnn_20kp"])
    ap.add_argument("--steps", type=int, default=3, help="timed calls per variant")
    ap.add_argument("--warmup", type=int, default=1, help="untimed calls per variant (the first one captures)")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 1:
        ap.error("--steps and --warmup must be >= 1 (the warm-up call captures the graphs)")
    if args.out:        # relative to where the caller ran it: build_model() changes into the repository root
        args.out = str(Path(args.out).resolve())
    if not torch.cuda.is_available():
        raise SystemExit("inpaint_bench.py needs a CUDA device")
    lines = []
    for name in args.workloads:
        r = run_workload(name, args.steps, args.warmup)
        r.update(card())
        r["steps"], r["warmup"] = args.steps, args.warmup
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
