#!/usr/bin/env python3
"""A/B of the two tile layouts of two-subsystem problems on the cnot2 example: the 2 x 2 tiles (TileLane<2,2>, 2 trajectories per
warp) against the first subsystem whole in the lane (TileLane<2,1,1>, 4 trajectories per warp).

    python tools/tile_inlane_ab.py [--sizes 4736,16384,32768] [--reps 5] [--out DIR]

Both variants live in one process (JQ_TILE_INLANE=0 / =1 at handle creation) and are timed alternately, size by size, on the same
device-resident synthetic pcof batch: kernel ms from the CUDA events around the launch (Working_Arrays.last_kernel_ms).  Prints one
line per (size, variant) with the median and spread, the ratio of the medians, and the card's name and power limit; with --out the
same as JSON in DIR/tile_inlane_ab.json.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="2368,3552,4736,7104,9472,14208,16384,18944,32768")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import juqbox_b200 as jq
    from juqbox_b200 import configs
    cfg = configs.example("cnot2")
    dev = torch.device("cuda", 0)
    sizes = [int(s) for s in a.sizes.split(",")]
    was = {}
    for name, env in (("tile 2x2", "0"), ("tile in-lane", "1")):
        os.environ["JQ_TILE_INLANE"] = env          # read when the handle is created
        was[name] = jq.Working_Arrays(cfg.params, cfg.nCoeff, device=0)
        was[name].set_kernel(4)
    os.environ.pop("JQ_TILE_INLANE")
    pc_all = torch.from_numpy(configs.synthetic_pcof(cfg, max(sizes))).to(dev)
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    rows = []
    for B in sizes:
        pc = pc_all[:B].contiguous()
        ms = {k: [] for k in was}
        facts = {}
        for k, wa in was.items():                  # warm-up: module load, scratch growth
            wa.evaluate_device(pc)
            torch.cuda.synchronize()
            facts[k] = {"tpc": int(wa.query(3)), "ctas": int(wa.query(4)), "regs": int(wa.query(5)), "smem": int(wa.query(6))}
        for _ in range(a.reps):
            for k, wa in was.items():
                wa.evaluate_device(pc)
                torch.cuda.synchronize()
                assert wa.last_kernel == 4
                ms[k].append(wa.last_kernel_ms)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        for k, v in ms.items():
            print(f"B={B:6d} {k:13s} median {med[k]:9.3f} ms  min {min(v):9.3f}  max {max(v):9.3f}  spread {100 * (max(v) - min(v)) / med[k]:5.2f}%"
                  f"  tpc {facts[k]['tpc']} ctas {facts[k]['ctas']} regs {facts[k]['regs']} smem {facts[k]['smem']} B", flush=True)
        ratio = med["tile 2x2"] / med["tile in-lane"]
        print(f"B={B:6d} speed-up of in-lane over 2x2 (ratio of medians): {ratio:.4f}", flush=True)
        rows.append({"candidates": B, "ms": ms, "median_ms": med, "speedup_inlane": ratio, "launch": facts})
    for wa in was.values():
        wa.close()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "tile_inlane_ab.json"), "w") as f:
            json.dump({"card": info, "workload": "cnot2", "reps": a.reps, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
