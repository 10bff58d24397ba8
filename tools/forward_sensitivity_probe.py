#!/usr/bin/env python3
"""Forward sensitivities (jq_forward_sensitivity): the whole forward-mode gradient (ndir = Npar unit directions) in one call per named
shape, against the adjoint gradient of the automatic evaluation path.  Prints a markdown report on stdout.

    python tools/forward_sensitivity_probe.py [reps]        (needs a GPU)

Per shape: CUDA-event time of the forward-sensitivity kernel (jq_query 1), host wall time around the blocking call (best of `reps`),
launch count, geometry (CTAs, groups per CTA, registers, dynamic shared memory), and the relative difference ||forward - adjoint|| /
||adjoint|| and max |forward - adjoint| / max |adjoint|.  The adjoint gradient's own call time (automatic kernel) is listed beside it.
"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import juqbox_b200 as jq                                    # noqa: E402
from juqbox_b200 import configs                             # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], text=True).strip()
    except Exception as e:                                 # the report says so instead of inventing a value
        return f"not read ({e})"


def best(fn):
    fn()                                                   # warm-up: module load, buffers, attributes
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return r, min(ts)


print("# Forward sensitivities: full forward-mode gradient in one call\n")
print(f"Card (nvidia-smi name, power limit): {card()}; best of {reps} calls after one warm-up call.\n")
print("| shape | Npar | samples | trajectories | kernel ms (events) | host call ms | launches | CTAs | groups/CTA | regs | smem B/CTA "
      "| rel. diff vs adjoint | max abs diff / max abs | adjoint call ms (kernel) |")
print("|---|---|---|---|---|---|---|---|---|---|---|---|---|---|")
for name in ("cnot2", "cnot3", "risk_neutral", "rabi"):
    cfg = configs.example(name)
    p = cfg.params
    pc = configs.synthetic_pcof(cfg, 1) * (20.0 if name == "risk_neutral" else 1.0)
    npar = pc.shape[1]
    shifts = weights = None
    if name == "risk_neutral":
        shifts, weights = configs.noise_shift(p.Ntot, cfg.nodes), np.asarray(cfg.weights)
    ns = 1 if shifts is None else shifts.shape[0]
    wa = jq.Working_Arrays(p, npar)
    dirs = np.eye(npar)[None]
    f, host_ms = best(lambda: wa.forward_sensitivity(pc, dirs, shifts, weights))
    assert wa.last_kernel == 8
    kern_ms, launches = wa.query(1), int(wa.query(2))
    ctas, gpc, regs, smem = (int(wa.query(k)) for k in (4, 3, 5, 6))
    a, adj_ms = best(lambda: wa.evaluate(pc, shifts, weights))
    adj_kernel = wa.last_kernel
    g = a["grad"][0] if weights is not None else a["grad"][0, 0]
    fw = f["dobjf"][0] if weights is not None else f["dobjf"][0, 0]
    rel = np.linalg.norm(fw - g) / np.linalg.norm(g)
    mx = np.abs(fw - g).max() / np.abs(g).max()
    print(f"| {name} | {npar} | {ns} | {npar * ns} | {kern_ms:.3f} | {host_ms:.3f} | {launches} | {ctas} | {gpc} | {regs} | {smem} "
          f"| {rel:.2e} | {mx:.2e} | {adj_ms:.3f} ({adj_kernel}) |", flush=True)
    wa.close()
