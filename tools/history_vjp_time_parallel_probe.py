#!/usr/bin/env python3
"""History vector-Jacobian products on the time-parallel path (jq_history_vjp_time_parallel, kernel 7 stages) against the serial VJP
kernel (jq_history_vjp, kernel 9) and against the final-state VJP on the same path, at batch 1 with one cotangent per shape.
Prints a markdown report on stdout.

    python tools/history_vjp_time_parallel_probe.py [reps]        (needs a GPU)

Per shape and save stride (every step, and the coarse stride of at most 41 saves): CUDA-event time of the trajectory work (jq_query 1)
and host wall time around the blocking call (best of `reps` after one warm-up call; kernel 9 one call after its warm-up) of the
time-parallel history VJP, of its history-only call (ncot = 0), of kernel 9's history VJP and of the time-parallel final-state VJP;
segments and launches; the relative difference to kernel 9's result.  The host time includes the copies of the cotangent history
(16 nsave n m bytes) and of the saved states.  Then the JQ_SEG_TIMING=1 stage breakdown of one time-parallel history VJP at each
stride per shape (a child process each: the library prints it).
"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import juqbox_b200 as jq                                    # noqa: E402
from juqbox_b200 import configs                             # noqa: E402

SHAPES = ("cnot1", "cnot2", "cnot3", "risk_neutral")


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], text=True).strip()
    except Exception as e:                                 # the report says so instead of inventing a value
        return f"not read ({e})"


def coarse(nsteps):
    return next(d for d in range(2, nsteps + 1) if nsteps % d == 0 and nsteps // d <= 40)


def setup(name, se):
    """One candidate (risk-neutral: with its quadrature nodes) and one random complex cotangent history per sample."""
    cfg = configs.example(name)
    p = cfg.params
    pc = configs.synthetic_pcof(cfg, 1)
    sh = configs.noise_shift(p.Ntot, cfg.nodes) if name == "risk_neutral" else None
    ns = 1 if sh is None else len(sh)
    nsave = p.nsteps // se + 1
    rng = np.random.default_rng(1)
    shape = (1, ns, 1, nsave, p.Ntot, p.N)
    c = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
    return p, pc, sh, c


def stages(name, se):
    """Child process: two time-parallel history VJPs, with JQ_SEG_TIMING=1 set by the parent."""
    p, pc, sh, c = setup(name, se)
    wa = jq.Working_Arrays(p, pc.shape[1])
    for _ in range(2):
        wa.history_vjp(pc, c, sh, se, time_parallel=True)
    wa.close()


def main(reps):
    def best(wa, fn, n=reps):
        fn()                                               # warm-up: module load, buffers, attributes
        ts, ks = [], []
        for _ in range(n):
            t0 = time.perf_counter()
            r = fn()
            ts.append((time.perf_counter() - t0) * 1e3)
            ks.append(wa.query(1))
        return r, min(ks), min(ts)

    print("# History VJPs on the time-parallel path\n")
    print(f"Card (nvidia-smi name, power limit): {card()}; best of {reps} calls after one warm-up call (kernel 9: one call after "
          "one warm-up), automatic segment count, one cotangent.\n")
    print("| shape | steps | save_every | nsave | kernel 9 history VJP ms (kernel / call) | time-parallel history VJP ms (kernel / call) "
          "| segments | launches | kernel 9 / time-parallel (kernel) | history only ms (kernel / call) "
          "| time-parallel final-state VJP ms (kernel) | history / final-state VJP (kernel) | rel. diff to kernel 9 |")
    print("|---|---|---|---|---|---|---|---|---|---|---|---|---|")
    rows = []
    for name in SHAPES:
        for se in (1, coarse(configs.example(name).params.nsteps)):
            p, pc, sh, c = setup(name, se)
            wa = jq.Working_Arrays(p, pc.shape[1])
            v9, k9, t9 = best(wa, lambda: wa.history_vjp(pc, c, sh, se), 1)
            assert wa.last_kernel == 9
            v7, k7, t7 = best(wa, lambda: wa.history_vjp(pc, c, sh, se, time_parallel=True))
            assert wa.last_kernel == 7
            nseg, nl = int(wa.query(7)), int(wa.query(2))
            _, kh, th = best(wa, lambda: wa.history_vjp(pc, None, sh, se, history=True, time_parallel=True))
            _, kf, _ = best(wa, lambda: wa.final_state_vjp(pc, c[:, :, :, -1], sh, time_parallel=True))
            wa.close()
            rel = np.linalg.norm(v7["vjp"] - v9["vjp"]) / np.linalg.norm(v9["vjp"])
            print(f"| {name} | {p.nsteps} | {se} | {p.nsteps // se + 1} | {k9:.2f} / {t9:.2f} | {k7:.3f} / {t7:.3f} | {nseg} | {nl} "
                  f"| {k9 / k7:.0f}x | {kh:.3f} / {th:.3f} | {kf:.3f} | {k7 / kf:.2f} | {rel:.2e} |", flush=True)
            rows.append((name, se))
    print("\n## Stage breakdown (JQ_SEG_TIMING=1, CUDA events, us; the second of two calls)\n")
    print("launch 1 (Phi, Adj) | join X | terminal values | launch 2 (saves, defect sweeps, particular solutions) "
          "| join Eta and refinement passes | join Lam2 with the particular solutions | launch 4 (mode 5 with jumps) | sum.\n")
    print("```")
    env = dict(os.environ, JQ_SEG_TIMING="1")
    for name, se in rows:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--stages", name, str(se)], env=env, capture_output=True,
                             text=True, check=True).stdout.splitlines()
        vjp = [l for l in out if l.startswith("seg vjp stages")]
        print(f"{name}, save_every {se}:\n  {vjp[-1]}")
    print("```")


if __name__ == "__main__":
    if len(sys.argv) > 3 and sys.argv[1] == "--stages":
        stages(sys.argv[2], int(sys.argv[3]))
    else:
        main(int(sys.argv[1]) if len(sys.argv) > 1 else 5)
