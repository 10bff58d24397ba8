#!/usr/bin/env python3
"""Final-state vector-Jacobian products on the time-parallel path (jq_final_state_vjp_time_parallel, kernel 7 stages) against the serial
VJP kernel (jq_final_state_vjp, kernel 9) and against kernel 7's own objective + gradient, at batch 1 with one cotangent per shape.
Prints a markdown report on stdout.

    python tools/final_state_vjp_time_parallel_probe.py [reps]        (needs a GPU)

Per shape: CUDA-event time of the trajectory work (jq_query 1) and host wall time around the blocking call (best of `reps` after one
warm-up call) of the time-parallel VJP, of its U(T)-only call (ncot = 0), of kernel 9 and of kernel 7's evaluation with gradient;
segments and launches of the time-parallel VJP; the relative difference of its result to kernel 9's.  Then the JQ_SEG_TIMING=1 stage
breakdown of one time-parallel VJP and one kernel-7 evaluation per shape (a child process each: the library prints it).
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


def setup(name):
    """One candidate (risk-neutral: with its quadrature nodes) and one random complex cotangent per sample."""
    cfg = configs.example(name)
    p = cfg.params
    pc = configs.synthetic_pcof(cfg, 1)
    sh = configs.noise_shift(p.Ntot, cfg.nodes) if name == "risk_neutral" else None
    ns = 1 if sh is None else len(sh)
    rng = np.random.default_rng(1)
    c = rng.standard_normal((1, ns, 1, p.Ntot, p.N)) + 1j * rng.standard_normal((1, ns, 1, p.Ntot, p.N))
    return cfg, p, pc, sh, c


def stages(name):
    """Child process: one time-parallel VJP and one kernel-7 evaluation after a warm-up each, with JQ_SEG_TIMING=1 set by the parent."""
    cfg, p, pc, sh, c = setup(name)
    wa = jq.Working_Arrays(p, pc.shape[1])
    for _ in range(2):
        wa.final_state_vjp(pc, c, sh, time_parallel=True)
    wa.set_kernel(7)
    for _ in range(2):
        wa.evaluate(pc, sh)
    wa.close()


def main(reps):
    def best(wa, fn):
        fn()                                               # warm-up: module load, buffers, attributes
        ts, ks = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = fn()
            ts.append((time.perf_counter() - t0) * 1e3)
            ks.append(wa.query(1))
        return r, min(ks), min(ts)

    print("# Final-state VJPs on the time-parallel path\n")
    print(f"Card (nvidia-smi name, power limit): {card()}; best of {reps} calls after one warm-up call, automatic segment count.\n")
    print("| shape | Ntot x N | Npar | steps | samples | kernel 9 ms (kernel / call) | time-parallel VJP ms (kernel / call) | segments "
          "| launches | kernel 9 / time-parallel (kernel) | U(T) only ms (kernel / call) | kernel 7 obj + grad ms (kernel / call) "
          "| rel. diff to kernel 9 |")
    print("|---|---|---|---|---|---|---|---|---|---|---|---|---|")
    for name in SHAPES:
        cfg, p, pc, sh, c = setup(name)
        wa = jq.Working_Arrays(p, pc.shape[1])
        v9, k9, t9 = best(wa, lambda: wa.final_state_vjp(pc, c, sh))
        assert wa.last_kernel == 9
        v7, k7, t7 = best(wa, lambda: wa.final_state_vjp(pc, c, sh, time_parallel=True))
        assert wa.last_kernel == 7
        nseg, nl = int(wa.query(7)), int(wa.query(2))
        _, ku, tu = best(wa, lambda: wa.final_state_vjp(pc, None, sh, final_state=True, time_parallel=True))
        wa.set_kernel(7)
        _, ke, te = best(wa, lambda: wa.evaluate(pc, sh))
        assert wa.last_kernel == 7
        wa.close()
        rel = np.linalg.norm(v7["vjp"] - v9["vjp"]) / np.linalg.norm(v9["vjp"])
        ns = 1 if sh is None else len(sh)
        print(f"| {name} | {p.Ntot} x {p.N} | {pc.shape[1]} | {p.nsteps} | {ns} | {k9:.2f} / {t9:.2f} | {k7:.3f} / {t7:.3f} | {nseg} | {nl} "
              f"| {k9 / k7:.0f}x | {ku:.3f} / {tu:.3f} | {ke:.3f} / {te:.3f} | {rel:.2e} |", flush=True)
    print("\n## Stage breakdown (JQ_SEG_TIMING=1, CUDA events, us; the second of two calls)\n")
    print("Time-parallel VJP: launch 1 (Phi, Adj) | join X | terminal values + U(T) | defect sweeps, join Eta and refinement passes "
          "| join Lam2 | launch 4 (mode 5) | sum.  Kernel 7 evaluation: launch 1 | join X | objective | launch 2 (penalty, defects) "
          "| join Eta and refinement passes | launch 3 | join Lam (and Lam2) | launch 4 | sum.\n")
    print("```")
    env = dict(os.environ, JQ_SEG_TIMING="1")
    for name in SHAPES:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--stages", name], env=env, capture_output=True, text=True,
                             check=True).stdout.splitlines()
        vjp = [l for l in out if l.startswith("seg vjp stages")]
        ev = [l for l in out if l.startswith("seg stages")]
        print(f"{name}:\n  {vjp[-1]}\n  {ev[-1]}")
    print("```")


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--stages":
        stages(sys.argv[2])
    else:
        main(int(sys.argv[1]) if len(sys.argv) > 1 else 5)
