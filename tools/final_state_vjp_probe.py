#!/usr/bin/env python3
"""Final-state vector-Jacobian products (jq_final_state_vjp): the gradient of one scalar objective of U(T) by one cotangent, against the
same gradient by jq_forward_sensitivity with Npar unit directions, and the full Jacobian of U(T) (ncot = 2 Ntot N) per named shape.
Prints a markdown report on stdout.

    python tools/final_state_vjp_probe.py [reps]        (needs a GPU)

The objective is L = Re vdot(c, U(T)) for a fixed random complex c, so its gradient is vjp(c) and, by the forward route,
Re vdot(c, dU . e_p) for every unit direction e_p.  Per shape: CUDA-event kernel time (jq_query 1) and host wall time around the
blocking call (best of `reps` after one warm-up call) of each route, the geometry of the VJP launch (CTAs, groups per CTA, registers,
dynamic shared memory per CTA) and the relative difference between the two gradients.
"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import juqbox_b200 as jq                                    # noqa: E402
from juqbox_b200 import configs                             # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], text=True).strip()
    except Exception as e:                                 # the report says so instead of inventing a value
        return f"not read ({e})"


def best(fn, n=reps):
    fn()                                                   # warm-up: module load, buffers, attributes
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        r = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return r, min(ts)


print("# Final-state VJPs: the gradient of one objective of U(T), and the full Jacobian\n")
print(f"Card (nvidia-smi name, power limit): {card()}; best of {reps} calls after one warm-up call (the Jacobian: one call after one "
      "warm-up call).\n")
print("| shape | Ntot x N | Npar | steps | VJP kernel ms | VJP call ms | CTAs | groups/CTA | regs | smem B/CTA "
      "| forward (Npar dirs) kernel ms | forward / VJP | rel. diff | Jacobian ncot | Jacobian kernel ms | Jacobian CTAs |")
print("|---|---|---|---|---|---|---|---|---|---|---|---|---|---|---|---|")
for name in ("cnot2", "cnot3", "risk_neutral", "rabi"):
    cfg = configs.example(name)
    p = cfg.params
    pc = configs.synthetic_pcof(cfg, 1) * (20.0 if name == "risk_neutral" else 1.0)
    npar = pc.shape[1]
    rng = np.random.default_rng(1)
    c = rng.standard_normal((1, 1, 1, p.Ntot, p.N)) + 1j * rng.standard_normal((1, 1, 1, p.Ntot, p.N))
    wa = jq.Working_Arrays(p, npar)
    v, vjp_ms = best(lambda: wa.final_state_vjp(pc, c))
    assert wa.last_kernel == 9
    vjp_kern = wa.query(1)
    ctas, gpc, regs, smem = (int(wa.query(k)) for k in (4, 3, 5, 6))
    f, _ = best(lambda: wa.forward_sensitivity(pc, np.eye(npar)[None], final_state=True))
    fwd_kern = wa.query(1)
    g_fwd = np.einsum("ab,kab->k", c[0, 0, 0].conj(), f["dstate"][0, 0]).real
    g_vjp = v["vjp"][0, 0, 0]
    rel = np.linalg.norm(g_vjp - g_fwd) / np.linalg.norm(g_fwd)
    ncot = 2 * p.Ntot * p.N                                # every entry of Re U and of Im U
    eye = np.eye(p.Ntot * p.N).reshape(p.Ntot * p.N, p.N, p.Ntot).swapaxes(-1, -2)
    cots = np.concatenate([eye, 1j * eye])[None, None]
    jac, _ = best(lambda: wa.final_state_vjp(pc, cots), n=1)
    jac_kern, jac_ctas = wa.query(1), int(wa.query(4))
    # the Jacobian's rows of Re U contracted with the real part of c (and Im U with Im c) give the same gradient
    w = np.concatenate([c[0, 0, 0].real.T.ravel(), c[0, 0, 0].imag.T.ravel()])
    assert np.linalg.norm(w @ jac["vjp"][0, 0] - g_vjp) <= 1e-10 * np.linalg.norm(g_vjp)
    wa.close()
    print(f"| {name} | {p.Ntot} x {p.N} | {npar} | {p.nsteps} | {vjp_kern:.3f} | {vjp_ms:.3f} | {ctas} | {gpc} | {regs} | {smem} "
          f"| {fwd_kern:.3f} | {fwd_kern / vjp_kern:.1f} | {rel:.2e} | {ncot} | {jac_kern:.3f} | {jac_ctas} |", flush=True)
