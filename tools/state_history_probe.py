#!/usr/bin/env python3
"""Derivatives of the state history (jq_history_vjp, jq_history_jvp) against the final-state routes they extend, per named shape.
Prints a markdown report on stdout, or writes it to the path given as second argument.

    python tools/state_history_probe.py [reps] [out.md]        (needs a GPU)

Per shape and one trajectory (batch 1, one cotangent or direction), the CUDA-event kernel time (jq_query 1, best of `reps` after one
warm-up call) of:
- jq_final_state_vjp, and jq_history_vjp at save_every = 1 and at a coarse save_every (at most 41 saves), each with a cotangent on
  every save; the difference to the final-state VJP is the cost of reading the cotangents and of the history adds;
- jq_forward_sensitivity with the final-state tangent, and jq_history_jvp at the same two save_every values.
It also prints the geometry of the launches (CTAs, groups per CTA, registers, dynamic shared memory per CTA) and, as a check, the
relative difference of the dot-product identity <vjp(c), d> = sum_j Re vdot(c_j, dU_j . d) at the coarse save_every.
"""
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import juqbox_b200 as jq                                    # noqa: E402
from juqbox_b200 import configs                             # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
out = open(sys.argv[2], "w") if len(sys.argv) > 2 else sys.stdout


def emit(s=""):
    print(s, file=out, flush=True)


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], text=True).strip()
    except Exception as e:                                 # the report says so instead of inventing a value
        return f"not read ({e})"


def coarse(nsteps):
    return next(d for d in range(2, nsteps + 1) if nsteps % d == 0 and nsteps // d <= 40)


def kernel_ms(wa, fn):
    """best CUDA-event kernel time of `reps` calls after one warm-up call; returns (result of the last call, ms)"""
    fn()
    ms = []
    for _ in range(reps):
        r = fn()
        ms.append(wa.query(1))
    return r, min(ms)


def geometry(wa):
    return tuple(int(wa.query(k)) for k in (4, 3, 5, 6))     # CTAs, groups per CTA, registers, smem bytes per CTA


emit("# State-history derivatives: VJPs and tangents of every saved state against the final-state routes\n")
emit(f"Card (nvidia-smi name, power limit, read in the same run): {card()}.  Batch 1, one cotangent or direction per call; kernel "
     f"times are CUDA-event times (jq_query 1), best of {reps} calls after one warm-up call.\n")
rows_v, rows_t = [], []
for name in ("cnot2", "cnot3", "risk_neutral", "rabi"):
    cfg = configs.example(name)
    p = cfg.params
    pc = configs.synthetic_pcof(cfg, 1) * (20.0 if name == "risk_neutral" else 1.0)
    npar = pc.shape[1]
    rng = np.random.default_rng(1)
    wa = jq.Working_Arrays(p, npar)
    sc = coarse(p.nsteps)
    c1 = rng.standard_normal((1, 1, 1, p.Ntot, p.N)) + 1j * rng.standard_normal((1, 1, 1, p.Ntot, p.N))
    d = rng.standard_normal((1, 1, npar))
    _, fs_ms = kernel_ms(wa, lambda: wa.final_state_vjp(pc, c1))
    fs_geo = geometry(wa)
    res = {}
    for se in (1, sc):
        nsave = p.nsteps // se + 1
        c = rng.standard_normal((1, 1, 1, nsave, p.Ntot, p.N)) + 1j * rng.standard_normal((1, 1, 1, nsave, p.Ntot, p.N))
        v, ms = kernel_ms(wa, lambda: wa.history_vjp(pc, c, save_every=se))
        assert wa.last_kernel == 9
        res[se] = (c, v["vjp"][0, 0, 0], ms, geometry(wa), nsave)
    _, fw_ms = kernel_ms(wa, lambda: wa.forward_sensitivity(pc, d, final_state=True))
    fw_geo = geometry(wa)
    tan = {}
    for se in (1, sc):
        dU, ms = kernel_ms(wa, lambda: wa.history_jvp(pc, d, save_every=se))
        assert wa.last_kernel == 8
        tan[se] = (dU[0, 0, 0], ms, geometry(wa))
    c, v, _, _, _ = res[sc]
    lhs, rhs = v @ d[0, 0], np.einsum("jab,jab->", c[0, 0, 0].conj(), tan[sc][0]).real
    rel = abs(lhs - rhs) / abs(rhs)
    wa.close()
    len_ = p.Ntot * p.N
    mb = 16.0 * (p.nsteps + 1) * len_ / 1e6                 # one history of every step, Re and Im
    (_, _, v1_ms, v1_geo, _), (_, _, vc_ms, _, nsc) = res[1], res[sc]
    rows_v.append(f"| {name} | {p.Ntot} x {p.N} | {npar} | {p.nsteps} | {fs_ms:.3f} | {v1_ms:.3f} | {100 * (v1_ms / fs_ms - 1):+.1f}% "
                  f"| {mb:.1f} | {sc} ({nsc}) | {vc_ms:.3f} | {100 * (vc_ms / fs_ms - 1):+.1f}% | {fs_geo[0]} / {v1_geo[0]} "
                  f"| {fs_geo[1]} | {fs_geo[2]} / {v1_geo[2]} | {fs_geo[3]} / {v1_geo[3]} | {rel:.2e} |")
    (_, t1_ms, t1_geo), (_, tc_ms, _) = tan[1], tan[sc]
    rows_t.append(f"| {name} | {fw_ms:.3f} | {t1_ms:.3f} | {100 * (t1_ms / fw_ms - 1):+.1f}% | {tc_ms:.3f} "
                  f"| {100 * (tc_ms / fw_ms - 1):+.1f}% | {fw_geo[0]} / {t1_geo[0]} | {fw_geo[2]} / {t1_geo[2]} | {fw_geo[3]} / {t1_geo[3]} |")

emit("## Reverse mode: `history_vjp` against `final_state_vjp`\n")
emit("| shape | Ntot x N | Npar | steps | final-state VJP ms | history VJP ms, save_every 1 | vs final | cotangent MB (save_every 1) "
     "| coarse save_every (saves) | history VJP ms, coarse | vs final | CTAs (final / history) | groups/CTA | regs (final / history) "
     "| smem B/CTA (final / history) | dot-product rel. diff (coarse) |")
emit("|---|---|---|---|---|---|---|---|---|---|---|---|---|---|---|---|")
for r in rows_v:
    emit(r)
emit("\n## Forward mode: `history_jvp` against `forward_sensitivity` (one direction, final-state tangent)\n")
emit("| shape | forward sensitivity ms | history JVP ms, save_every 1 | vs forward | history JVP ms, coarse | vs forward "
     "| CTAs (forward / history) | regs | smem B/CTA |")
emit("|---|---|---|---|---|---|---|---|---|")
for r in rows_t:
    emit(r)
