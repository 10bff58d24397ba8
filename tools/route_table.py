"""Kernel choice and outputs over a fixed, seeded matrix of problems, batch sizes, kernel preferences, entries and environment knobs.

    python tools/route_table.py [problem ...] > routes.jsonl        (needs a GPU; default: every problem)

One JSON line per case: the jq_set_kernel result, jq_query items 0 and 2-7 after the entry, and a hash of the entry's outputs (or its
error).  Two builds that select kernels alike and compute alike print identical lines, so a diff of two runs checks a change of the
selection logic.  The batch sizes are 1, 2, 16384 and both sides of every automatic cut-over; a cut-over is found by bisection over
the batch size on what automatic mode runs (kernel id, trajectories per CTA), so it needs no knowledge of the thresholds.
"""
import hashlib
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
import torch                                                # noqa: E402

import juqbox_b200 as jq                                    # noqa: E402
from juqbox_b200 import configs                             # noqa: E402
from juqbox_b200.params import objparams                    # noqa: E402

NSTEPS = 256              # the shortest horizon automatic mode sends to the time-parallel evaluation
MAX_BATCH = 16384
KNOBS = [{}, {"JQ_TILE_INLANE": "0"}, {"JQ_TILE_INLANE": "1"}, {"JQ_SEG_NTRAJ": "0"}]


def golden(name):
    with open(os.path.join(ROOT, "tests", "golden", f"{name}.json")) as f:
        return configs.test_case(name, json.load(f).get("pcof0"))


def dense(n, m, Nc=2, Nfreq=2, seed=12):
    rng = np.random.default_rng(seed)
    sym = lambda a: (a + a.T) / 2
    p = objparams([m], [n - m], 3.0, NSTEPS, Uinit=np.eye(n, m),
                  Utarget=np.linalg.qr(rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)))[0][:, :m],
                  Cfreq=rng.standard_normal((Nc, Nfreq)), Rfreq=[1.0, 2.0], Hconst=sym(rng.standard_normal((n, n))) * 0.3,
                  Hsym_ops=[sym(rng.standard_normal((n, n))) / np.sqrt(n) for _ in range(Nc)],
                  Hanti_ops=[(lambda a: (a - a.T) / 2)(rng.standard_normal((n, n))) / np.sqrt(n) for _ in range(Nc)])
    return p, 2 * Nc * Nfreq * 5, 0.2


def problems():
    """name -> (params, npar, pcof scale, shifts, weights)"""
    out = {}
    for name in ("cnot1", "cnot2", "cnot3", "rabi"):
        cfg = configs.example(name)
        out[name] = (cfg.params, cfg.nCoeff, float(np.max(np.abs(configs.synthetic_pcof(cfg, 1)))), None, None)
    cfg = configs.example("risk_neutral")
    out["risk_neutral_weighted"] = (cfg.params, cfg.nCoeff, float(np.max(np.abs(configs.synthetic_pcof(cfg, 1)))),
                                    configs.noise_shift(cfg.params.Ntot, cfg.nodes), cfg.weights)
    for name in ("flux", "cnot2-jacobi", "cnot2-leakieq"):
        cfg = golden(name)
        out[name] = (cfg.params, len(cfg.pcof0), float(np.max(np.abs(cfg.pcof0))), None, None)
    p, npar, sc = dense(24, 6)
    out["dense_24x6"] = (p, npar, sc, np.random.default_rng(5).uniform(-0.05, 0.05, (3, 24)), None)
    cfg = configs.example("rabi_lab", T=20.0, Pmin=60)
    out["uncoupled"] = (cfg.params, cfg.nCoeff, float(np.max(np.abs(cfg.pcof0))), None, None)
    cfg = configs.qudit_system([3, 2, 2], [2, 1, 1])
    out["qudits_45x12"] = (cfg.params, cfg.nCoeff, 0.5 * cfg.maxpar[0], None, None)
    cfg = configs.example("risk_neutral")
    cfg.params.T = 40.0
    out["long_pcof"] = (cfg.params, 2 * cfg.params.Ncoupled * cfg.params.Nfreq * 200, 0.01, None, None)
    for p, *_ in out.values():
        p.nsteps = NSTEPS
    return out


def pcofs(npar, scale, nbatch, seed):
    return np.random.default_rng(seed).uniform(-scale, scale, (nbatch, npar))


def digest(res):
    h = hashlib.sha256()
    for k in sorted(res):
        v = res[k]
        v = v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
        h.update(k.encode())
        h.update(np.ascontiguousarray(v).tobytes())
    return h.hexdigest()[:24]


def message(e):
    return re.sub(r" \([^()]*\.cu:\d+\)", "", str(e))      # source positions move with every edit


def run_entry(wa, entry, pc, shifts, weights):
    if entry == "evaluate":
        return wa.evaluate(pc, shifts, weights)
    if entry == "evaluate_device":
        dev = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda(wa.device)
        r = wa.evaluate_device(dev(pc), dev(shifts), dev(weights))
        torch.cuda.synchronize()
        return r
    if entry == "eval_f_grad":
        return wa.eval_f_grad(pc[0], shifts, weights, tik0=0.01)
    if entry == "forward_history":
        hist, infid, leak = wa.forward_history(pc, shifts, save_every=wa.params.nsteps)
        return {"hist": hist, "infid": infid, "leak": leak}
    dirs = np.random.default_rng(7).standard_normal((pc.shape[0], 2, pc.shape[1]))
    return wa.forward_sensitivity(pc, dirs, shifts, weights, final_state=weights is None and pc.shape[0] <= 2)


def cutovers(wa, npar, scale, shifts, weights):
    """Batch sizes b where what automatic mode runs for b differs from what it runs for b + 1."""
    seen = {}

    def sig(b):
        if b not in seen:
            wa.evaluate(pcofs(npar, scale, b, 1), shifts, weights)
            seen[b] = (wa.last_kernel, int(wa.query(3)))
        return seen[b]

    cuts = []

    def split(lo, hi):
        if sig(lo) == sig(hi):
            return
        if hi - lo == 1:
            cuts.append(lo)
            return
        mid = (lo + hi) // 2
        split(lo, mid)
        split(mid, hi)
    wa.set_kernel(0)
    split(1, MAX_BATCH)
    return sorted(cuts)


def main(names):
    for name, (p, npar, scale, shifts, weights) in problems().items():
        if names and name not in names:
            continue
        wa = jq.Working_Arrays(p, npar)
        cuts = cutovers(wa, npar, scale, shifts, weights)
        wa.close()
        batches = sorted({1, 2, MAX_BATCH} | {b for c in cuts for b in (c - 1, c, c + 1, c + 2) if 1 <= b <= MAX_BATCH})
        print(json.dumps({"problem": name, "cutovers": cuts, "batches": batches}), flush=True)
        for knob in KNOBS:
            old = {k: os.environ.get(k) for k in knob}
            os.environ.update(knob)                         # read when the handle is created
            wa = jq.Working_Arrays(p, npar)
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k)
                else:
                    os.environ[k] = v
            for pref in range(8):
                try:
                    wa.set_kernel(pref)
                    setk = "ok"
                except Exception as e:
                    print(json.dumps({"problem": name, "knob": knob, "pref": pref, "set_kernel": message(e)}), flush=True)
                    continue
                for nbatch in batches:
                    for entry in ("evaluate", "evaluate_device", "eval_f_grad", "forward_history", "forward_sensitivity"):
                        if entry == "eval_f_grad" and nbatch != 1:
                            continue                        # one pcof per call
                        case = {"problem": name, "knob": knob, "pref": pref, "set_kernel": setk, "nbatch": nbatch, "entry": entry}
                        try:
                            res = run_entry(wa, entry, pcofs(npar, scale, nbatch, 100 * pref + nbatch), shifts, weights)
                            case["out"] = digest(res)
                            case["query"] = [wa.query(i) for i in (0, 2, 3, 4, 5, 6, 7)]
                        except Exception as e:
                            case["error"] = message(e)
                        print(json.dumps(case), flush=True)
            wa.close()


if __name__ == "__main__":
    main(sys.argv[1:])
