"""Small runs of every kernel for compute-sanitizer (memcheck / racecheck / synccheck):
    compute-sanitizer --tool racecheck python tools/sanitize_small.py"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import juqbox_b200 as jq
from juqbox_b200 import configs

for name, T, nsteps in (("risk_neutral", 3.0, 40), ("cnot2", 2.0, 40), ("cnot3", 2.0, 24), ("cnot1", 2.0, 40), ("rabi", 10.0, 12)):
    cfg = configs.example(name)
    cfg.params.T, cfg.params.nsteps = T, nsteps
    pc = configs.synthetic_pcof(cfg, 5) * 20
    sh = configs.noise_shift(cfg.params.Ntot, [-0.03, 0.05]) if name == "risk_neutral" else None
    res = {}
    for obj in (1, 3):
        cfg.params.objFuncType = obj
        wa = jq.Working_Arrays(cfg.params, cfg.nCoeff)
        for k in (1, 2, 3, 4, 5, 7):
            try:
                wa.set_kernel(k)
                if k == 7:
                    wa.set_time_segments(3)      # ragged segments: 40 = 13 + 13 + 14 steps
                r = wa.evaluate(pc, sh)
            except Exception:      # no instantiation of this layout for the shape / objFuncType
                continue
            res[(obj, k)] = r["grad"]
        wa.close()
    ref = res[(1, 1)]
    for key, g in res.items():
        err = np.linalg.norm(g - ref) / np.linalg.norm(ref)
        print(name, key, "rel diff vs generic", err)
        assert err < 1e-10
# the other kernels: state history from every trajectory kernel, weighted sums over many samples, control read-out
cfg = configs.example("cnot2")
cfg.params.T, cfg.params.nsteps = 2.0, 40
pc = configs.synthetic_pcof(cfg, 3) * 20
wa = jq.Working_Arrays(cfg.params, cfg.nCoeff)
hists = {}
for k in (1, 2, 3, 4, 5):
    wa.set_kernel(k)
    hists[k] = wa.forward_history(pc, save_every=4)[0]
assert all(np.abs(hists[k] - hists[1]).max() < 1e-12 for k in hists)
wa.set_kernel(0)
p, q = wa.controls(pc[0], np.linspace(0, cfg.params.T, 77))
wa.close()
cfg = configs.example("risk_neutral")
cfg.params.T, cfg.params.nsteps = 3.0, 40
sh = configs.noise_shift(cfg.params.Ntot, np.linspace(-0.05, 0.05, 130))
w = np.full(130, 1.0 / 130)
wa = jq.Working_Arrays(cfg.params, cfg.nCoeff)
pc = configs.synthetic_pcof(cfg, 2) * 20
tot = wa.evaluate(pc, sh, w)
per = wa.evaluate(pc, sh)
assert np.allclose(tot["grad"], (per["grad"] * w[None, :, None]).sum(1), rtol=1e-12, atol=1e-16)
wa.close()
# round 2: fused callback entry, pFidType 3, dense forbidden-state weights and uncoupled controls on the generic kernel (TMA-staged
# operator table, several trajectory groups per CTA)
r = wa = None
cfg = configs.example("risk_neutral")
cfg.params.T, cfg.params.nsteps = 3.0, 40
wa = jq.Working_Arrays(cfg.params, cfg.nCoeff)
pc = configs.synthetic_pcof(cfg, 1)[0] * 20
sh = configs.noise_shift(cfg.params.Ntot, cfg.nodes)
a = wa.eval_f_grad(pc, sh, cfg.weights, tik0=0.01)
b = wa.eval_f_grad(pc, sh, cfg.weights, tik0=0.01)
assert a["evaluated"] and not b["evaluated"]
wa.close()
cfg.params.pFidType = 3
wa = jq.Working_Arrays(cfg.params, cfg.nCoeff + 1)
pcs = np.concatenate([configs.synthetic_pcof(cfg, 4) * 20, np.linspace(-1, 1, 4)[:, None]], axis=1)
for k in (1, 3, 5):
    try:
        wa.set_kernel(k)
    except Exception:      # no instantiation of this layout for the shape
        continue
    wa.evaluate(pcs)
wa.close()
from juqbox_b200.params import objparams
lab = configs.example("rabi_lab", T=2.0, Pmin=20)
wa = jq.Working_Arrays(lab.params, lab.nCoeff)
wa.evaluate(np.tile(lab.pcof0, (7, 1)) * np.linspace(0.5, 2, 7)[:, None])
wa.close()
p = configs.example("risk_neutral").params
F = np.random.default_rng(0).standard_normal((p.Ntot, 2)) + 1j * np.random.default_rng(1).standard_normal((p.Ntot, 2))
pd = objparams(p.Ne, p.Ng, 3.0, 40, Uinit=p.Uinit, Utarget=p.Utarget_r + 1j * p.Utarget_i, Cfreq=p.Cfreq, Rfreq=p.Rfreq, Hconst=p.Hconst,
               Hsym_ops=p.Hsym_ops, Hanti_ops=p.Hanti_ops, use_custom_forbidden=True, forb_states=F / np.linalg.norm(F, axis=0), forb_weights=[0.5, 0.1])
wa = jq.Working_Arrays(pd, 48)
wa.evaluate(configs.synthetic_pcof(configs.example("risk_neutral"), 9) * 20)
wa.close()
print("sanitize_small OK")
