"""Final-state vector-Jacobian products on the time-parallel path (jq_final_state_vjp_time_parallel, kernel 7 stages).

Pinned against the serial VJP kernel (jq_final_state_vjp, kernel 9), which computes the same unforced adjoint sweep from the same
terminal value in one pass; against kernel 7's and kernel 1's own infidelity gradients (the infidelity cotangent); and U(T) against
forward_history.  Tests marked gpu need a device; the others check the binding and the wrappers without one."""
import ctypes as C

import numpy as np
import pytest

from helpers import golden_config
from test_gpu_final_state_vjp import SHIFTS, _infid_cot, _LinearStandIn, _random_cot, _rel, _small_swap, _uncoupled_params
from test_gpu_forward_sensitivity import _dense_weight_params

TOL_K9 = 1e-11       # against kernel 9: the same sweep, cut into segments joined through their propagators
TOL_K7 = 1e-12       # infidelity cotangent against kernel 7's own infidgrad at the same segments (the same stages)
TOL_STATE = 1e-12    # U(T) against forward_history on kernel 1
MUST_SERVE = ("cnot1", "cnot2", "cnot3", "risk_neutral")      # shapes the time-parallel VJP must serve: never skipped


class _TimeParallelStandIn(_LinearStandIn):
    """The linear stand-in with the time-parallel entry: U(T) alone for cot=None, the same adjoint otherwise."""

    def __init__(self):
        super().__init__()
        self.calls = []

    def final_state_vjp(self, pcof, cot, shifts=None, final_state=False, time_parallel=False):
        self.calls.append((cot is None, final_state, time_parallel))
        out = {} if cot is None else super().final_state_vjp(pcof, cot, shifts)
        if final_state:
            out["state"] = np.einsum("sijp,bp->bsij", self._a(shifts), pcof)
        return out


# ---------------------------------------------------------------------------------------------------------------- no device needed
def test_symbol_exported_and_null_handle_rejected():
    from juqbox_b200 import _lib
    lib = _lib.load()
    assert "jq_final_state_vjp_time_parallel" in _lib.EXPORTS and hasattr(lib, "jq_final_state_vjp_time_parallel")
    one = np.zeros(64)
    p = one.ctypes.data_as(C.c_void_p)
    assert lib.jq_final_state_vjp_time_parallel(None, 1, p, 64, 1, None, 1, p, p, p, None, None) == -1       # JQ_ERR_ARG
    assert "handle" in _lib.last_error()


def _no_lib_wa():
    import juqbox_b200 as jq
    from juqbox_b200 import configs

    class NoLib:                            # any call into the library fails the test
        def __getattr__(self, name):
            raise AssertionError(f"library called: {name}")
    cfg = configs.example("rabi")
    wa = jq.Working_Arrays.__new__(jq.Working_Arrays)
    wa.params, wa._lib, wa._handle = cfg.params, NoLib(), None
    wa._snapshot = wa._fingerprint(cfg.params)
    return wa, cfg.nCoeff, cfg.params.Ntot, cfg.params.N


def test_wrapper_rejects_malformed_inputs_before_the_library():
    wa, npar, n, m = _no_lib_wa()
    pc = np.zeros((2, npar))
    for bad in (np.zeros((2, 1, 1, n, m, 1)), np.zeros((2, 1, n, m)), np.zeros((2, 1, 0, n, m)), np.zeros((1, 1, 1, n, m)),
                np.zeros((2, 2, 1, n, m)), np.zeros((2, 1, 1, m, n + 1)), np.zeros((2, 1, 1, n, m + 1))):
        with pytest.raises(ValueError):
            wa.final_state_vjp(pc, bad, time_parallel=True)
    with pytest.raises(ValueError):         # shifts not [nsamples, Ntot]
        wa.final_state_vjp(pc, np.zeros((2, 3, 1, n, m)), np.zeros((3, n + 1)), time_parallel=True)
    with pytest.raises(ValueError):         # cot for 2 samples, shifts for 3
        wa.final_state_vjp(pc, np.zeros((2, 2, 1, n, m)), np.zeros((3, n)), time_parallel=True)
    with pytest.raises(ValueError):         # shifts of the U(T)-only call
        wa.final_state_vjp(pc, None, np.zeros((3, n + 1)), final_state=True, time_parallel=True)


@pytest.mark.parametrize("final_state,time_parallel", [(False, False), (True, False), (False, True)])
def test_cot_none_needs_the_time_parallel_state_call(final_state, time_parallel):
    wa, npar, _, _ = _no_lib_wa()
    with pytest.raises(ValueError, match="cot=None"):
        wa.final_state_vjp(np.zeros((1, npar)), None, final_state=final_state, time_parallel=time_parallel)


@pytest.mark.parametrize("shifts", [None, np.zeros((2, 3))])
def test_final_state_time_parallel_plumbing_on_a_linear_stand_in(shifts):
    """The torch function with time_parallel=True: the forward pass is the U(T)-only call, the backward pass one time-parallel VJP."""
    torch = pytest.importorskip("torch")
    import juqbox_b200 as jq
    wa = _TimeParallelStandIn()
    pc = torch.tensor(np.random.default_rng(1).standard_normal((3, 5)), dtype=torch.float64, requires_grad=True)
    U = jq.final_state(wa, pc, shifts, time_parallel=True)
    assert U.shape == (3, 1 if shifts is None else 2, 3, 2) and U.dtype == torch.complex128
    assert wa.calls == [(True, True, True)]
    (U.abs() ** 2).sum().backward()
    assert wa.calls[-1] == (False, False, True)
    assert torch.autograd.gradcheck(lambda x: jq.final_state(wa, x, shifts, time_parallel=True), (pc,), eps=1e-6, atol=1e-9, rtol=1e-7)


# ---------------------------------------------------------------------------------------------------------------- on the GPU
def _case(name):
    """(params, pcof, shifts) of a named case: the example configs (risk-neutral with its quadrature nodes) or a golden."""
    from juqbox_b200 import configs
    if name in MUST_SERVE:
        cfg = configs.example(name)
        sh = configs.noise_shift(cfg.params.Ntot, cfg.nodes) if name == "risk_neutral" else None
        return cfg.params, configs.synthetic_pcof(cfg, 1)[0], sh
    cfg, _ = golden_config(name)
    return cfg.params, np.asarray(cfg.pcof0, dtype=np.float64), None


def _wa(p, npar, name, nseg=0, required=False):
    """A handle with kernel 7's segment count set; skips a problem that kernel 7 does not serve, never a required one (MUST_SERVE)."""
    import juqbox_b200 as jq
    wa = jq.Working_Arrays(p, npar)
    try:
        wa.set_kernel(7)
    except Exception as e:
        wa.close()
        assert not required and name not in MUST_SERVE, (name, str(e))
        pytest.skip(f"no time-parallel evaluation for {name}: {e}")
    wa.set_kernel(0)
    wa.set_time_segments(nseg)
    return wa


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cnot1", "cnot2", "cnot3", "risk_neutral", "swap02", "flux", "rabi", "cnot2-leakieq"])
def test_agrees_with_the_serial_vjp_kernel(name):
    """Random complex cotangents through the time-parallel VJP (automatic, 3 and 1 segments) and kernel 9."""
    p, pc, sh = _case(name)
    ns = 1 if sh is None else len(sh)
    c = _random_cot(np.random.default_rng(5), (1, ns, 2, p.Ntot, p.N))
    wa = _wa(p, len(pc), name)
    want = wa.final_state_vjp(pc[None, :], c, sh)["vjp"]
    assert wa.last_kernel == 9
    errs = {}
    for nseg in (0, 3, 1):
        wa.set_time_segments(nseg)
        try:
            got = wa.final_state_vjp(pc[None, :], c, sh, time_parallel=True)["vjp"]
        except Exception as e:
            assert name not in MUST_SERVE, (name, str(e))
            wa.close()
            pytest.skip(f"{name}: {e}")
        assert wa.last_kernel == 7 and (nseg == 0 or int(wa.query(7)) == nseg)
        errs[int(wa.query(7))] = _rel(got, want)
    wa.close()
    print(f"{name}: relative difference to kernel 9 by segment count {errs}")
    assert max(errs.values()) <= TOL_K9, (name, errs)


@pytest.mark.gpu
def test_infidelity_cotangent_reproduces_kernel7_infidgrad():
    """c = dinfid/d(Re U, Im U) pins the sign and layout of the terminal value: kernel 7's own infidgrad at the same segments."""
    cfg, _ = golden_config("cnot2-leakieq")
    p = cfg.params
    p.objFuncType = 3
    pc = np.asarray(cfg.pcof0, dtype=np.float64)
    wa = _wa(p, len(pc), "cnot2-leakieq", 5, required=True)      # kernel 7 serves this golden (test_gpu_timeparallel.py)
    U = wa.final_state_vjp(pc[None, :], None, final_state=True, time_parallel=True)["state"]
    c = _infid_cot(p, U, p.globalPhase)[:, :, None]
    got = wa.final_state_vjp(pc[None, :], c, time_parallel=True)["vjp"][0, 0, 0]
    wa.set_kernel(7)
    want = wa.evaluate(pc[None, :])["infidgrad"][0, 0]
    assert wa.last_kernel == 7 and int(wa.query(7)) == 5
    wa.close()
    err = _rel(got, want)
    print(f"cnot2-leakieq: relative |vjp(dinfid/dU) - kernel 7 infidgrad| = {err:.3e}")
    assert err <= TOL_K7, err


@pytest.mark.gpu
@pytest.mark.parametrize("pfid", [1, 3, 4])
def test_infidelity_cotangent_reproduces_kernel1_infidgrad(pfid):
    cfg, pc = _small_swap()
    p = cfg.params
    p.pFidType, p.globalPhase, p.objFuncType = pfid, 0.37, 3
    pc = np.concatenate([pc, [0.37]]) if pfid == 3 else pc
    wa = _wa(p, len(pc), "swap02", required=True)
    U = wa.final_state_vjp(pc[None, :], None, final_state=True, time_parallel=True)["state"]
    c = _infid_cot(p, U, pc[-1] if pfid == 3 else p.globalPhase)[:, :, None]
    got = wa.final_state_vjp(pc[None, :], c, time_parallel=True)["vjp"][0, 0, 0]
    wa.set_kernel(1)
    want = wa.evaluate(pc[None, :])["infidgrad"][0, 0]
    wa.close()
    if pfid == 3:                           # U(T) does not depend on the phase
        assert got[-1] == 0.0
        got, want = got[:-1], want[:-1]
    err = _rel(got, want)
    print(f"pFidType {pfid}: relative |vjp(dinfid/dU) - kernel 1 infidgrad| = {err:.3e}")
    assert err <= TOL_K9, err


@pytest.mark.gpu
@pytest.mark.parametrize("name,T,nsteps,scale", [("rabi", 10.0, 12, 20.0), ("risk_neutral", 30.0, 160, 40.0), ("cnot2", 6.0, 90, 60.0)])
def test_coarse_time_steps_engage_the_refinement(name, T, nsteps, scale):
    """The coarse-step problems of test_gpu_timeparallel.py, where the refinement passes of the backward boundary states must run."""
    from juqbox_b200 import configs
    cfg = configs.example(name)
    cfg.params.T, cfg.params.nsteps = T, nsteps
    pc = configs.synthetic_pcof(cfg, 2) * scale
    c = _random_cot(np.random.default_rng(9), (2, 1, 2, cfg.params.Ntot, cfg.params.N))
    wa = _wa(cfg.params, cfg.nCoeff, name, 3)
    got = wa.final_state_vjp(pc, c, time_parallel=True)["vjp"]
    want = wa.final_state_vjp(pc, c)["vjp"]
    wa.close()
    err = _rel(got, want)
    print(f"{name} ({nsteps} steps): relative difference to kernel 9 = {err:.3e}")
    assert err <= TOL_K9, err


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cnot2", "risk_neutral"])
def test_state_matches_forward_history_and_the_state_only_call(name):
    p, pc, sh = _case(name)
    ns = 1 if sh is None else len(sh)
    pcs = np.stack([pc, 0.6 * pc])
    wa = _wa(p, len(pc), name, 4)
    only = wa.final_state_vjp(pcs, None, sh, final_state=True, time_parallel=True)["state"]
    assert wa.last_kernel == 7 and int(wa.query(2)) == 3
    with_cot = [wa.final_state_vjp(pcs, _random_cot(np.random.default_rng(k), (2, ns, k, p.Ntot, p.N)), sh, final_state=True,
                                   time_parallel=True)["state"] for k in (1, 2)]
    wa.set_kernel(1)
    hist = wa.forward_history(pcs, sh, save_every=p.nsteps)[0][:, :, -1].swapaxes(-1, -2)
    wa.close()
    assert all(np.array_equal(only, u) for u in with_cot)
    err = _rel(only, hist)
    print(f"{name}: relative |U(T) - forward_history| = {err:.3e}")
    assert err <= TOL_STATE, err


@pytest.mark.gpu
def test_batching_repeatability_and_linearity():
    cfg, pc = _small_swap()
    p = cfg.params
    rng = np.random.default_rng(13)
    pcs = np.stack([pc, -0.8 * pc])
    cots = _random_cot(rng, (2, 2, 3, p.Ntot, p.N))
    wa = _wa(p, len(pc), "swap02", 6, required=True)
    full = wa.final_state_vjp(pcs, cots, SHIFTS, final_state=True, time_parallel=True)
    again = wa.final_state_vjp(pcs, cots, SHIFTS, final_state=True, time_parallel=True)
    assert np.array_equal(full["vjp"], again["vjp"]) and np.array_equal(full["state"], again["state"])
    errs = []
    for b in range(2):
        for s in range(2):
            for k in range(3):
                one = wa.final_state_vjp(pcs[b:b + 1], cots[b:b + 1, s:s + 1, k:k + 1], SHIFTS[s:s + 1], final_state=True, time_parallel=True)
                errs.append(_rel(one["vjp"][0, 0, 0], full["vjp"][b, s, k]))
                assert np.array_equal(one["state"][0, 0], full["state"][b, s])
    c, e = _random_cot(rng, (2, p.Ntot, p.N))
    al, be = 0.7, -2.3
    v = wa.final_state_vjp(pc[None, :], np.stack([c, e, al * c + be * e])[None, None], time_parallel=True)["vjp"][0, 0]
    wa.close()
    lin = _rel(v[2], al * v[0] + be * v[1])
    print(f"batched vs one at a time: {max(errs):.3e}; linearity {lin:.3e}")
    assert max(errs) <= 1e-13, errs
    assert lin <= 1e-12, lin


@pytest.mark.gpu
def test_reporting_and_the_kernel_preference():
    cfg, pc = _small_swap()
    p = cfg.params
    c = _random_cot(np.random.default_rng(2), (1, 1, 1, p.Ntot, p.N))
    wa = _wa(p, len(pc), "swap02", 5, required=True)
    wa.set_kernel(3)                        # a preference the time-parallel VJP ignores and leaves in place
    wa.final_state_vjp(pc[None, :], c, time_parallel=True)
    assert wa.last_kernel == 7 and int(wa.query(7)) == 5 and wa.last_kernel_ms > 0.0 and int(wa.query(2)) == 12
    wa.final_state_vjp(pc[None, :], c)
    assert wa.last_kernel == 9
    wa.evaluate(pc[None, :])
    assert wa.last_kernel == 3
    wa.close()


def _rejection_codes(p, npar, ncot=1, both_null=False, null_vjp=False, no_state=False):
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    wa = jq.Working_Arrays(p, npar)
    buf = np.zeros(16 * npar * p.Ntot * p.N)
    P = buf.ctypes.data_as(C.c_void_p)
    pcof = np.zeros(npar)
    cot = None if both_null else P
    rc = lib.jq_final_state_vjp_time_parallel(wa._handle, 1, pcof.ctypes.data_as(C.c_void_p), npar, 1, None, ncot, cot, cot,
                                              None if null_vjp else P, None if no_state else P, None if no_state else P)
    msg = _lib.last_error()
    wa.close()
    return rc, msg


@pytest.mark.gpu
def test_rejections():
    cfg, _ = golden_config("cnot2-jacobi")
    rc, msg = _rejection_codes(cfg.params, len(cfg.pcof0))
    assert rc == -1 and "time-parallel" in msg, msg
    pd, pc = _dense_weight_params(2)
    rc, msg = _rejection_codes(pd, len(pc))
    assert rc == -1 and "time-parallel" in msg, msg
    pu, pc = _uncoupled_params("antisymmetric")
    rc, msg = _rejection_codes(pu, len(pc))
    assert rc == -1 and "time-parallel" in msg, msg
    cfg, pc = _small_swap()
    p, npar = cfg.params, len(pc)
    assert _rejection_codes(p, npar)[0] == 0
    for kw, what in (({"ncot": -1}, "ncot >= 0"), ({"both_null": True}, "cot_r, cot_i"), ({"null_vjp": True}, "null vjp"),
                     ({"ncot": 0, "no_state": True}, "state_r or state_i")):
        rc, msg = _rejection_codes(p, npar, **kw)
        assert rc == -1 and what in msg and "jq_final_state_vjp_time_parallel" in msg, (kw, msg)
    assert _rejection_codes(p, npar, ncot=0, null_vjp=True, both_null=True)[0] == 0      # U(T) only: cotangents and vjp ignored


def _torch_loss(p, U):
    """A custom loss of U(T): the population of column 0 outside the first two levels plus a gate infidelity on the first N rows."""
    import torch
    V = torch.tensor(p.Utarget_r + 1j * p.Utarget_i, device=U.device)[: p.N]
    pop = (U[..., 2:, 0].abs() ** 2).sum(dim=-1)
    S = (U[..., : p.N, :].conj() * V).sum(dim=(-2, -1)) / p.N
    return (pop + 1.0 - S.abs() ** 2).sum()


@pytest.mark.gpu
@pytest.mark.parametrize("shifts", [None, SHIFTS])
def test_torch_custom_loss_matches_the_serial_path(shifts):
    import torch
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    wa = _wa(p, len(pc), "swap02", required=True)
    out = {}
    for tp in (False, True):
        x = torch.tensor(pc[None, :], dtype=torch.float64, device="cuda", requires_grad=True)
        loss = _torch_loss(p, jq.final_state(wa, x, shifts, time_parallel=tp))
        loss.backward()
        assert wa.last_kernel == (7 if tp else 9)
        out[tp] = (float(loss.detach()), x.grad.cpu().numpy()[0])
    wa.close()
    ev = abs(out[True][0] - out[False][0]) / abs(out[False][0])
    eg = _rel(out[True][1], out[False][1])
    print(f"torch custom loss, {1 if shifts is None else len(shifts)} sample(s): value {ev:.3e}, gradient {eg:.3e}")
    assert ev <= 1e-12 and eg <= TOL_K9, (ev, eg)
