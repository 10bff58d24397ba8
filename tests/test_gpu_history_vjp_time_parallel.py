"""History vector-Jacobian products on the time-parallel path (jq_history_vjp_time_parallel, kernel 7 stages).

Pinned against the serial VJP kernel (jq_history_vjp, kernel 9), which applies the same cotangent jumps to the same unforced adjoint
sweep in one pass; against the final-state VJP on the same path (the last block alone, bit for bit); and the saved states against
forward_history on kernel 1.  Tests marked gpu need a device; the others check the binding and the wrappers without one."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_final_state_vjp import SHIFTS, _random_cot, _rel, _small_swap, _uncoupled_params
from test_gpu_final_state_vjp_time_parallel import MUST_SERVE, TOL_K9, TOL_STATE, _case, _no_lib_wa, _wa
from test_gpu_forward_sensitivity import _dense_weight_params
from test_gpu_state_history import _LinearStandIn, _coarse, _population_loss
from helpers import golden_config


class _TimeParallelStandIn(_LinearStandIn):
    """The linear stand-in of test_gpu_state_history with the time-parallel entry: the history alone for cot=None."""

    def __init__(self):
        super().__init__()
        self.calls = []

    def history_vjp(self, pcof, cot, shifts=None, save_every=1, history=False, time_parallel=False):
        self.calls.append((cot is None, history, time_parallel))
        out = {} if cot is None else super().history_vjp(pcof, cot, shifts, save_every)
        if history:
            out["history"] = np.einsum("sjiap,bp->bsjia", self._a(shifts, save_every), pcof)
        return out


# ---------------------------------------------------------------------------------------------------------------- no device needed
def test_symbol_exported_and_null_handle_rejected():
    from juqbox_b200 import _lib
    lib = _lib.load()
    assert "jq_history_vjp_time_parallel" in _lib.EXPORTS and hasattr(lib, "jq_history_vjp_time_parallel")
    one = np.zeros(64)
    p = one.ctypes.data_as(C.c_void_p)
    assert lib.jq_history_vjp_time_parallel(None, 1, p, 64, 1, None, 1, 1, p, p, p, None, None) == -1       # JQ_ERR_ARG
    assert "handle" in _lib.last_error()


def test_wrapper_rejects_malformed_inputs_before_the_library():
    wa, npar, n, m = _no_lib_wa()
    nsteps = wa.params.nsteps
    nsave = nsteps + 1
    pc = np.zeros((2, npar))
    for bad in (np.zeros((2, 1, 1, nsave, n, m, 1)), np.zeros((2, 1, nsave, n, m)), np.zeros((2, 1, 0, nsave, n, m)),
                np.zeros((1, 1, 1, nsave, n, m)), np.zeros((2, 2, 1, nsave, n, m)), np.zeros((2, 1, 1, nsave + 1, n, m)),
                np.zeros((2, 1, 1, nsave, m, n + 1)), np.zeros((2, 1, 1, nsave, n, m + 1))):
        with pytest.raises(ValueError):
            wa.history_vjp(pc, bad, save_every=1, time_parallel=True)
    with pytest.raises(ValueError):         # shifts not [nsamples, Ntot]
        wa.history_vjp(pc, np.zeros((2, 3, 1, nsave, n, m)), np.zeros((3, n + 1)), 1, time_parallel=True)
    with pytest.raises(ValueError):         # cot for 2 samples, shifts for 3
        wa.history_vjp(pc, np.zeros((2, 2, 1, nsave, n, m)), np.zeros((3, n)), 1, time_parallel=True)
    for se in (0, -1, nsteps + 1, 1.5):    # save_every, also for the history-only call
        with pytest.raises(ValueError, match="saveEvery"):
            wa.history_vjp(pc, np.zeros((2, 1, 1, nsave, n, m)), save_every=se, time_parallel=True)
        with pytest.raises(ValueError, match="saveEvery"):
            wa.history_vjp(pc, None, save_every=se, history=True, time_parallel=True)
    with pytest.raises(ValueError):         # shifts of the history-only call
        wa.history_vjp(pc, None, np.zeros((3, n + 1)), 1, history=True, time_parallel=True)


@pytest.mark.parametrize("history,time_parallel", [(False, False), (True, False), (False, True)])
def test_cot_none_needs_the_time_parallel_history_call(history, time_parallel):
    wa, npar, _, _ = _no_lib_wa()
    with pytest.raises(ValueError, match="cot=None"):
        wa.history_vjp(np.zeros((1, npar)), None, save_every=1, history=history, time_parallel=time_parallel)


@pytest.mark.parametrize("shifts,save_every", [(None, 1), (np.zeros((2, 3)), 2)])
def test_state_history_time_parallel_plumbing_on_a_linear_stand_in(shifts, save_every):
    """The torch function with time_parallel=True: the forward pass is the history-only call, the backward pass one time-parallel
    history VJP."""
    torch = pytest.importorskip("torch")
    import juqbox_b200 as jq
    wa = _TimeParallelStandIn()
    pc = torch.tensor(np.random.default_rng(1).standard_normal((3, 5)), dtype=torch.float64, requires_grad=True)
    U = jq.state_history(wa, pc, shifts, save_every, time_parallel=True)
    assert U.shape == (3, 1 if shifts is None else 2, 4 // save_every + 1, 3, 2) and U.dtype == torch.complex128
    assert wa.calls == [(True, True, True)]
    (U.abs() ** 2).sum().backward()
    assert wa.calls[-1] == (False, False, True)
    assert torch.autograd.gradcheck(lambda x: jq.state_history(wa, x, shifts, save_every, time_parallel=True), (pc,), eps=1e-6,
                                    atol=1e-9, rtol=1e-7)


# ---------------------------------------------------------------------------------------------------------------- on the GPU
def _boundary_stride(nsteps):
    """(nseg, save_every) with saves exactly on every segment boundary: nseg a divisor of nsteps, save_every = nsteps / nseg; for a
    prime nsteps (risk-neutral: 7937) save_every = 1, where every boundary carries a save."""
    nseg = next((d for d in (7, 6, 5, 4, 3, 2) if nsteps % d == 0), None)
    return (nseg, nsteps // nseg) if nseg else (3, 1)


def _odd_stride(nsteps):
    """A coarse save_every that does not divide the length of 3 segments (so saves fall anywhere inside them)."""
    for d in range(2, nsteps + 1):
        if nsteps % d == 0 and nsteps // d <= 60 and (nsteps // 3) % d != 0:
            return d
    return _coarse(nsteps)


@pytest.mark.gpu
@pytest.mark.parametrize("stride", ["every", "coarse", "boundary"])
@pytest.mark.parametrize("name", ["cnot1", "cnot2", "cnot3", "risk_neutral", "swap02", "rabi", "cnot2-leakieq"])
def test_agrees_with_the_serial_history_vjp(name, stride):
    """Random complex cotangents at every save through the time-parallel history VJP (automatic, 3 and 1 segments; for the boundary
    stride also the segment count that puts a save on every boundary) and kernel 9."""
    p, pc, sh = _case(name)
    ns = 1 if sh is None else len(sh)
    segs = [0, 3, 1]
    if stride == "every":
        se = 1
    elif stride == "coarse":
        se = _odd_stride(p.nsteps)
    else:
        nb, se = _boundary_stride(p.nsteps)
        segs = sorted({nb, 2 * nb if p.nsteps % (2 * nb) == 0 else nb})
    nsave = p.nsteps // se + 1
    c = _random_cot(np.random.default_rng(5), (1, ns, 1, nsave, p.Ntot, p.N))
    wa = _wa(p, len(pc), name)
    want = wa.history_vjp(pc[None, :], c, sh, se)["vjp"]
    assert wa.last_kernel == 9
    errs = {}
    for nseg in segs:
        wa.set_time_segments(nseg)
        try:
            got = wa.history_vjp(pc[None, :], c, sh, se, time_parallel=True)["vjp"]
        except Exception as e:
            assert name not in MUST_SERVE, (name, str(e))
            wa.close()
            pytest.skip(f"{name}: {e}")
        assert wa.last_kernel == 7 and (nseg == 0 or int(wa.query(7)) == nseg)
        errs[int(wa.query(7))] = _rel(got, want)
    wa.close()
    print(f"{name}, save_every {se}: relative difference to kernel 9 by segment count {errs}")
    assert max(errs.values()) <= TOL_K9, (name, se, errs)


@pytest.mark.gpu
def test_one_step_per_segment():
    """rabi with nseg = nsteps: every segment is one step, every boundary carries a jump."""
    p, pc, sh = _case("rabi")
    c = _random_cot(np.random.default_rng(6), (1, 1, 2, p.nsteps + 1, p.Ntot, p.N))
    wa = _wa(p, len(pc), "rabi", p.nsteps, required=True)
    got = wa.history_vjp(pc[None, :], c, sh, 1, time_parallel=True)["vjp"]
    assert wa.last_kernel == 7 and int(wa.query(7)) == p.nsteps
    want = wa.history_vjp(pc[None, :], c, sh, 1)["vjp"]
    wa.close()
    err = _rel(got, want)
    print(f"rabi, {p.nsteps} segments of one step: relative difference to kernel 9 = {err:.3e}")
    assert err <= TOL_K9, err


@pytest.mark.gpu
def test_single_jumps_around_a_segment_boundary():
    """A cotangent nonzero in one intermediate block only: on a segment boundary, one step either side of it, and mid-segment."""
    cfg, pc = _small_swap()
    p = cfg.params
    nseg = 3
    k0 = p.nsteps // nseg                   # first boundary: the start of segment 1
    rng = np.random.default_rng(17)
    wa = _wa(p, len(pc), "swap02", nseg, required=True)
    errs = {}
    for j in (k0, k0 - 1, k0 + 1, k0 + k0 // 2):
        c = np.zeros((1, 1, 1, p.nsteps + 1, p.Ntot, p.N), dtype=complex)
        c[0, 0, 0, j] = _random_cot(rng, (p.Ntot, p.N))
        got = wa.history_vjp(pc[None, :], c, save_every=1, time_parallel=True)["vjp"]
        assert int(wa.query(7)) == nseg
        want = wa.history_vjp(pc[None, :], c, save_every=1)["vjp"]
        errs[j] = _rel(got, want)
    wa.close()
    print(f"single jumps (boundary at step {k0}): {errs}")
    assert max(errs.values()) <= TOL_K9, errs


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cnot2", "risk_neutral"])
def test_last_block_cotangent_gives_the_final_state_vjp_bits(name):
    p, pc, sh = _case(name)
    ns = 1 if sh is None else len(sh)
    se = _coarse(p.nsteps)
    nsave = p.nsteps // se + 1
    c = _random_cot(np.random.default_rng(3), (1, ns, 2, p.Ntot, p.N))
    ch = np.zeros((1, ns, 2, nsave, p.Ntot, p.N), dtype=complex)
    ch[:, :, :, -1] = c
    wa = _wa(p, len(pc), name, 5)
    want = wa.final_state_vjp(pc[None, :], c, sh, time_parallel=True)["vjp"]
    got = wa.history_vjp(pc[None, :], ch, sh, se, time_parallel=True)["vjp"]
    wa.close()
    assert np.array_equal(got, want), _rel(got, want)


@pytest.mark.gpu
def test_batching_and_the_history_only_call():
    """Batch 2 x 2 samples x 3 cotangents gives the bits of one trajectory at a time; the history of the ncot = 0 call is the history
    returned with 1 and 2 cotangents, and agrees with forward_history on kernel 1 (block 0 exactly Uinit)."""
    cfg, pc = _small_swap()
    p = cfg.params
    se = 50
    nsave = p.nsteps // se + 1
    rng = np.random.default_rng(13)
    pcs = np.stack([pc, -0.8 * pc])
    cots = _random_cot(rng, (2, 2, 3, nsave, p.Ntot, p.N))
    wa = _wa(p, len(pc), "swap02", 6, required=True)
    full = wa.history_vjp(pcs, cots, SHIFTS, se, history=True, time_parallel=True)
    for b in range(2):
        for s in range(2):
            for k in range(3):
                one = wa.history_vjp(pcs[b:b + 1], cots[b:b + 1, s:s + 1, k:k + 1], SHIFTS[s:s + 1], se, history=True, time_parallel=True)
                assert np.array_equal(one["vjp"][0, 0, 0], full["vjp"][b, s, k]), (b, s, k)
                assert np.array_equal(one["history"][0, 0], full["history"][b, s])
    only = wa.history_vjp(pcs, None, SHIFTS, se, history=True, time_parallel=True)
    assert set(only) == {"history"} and wa.last_kernel == 7 and int(wa.query(2)) == 3
    with1 = wa.history_vjp(pcs, cots[:, :, :1], SHIFTS, se, history=True, time_parallel=True)["history"]
    with2 = wa.history_vjp(pcs, cots[:, :, :2], SHIFTS, se, history=True, time_parallel=True)["history"]
    assert np.array_equal(only["history"], with1) and np.array_equal(only["history"], with2)
    assert np.array_equal(only["history"], full["history"])
    wa.set_kernel(1)
    ref = wa.forward_history(pcs, SHIFTS, save_every=se)[0].swapaxes(-1, -2)
    wa.close()
    U0 = np.asarray(p.Uinit)
    assert np.array_equal(only["history"][:, :, 0], np.broadcast_to(U0, only["history"][:, :, 0].shape))
    err = _rel(only["history"], ref)
    print(f"history against forward_history on kernel 1: {err:.3e}")
    assert err <= TOL_STATE, err


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cnot2", "cnot3", "risk_neutral"])
def test_history_matches_forward_history(name):
    p, pc, sh = _case(name)
    se = _coarse(p.nsteps)
    wa = _wa(p, len(pc), name)
    got = wa.history_vjp(pc[None, :], None, sh, se, history=True, time_parallel=True)["history"]
    wa.set_kernel(1)
    ref = wa.forward_history(pc[None, :], sh, save_every=se)[0].swapaxes(-1, -2)
    wa.close()
    assert np.array_equal(got[:, :, 0], ref[:, :, 0])
    err = _rel(got, ref)
    print(f"{name}: relative |history - forward_history| = {err:.3e}")
    assert err <= TOL_STATE, err


def _rejection(p, npar, save_every=1, ncot=1, both_null=False, null_vjp=False, no_hist=False):
    """(return code, message, launches reported before, after) of one call of the C entry."""
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    wa = jq.Working_Arrays(p, npar)
    pcof = np.zeros(npar)
    wa.evaluate(pcof[None, :])              # some launch count to compare with
    before = int(wa.query(2))
    nsave = p.nsteps // max(save_every, 1) + 1
    buf = np.zeros(4 * max(ncot, 1) * nsave * p.Ntot * p.N + 4 * npar)
    P = buf.ctypes.data_as(C.c_void_p)
    cot = None if both_null else P
    rc = lib.jq_history_vjp_time_parallel(wa._handle, 1, pcof.ctypes.data_as(C.c_void_p), npar, 1, None, save_every, ncot, cot, cot,
                                          None if null_vjp else P, None if no_hist else P, None if no_hist else P)
    msg = _lib.last_error()
    after = int(wa.query(2))
    wa.close()
    return rc, msg, before, after


@pytest.mark.gpu
def test_rejections():
    cfg, _ = golden_config("cnot2-jacobi")
    for p, pc in ((cfg.params, cfg.pcof0), _dense_weight_params(2), _uncoupled_params("antisymmetric")):
        rc, msg, before, after = _rejection(p, len(pc))
        assert rc == -1 and "time-parallel" in msg and before == after, msg
    cfg, pc = _small_swap()
    p, npar = cfg.params, len(pc)
    assert _rejection(p, npar)[0] == 0
    for kw, what in (({"save_every": 0}, "saveEvery"), ({"save_every": p.nsteps + 1}, "saveEvery"), ({"ncot": -1}, "ncot >= 0"),
                     ({"both_null": True}, "cot_r, cot_i"), ({"null_vjp": True}, "null vjp"), ({"ncot": 0, "no_hist": True}, "hist_r or hist_i")):
        rc, msg, before, after = _rejection(p, npar, **kw)
        assert rc == -1 and what in msg and before == after, (kw, msg)
    assert _rejection(p, npar, ncot=0, null_vjp=True, both_null=True)[0] == 0      # the history only: cotangents and vjp ignored


@pytest.mark.gpu
def test_trajectory_limit_is_rejected_without_a_launch():
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    cfg, pc = _small_swap()
    p, npar = cfg.params, len(pc)
    wa = jq.Working_Arrays(p, npar)
    wa.evaluate(pc[None, :])
    before = int(wa.query(2))
    one = np.zeros((1 << 12) * max(npar, p.Ntot))
    P = one.ctypes.data_as(C.c_void_p)
    rc = lib.jq_history_vjp_time_parallel(wa._handle, 1 << 12, P, npar, 1 << 10, P, 1, 1 << 10, P, P, P, None, None)
    msg = _lib.last_error()
    after = int(wa.query(2))
    wa.close()
    assert rc == -1 and "2^31 - 1" in msg and before == after, msg


@pytest.mark.gpu
@pytest.mark.parametrize("nsamples", [1, 2])
def test_torch_loss_on_intermediate_populations_matches_the_serial_path(nsamples):
    import torch
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    se = 100
    nsave = p.nsteps // se + 1
    w = torch.linspace(0.0, 2.0, nsave, dtype=torch.float64) ** 2
    sh = SHIFTS[:nsamples]
    wa = _wa(p, len(pc), "swap02", required=True)
    out = {}
    for tp in (False, True):
        x = torch.tensor(pc[None, :], dtype=torch.float64, device="cuda", requires_grad=True)
        loss = _population_loss(jq.state_history(wa, x, sh, se, time_parallel=tp), w.to("cuda"))
        loss.backward()
        assert wa.last_kernel == (7 if tp else 9)
        out[tp] = (float(loss.detach()), x.grad.cpu().numpy()[0])
    wa.close()
    ev = abs(out[True][0] - out[False][0]) / abs(out[False][0])
    eg = _rel(out[True][1], out[False][1])
    print(f"torch population loss, {nsamples} sample(s): value {ev:.3e}, gradient {eg:.3e}")
    assert ev <= 1e-12 and eg <= TOL_K9, (ev, eg)


@pytest.mark.gpu
def test_no_two_set_gradient_sweep_is_rejected_for_cotangents():
    """A single 3-level qudit: kernel 7 serves it (fibre layout, three rows per lane), the history alone is returned, but no two-set
    fibre segment sweep exists for that layout, so a call with cotangents is rejected without a launch."""
    import juqbox_b200 as jq
    from juqbox_b200 import _lib, configs
    lib = _lib.load()
    cfg = configs.qudit_system([2], [1], T=10.0)
    p, npar = cfg.params, cfg.nCoeff
    wa = jq.Working_Arrays(p, npar)
    wa.set_kernel(7)                        # kernel 7 serves the shape ...
    wa.set_kernel(0)
    pc = configs.synthetic_pcof(cfg, 1)
    hist = wa.history_vjp(pc, None, save_every=p.nsteps, history=True, time_parallel=True)["history"]
    assert wa.last_kernel == 7 and hist.shape == (1, 1, 2, p.Ntot, p.N)
    before = int(wa.query(2))
    nsave = 2
    buf = np.zeros(4 * nsave * p.Ntot * p.N + 4 * npar)
    P = buf.ctypes.data_as(C.c_void_p)
    rc = lib.jq_history_vjp_time_parallel(wa._handle, 1, pc.ctypes.data_as(C.c_void_p), npar, 1, None, p.nsteps, 1, P, P, P, None, None)
    msg = _lib.last_error()
    after = int(wa.query(2))
    wa.close()
    assert rc == -1 and "second adjoint set" in msg and before == after, msg


@pytest.mark.gpu
def test_histories_larger_than_the_device_are_an_allocation_error():
    """Cotangent histories of ~200 GB: JQ_ERR_ALLOC with the size, before anything is copied or launched."""
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    cfg, pc = _small_swap()
    p, npar = cfg.params, len(pc)
    nsave = p.nsteps + 1
    nbatch = int(2.0e11 / (16.0 * nsave * p.Ntot * p.N)) + 1         # two cotangent parts of 8 bytes per entry
    wa = jq.Working_Arrays(p, npar)
    wa.set_time_segments(1)
    wa.evaluate(pc[None, :])
    before = int(wa.query(2))
    pcof = np.tile(pc, (nbatch, 1))
    small = np.zeros(64)
    S = small.ctypes.data_as(C.c_void_p)
    rc = lib.jq_history_vjp_time_parallel(wa._handle, nbatch, pcof.ctypes.data_as(C.c_void_p), npar, 1, None, 1, 1, S, S, S, None, None)
    msg = _lib.last_error()
    after = int(wa.query(2))
    wa.close()
    assert rc == -4 and "GB" in msg and "jq_history_vjp_time_parallel" in msg and before == after, msg
