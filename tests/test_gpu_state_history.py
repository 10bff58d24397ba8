"""Derivatives of the state history: jq_history_vjp (reverse mode), jq_history_jvp (forward mode) and juqbox_b200.state_history.

Save j is the state U_j after step j * save_every (U_0 = Uinit).  The VJP is pinned against the forward tangent of every save (the
dot-product identity <vjp(c), d> = sum_j Re vdot(c_j, dU_j . d)), the tangents against central differences of forward_history, and
both against the final-state routes they extend (bit for bit).  Tests marked gpu need a device; the others check the binding and the
torch wrapper without one."""
import ctypes as C
import types

import numpy as np
import pytest

from helpers import golden_config
from test_gpu_final_state_vjp import SHIFTS, _dot_case, _random_cot, _rel, _small_swap

TOL_DOT = 1e-9      # dot-product identity against the forward tangent (two independent routes)
# cnot3 (32386 steps): the backward sweep's recomputed states drift from the forward ones over the long loop.  A cotangent on U(T)
# alone, which is final_state_vjp bit for bit, gives 9e-11 ... 2.2e-8 here depending on the random cotangent; these fixed inputs give
# 1.24e-9 at the coarse stride and 2.0e-10 at save_every = 1 (profiles/r06_state_history.md).
TOL_DOT_CNOT3 = 2e-9


def _coarse(nsteps):
    """The smallest save_every that leaves at most 41 saves."""
    return next(d for d in range(2, nsteps + 1) if nsteps % d == 0 and nsteps // d <= 40)


class _LinearStandIn:
    """A stand-in for Working_Arrays: U(t_k) = A_k pcof, a fixed complex linear map per sample and step, with history_vjp its exact
    adjoint under the library's convention vjp_p = sum_j Re vdot(c_j, A_j[..., p])."""

    def __init__(self, nsamples=2, Ntot=3, N=2, npar=5, nsteps=4):
        rng = np.random.default_rng(0)
        self.params = types.SimpleNamespace(nsteps=nsteps, Ntot=Ntot, N=N)
        self.A = _random_cot(rng, (nsamples, nsteps + 1, Ntot, N, npar))
        self.A[:, 0] = 0.0                                                  # U_0 = Uinit does not depend on pcof

    def _a(self, shifts, save_every):
        return self.A[:1 if shifts is None else len(shifts), ::save_every]

    def forward_history(self, pcof, shifts=None, save_every=1):
        U = np.einsum("sjiap,bp->bsjia", self._a(shifts, save_every), pcof)
        return U.swapaxes(-1, -2), None, None                               # [nbatch, nsamples, nsave, N, Ntot]

    def history_vjp(self, pcof, cot, shifts=None, save_every=1, history=False):
        return {"vjp": np.einsum("bskjia,sjiap->bskp", cot.conj(), self._a(shifts, save_every)).real}


# ---------------------------------------------------------------------------------------------------------------- no device needed
def test_symbols_exported_and_null_handle_rejected():
    from juqbox_b200 import _lib
    lib = _lib.load()
    one = np.zeros(64)
    p = one.ctypes.data_as(C.c_void_p)
    for name in ("jq_history_vjp", "jq_history_jvp"):
        assert name in _lib.EXPORTS and hasattr(lib, name)
    assert lib.jq_history_vjp(None, 1, p, 64, 1, None, 1, 1, p, p, p, None, None) == -1          # JQ_ERR_ARG
    assert "handle" in _lib.last_error()
    assert lib.jq_history_jvp(None, 1, p, 64, 1, None, 1, 1, p, p, p) == -1
    assert "handle" in _lib.last_error()


def test_wrappers_reject_malformed_inputs_before_the_library():
    import juqbox_b200 as jq
    from juqbox_b200 import configs

    class NoLib:                            # any call into the library fails the test
        def __getattr__(self, name):
            raise AssertionError(f"library called: {name}")
    cfg = configs.example("rabi")
    p = cfg.params
    wa = jq.Working_Arrays.__new__(jq.Working_Arrays)
    wa.params, wa._lib, wa._handle = p, NoLib(), None
    wa._snapshot = wa._fingerprint(p)
    npar, n, m, ns = cfg.nCoeff, p.Ntot, p.N, p.nsteps + 1
    pc = np.zeros((2, npar))
    for bad in (np.zeros((2, 1, 1, ns, n, m, 1)), np.zeros((2, 1, 1, n, m)), np.zeros((2, 1, 0, ns, n, m)),
                np.zeros((1, 1, 1, ns, n, m)), np.zeros((2, 2, 1, ns, n, m)), np.zeros((2, 1, 1, ns - 1, n, m)),
                np.zeros((2, 1, 1, ns, m, n + 1)), np.zeros((2, 1, 1, ns, n, m + 1))):
        with pytest.raises(ValueError):
            wa.history_vjp(pc, bad)
    for bad in (np.zeros((2, npar)), np.zeros((2, 0, npar)), np.zeros((1, 1, npar)), np.zeros((2, 1, npar + 1))):
        with pytest.raises(ValueError):
            wa.history_jvp(pc, bad)
    good_c, good_d = np.zeros((2, 1, 1, ns, n, m)), np.zeros((2, 1, npar))
    for call in (lambda **k: wa.history_vjp(pc, good_c, **k), lambda **k: wa.history_jvp(pc, good_d, **k)):
        for se in (0, -1, p.nsteps + 1, 1.5):
            with pytest.raises(ValueError):
                call(save_every=se)
        with pytest.raises(ValueError):     # shifts not [nsamples, Ntot]
            call(shifts=np.zeros((1, n + 1)))
    with pytest.raises(ValueError):         # pcof not [nbatch, npar]
        wa.history_vjp(np.zeros(npar), good_c)
    with pytest.raises(ValueError):         # cot for 1 sample, shifts for 3
        wa.history_vjp(pc, good_c, np.zeros((3, n)))
    with pytest.raises(ValueError):         # cot for save_every = 1, called with save_every = nsteps
        wa.history_vjp(pc, good_c, save_every=p.nsteps)


@pytest.mark.parametrize("shifts,save_every", [(None, 1), (np.zeros((2, 3)), 1), (np.zeros((2, 3)), 2)])
def test_state_history_gradcheck_against_a_linear_stand_in(shifts, save_every):
    """The torch wrapper on CPU: gradcheck of U_j = A_j pcof pins the complex convention (cot_j = dL/dRe U_j + i dL/dIm U_j) and the
    axis order [nbatch, nsamples, nsave, Ntot, N]."""
    torch = pytest.importorskip("torch")
    import juqbox_b200 as jq
    wa = _LinearStandIn()
    pc = torch.tensor(np.random.default_rng(1).standard_normal((3, 5)), dtype=torch.float64, requires_grad=True)
    U = jq.state_history(wa, pc, shifts, save_every)
    ns = 1 if shifts is None else 2
    assert U.shape == (3, ns, 4 // save_every + 1, 3, 2) and U.dtype == torch.complex128
    want = np.einsum("sjiap,bp->bsjia", wa._a(shifts, save_every), pc.detach().numpy())
    assert np.array_equal(U.detach().numpy(), want)
    assert torch.autograd.gradcheck(lambda x: jq.state_history(wa, x, shifts, save_every), (pc,), eps=1e-6, atol=1e-9, rtol=1e-7)
    with pytest.raises(ValueError):
        jq.state_history(wa, pc.float())


# ---------------------------------------------------------------------------------------------------------------- on the GPU
@pytest.mark.gpu
@pytest.mark.parametrize("coarse", [False, True], ids=["every-step", "coarse"])
@pytest.mark.parametrize("name", ["swap02", "flux", "cnot2", "cnot3", "unc_symmetric", "unc_antisymmetric", "pfid3", "samples"])
def test_dot_product_identity_against_the_history_tangent(name, coarse):
    """<vjp(c), d> = sum_j Re vdot(c_j, dU_j . d) for 2 random cotangents on every save and 2 random directions per sample."""
    import juqbox_b200 as jq
    p, pc, shifts = _dot_case(name)
    se = _coarse(p.nsteps) if coarse else 1
    nsave = p.nsteps // se + 1
    ns = 1 if shifts is None else len(shifts)
    rng = np.random.default_rng(23)
    d = rng.standard_normal((2, len(pc)))
    c = _random_cot(rng, (1, ns, 2, nsave, p.Ntot, p.N))
    wa = jq.Working_Arrays(p, len(pc))
    v = wa.history_vjp(pc[None, :], c, shifts, se)["vjp"][0]              # [ns, ncot, npar]
    assert wa.last_kernel == 9 and v.shape == (ns, 2, len(pc))
    dU = wa.history_jvp(pc[None, :], d[None], shifts, se)[0]               # [ns, ndir, nsave, Ntot, N]
    assert wa.last_kernel == 8 and dU.shape == (ns, 2, nsave, p.Ntot, p.N)
    wa.close()
    assert np.all(dU[:, :, 0] == 0.0)
    lhs = np.einsum("skp,jp->skj", v, d)
    rhs = np.einsum("sktab,sjtab->skj", c[0].conj(), dU).real
    err = _rel(lhs, rhs)
    print(f"{name}, save_every {se}: relative |<vjp(c), d> - sum_j Re vdot(c_j, dU_j d)| = {err:.3e}")
    assert err <= (TOL_DOT_CNOT3 if name == "cnot3" else TOL_DOT), (name, se, err)
    if p.pFidType == 3:
        assert np.all(v[..., -1] == 0.0)


@pytest.mark.gpu
def test_intermediate_tangents_are_second_order_limit_of_central_differences():
    """The tangent of every save against (U_j(pc + eps d) - U_j(pc - eps d)) / 2 eps of forward_history.  The difference is O(eps^2):
    halving eps must divide it by 3 to 5, and at eps = 1e-2 (d of the size of the controls) it must be below 1e-7 relative."""
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    se = 100
    d = np.random.default_rng(7).standard_normal(len(pc))
    d *= np.abs(pc).max() / np.abs(d).max()
    wa = jq.Working_Arrays(p, len(pc))
    dU = wa.history_jvp(pc[None, :], d[None, None, :], save_every=se)[0, 0, 0][1:]      # saves 1 ... nsave - 1
    U = lambda x: wa.forward_history(x[None, :], save_every=se)[0][0, 0, 1:].swapaxes(-1, -2)
    errs, worst = [], []
    for eps in (2e-2, 1e-2):
        fd = (U(pc + eps * d) - U(pc - eps * d)) / (2 * eps)
        errs.append(_rel(dU, fd))
        worst.append(max(_rel(dU[j], fd[j]) for j in range(len(dU))))
    wa.close()
    print(f"history tangent vs central differences: {errs[0]:.3e} (eps), {errs[1]:.3e} (eps/2), ratio {errs[0] / errs[1]:.2f}; "
          f"worst single save {worst[1]:.3e}")
    assert 3.0 < errs[0] / errs[1] < 5.0 and errs[1] <= 1e-7 and worst[1] <= 1e-6, (errs, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["samples", "pfid3", "cnot2-jacobi"])
def test_last_block_cotangent_gives_the_final_state_vjp_bits(name):
    import juqbox_b200 as jq
    if name == "cnot2-jacobi":
        cfg, _ = golden_config(name)
        p, pc, sh = cfg.params, np.asarray(cfg.pcof0, dtype=np.float64), None
    else:
        p, pc, sh = _dot_case(name)
    ns = 1 if sh is None else len(sh)
    pcs = np.stack([pc, -0.7 * pc])
    se = _coarse(p.nsteps)
    nsave = p.nsteps // se + 1
    c = _random_cot(np.random.default_rng(5), (2, ns, 3, p.Ntot, p.N))
    ch = np.zeros((2, ns, 3, nsave, p.Ntot, p.N), dtype=complex)
    ch[:, :, :, -1] = c
    wa = jq.Working_Arrays(p, len(pc))
    want = wa.final_state_vjp(pcs, c, sh)["vjp"]
    got = wa.history_vjp(pcs, ch, sh, se)["vjp"]
    wa.close()
    assert np.array_equal(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["samples", "cnot2"])
def test_histories_equal_the_existing_routes_bit_for_bit(name):
    """hist of history_vjp = forward_history on kernel 1; the last tangent of history_jvp = forward_sensitivity's dstate."""
    import juqbox_b200 as jq
    if name == "cnot2":
        cfg, _ = golden_config("cnot2")
        p, pcs, sh = cfg.params, np.asarray(cfg.pcof0)[None, :], None
    else:
        cfg, pc = _small_swap()
        p, pcs, sh = cfg.params, np.stack([pc, -0.7 * pc]), SHIFTS
    ns = 1 if sh is None else len(sh)
    rng = np.random.default_rng(3)
    wa = jq.Working_Arrays(p, pcs.shape[1])
    for se in (1, _coarse(p.nsteps)):
        nsave = p.nsteps // se + 1
        c = _random_cot(rng, (len(pcs), ns, 2, nsave, p.Ntot, p.N))
        d = rng.standard_normal((len(pcs), 3, pcs.shape[1]))
        H = wa.history_vjp(pcs, c, sh, se, history=True)["history"]
        dH = wa.history_jvp(pcs, d, sh, se)
        wa.set_kernel(1)
        hist = wa.forward_history(pcs, sh, save_every=se)[0]
        assert wa.last_kernel == 1
        wa.set_kernel(0)
        dstate = wa.forward_sensitivity(pcs, d, sh, final_state=True)["dstate"]
        assert np.array_equal(H, hist.swapaxes(-1, -2)), se
        assert np.array_equal(dH[:, :, :, -1], dstate), se
    wa.close()


@pytest.mark.gpu
def test_state_history_last_save_equals_final_state():
    import torch
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    wa = jq.Working_Arrays(p, len(pc))
    x = torch.tensor(np.stack([pc, 0.5 * pc]), dtype=torch.float64, device="cuda")
    for sh in (None, SHIFTS):
        H = jq.state_history(wa, x, sh, save_every=200)
        assert H.device == x.device and H.shape == (2, 1 if sh is None else 2, p.nsteps // 200 + 1, p.Ntot, p.N)
        assert torch.equal(H[:, :, -1], jq.final_state(wa, x, sh))
    wa.close()


def _spline_index(p, pc):
    """(D1, k(t)): the coefficient i of a spline block (pcof index % D1 == i) enters the controls at time t only if i < k(t), with
    k(t) = min(max(ceil(t / dtknot + 2), 3), D1) as in bcarrier2."""
    nspl = len(pc) - (1 if p.pFidType == 3 else 0)
    D1 = nspl // (2 * (p.Ncoupled + p.Nunc) * p.Nfreq)
    dtknot = p.T / (D1 - 2)
    return D1, lambda t: min(max(int(np.ceil(t / dtknot + 2.0)), 3), D1)


@pytest.mark.gpu
def test_jump_placement():
    """A cotangent only at save j leaves every vjp entry whose spline support lies wholly after t_j + dt exactly 0; a direction
    supported wholly after t_j + dt leaves the tangents of saves 0 ... j exactly 0."""
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    se, j = 200, 3
    nsave = p.nsteps // se + 1
    dt = p.T / p.nsteps
    tj = j * se * dt
    D1, k = _spline_index(p, pc)
    late = (np.arange(len(pc)) % D1) >= k(tj + dt)           # never read at t <= t_j + dt
    assert late.any() and (~late).any()
    rng = np.random.default_rng(9)
    c = np.zeros((1, 1, 1, nsave, p.Ntot, p.N), dtype=complex)
    c[0, 0, 0, j] = _random_cot(rng, (p.Ntot, p.N))
    d = np.where(late, rng.standard_normal(len(pc)), 0.0)
    wa = jq.Working_Arrays(p, len(pc))
    v = wa.history_vjp(pc[None, :], c, save_every=se)["vjp"][0, 0, 0]
    dU = wa.history_jvp(pc[None, :], d[None, None, :], save_every=se)[0, 0, 0]
    wa.close()
    assert np.all(v[late] == 0.0) and np.any(v[~late] != 0.0)
    assert np.all(dU[:j + 1] == 0.0) and np.all(np.abs(dU[j + 2:]).max(axis=(-2, -1)) > 0.0)


@pytest.mark.gpu
def test_linear_across_saves_and_trajectories_independent_of_batch():
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    se = 400
    nsave = p.nsteps // se + 1
    rng = np.random.default_rng(11)
    c, e = _random_cot(rng, (2, nsave, p.Ntot, p.N))
    al, be = 0.7, -2.3
    per_save = np.zeros((nsave, nsave, p.Ntot, p.N), dtype=complex)      # cotangent j: c at save j only
    per_save[np.arange(nsave), np.arange(nsave)] = c
    wa = jq.Working_Arrays(p, len(pc))
    v = wa.history_vjp(pc[None, :], np.concatenate([np.stack([c, e, al * c + be * e]), per_save])[None, None], save_every=se)
    v = v["vjp"][0, 0]
    err_lin, err_sum = _rel(v[2], al * v[0] + be * v[1]), _rel(v[3:].sum(axis=0), v[0])
    print(f"linearity in the cotangent: {err_lin:.3e}; across saves: {err_sum:.3e}")
    assert max(err_lin, err_sum) <= 1e-12, (err_lin, err_sum)
    assert np.all(v[3] == 0.0)                                           # save 0 (Uinit) has no effect
    # trajectory (b, s, k) does not depend on the batch around it: ragged batch sizes and positions give the same bits
    pcs = np.stack([pc, 0.5 * pc, -1.2 * pc])
    cots = _random_cot(rng, (3, 2, 5, nsave, p.Ntot, p.N))
    dirs = rng.standard_normal((3, 5, len(pc)))
    full = wa.history_vjp(pcs, cots, SHIFTS, se, history=True)
    part = wa.history_vjp(pcs[2:], cots[2:, 1:, 1:4], SHIFTS[1:], se, history=True)
    dfull = wa.history_jvp(pcs, dirs, SHIFTS, se)
    dpart = wa.history_jvp(pcs[2:], dirs[2:, 1:4], SHIFTS[1:], se)
    wa.close()
    assert np.array_equal(part["vjp"][0, 0], full["vjp"][2, 1, 1:4])
    assert np.array_equal(part["history"][0, 0], full["history"][2, 1])
    assert np.array_equal(dpart[0, 0], dfull[2, 1, 1:4])


@pytest.mark.gpu
def test_rejections():
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    cfg, pc = _small_swap()
    p = cfg.params
    npar = len(pc)
    wa = jq.Working_Arrays(p, npar)
    nsave = p.nsteps + 1
    buf = np.zeros(2 * npar * nsave * p.Ntot * p.N)                       # every call below fits (1 trajectory, save_every = 1)
    P = buf.ctypes.data_as(C.c_void_p)
    sh = np.zeros((2, p.Ntot))
    S = sh.ctypes.data_as(C.c_void_p)
    vjp = lambda nbatch, npar_, ns, shift, se, ncot, cr, ci, out: lib.jq_history_vjp(wa._handle, nbatch, P, npar_, ns, shift, se, ncot,
                                                                                      cr, ci, out, None, None)
    jvp = lambda nbatch, npar_, ns, shift, se, ndir, dirs, outr, outi: lib.jq_history_jvp(wa._handle, nbatch, P, npar_, ns, shift, se,
                                                                                           ndir, dirs, outr, outi)
    assert vjp(1, npar, 1, None, 1, 1, P, P, P) == 0
    assert vjp(1, npar, 1, None, 1, 1, None, P, P) == 0                  # a NULL part is zero
    assert vjp(1, npar, 1, None, 1, 1, P, None, P) == 0
    assert wa.last_kernel == 9 and wa.last_kernel_ms > 0.0
    assert jvp(1, npar, 1, None, 1, 1, P, P, P) == 0
    assert wa.last_kernel == 8 and wa.last_kernel_ms > 0.0
    for se in (0, -4, 7):                                                 # 1600 steps: 7 does not divide
        assert vjp(1, npar, 1, None, se, 1, P, P, P) == -1
        assert "divisible by saveEvery" in _lib.last_error()
        assert jvp(1, npar, 1, None, se, 1, P, P, P) == -1
        assert "divisible by saveEvery" in _lib.last_error()
    assert vjp(1, npar, 1, None, 1, 0, P, P, P) == -1                     # ncot = 0
    assert vjp(1, npar, 1, None, 1, 1, None, None, P) == -1               # both cotangent parts NULL
    assert vjp(1, npar, 1, None, 1, 1, P, P, None) == -1                  # NULL vjp
    assert jvp(1, npar, 1, None, 1, 0, P, P, P) == -1                     # ndir = 0
    assert jvp(1, npar, 1, None, 1, 1, None, P, P) == -1                  # NULL dirs
    assert jvp(1, npar, 1, None, 1, 1, P, None, P) == -1                  # NULL outputs
    assert jvp(1, npar, 1, None, 1, 1, P, P, None) == -1
    assert vjp(1, npar + 1, 1, None, 1, 1, P, P, P) == -2                 # wrong npar: JQ_ERR_PCOF_LENGTH
    assert jvp(1, npar + 1, 1, None, 1, 1, P, P, P) == -2
    assert vjp(2, npar, 2, S, 1, 0x20000000, P, P, P) == -1               # 2 * 2 * 2^29 = 2^31 trajectories
    assert "2^31" in _lib.last_error()
    assert jvp(2, npar, 2, S, 1, 0x20000000, P, P, P) == -1
    assert "2^31" in _lib.last_error()
    # 2^20 directions of 1601 blocks of 4 x 3 need 322 GB of tangent histories: more than the device has, no launch
    assert jvp(1, npar, 1, None, 1, 1 << 20, P, P, P) == -4               # JQ_ERR_ALLOC
    assert "GB" in _lib.last_error()
    assert jvp(1, npar, 1, None, 1, 1, P, P, P) == 0                      # the handle still works
    wa.close()
    # the Jacobi solver has no tangent; its VJP is fine
    cfg, _ = golden_config("cnot2-jacobi")
    pj = np.asarray(cfg.pcof0, dtype=np.float64)
    wj = jq.Working_Arrays(cfg.params, len(pj))
    small = np.zeros(4 * len(pj) * cfg.params.Ntot * cfg.params.N)          # save_every = nsteps: 2 saves
    B, Q = small.ctypes.data_as(C.c_void_p), pj.ctypes.data_as(C.c_void_p)
    assert lib.jq_history_jvp(wj._handle, 1, Q, len(pj), 1, None, cfg.params.nsteps, 1, Q, B, B) == -1
    assert "Jacobi" in _lib.last_error()
    assert lib.jq_history_vjp(wj._handle, 1, Q, len(pj), 1, None, cfg.params.nsteps, 1, B, B, B, None, None) == 0
    wj.close()
    # a trajectory over 227 KB of shared memory: one 48-level qudit, all 48 columns (14 and 20 blocks of 48 x 48 doubles)
    from juqbox_b200.params import objparams
    n = 48
    a = np.diag(np.sqrt(np.arange(1, n)), 1)
    pb = objparams([n], [0], 1.0, 10, Uinit=np.eye(n), Utarget=np.eye(n) + 0j, Cfreq=np.array([[0.0]]), Rfreq=[0.0],
                   Hconst=np.zeros((n, n)), Hsym_ops=[a + a.T], Hanti_ops=[a - a.T])
    pcb = np.zeros(6)
    wb = jq.Working_Arrays(pb, len(pcb))
    small = np.zeros(4 * 11 * n * n)
    B, Q = small.ctypes.data_as(C.c_void_p), pcb.ctypes.data_as(C.c_void_p)
    assert lib.jq_history_vjp(wb._handle, 1, Q, len(pcb), 1, None, 10, 1, B, B, B, None, None) == -1
    assert "shared memory" in _lib.last_error()
    assert lib.jq_history_jvp(wb._handle, 1, Q, len(pcb), 1, None, 10, 1, Q, B, B) == -1
    assert "shared memory" in _lib.last_error()
    wb.close()


def _population_loss(U, w):
    """sum_j w_j sum |U_j|^2 over the guard rows (the last row of each block): leakage weighted differently at every save."""
    return (w * (U[..., -1, :].abs() ** 2).sum(dim=-1)).sum()


@pytest.mark.gpu
def test_torch_loss_on_intermediate_populations():
    """A torch loss of the intermediate populations, backpropagated through state_history, against the same loss contracted with the
    tangents of history_jvp (unit directions), with one and with two samples; two samples give the per-sample gradients summed."""
    import torch
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    se = 100
    nsave = p.nsteps // se + 1
    w = torch.linspace(0.0, 2.0, nsave, dtype=torch.float64) ** 2
    wa = jq.Working_Arrays(p, len(pc))
    dU = wa.history_jvp(pc[None, :], np.eye(len(pc))[None], SHIFTS, se)[0]              # [ns, npar, nsave, Ntot, N]
    H = wa.forward_history(pc[None, :], SHIFTS, save_every=se)[0][0].swapaxes(-1, -2)  # [ns, nsave, Ntot, N]
    # dL/dU_j = 2 w_j U_j on the guard row: the forward route is sum Re(conj(dL/dU) dU)
    G = np.zeros_like(H)
    G[..., -1, :] = 2.0 * w.numpy()[None, :, None] * H[..., -1, :]
    want = np.einsum("sjab,spjab->sp", G.conj(), dU).real                              # [ns, npar]
    errs = []
    x = torch.tensor(pc[None, :], dtype=torch.float64, device="cuda", requires_grad=True)
    U = jq.state_history(wa, x, SHIFTS[:1], se)
    _population_loss(U, w.to(U.device)).backward()
    assert wa.last_kernel == 9 and x.grad.device == x.device
    errs.append(_rel(x.grad.cpu().numpy()[0], want[0]))
    x2 = torch.tensor(pc[None, :], dtype=torch.float64, requires_grad=True)
    _population_loss(jq.state_history(wa, x2, SHIFTS, se), w).backward()
    errs.append(_rel(x2.grad.numpy()[0], want.sum(axis=0)))
    per = []
    for s in range(len(SHIFTS)):
        xs = torch.tensor(pc[None, :], dtype=torch.float64, requires_grad=True)
        _population_loss(jq.state_history(wa, xs, SHIFTS[s:s + 1], se), w).backward()
        per.append(xs.grad.numpy()[0])
    wa.close()
    err_sum = _rel(x2.grad.numpy()[0], per[0] + per[1])
    print(f"torch population loss: one sample {errs[0]:.3e}, two samples {errs[1]:.3e} vs history_jvp, {err_sum:.3e} vs per-sample sum")
    assert max(errs) <= 1e-9 and err_sum <= 1e-12, (errs, err_sum)
