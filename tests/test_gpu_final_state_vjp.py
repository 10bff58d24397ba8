"""Final-state vector-Jacobian products (jq_final_state_vjp) and U(T) as a differentiable torch function (juqbox_b200.final_state).

The VJP is pinned against two routes the library already trusts: the forward tangent of jq_forward_sensitivity (the dot-product
identity <vjp(c), d> = Re vdot(c, dU . d) for random c and d), and the generic kernel's infidelity gradient (the cotangent
dinfid/d(Re U, Im U) reproduces it).  Tests marked gpu need a device; the others check the binding and the torch wrapper without one."""
import ctypes as C
import types

import numpy as np
import pytest

from helpers import golden_config

TOL_DOT = 1e-9      # dot-product identity against the forward tangent (two independent routes)
TOL_INFID = 1e-12   # infidelity cotangent against the generic kernel's infidgrad (the same sweep)
SHIFTS = np.array([[0.0, 0.001, 0.01, 0.1], [0.0, -0.002, -0.02, -0.2]])


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300))


def _small_swap():
    cfg, _ = golden_config("swap02")
    cfg.params.T, cfg.params.nsteps = 30.0, 1600
    return cfg, np.asarray(cfg.pcof0) * 3.0


def _uncoupled_params(kind):
    """The two uncoupled-control problems of the forward-sensitivity tests."""
    from juqbox_b200 import configs
    from juqbox_b200.params import objparams
    rng = np.random.default_rng(1)
    if kind == "symmetric":                 # rabi in the lab frame: one symmetric uncoupled control
        cfg = configs.example("rabi_lab", T=20.0, Pmin=60)
        return cfg.params, cfg.pcof0 * 5.0 + 0.3 * cfg.maxpar[0] * rng.standard_normal(cfg.nCoeff)
    base, _ = _small_swap()                 # an antisymmetric uncoupled operator next to a coupled pair, sparse storage
    p = base.params
    a = np.diag(np.sqrt(np.arange(1, p.Ntot)), 1)
    om = np.vstack([p.Cfreq[:1], p.Cfreq[:1] * 0.5])
    pm = objparams(p.Ne, p.Ng, 10.0, 4000, Uinit=p.Uinit, Utarget=p.Utarget_r + 1j * p.Utarget_i, Cfreq=om, Rfreq=[0.0, 0.7],
                   Hconst=p.Hconst, Hsym_ops=[a + a.T], Hanti_ops=[a - a.T], Hunc_ops=[0.3 * (a - a.T)], use_sparse=True, objFuncType=2)
    pm.Rfreq = [0.7, 0.0]
    return pm, rng.uniform(-1, 1, 2 * 2 * pm.Nfreq * 6) * 0.02


def _random_cot(rng, shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def _infid_cot(p, U, phase):
    """c = dinfid/dRe U + i dinfid/dIm U of the pFidType formulas (src/evalobjgrad.jl:755-763) at U [..., Ntot, N].  With
    S = tr(U^H V) / N and G = dinfid/dRe S + i dinfid/dIm S, c = V conj(G) / N."""
    V = p.Utarget_r + 1j * p.Utarget_i
    S = np.einsum("...ij,ij->...", U.conj(), V)[..., None, None] / p.N
    G = {1: 2.0 * (S - np.exp(1j * phase)), 2: -2.0 * S, 3: -np.exp(-1j * phase) + 0 * S, 4: -np.exp(-1j * phase) + 0 * S}[p.pFidType]
    return V * np.conj(G) / p.N


class _LinearStandIn:
    """A stand-in for Working_Arrays: U = A pcof, a fixed complex linear map per sample, with final_state_vjp its exact adjoint
    under the library's convention vjp_p = sum Re(c) dRe U / dp + Im(c) dIm U / dp = Re vdot(c, A[..., p])."""

    def __init__(self, nsamples=2, Ntot=3, N=2, npar=5):
        rng = np.random.default_rng(0)
        self.params = types.SimpleNamespace(nsteps=4, Ntot=Ntot, N=N)
        self.A = _random_cot(rng, (nsamples, Ntot, N, npar))

    def _a(self, shifts):
        return self.A[:1 if shifts is None else len(shifts)]

    def forward_history(self, pcof, shifts=None, save_every=1):
        U = np.einsum("sijp,bp->bsij", self._a(shifts), pcof)
        nsave = self.params.nsteps // save_every + 1
        hist = np.stack([np.zeros_like(U)] * (nsave - 1) + [U], axis=2).swapaxes(-1, -2)    # [nbatch, nsamples, nsave, N, Ntot]
        return hist, None, None

    def final_state_vjp(self, pcof, cot, shifts=None, final_state=False):
        return {"vjp": np.einsum("bskij,sijp->bskp", cot.conj(), self._a(shifts)).real}


# ---------------------------------------------------------------------------------------------------------------- no device needed
def test_symbol_exported_and_null_handle_rejected():
    from juqbox_b200 import _lib
    lib = _lib.load()
    assert "jq_final_state_vjp" in _lib.EXPORTS and hasattr(lib, "jq_final_state_vjp")
    one = np.zeros(64)
    p = one.ctypes.data_as(C.c_void_p)
    rc = lib.jq_final_state_vjp(None, 1, p, 64, 1, None, 1, p, p, p, None, None)
    assert rc == -1                                                         # JQ_ERR_ARG
    assert "handle" in _lib.last_error()


def test_wrapper_rejects_malformed_shapes_before_the_library():
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
    npar, n, m = cfg.nCoeff, p.Ntot, p.N
    pc = np.zeros((2, npar))
    for bad in (np.zeros((2, 1, 1, n, m, 1)), np.zeros((2, 1, n, m)), np.zeros((2, 1, 0, n, m)), np.zeros((1, 1, 1, n, m)),
                np.zeros((2, 2, 1, n, m)), np.zeros((2, 1, 1, m, n + 1)), np.zeros((2, 1, 1, n, m + 1))):
        with pytest.raises(ValueError):
            wa.final_state_vjp(pc, bad)
    with pytest.raises(ValueError):         # pcof not [nbatch, npar]
        wa.final_state_vjp(np.zeros(npar), np.zeros((1, 1, 1, n, m)))
    with pytest.raises(ValueError):         # shifts not [nsamples, Ntot]
        wa.final_state_vjp(pc, np.zeros((2, 3, 1, n, m)), np.zeros((3, n + 1)))
    with pytest.raises(ValueError):         # cot for 2 samples, shifts for 3
        wa.final_state_vjp(pc, np.zeros((2, 2, 1, n, m)), np.zeros((3, n)))


@pytest.mark.parametrize("shifts", [None, np.zeros((2, 3))])
def test_final_state_gradcheck_against_a_linear_stand_in(shifts):
    """The torch wrapper on CPU: gradcheck of U = A pcof pins the complex convention (cot = dL/dRe U + i dL/dIm U) and the shapes."""
    torch = pytest.importorskip("torch")
    import juqbox_b200 as jq
    wa = _LinearStandIn()
    pc = torch.tensor(np.random.default_rng(1).standard_normal((3, 5)), dtype=torch.float64, requires_grad=True)
    U = jq.final_state(wa, pc, shifts)
    assert U.shape == (3, 1 if shifts is None else 2, 3, 2) and U.dtype == torch.complex128
    assert torch.autograd.gradcheck(lambda x: jq.final_state(wa, x, shifts), (pc,), eps=1e-6, atol=1e-9, rtol=1e-7)
    with pytest.raises(ValueError):
        jq.final_state(wa, pc.float())


# ---------------------------------------------------------------------------------------------------------------- on the GPU
def _dot_case(name):
    if name in ("swap02", "flux", "cnot2", "cnot3"):
        cfg, _ = golden_config(name)
        return cfg.params, np.asarray(cfg.pcof0, dtype=np.float64), None
    if name.startswith("unc_"):
        p, pc = _uncoupled_params(name[4:])
        return p, pc, None
    cfg, pc = _small_swap()
    if name == "pfid3":
        cfg.params.pFidType, cfg.params.globalPhase = 3, 0.37
        return cfg.params, np.concatenate([pc, [0.37]]), None
    return cfg.params, pc, SHIFTS                                          # "samples"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["swap02", "flux", "cnot2", "cnot3", "unc_symmetric", "unc_antisymmetric", "pfid3", "samples"])
def test_dot_product_identity_against_the_forward_tangent(name):
    """<vjp(c), d> = Re vdot(c, dU . d) for 2 random cotangents and 2 random directions per sample."""
    import juqbox_b200 as jq
    p, pc, shifts = _dot_case(name)
    ns = 1 if shifts is None else len(shifts)
    rng = np.random.default_rng(17)
    d = rng.standard_normal((2, len(pc)))
    c = _random_cot(rng, (1, ns, 2, p.Ntot, p.N))
    wa = jq.Working_Arrays(p, len(pc))
    v = wa.final_state_vjp(pc[None, :], c, shifts)["vjp"][0]               # [ns, ncot, npar]
    assert wa.last_kernel == 9 and v.shape == (ns, 2, len(pc))
    dU = wa.forward_sensitivity(pc[None, :], d[None], shifts, final_state=True)["dstate"][0]      # [ns, ndir, Ntot, N]
    wa.close()
    lhs = np.einsum("skp,jp->skj", v, d)
    rhs = np.einsum("skab,sjab->skj", c[0].conj(), dU).real
    err = _rel(lhs, rhs)
    print(f"{name}: relative |<vjp(c), d> - Re vdot(c, dU d)| = {err:.3e}")
    assert err <= TOL_DOT, (name, err)
    if p.pFidType == 3:
        assert np.all(v[..., -1] == 0.0)


def _infid_case(name):
    if name in ("cnot2-leakieq", "cnot2-jacobi"):
        cfg, _ = golden_config(name)
        cfg.params.objFuncType = 3
        return cfg.params, np.asarray(cfg.pcof0, dtype=np.float64)
    cfg, pc = _small_swap()
    p = cfg.params
    p.pFidType, p.globalPhase, p.objFuncType = int(name[4]), 0.37, 3
    return p, (np.concatenate([pc, [0.37]]) if p.pFidType == 3 else pc)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cnot2-leakieq", "pfid1", "pfid3", "pfid4", "cnot2-jacobi"])
def test_infidelity_cotangent_reproduces_infidgrad(name):
    import juqbox_b200 as jq
    p, pc = _infid_case(name)
    wa = jq.Working_Arrays(p, len(pc))
    zero = np.zeros((1, 1, 1, p.Ntot, p.N))
    U = wa.final_state_vjp(pc[None, :], zero, final_state=True)["state"]       # [1, 1, Ntot, N]
    c = _infid_cot(p, U, pc[-1] if p.pFidType == 3 else p.globalPhase)[:, :, None]
    r = wa.final_state_vjp(pc[None, :], c, final_state=True)
    assert np.array_equal(r["state"], U)
    wa.set_kernel(1)
    a = wa.evaluate(pc[None, :])
    assert wa.last_kernel == 1
    wa.close()
    got, want = r["vjp"][0, 0, 0], a["infidgrad"][0, 0]
    if p.pFidType == 3:                     # U(T) does not depend on the phase; infidgrad's last entry is the phase derivative
        assert got[-1] == 0.0
        got, want = got[:-1], want[:-1]
    err = _rel(got, want)
    print(f"{name}: relative |vjp(dinfid/dU) - infidgrad| = {err:.3e}")
    assert err <= TOL_INFID, (name, err)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["swap_samples", "cnot2"])
def test_state_equals_forward_history_on_the_generic_kernel(name):
    import juqbox_b200 as jq
    if name == "cnot2":
        cfg, _ = golden_config("cnot2")
        p, pcs, sh = cfg.params, np.asarray(cfg.pcof0)[None, :], None
    else:
        cfg, pc = _small_swap()
        p, pcs, sh = cfg.params, np.stack([pc, -0.7 * pc]), SHIFTS
    ns = 1 if sh is None else len(sh)
    wa = jq.Working_Arrays(p, pcs.shape[1])
    c = _random_cot(np.random.default_rng(3), (len(pcs), ns, 2, p.Ntot, p.N))
    U = wa.final_state_vjp(pcs, c, sh, final_state=True)["state"]
    wa.set_kernel(1)
    hist = wa.forward_history(pcs, sh, save_every=p.nsteps)[0]
    assert wa.last_kernel == 1
    wa.close()
    assert np.array_equal(U, hist[:, :, -1].swapaxes(-1, -2))


@pytest.mark.gpu
def test_linear_in_the_cotangent_and_trajectories_independent_of_batch():
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    rng = np.random.default_rng(11)
    c, e = _random_cot(rng, (2, p.Ntot, p.N))
    al, be = 0.7, -2.3
    wa = jq.Working_Arrays(p, len(pc))
    v = wa.final_state_vjp(pc[None, :], np.stack([c, e, al * c + be * e])[None, None])["vjp"][0, 0]
    err = _rel(v[2], al * v[0] + be * v[1])
    print(f"linearity in the cotangent: {err:.3e}")
    assert err <= 1e-12, err
    # a real cotangent (no imaginary part crosses the ABI) gives the bits of the same cotangent with a zero imaginary part
    re = wa.final_state_vjp(pc[None, :], c.real[None, None, None])["vjp"]
    assert np.array_equal(re, wa.final_state_vjp(pc[None, :], c.real[None, None, None] + 0j)["vjp"])
    # trajectory (b, s, k) does not depend on the batch around it: ragged batch sizes and positions give the same bits
    pcs = np.stack([pc, 0.5 * pc, -1.2 * pc])
    cots = _random_cot(rng, (3, 2, 5, p.Ntot, p.N))
    full = wa.final_state_vjp(pcs, cots, SHIFTS, final_state=True)
    part = wa.final_state_vjp(pcs[2:], cots[2:, 1:, 1:4], SHIFTS[1:], final_state=True)
    wa.close()
    assert np.array_equal(part["vjp"][0, 0], full["vjp"][2, 1, 1:4])
    assert np.array_equal(part["state"][0, 0], full["state"][2, 1])


@pytest.mark.gpu
def test_rejections():
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    cfg, pc = _small_swap()
    p = cfg.params
    npar = len(pc)
    wa = jq.Working_Arrays(p, npar)
    buf = np.zeros(16 * npar * p.Ntot * p.N)
    P = buf.ctypes.data_as(C.c_void_p)
    sh = np.zeros((2, p.Ntot))
    S = sh.ctypes.data_as(C.c_void_p)
    call = lambda nbatch, npar_, ns, shift, ncot, cr, ci, out: lib.jq_final_state_vjp(wa._handle, nbatch, P, npar_, ns, shift, ncot,
                                                                                       cr, ci, out, None, None)
    assert call(1, npar, 1, None, 1, P, P, P) == 0
    assert call(1, npar, 1, None, 1, None, P, P) == 0                          # a NULL part is zero
    assert call(1, npar, 1, None, 1, P, None, P) == 0
    assert wa.last_kernel == 9 and wa.last_kernel_ms > 0.0
    assert call(1, npar, 1, None, 0, P, P, P) == -1                            # ncot = 0
    assert call(1, npar, 1, None, 1, None, None, P) == -1                      # both cotangent parts NULL
    assert call(1, npar, 1, None, 1, P, P, None) == -1                         # NULL vjp
    assert call(1, npar + 1, 1, None, 1, P, P, P) == -2                        # wrong npar: JQ_ERR_PCOF_LENGTH
    assert call(2, npar, 2, S, 0x20000000, P, P, P) == -1                      # 2 * 2 * 2^29 = 2^31 trajectories
    assert "2^31" in _lib.last_error()
    wa.close()


def _torch_infid(p, U):
    import torch
    V = torch.tensor(p.Utarget_r + 1j * p.Utarget_i, device=U.device)
    S = (U.conj() * V).sum(dim=(-2, -1)) / p.N
    return 1.0 - S.abs() ** 2


@pytest.mark.gpu
def test_torch_infidelity_gradient_matches_infidgrad():
    """pFidType 2 infidelity written in torch on top of final_state, backpropagated through one VJP per sample."""
    import torch
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    p.objFuncType = 3
    assert p.pFidType == 2
    wa = jq.Working_Arrays(p, len(pc))
    wa.set_kernel(1)
    a1 = wa.evaluate(pc[None, :])["infidgrad"][0, 0]
    a2 = wa.evaluate(pc[None, :], SHIFTS)["infidgrad"][0]
    x = torch.tensor(pc[None, :], dtype=torch.float64, device="cuda", requires_grad=True)
    U = jq.final_state(wa, x)
    assert U.device == x.device and U.shape == (1, 1, p.Ntot, p.N)
    _torch_infid(p, U).sum().backward()
    assert wa.last_kernel == 9 and x.grad.device == x.device
    err1 = _rel(x.grad.cpu().numpy()[0], a1)
    # a loss summed over two noise samples
    x2 = torch.tensor(pc[None, :], dtype=torch.float64, requires_grad=True)
    _torch_infid(p, jq.final_state(wa, x2, SHIFTS)).sum().backward()
    err2 = _rel(x2.grad.numpy()[0], a2.sum(axis=0))
    per = []
    for s in range(len(SHIFTS)):
        xs = torch.tensor(pc[None, :], dtype=torch.float64, requires_grad=True)
        _torch_infid(p, jq.final_state(wa, xs, SHIFTS[s:s + 1])).sum().backward()
        per.append(xs.grad.numpy()[0])
    wa.close()
    err3 = _rel(x2.grad.numpy()[0], per[0] + per[1])
    print(f"torch pFidType 2 infidelity: one sample {err1:.3e}, two samples {err2:.3e} vs infidgrad, {err3:.3e} vs per-sample sum")
    assert max(err1, err2, err3) <= TOL_INFID, (err1, err2, err3)
