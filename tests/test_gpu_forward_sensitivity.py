"""Forward sensitivities (jq_forward_sensitivity): the tangent of the forward sweep along ndir directions per candidate.

The tangent sweep and the discrete adjoint reach the same derivative by independent routes, so agreement between them pins both,
including the extension branches (pFidType 1/3/4, dense forbidden-state weights, uncoupled controls) that finite differences of the
oracle pin only to ~1e-6.  Tests marked gpu need a device; the others check the binding without one."""
import ctypes as C

import numpy as np
import pytest

from helpers import golden_config

TOL = 1e-9          # ||forward - adjoint|| / ||adjoint||


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)                                       # real or complex (final-state tangents)
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300))


def _small_swap():
    cfg, _ = golden_config("swap02")
    cfg.params.T, cfg.params.nsteps = 30.0, 1600
    return cfg, np.asarray(cfg.pcof0) * 3.0


def _forward_vs_adjoint(params, pc, dirs, shifts=None):
    """dobjf along `dirs` [ndir, npar] against grad . d of the automatic evaluation; returns (relative difference, both results)."""
    import juqbox_b200 as jq
    wa = jq.Working_Arrays(params, len(pc))
    f = wa.forward_sensitivity(pc[None, :], dirs[None], shifts)
    assert wa.last_kernel == 8
    a = wa.evaluate(pc[None, :], shifts)
    wa.close()
    want = a["grad"][0] @ dirs.T                                             # [nsamples, ndir]
    return _rel(f["dobjf"][0], want), f, a


# ---------------------------------------------------------------------------------------------------------------- no device needed
def test_symbol_exported_and_null_handle_rejected():
    from juqbox_b200 import _lib
    lib = _lib.load()
    assert "jq_forward_sensitivity" in _lib.EXPORTS and hasattr(lib, "jq_forward_sensitivity")
    one = np.zeros(64)
    p = one.ctypes.data_as(C.c_void_p)
    rc = lib.jq_forward_sensitivity(None, 1, p, 64, 1, None, None, 1, p, p, p, p, p, None, None)
    assert rc == -1                                                         # JQ_ERR_ARG
    assert "handle" in _lib.last_error()


def test_wrapper_rejects_malformed_dirs_before_the_library():
    import juqbox_b200 as jq
    from juqbox_b200 import configs

    class NoLib:                            # any call into the library fails the test
        def __getattr__(self, name):
            raise AssertionError(f"library called: {name}")
    cfg = configs.example("rabi")
    wa = jq.Working_Arrays.__new__(jq.Working_Arrays)
    wa.params, wa._lib, wa._handle = cfg.params, NoLib(), None
    wa._snapshot = wa._fingerprint(cfg.params)
    npar = cfg.nCoeff
    pc = np.zeros((2, npar))
    for bad in (np.zeros((2, npar)), np.zeros((2, 3, npar + 1)), np.zeros((1, 3, npar)), np.zeros((2, 0, npar)), np.zeros((2, 3, npar, 1))):
        with pytest.raises(ValueError):
            wa.forward_sensitivity(pc, bad)
    with pytest.raises(ValueError):         # a weighted sum of final states is not defined
        wa.forward_sensitivity(pc, np.zeros((2, 1, npar)), np.zeros((3, cfg.params.Ntot)), np.ones(3), final_state=True)
    with pytest.raises(ValueError):
        wa.forward_sensitivity(pc, np.zeros((2, 1, npar)), np.zeros((3, cfg.params.Ntot)), np.ones(2))
    with pytest.raises(ValueError):
        jq.forward_sensitivity(np.zeros(npar), cfg.params, wa, np.zeros((3, npar - 1)))


# ---------------------------------------------------------------------------------------------------------------- on the GPU
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["rabi", "swap02", "flux", "cnot2", "cnot3"])
def test_forward_gradient_matches_adjoint(case):
    """Unit directions (the whole forward-mode gradient in one call), 8 random directions for cnot3."""
    cfg, _ = golden_config(case)
    pc = np.asarray(cfg.pcof0, dtype=np.float64)
    dirs = np.random.default_rng(5).standard_normal((8, len(pc))) if case == "cnot3" else np.eye(len(pc))
    err, f, a = _forward_vs_adjoint(cfg.params, pc, dirs)
    print(f"{case}: ndir {len(dirs)}  max relative |forward - adjoint| = {err:.3e}")
    assert err <= TOL, (case, err)
    assert f["infid"][0, 0] == pytest.approx(a["infid"][0, 0], rel=1e-12) and f["leak"][0, 0] == pytest.approx(a["leak"][0, 0], rel=1e-12, abs=1e-18)


@pytest.mark.gpu
def test_leakieq_infidelity_and_leak_tangents_match_their_adjoints():
    cfg, _ = golden_config("cnot2-leakieq")
    p = cfg.params
    assert p.objFuncType != 1
    pc = np.asarray(cfg.pcof0, dtype=np.float64)
    import juqbox_b200 as jq
    wa = jq.Working_Arrays(p, len(pc))
    f = wa.forward_sensitivity(pc[None, :], np.eye(len(pc))[None])
    a = wa.evaluate(pc[None, :])
    wa.close()
    ei, el = _rel(f["dinfid"][0, 0], a["infidgrad"][0, 0]), _rel(f["dleak"][0, 0], a["leakgrad"][0, 0])
    print(f"cnot2-leakieq: infidelity {ei:.3e}, leak {el:.3e}")
    assert ei <= TOL and el <= TOL, (ei, el)


def _dense_weight_params(objFuncType):
    from juqbox_b200.params import objparams
    cfg, pc = _small_swap()
    p = cfg.params
    rng = np.random.default_rng(3)
    F = rng.standard_normal((p.Ntot, 2)) + 1j * rng.standard_normal((p.Ntot, 2))
    F /= np.linalg.norm(F, axis=0)
    pd = objparams(p.Ne, p.Ng, p.T, p.nsteps, Uinit=p.Uinit, Utarget=p.Utarget_r + 1j * p.Utarget_i, Cfreq=p.Cfreq, Rfreq=p.Rfreq,
                   Hconst=p.Hconst, Hsym_ops=p.Hsym_ops, Hanti_ops=p.Hanti_ops, linear_solver=p.linear_solver, objFuncType=objFuncType,
                   use_custom_forbidden=True, forb_states=F, forb_weights=[0.7, 0.2])
    return pd, pc


def _uncoupled_params(kind):
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


def _extension(name):
    if name.startswith("pfid"):
        cfg, pc = _small_swap()
        p = cfg.params
        p.pFidType, p.globalPhase, p.objFuncType = int(name[4]), 0.37, 3 if name.endswith("obj3") else 1
        if p.pFidType == 3:
            pc = np.concatenate([pc, [0.37]])                                  # the global phase rides along as the last entry
        return p, pc, None
    if name.startswith("dense_w"):
        p, pc = _dense_weight_params(int(name[-1]))
        assert p.wmat_imag is not None and np.any(p.wmat_imag)
        return p, pc, np.array([[0.0, 0.001, 0.01, 0.1], [0.0, -0.002, -0.02, -0.2]])
    p, pc = _uncoupled_params(name.split("_")[1])
    return p, pc, None


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["pfid1", "pfid3", "pfid4", "pfid1_obj3", "pfid3_obj3", "pfid4_obj3", "dense_w1", "dense_w2",
                                  "unc_symmetric", "unc_antisymmetric"])
def test_extension_branches_forward_matches_adjoint(name):
    """The exact pin of the extension branches: every direction of the forward gradient (the phase entry too for pFidType 3)."""
    p, pc, shifts = _extension(name)
    err, f, a = _forward_vs_adjoint(p, pc, np.eye(len(pc)), shifts)
    print(f"{name}: max relative |forward - adjoint| = {err:.3e}")
    assert err <= TOL, (name, err)
    if p.objFuncType != 1:
        assert _rel(f["dinfid"][0], a["infidgrad"][0]) <= TOL and _rel(f["dleak"][0], a["leakgrad"][0]) <= TOL


@pytest.mark.gpu
def test_final_state_tangent_is_second_order_limit_of_central_differences():
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    d = np.random.default_rng(7).standard_normal(len(pc))
    d *= np.abs(pc).max() / np.abs(d).max()                                   # a perturbation of the size of the controls
    wa = jq.Working_Arrays(p, len(pc))
    dU = wa.forward_sensitivity(pc[None, :], d[None, None, :], final_state=True)["dstate"][0, 0, 0]
    assert dU.shape == (p.Ntot, p.N)
    U = lambda x: wa.forward_history(x[None, :], save_every=p.nsteps)[0][0, 0, -1].T     # Ntot x N
    errs = []
    for eps in (2e-2, 1e-2):
        fd = (U(pc + eps * d) - U(pc - eps * d)) / (2 * eps)
        errs.append(_rel(dU, fd))
    wa.close()
    print(f"final-state tangent vs central differences: {errs[0]:.3e} (eps), {errs[1]:.3e} (eps/2), ratio {errs[0] / errs[1]:.2f}")
    assert 3.0 < errs[0] / errs[1] < 5.0 and errs[1] <= 1e-7, errs


@pytest.mark.gpu
def test_coarse_steps_tangent_is_the_derivative_of_the_discrete_objective():
    """The rabi example takes 57 steps of dt = 1.75 with 3 Neumann terms.  There the tangent and Richardson-extrapolated central
    differences of the objective agree to ~1e-10.  The adjoint gradient (the reference's formula, the same in the CPU oracle)
    sits ~5e-7 away from both: it is not the exact derivative of the discrete map at such steps."""
    import juqbox_b200 as jq
    from juqbox_b200 import configs
    cfg = configs.example("rabi")
    p = cfg.params
    pc = configs.synthetic_pcof(cfg, 1)[0]
    n = len(pc)
    wa = jq.Working_Arrays(p, n)
    tan = wa.forward_sensitivity(pc[None, :], np.eye(n)[None])["dobjf"][0, 0]
    adj = wa.evaluate(pc[None, :])["grad"][0, 0]

    def cd(eps):
        r = wa.evaluate(np.concatenate([pc + eps * np.eye(n), pc - eps * np.eye(n)]), evaladjoint=False)["objf"][:, 0]
        return (r[:n] - r[n:]) / (2 * eps)
    d1, d2, d4 = cd(1e-5), cd(2e-5), cd(4e-5)
    wa.close()
    rich, rich2 = (4 * d1 - d2) / 3, (4 * d2 - d4) / 3
    e_fd, e_tan, e_adj = _rel(rich2, rich), _rel(tan, rich), _rel(adj, rich)
    print(f"rabi example: Richardson self-consistency {e_fd:.2e}, tangent {e_tan:.2e}, adjoint {e_adj:.2e} (relative to Richardson)")
    assert e_fd <= 1e-9 and e_tan <= 1e-8, (e_fd, e_tan, e_adj)


@pytest.mark.gpu
def test_pfid2_infidelity_tangent_is_minus_two_re_sbar_sdot():
    import juqbox_b200 as jq
    cfg, _ = golden_config("cnot2")
    p = cfg.params
    assert p.pFidType == 2
    pc = np.asarray(cfg.pcof0, dtype=np.float64)
    dirs = np.random.default_rng(9).standard_normal((3, len(pc)))
    wa = jq.Working_Arrays(p, len(pc))
    f = wa.forward_sensitivity(pc[None, :], dirs[None], final_state=True)
    U = wa.forward_history(pc[None, :], save_every=p.nsteps)[0][0, 0, -1].T
    wa.close()
    Vt = p.Utarget_r + 1j * p.Utarget_i
    s = np.vdot(Vt, U) / p.N
    for k in range(3):
        sdot = np.vdot(Vt, f["dstate"][0, 0, k]) / p.N
        want = -2.0 * np.real(np.conj(s) * sdot)
        assert abs(f["dinfid"][0, 0, k] - want) <= 1e-12 * max(abs(want), 1e-300), (k, f["dinfid"][0, 0, k], want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["swap_samples", "dense_w2", "pfid3"])
def test_primal_outputs_equal_the_generic_kernel_bit_for_bit(name):
    import juqbox_b200 as jq
    if name == "swap_samples":
        cfg, pc = _small_swap()
        p, shifts = cfg.params, np.array([[0.0, 0.001, 0.01, 0.1], [0.0, -0.002, -0.02, -0.2]])
    else:
        p, pc, shifts = _extension(name)
    pcs = np.stack([pc, 0.5 * pc, -1.2 * pc])
    dirs = np.random.default_rng(2).standard_normal((3, 2, len(pc)))
    wa = jq.Working_Arrays(p, len(pc))
    f = wa.forward_sensitivity(pcs, dirs, shifts)
    wa.set_kernel(1)
    r = wa.evaluate(pcs, shifts, evaladjoint=False)
    assert wa.last_kernel == 1
    wa.close()
    assert np.array_equal(f["infid"], r["infid"]) and np.array_equal(f["leak"], r["leak"])


@pytest.mark.gpu
def test_weighted_sums_equal_host_weighted_samples():
    import juqbox_b200 as jq
    from juqbox_b200 import configs
    cfg = configs.example("risk_neutral")
    cfg.params.T, cfg.params.nsteps = 30.0, 800
    p = cfg.params
    pcs = configs.synthetic_pcof(cfg, 2) * 20
    sh = configs.noise_shift(p.Ntot, cfg.nodes)
    dirs = np.random.default_rng(4).standard_normal((2, 5, cfg.nCoeff))
    wa = jq.Working_Arrays(p, cfg.nCoeff)
    per = wa.forward_sensitivity(pcs, dirs, sh)
    w = wa.forward_sensitivity(pcs, dirs, sh, cfg.weights)
    wts = np.asarray(cfg.weights)
    for key in ("infid", "leak"):
        assert _rel(w[key], per[key] @ wts) <= 1e-14, key
    for key in ("dinfid", "dleak"):
        assert w[key].shape == (2, 5)
        assert _rel(w[key], np.einsum("bsk,s->bk", per[key], wts)) <= 1e-14, key
    # the module-level form: one pcof, nodes and weights
    wa = jq.Working_Arrays(p, cfg.nCoeff)
    m = jq.forward_sensitivity(pcs[1], p, wa, dirs[1], nodes=cfg.nodes, weights=cfg.weights)
    wa.close()
    assert np.array_equal(m["dinfid"], w["dinfid"][1]) and m["infid"] == w["infid"][1]


@pytest.mark.gpu
def test_linear_in_the_direction_and_trajectories_independent_of_batch():
    import juqbox_b200 as jq
    cfg, pc = _small_swap()
    p = cfg.params
    rng = np.random.default_rng(11)
    d, e = rng.standard_normal((2, len(pc)))
    al, be = 0.7, -2.3
    wa = jq.Working_Arrays(p, len(pc))
    f = wa.forward_sensitivity(pc[None, :], np.stack([d, e, al * d + be * e])[None], final_state=True)
    for key in ("dinfid", "dleak"):
        v = f[key][0, 0]
        assert abs(v[2] - (al * v[0] + be * v[1])) <= 1e-12 * np.abs([al * v[0], be * v[1]]).max(), key
    ds = f["dstate"][0, 0]
    assert _rel(ds[2], al * ds[0] + be * ds[1]) <= 1e-12
    # trajectory (b, s, k) does not depend on the batch around it: ragged batch sizes and positions give the same bits
    pcs = np.stack([pc, 0.5 * pc, -1.2 * pc])
    sh = np.array([[0.0, 0.001, 0.01, 0.1], [0.0, -0.002, -0.02, -0.2]])
    dirs = rng.standard_normal((3, 5, len(pc)))
    full = wa.forward_sensitivity(pcs, dirs, sh, final_state=True)
    part = wa.forward_sensitivity(pcs[2:], dirs[2:, 1:4], sh[1:], final_state=True)
    wa.close()
    for key in ("dinfid", "dleak", "dstate"):
        assert np.array_equal(part[key][0, 0], full[key][2, 1, 1:4]), key
    assert np.array_equal(part["infid"][0, 0], full["infid"][2, 1])


@pytest.mark.gpu
def test_rejections():
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    lib = _lib.load()
    cfg, pc = _small_swap()
    p = cfg.params
    npar = len(pc)
    wa = jq.Working_Arrays(p, npar)
    buf = np.zeros(4 * npar * 8)
    P = buf.ctypes.data_as(C.c_void_p)
    sh = np.zeros((2, p.Ntot))
    S = sh.ctypes.data_as(C.c_void_p)
    call = lambda nbatch, npar_, ns, shift, w, ndir, dirs, sr=None: lib.jq_forward_sensitivity(
        wa._handle, nbatch, P, npar_, ns, shift, w, ndir, dirs, P, P, P, P, sr, None)
    assert call(1, npar, 1, None, None, 1, P) == 0
    assert call(1, npar, 1, None, None, 0, P) == -1                            # ndir = 0
    assert call(1, npar, 1, None, None, 2, None) == -1                         # NULL dirs
    assert call(1, npar, 2, S, P, 1, P, sr=P) == -1                            # weights with dstate
    assert "weighted sum" in _lib.last_error()
    assert call(1, npar + 1, 1, None, None, 1, P) == -2                        # wrong npar: JQ_ERR_PCOF_LENGTH
    assert call(2, npar, 2, S, None, 0x40000000, P) == -1                      # 2 * 2 * 2^30 trajectories
    assert "2^31" in _lib.last_error()
    wa.close()
    cfg, _ = golden_config("cnot2-jacobi")
    assert cfg.params.linear_solver.solver_id == 2
    wa = jq.Working_Arrays(cfg.params, len(cfg.pcof0))
    with pytest.raises(_lib.JuqboxCudaError, match="Jacobi"):
        wa.forward_sensitivity(np.asarray(cfg.pcof0)[None, :], np.eye(len(cfg.pcof0))[None, :2])
    wa.close()
