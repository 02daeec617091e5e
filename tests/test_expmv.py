"""prop_method=Expmv: the truncated-Taylor propagator (krotov.jl_b200/expmv.py, taylor_step in warp_kernel.cuh) against
scipy.linalg.expm and the exact-propagator vectors; its host driver on an oracle-backed engine; argument errors; on the
GPU the device path against the same references, on several CTAs and emulated ranks, and its C ABI."""
import json
import os

import numpy as np
import pytest
from scipy.linalg import expm

import expmv_reference as X
import krotov_jl_b200 as K
import workloads as W
from krotov_jl_b200 import _lib as B
from krotov_jl_b200 import expmv as E
from util import run_product, to_problem

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SX = np.array([[0, 1], [1, 0]], complex)
SZ = np.diag([1.0, -1.0]).astype(complex)
SM = np.array([[0, 1], [0, 0]], complex)


def gold(name):
    with open(os.path.join(GOLD, name + ".json")) as fh:
        return json.load(fh)


def _cheby_step(G, v, dt):
    """One step of the Chebyshev recursion with the repository's window rule (real parts of the eigenvalues)."""
    ev = np.linalg.eigvals(G)
    lo, hi = ev.real.min(), ev.real.max()
    Delta = 1.01 * (hi - lo)
    E_min = lo - 0.005 * (hi - lo)
    a = K.cheby_coeffs(Delta, dt)
    beta, c = Delta / 2 + E_min, (-2j / Delta) * np.sign(dt)
    v0, v1 = v, c * (G @ v - beta * v)
    psi = a[0] * v0 + a[1] * v1
    for j in range(2, len(a)):
        v0, v1 = v1, 2 * c * (G @ v1 - beta * v1) + v0
        psi = psi + a[j] * v1
    return np.exp(-1j * beta * dt) * psi


# ---- CPU 1: the restated device step with host-chosen parameters against expm ------------------------------------------
def test_taylor_step_matches_expm_on_the_liouvillian_grid_where_chebyshev_does_not():
    rng = np.random.default_rng(3)
    worst_taylor, cheby = 0.0, {}
    for gamma in (0.01, 0.1, 1.0, 2.0):
        for dt in (0.01, 0.1, 0.5, 2.0):
            G = X.liouvillian(-0.5 * SZ + 0.3 * SX, [np.sqrt(gamma) * SM])
            v = rng.standard_normal(4) + 1j * rng.standard_normal(4)
            for Gd, h in ((G, dt), (G.conj().T, -dt)):  # forward, and the backward sweep's adjoint with dt < 0
                ref = expm(-1j * Gd * h) @ v
                got, _ = X.step_with_host_params(Gd, v, h)
                worst_taylor = max(worst_taylor, np.abs(got - ref).max() / np.linalg.norm(v))
            cheby[(gamma, dt)] = np.abs(_cheby_step(G, v, dt) - expm(-1j * G * dt) @ v).max() / np.linalg.norm(v)
    assert worst_taylor <= 1e-14, worst_taylor
    # why the propagator exists: strong decay and long steps miss by orders of magnitude more with Chebyshev
    assert cheby[(2.0, 2.0)] > 1e-8 and cheby[(1.0, 2.0)] > 1e-11, cheby


@pytest.mark.parametrize("case", ["c1", "c2", "c3"])
def test_taylor_step_matches_expm_for_the_config_generators_at_their_range_corners(case):
    w = {"c1": W.c1_tls, "c2": lambda: W.c2_transmon_x(n_grid=101), "c3": lambda: W.c3_two_transmon(n_grid=41, T=8.0)}[case]()
    t = np.asarray(w.tlist)
    pulses = [np.array([c(x) for x in 0.5 * (t[1:] + t[:-1])]) for c in w.controls]
    fw = E.TaylorDirection(w.H0, w.Hc, t, False, pulses)
    fw.control_ranges = [(5 * lo, 5 * hi) if hi > 0 else (5 * lo, 5 * abs(lo)) for lo, hi in fw.control_ranges]
    fw._derive()
    rng = np.random.default_rng(4)
    dt, c = float(fw.dt_of_class[0]), 0
    for corner in [[r[0] for r in fw.control_ranges], [r[1] for r in fw.control_ranges]]:
        Hm = w.H0[0] + sum(a * Hl for a, Hl in zip(corner, w.Hc[0]) if Hl is not None)
        v = rng.standard_normal(w.d) + 1j * rng.standard_normal(w.d)
        m, s = int(fw.m[0, c]), int(fw.s[0, c])
        got = X.taylor_step(Hm, v, dt, fw.mu[0], fw.scale[0], m, s, fw.coeff_table[0, c])
        assert np.abs(got - expm(-1j * Hm * dt) @ v).max() <= 1e-14 * np.linalg.norm(v)


def test_taylor_step_on_a_non_uniform_grid_uses_the_exact_step_of_every_interval():
    t = np.concatenate([np.linspace(0, 1, 11)[:-1], np.linspace(1, 3, 6)])
    G = X.liouvillian(-0.5 * SZ, [SM])
    for backward in (False, True):
        Gd = G.conj().T if backward else G
        tw = E.TaylorDirection([Gd], [[np.kron(np.eye(2), SX) - np.kron(SX.T, np.eye(2))]], t, backward, [np.full(15, 0.3)])
        assert len(set(np.round(np.abs(tw.dt_of_class), 12))) == 2  # (classes: the exact steps of the grid)
        v = np.array([1, 0, 0, 0], complex)
        for n in range(len(t) - 1):
            c = int(tw.dt_class_of_step[n])
            dt = float(tw.dt_of_class[c])
            assert dt == (-1 if backward else 1) * (t[n + 1] - t[n])
            Hm = Gd + 0.3 * (np.kron(np.eye(2), SX) - np.kron(SX.T, np.eye(2)))
            got = X.taylor_step(Hm, v, dt, tw.mu[0], tw.scale[0], int(tw.m[0, c]), int(tw.s[0, c]), tw.coeff_table[0, c])
            assert np.abs(got - expm(-1j * Hm * dt) @ v).max() <= 1e-14


def test_theta_table_and_parameter_choice():
    assert E.taylor_params(0.0) == (1, 1)
    for norm in (1e-3, 0.5, 3.0, 40.0, 700.0):
        m, s = E.taylor_params(norm)
        assert norm / s <= min(E.THETA[m - 1], E.THETA_CAP) and m - 1 <= E.M_MAX
        # no other (p, s) of the table with the cap reaches the bound with fewer products
        for p, th in E.THETA.items():
            assert p * max(1, int(np.ceil(norm / min(th, E.THETA_CAP)))) >= (m - 1) * s


# ---- CPU 2: the 1-norm bound over the control range ----------------------------------------------------------------------
POLY = [0.1, 1.0, -0.8]  # vertex at eps = 0.625, inside the range [0, 0.8] of the guess below: |P| peaks there, not at a corner


def _amp_case(amp):
    """(ControlProblem, terms) for the damped qubit with control 0 entering as `amp`; terms[g] = [(operator, a(eps, t))]
    with the amplitude written out independently of the library."""
    w = X.damped_qubit()
    T = float(w.tlist[-1])
    shape = lambda t: 0.5 + 0.1 * t  # noqa: E731
    e = lambda t: 0.8 * W.flattop(t, T=T, t_rise=0.3 * T)  # noqa: E731
    if amp == "linear":
        amps = [[(w.Hc[g][0], e, lambda x, t: x)] for g in range(2)]
    elif amp == "polynomial":
        amps = [[(w.Hc[g][0], K.PolynomialAmplitude(e, POLY, shape), lambda x, t: np.polyval(POLY[::-1], x) * shape(t))]
                for g in range(2)]
    elif amp == "tanh":
        amps = [[(w.Hc[g][0], K.ParametrizedAmplitude(e, K.TanhParametrization(-0.5, 0.5)), lambda x, t: 0.5 * np.tanh(x))]
                for g in range(2)]
    else:  # a tied cos / sin pair of one control
        amps = [[(w.Hc[g][0], K.ShapedAmplitude(e, np.cos), lambda x, t: np.cos(t) * x),
                 (0.5 * w.Hc[g][0], K.ShapedAmplitude(e, np.sin), lambda x, t: np.sin(t) * x)] for g in range(2)]
    gens = [K.hamiltonian(w.H0[g], *[(op, a) for op, a, _ in amps[g]]) for g in range(2)]
    trajs = [K.Trajectory(w.psi0[k], gens[k], target_state=w.target[k]) for k in range(2)]
    prob = K.ControlProblem(trajs, w.tlist, J_T=K.J_T_re, lambda_a=2.0, print_iters=False, iter_stop=1,
                            prop_method=K.Expmv)
    return prob, w, [[(op, f) for op, _, f in amps[g]] for g in range(2)]


@pytest.mark.parametrize("amp", ["linear", "polynomial", "tanh", "tied"])
def test_norm_bound_holds_inside_the_envelope(amp, monkeypatch):
    monkeypatch.setattr(K.workspace, "KrotovCuda", X.ExpmvOracleEngine)
    rng = np.random.default_rng(11)
    prob, w, terms = _amp_case(amp)
    wrk = K.KrotovWrk(prob)
    t = np.asarray(w.tlist)
    mids = 0.5 * (t[1:] + t[:-1])
    for tw in (wrk.fw_settings, wrk.bw_settings):
        nu = tw.norm_rate()
        lo, hi = tw.control_ranges[0]  # (tied terms carry their control's range)
        if amp == "polynomial":
            assert lo <= 0.625 <= hi  # the critical point of P lies inside the range ...
            corners = max(abs(np.polyval(POLY[::-1], x)) for x in (lo, hi))
            assert corners < abs(np.polyval(POLY[::-1], 0.625))  # ... and |P| there exceeds both corners
        worst = 0.0
        for g in range(2):
            for x in np.concatenate([rng.uniform(lo, hi, 300), [lo, hi, 0.625 if lo <= 0.625 <= hi else lo]]):
                n = int(rng.integers(len(mids)))
                Hm = w.H0[g] + sum(f(x, mids[n]) * op for op, f in terms[g])
                if tw.backward:
                    Hm = Hm.conj().T
                M = Hm - tw.mu[g] * np.eye(Hm.shape[0])
                ratio = np.abs(M).sum(axis=0).max() / nu[g]
                worst = max(worst, ratio)
        assert worst <= 1 + 1e-12, worst
        assert worst > 0.5  # (the bound is not vacuous: it is reached to within a factor 2)


# ---- the exact-propagator vectors (tests/golden/*_exact*.json) ------------------------------------------------------------
# every vector the device path accepts, built as the tests of its feature build it; the two *_sigma_exact40 vectors use the
# general second-order update (sigma(t) varying over the grid, a non-Hermitian generator), which the device path refuses
# for either propagator (test_the_general_second_order_vectors_are_refused_as_with_cheby)
VECTORS = ["c1_tls_exact50", "c1_tls_sigma_exact50", "c1_tls_tanh_exact50", "damped_qubit_exact40",
           "c2_transmon_x_g101_exact40", "two_generators_d5_exact40", "non_hermitian_d4_exact40",
           "nonlinear_two_generators_d5_exact40", "c3_two_transmon_g41_exact30", "tls_rotating_frame_terms_exact40",
           "transmon_stark_terms_exact40", "two_generators_shapes_terms_exact40"]


def _recorder():
    hist = dict(J_T=[], g_a_int=[], tau=[])

    def cb(wrk, it, eps_new, eps_old):
        hist["J_T"].append(wrk.result.J_T)
        hist["tau"].append(np.array(wrk.result.tau_vals))
        if it > 0:
            hist["g_a_int"].append(np.array(wrk.g_a_int))
        hist["pulses"] = np.array([np.array(e) for e in eps_new])
        hist["info"] = wrk.engine.info()

    return hist, cb


def _vector_problem(name, **kw):
    """The ControlProblem behind the committed vector `name`, with prop_method=Expmv."""
    import mp_reference as M
    import sat_reference as S
    import terms_reference as R

    kw = dict(prop_method=K.Expmv, **kw)
    if name == "c1_tls_exact50":
        return to_problem(W.c1_tls(), iter_stop=5, **kw)
    if name == "c1_tls_sigma_exact50":
        return to_problem(W.c1_tls(), iter_stop=3, sigma=-2.0, **kw)
    if name == "c1_tls_tanh_exact50":
        return S.param_problem(W.c1_tls(), [K.TanhParametrization(-0.5, 0.5)], iter_stop=5, **kw)
    if name == "damped_qubit_exact40":
        return to_problem(X.damped_qubit(), iter_stop=3, **kw)
    if name == "c3_two_transmon_g41_exact30":
        return to_problem(W.c3_two_transmon(n_grid=41, T=8.0), iter_stop=2, **kw)
    if name.endswith("_terms_exact40"):
        return R.CASES[name[: -len("_terms_exact40")]]().problem(**kw)
    make, iters = M.exact_cases()[name[: -len("_exact40")]]
    return to_problem(make(), iter_stop=iters, **kw)


def _run_vector(name, **kw):
    hist, cb = _recorder()
    K.optimize(_vector_problem(name, callback=cb, **kw), method=K.Krotov)
    g = gold(name)
    err = dict(J_T=np.abs(np.array(hist["J_T"]) - np.array(g["J_T"])).max(),
               pulses=np.abs(hist["pulses"] - np.array(g["pulses"]).reshape(hist["pulses"].shape)).max(),
               g_a=np.abs(np.array(hist["g_a_int"]).reshape(-1) - np.array(g["g_a_int"]).reshape(-1)).max())
    if "tau_re" in g:
        err["tau"] = np.abs(hist["tau"][-1] - (np.array(g["tau_re"]) + 1j * np.array(g["tau_im"]))).max()
    return hist, err


# ---- CPU 3: the host driver (Taylor settings, range events) against the exact-propagator vectors -------------------------
@pytest.mark.parametrize("name", VECTORS)
def test_host_driver_on_the_oracle_engine_meets_the_exact_vectors(name, monkeypatch):
    monkeypatch.setattr(K.workspace, "KrotovCuda", X.ExpmvOracleEngine)
    X.ExpmvOracleEngine.pushed.clear()
    _, err = _run_vector(name)
    assert {d for d, _ in X.ExpmvOracleEngine.pushed} == {0, 1}
    assert max(err.values()) < 1e-12, err


def test_the_general_second_order_vectors_are_refused_as_with_cheby(monkeypatch):
    """non_hermitian_d4_sigma_exact40 and two_generators_d5_sigma_exact40 need sigma(t) varying over the grid (and the
    first a non-Hermitian generator): the device path folds only a constant sigma of a Hermitian problem into chi(T)."""
    import mp_reference as M

    monkeypatch.setattr(K.workspace, "KrotovCuda", X.ExpmvOracleEngine)
    for name in ("non_hermitian_d4", "two_generators_d5"):
        g = gold(name + "_sigma_exact40")
        make, iters = M.exact_cases()[name]
        w = make()
        t = np.asarray(w.tlist)
        sigma = lambda x: -0.6 - 0.3 * x  # noqa: E731  (the sigma(t) of the vector, g["sigma"] on the midpoints)
        assert np.allclose(K.discretize_on_midpoints(sigma, t), g["sigma"])
        for method in (K.Cheby, K.Expmv):
            with pytest.raises(K.ArgumentError, match="sigma"):
                K.optimize(to_problem(w, iter_stop=iters, prop_method=method, sigma=sigma), method=K.Krotov)
        if name == "non_hermitian_d4":  # ... and a constant sigma on the non-Hermitian generator
            for method in (K.Cheby, K.Expmv):
                with pytest.raises(K.ArgumentError, match="Hermitian"):
                    K.optimize(to_problem(w, iter_stop=iters, prop_method=method, sigma=-0.6), method=K.Krotov)


# ---- CPU 4: argument errors before any device work -----------------------------------------------------------------------
def test_argument_errors(monkeypatch):
    monkeypatch.setattr(K.workspace, "KrotovCuda", X.ExpmvOracleEngine)
    w = X.damped_qubit()
    with pytest.raises(K.ArgumentError, match="d <= 32"):
        K.KrotovWrk(to_problem(W.spin_chain(n_spins=6, n_traj=2), prop_method=K.Expmv))
    with pytest.raises(K.ArgumentError, match="replicated"):
        K.KrotovWrk(to_problem(w, prop_method=K.Expmv, multi_gpu="replicate", emulate_ranks=2))
    with pytest.raises(K.ArgumentError, match="same method"):
        K.KrotovWrk(to_problem(w, prop_method=K.Cheby, bw_prop_method=K.Expmv))
    for m in ("ExpProp", "Newton"):
        with pytest.raises(K.ArgumentError, match="Cheby.*Expmv"):
            K.KrotovWrk(to_problem(w, prop_method=m))
    wrk = K.KrotovWrk(to_problem(w, prop_method="Expmv", multi_gpu="auto", emulate_ranks=0))
    assert isinstance(wrk.fw_settings, E.TaylorDirection) and not wrk._replicated


# ============================================================================== GPU
# achieved maxima on one B200 are recorded in DESIGN.md 4.7
@pytest.mark.gpu
@pytest.mark.parametrize("name", VECTORS)
def test_device_expmv_meets_the_exact_vectors(name):
    hist, err = _run_vector(name)
    assert hist["info"]["kernel"] == B.KERNEL_TAYLOR
    print(name, {k: f"{v:.2e}" for k, v in err.items()})
    assert max(err.values()) <= 1e-12, err


@pytest.mark.gpu
def test_reference_tls_test_with_expmv():
    """test/test_tls_optimization.jl:47-70 with prop_method=Expmv; J_T history against the float64 expm oracle."""
    from oracle import krotov_oracle as O

    w = W.c1_tls()
    got = run_product(w, 5, prop_method=K.Expmv)
    res = got["result"]
    assert res.J_T < 1e-3 and 1.0 < np.abs(res.optimized_controls[0]).max() < 1.2
    ref = O.optimize_krotov(W.to_oracle(w), 5, prop_method="expm")
    # 1e-10 relative, with an absolute floor for the last iterations (J_T ~ 1e-5): there both float64 propagators sit
    # ~2e-14 from the 50-digit exact loop (test_device_expmv_meets_the_exact_vectors[c1_tls_exact50])
    assert np.all(np.abs(np.array(got["J_T"]) - ref["J_T"]) <= 1e-10 * np.abs(ref["J_T"]) + 1e-13)


@pytest.mark.gpu
def test_damped_ensemble_on_several_ctas_against_expm():
    from oracle import krotov_oracle as O

    w = X.damped_ensemble()
    got = run_product(w, 2, prop_method=K.Expmv)
    assert got["info"]["grid_blocks"] > 1 and got["info"]["kernel"] == B.KERNEL_TAYLOR
    ref = O.optimize_krotov(W.to_oracle(w), 2, prop_method="expm")
    dj = np.abs(np.array(got["J_T"]) - ref["J_T"])
    assert np.all(dj <= 1e-10 * np.abs(ref["J_T"]) + 2e-15), dj
    assert np.abs(got["pulses"] - ref["pulses"]).max() <= 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [2, 3])
def test_emulated_ranks_shard_bitwise(ranks):
    w = X.damped_ensemble(n_samples=48)
    one = run_product(w, 2, prop_method=K.Expmv)
    hist = {}

    def cb(wrk, it, eps_new, eps_old):
        hist["all"] = np.array(wrk.engine.pulses_all) if it > 0 else None

    got = run_product(w, 2, prop_method=K.Expmv, emulate_ranks=ranks, multi_gpu="auto", callback=cb)
    allp = hist["all"]
    assert allp.shape[0] == ranks
    for r in range(1, ranks):
        assert np.array_equal(allp[r], allp[0])
    assert np.abs(got["pulses"] - one["pulses"]).max() <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tanh", "tied", "host_chi"])
def test_expmv_under_amplitudes_tied_terms_and_host_chi(case):
    from oracle import krotov_oracle as O

    w = X.damped_qubit()
    if case == "host_chi":
        base = K.chi_re
        got = run_product(w, 2, prop_method=K.Expmv, chi=lambda Psi, trajectories, tau=None: base(Psi, trajectories, tau=tau))
        ref = run_product(w, 2, prop_method=K.Expmv)
        assert np.abs(got["pulses"] - ref["pulses"]).max() <= 1e-13
        exp = O.optimize_krotov(W.to_oracle(w), 2, prop_method="expm")
        assert np.abs(got["pulses"] - exp["pulses"]).max() <= 1e-9
        return
    hist = {}

    def cb(wrk, it, eps_new, eps_old):
        hist.setdefault("J", []).append(wrk.result.J_T)
        hist["pulses"] = np.array([np.array(e) for e in eps_new])

    outs = {}
    for method in (K.Expmv, K.Cheby):
        hist.clear()
        e = w.controls[0]
        gens = []
        for g in range(2):
            if case == "tanh":
                terms = [w.H0[g], (w.Hc[g][0], K.ParametrizedAmplitude(e, K.TanhParametrization(-0.5, 0.5)))]
            else:
                terms = [w.H0[g], (w.Hc[g][0], K.ShapedAmplitude(e, lambda t: np.cos(0.3 * t))),
                         (0.5 * w.Hc[g][0], K.ShapedAmplitude(e, lambda t: np.sin(0.3 * t)))]
            gens.append(K.hamiltonian(*terms))
        trajs = [K.Trajectory(w.psi0[k], gens[k], target_state=w.target[k]) for k in range(2)]
        K.optimize(K.ControlProblem(trajs, w.tlist, J_T=K.J_T_re, lambda_a=2.0, print_iters=False, iter_stop=2,
                                    prop_method=method, callback=cb), method=K.Krotov)
        outs[method.__name__] = (np.array(hist["J"]), hist["pulses"].copy())
    # weak-enough decay for Chebyshev at this step: the two propagators agree to the Chebyshev error of the grid
    assert np.abs(outs["Expmv"][1] - outs["Cheby"][1]).max() < 1e-8
    assert np.abs(outs["Expmv"][0] - outs["Cheby"][0]).max() < 1e-10


@pytest.mark.gpu
def test_c_abi_of_expmv():
    from krotov_jl_b200.engine import KrotovCuda

    lib = B.lib()
    base = lib.krotov_live_device_objects()
    w = X.damped_qubit()
    t = np.asarray(w.tlist)
    pulses = np.array([[w.controls[0](x) for x in 0.5 * (t[1:] + t[:-1])]])
    kw = dict(tlist=t, H0=w.H0, Hc=w.Hc, gen_of_traj=w.gen_of_traj, psi0=w.psi0, target=w.target,
              update_shape=np.ones((1, len(t) - 1)), lambda_a=[2.0], functional=B.CHI_RE)
    eng = KrotovCuda(propagator=B.PROP_EXPMV, **kw)
    fw = E.TaylorDirection(w.H0, w.Hc, t, False, pulses)
    bw = E.TaylorDirection([h.conj().T for h in w.H0], [[h.conj().T for h in r] for r in w.Hc], t, True, pulses)
    with pytest.raises(B.KrotovCudaError, match="ERR_STATE"):
        eng.forward(pulses)
    with pytest.raises(B.KrotovCudaError, match="ERR_STATE"):
        nc = len(fw.dt_of_class)
        eng.set_cheby(B.FORWARD, fw.dt_class_of_step, fw.dt_of_class, [0.0, 0.0], [1.0, 1.0], np.ones((2, nc)), np.ones((2, nc, 1)))
    for bad in (dict(m=fw.m * 0), dict(s=fw.s * 0), dict(scale=fw.scale * 0), dict(mu=fw.mu + np.inf),
                dict(scale=fw.scale * np.nan)):
        args = dict(mu=fw.mu, scale=fw.scale, s=fw.s, m=fw.m)
        args.update(bad)
        with pytest.raises(B.KrotovCudaError, match="ERR_ARG"):
            eng.set_taylor(B.FORWARD, fw.dt_class_of_step, fw.dt_of_class, args["mu"], args["scale"], args["s"], args["m"],
                           fw.coeff_table)
    fw.push(eng, B.FORWARD)
    eng.forward(pulses)
    with pytest.raises(B.KrotovCudaError, match="ERR_STATE"):
        eng.iterate(pulses)
    bw.push(eng, B.BACKWARD)
    eng.iterate(pulses)
    info = eng.info()
    assert info["kernel"] == B.KERNEL_TAYLOR and info["m_fw"] == int((fw.m * fw.s).max())
    cheb = KrotovCuda(**kw)
    with pytest.raises(B.KrotovCudaError, match="ERR_STATE"):
        fw.push(cheb, B.FORWARD)
    cheb.close()
    with pytest.raises(B.KrotovCudaError, match="ERR_UNSUPPORTED"):
        KrotovCuda(propagator=B.PROP_EXPMV, replicated_forward=True, **kw)
    with pytest.raises(B.KrotovCudaError, match="ERR_UNSUPPORTED"):
        KrotovCuda(propagator=B.PROP_EXPMV, force_path=B.PATH_DENSE, **kw)
    # more trajectories than one per warp of a co-resident grid (the Chebyshev handle runs them several per warp)
    big = dict(kw, gen_of_traj=np.zeros(14 * 148 * 2, int), psi0=np.repeat(w.psi0[:1], 14 * 148 * 2, 0),
               target=np.repeat(w.target[:1], 14 * 148 * 2, 0), H0=w.H0[:1], Hc=w.Hc[:1])
    with pytest.raises(B.KrotovCudaError, match="ERR_UNSUPPORTED"):
        KrotovCuda(propagator=B.PROP_EXPMV, **big)
    seq = KrotovCuda(**big)
    assert seq.info()["path"] == B.PATH_WARP
    seq.close()
    eng.close()
    assert lib.krotov_live_device_objects() == base


# ---- two real GPUs, shard mode ---------------------------------------------------------------------------------------------
def _mg_run(comm=None):
    hist, cb = _recorder()
    K.optimize(to_problem(X.damped_ensemble(n_samples=64), iter_stop=2, prop_method=K.Expmv, multi_gpu="shard",
                          callback=cb, rethrow_exceptions=True), method=K.Krotov, comm=comm)
    return hist


def _mg_worker(rank, world, port, q):
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "tests")]
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from krotov_jl_b200.distributed import Comm

        got = _mg_run(Comm(device=rank))
        q.put((rank, got["pulses"].tolist(), list(got["J_T"]), np.asarray(got["g_a_int"]).tolist(), got["info"]["kernel"]))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_gpus_shard():
    """The regular Taylor instances under the real cross-rank exchange (krotov_comm_connect, in-kernel NVLink sum)."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp

    one = _mg_run()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 35500 + os.getpid() % 2000
    procs = [ctx.Process(target=_mg_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, pulses, J, ga, kernel in res:
        assert kernel == B.KERNEL_TAYLOR
        assert np.abs(np.asarray(pulses) - one["pulses"]).max() < 1e-12
        assert np.abs(np.array(J) - np.array(one["J_T"])).max() < 1e-12
        assert np.abs(np.array(ga) - np.array(one["g_a_int"])).max() < 1e-12
