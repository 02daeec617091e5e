"""Bounded control amplitudes: pulse parametrizations (square, tanh, tanh**2, logistic, logistic**2) entering the
generator as ``shape[n] * P(tanh(s u))`` (``ParametrizedAmplitude``, ``krotov_set_amplitude_saturation``)."""
import json
import os

import mpmath as mp
import numpy as np
import pytest

import krotov_jl_b200 as K
import sat_reference as S
import workloads as W
from oracle import krotov_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
RTOL_JT, ATOL_JT, ATOL_PULSE = 1e-10, 2e-15, 1e-9


def gold(name):
    with open(os.path.join(GOLD, name + ".json")) as fh:
        return json.load(fh)


def assert_parity(got, ref, rtol=RTOL_JT, atol=ATOL_JT, ga=True):
    ref_JT = np.asarray(ref["J_T"])
    dj = np.abs(np.asarray(got["J_T"]) - ref_JT)
    assert np.all(dj <= rtol * np.abs(ref_JT) + atol), (list(got["J_T"]), list(ref_JT))
    assert np.abs(got["pulses"] - np.asarray(ref["pulses"])).max() <= ATOL_PULSE
    if ga:
        assert np.abs(np.asarray(got["g_a_int"]) - np.asarray(ref["g_a_int"])).max() <= 1e-11


def kinds():
    """(parametrization, closed form of a(u) in mpmath)."""
    return [
        (K.SquareParametrization(), lambda u: u**2),
        (K.TanhParametrization(-0.5, 0.8), lambda u: mp.mpf("0.15") + mp.mpf("0.65") * mp.tanh(u)),
        (K.TanhSqParametrization(0.7), lambda u: mp.mpf("0.7") * mp.tanh(u) ** 2),
        (K.LogisticParametrization(0.1, 0.9, k=1.5), lambda u: mp.mpf("0.1") + mp.mpf("0.8") / (1 + mp.exp(-1.5 * u))),
        (K.LogisticSqParametrization(0.6, k=2.5), lambda u: mp.mpf("0.6") * (2 / (1 + mp.exp(-2.5 * u)) - 1) ** 2),
    ]


# ---- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("i", range(5))
def test_parametrizations_against_closed_forms(i):
    mp.mp.dps = 40
    par, exact = kinds()[i]
    for u in (-3.0, -1.3, -0.5, 0.25, 0.7, 1.9, 3.0):
        a_ref = exact(mp.mpf(u))
        da_ref = mp.diff(exact, mp.mpf(u))
        a, da = float(par.a_of_epsilon(u)), float(par.da_deps_derivative(u))
        assert abs(a - a_ref) <= 1e-14 * abs(a_ref), (u, a, a_ref)
        assert abs(da - da_ref) <= 1e-14 * abs(da_ref), (u, da, da_ref)
        # the device form: P(tanh(s u)) (s = 0: P(u))
        P, s = par.device_form()
        x = np.tanh(s * u) if s > 0 else u
        v = sum(c * x**q for q, c in enumerate(P))
        assert abs(v - a) <= 1e-15 * max(abs(a), 1.0), (u, v, a)
        amp = K.ParametrizedAmplitude(object(), par)
        assert amp.saturation == s and amp.coeffs == [float(c) for c in P] and amp(u) == par.a_of_epsilon(u)
        # epsilon_of_a: the clamped inverse (the squared forms lose the sign of u)
        back = float(par.epsilon_of_a(a))
        want = abs(u) if isinstance(par, (K.SquareParametrization, K.TanhSqParametrization,
                                         K.LogisticSqParametrization)) else u
        assert abs(back - want) <= 1e-11 * max(1.0, abs(want)), (u, back)
    # beyond the range: finite, at the edge
    hi = {K.SquareParametrization: 4.0}.get(type(par), 10.0)
    assert np.isfinite(par.epsilon_of_a(hi)) and np.isfinite(par.epsilon_of_a(-hi))


def test_parametrization_argument_errors():
    for bad in (lambda: K.TanhParametrization(1.0, 1.0), lambda: K.TanhParametrization(2.0, 1.0),
                lambda: K.TanhSqParametrization(0.0), lambda: K.TanhSqParametrization(-1.0),
                lambda: K.LogisticParametrization(1.0, 0.0), lambda: K.LogisticParametrization(0.0, 1.0, k=0.0),
                lambda: K.LogisticParametrization(0.0, 1.0, k=-1.0), lambda: K.LogisticSqParametrization(0.0),
                lambda: K.LogisticSqParametrization(1.0, k=0.0), lambda: K.TanhParametrization(0.0, np.inf)):
        with pytest.raises(ValueError):
            bad()
    with pytest.raises(TypeError):
        K.ParametrizedAmplitude(object(), lambda u: u)
    # a control entering two generators through different parametrizations
    w = W.c1_tls()
    u = w.controls[0]
    H_a = K.hamiltonian(w.H0[0], (w.Hc[0][0], K.ParametrizedAmplitude(u, K.TanhParametrization(-1, 1))))
    H_b = K.hamiltonian(w.H0[0], (w.Hc[0][0], K.ParametrizedAmplitude(u, K.LogisticParametrization(-1, 1, k=2.0))))
    trajs = [K.Trajectory(w.psi0[0], H_a, target_state=w.target[0]), K.Trajectory(w.psi0[0], H_b, target_state=w.target[0])]
    with pytest.raises(K.ArgumentError):
        K.optimize(K.ControlProblem(trajs, w.tlist, prop_method=K.Cheby, J_T=K.J_T_sm, lambda_a=1.0, iter_stop=1,
                                    print_iters=False, rethrow_exceptions=True), method=K.Krotov)


def test_oracle_meets_the_exact_tanh_vector():
    """The NumPy oracle with TanhParametrization(-0.5, 0.5) on the two-level system against the 50-digit
    exact-propagator optimisation (tests/golden/make_golden_sat.py); the committed copy equals a fresh run."""
    g = gold("c1_tls_tanh_exact50")
    fresh = S.tls_tanh_exact(5, amp_poly=tuple(g["amp_poly"]), amp_sat=g["amp_sat"])
    assert fresh["J_T"] == g["J_T"] and fresh["pulses"] == g["pulses"]
    p = S.oracle_problem(W.c1_tls(), [K.TanhParametrization(-0.5, 0.5)])
    for method, tol in (("expm", 2e-14), ("cheby", 5e-13)):
        h = S.optimize_sat(p, 5, method)
        assert np.abs(np.array(h["J_T"]) - np.array(g["J_T"])).max() < tol
        assert np.abs(h["pulses"][0] - np.array(g["pulses"])).max() < tol
        assert np.abs(np.array(h["g_a_int"])[:, 0] - np.array(g["g_a_int"])).max() < tol


def test_host_driver_on_the_oracle_engine_meets_the_exact_tanh_vector(monkeypatch):
    """optimize() -> ParametrizedAmplitude -> set_amplitude_saturation, arithmetic by the oracle."""
    import krotov_jl_b200.workspace as WS

    monkeypatch.setattr(WS, "KrotovCuda", S.SatOracleEngine)
    S.SatOracleEngine.saturations.clear()
    g = gold("c1_tls_tanh_exact50")
    got = S.run_param(W.c1_tls(), [K.TanhParametrization(-0.5, 0.5)], 5)
    assert [list(s) for s in S.SatOracleEngine.saturations] == [[1.0]]
    assert np.abs(np.array(got["J_T"]) - np.array(g["J_T"])).max() < 5e-13
    assert np.abs(got["pulses"][0] - np.array(g["pulses"])).max() < 5e-13
    res = got["result"]  # optimized_controls hold u, on the time grid
    assert len(res.optimized_controls[0]) == 501
    assert np.abs(K.discretize_on_midpoints(res.optimized_controls[0], W.c1_tls().tlist) - got["pulses"][0]).max() < 1e-12


def _wrk(monkeypatch, amp):
    import krotov_jl_b200.workspace as WS

    monkeypatch.setattr(WS, "KrotovCuda", S.SatOracleEngine)
    w = W.c1_tls()
    H = K.hamiltonian(w.H0[0], (w.Hc[0][0], amp(w.controls[0])))
    problem = K.ControlProblem([K.Trajectory(w.psi0[0], H, target_state=w.target[0])], w.tlist, prop_method=K.Cheby,
                               J_T=K.J_T_sm, lambda_a=1.0, iter_stop=1)
    return K.KrotovWrk(problem)


def test_envelope_corners(monkeypatch):
    # tanh**2 over a range straddling 0: the amplitude 0 is part of the range
    par = K.TanhSqParametrization(0.7)
    wrk = _wrk(monkeypatch, lambda c: K.ParametrizedAmplitude(c, par))
    lo, hi = wrk._amp_envelope_corners(0, -0.4, 1.1)
    assert lo == 0.0 and hi == pytest.approx(float(par.a_of_epsilon(1.1)), rel=1e-15)
    assert wrk._amp_envelope_corners(0, 0.2, 1.1) == pytest.approx((par.a_of_epsilon(0.2), par.a_of_epsilon(1.1)), rel=1e-15)
    # logistic**2 likewise
    par = K.LogisticSqParametrization(0.6, k=2.0)
    assert S.saturated_corners(*par.device_form(), -2.0, 0.5)[0] == 0.0
    # tanh: exactly (a(lo), a(hi))
    par = K.TanhParametrization(-0.5, 0.5)
    wrk = _wrk(monkeypatch, lambda c: K.ParametrizedAmplitude(c, par))
    for lo, hi in ((-0.3, 1.2), (0.1, 0.4), (-2.0, -1.0)):
        assert wrk._amp_envelope_corners(0, lo, hi) == (par.a_of_epsilon(lo), par.a_of_epsilon(hi))
    # polynomial amplitudes: the same bits as the per-corner rule (and as the oracle's pinned convention)
    for coeffs in ([0.0, 1.0, 0.5], [0.05, 1.0, 2.0, -0.5], [0.3, -1.0]):
        wrk = _wrk(monkeypatch, lambda c: K.PolynomialAmplitude(c, coeffs))
        p = O.ProblemArrays(tlist=None, H0=None, Hc=None, gen_of_traj=None, psi0=None, target=None, pulses=None, S=None,
                            lam=None, amp_poly=[coeffs])
        for lo, hi in ((-0.3, 1.2), (0.1, 0.4)):
            got = wrk._amp_envelope_corners(0, lo, hi)
            assert got == (wrk._amp_envelope(0, lo), wrk._amp_envelope(0, hi))
            assert got == (p.amplitude_envelope(0, lo), p.amplitude_envelope(0, hi))


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _ensemble():
    w = W.c4_ensemble(n_samples=8, n_grid=201)
    a = [max(float(np.abs(K.discretize(c, w.tlist)).max()), 0.1) for c in w.controls]
    return w, a


@pytest.mark.gpu
def test_tls_tanh_against_oracle_exact_vector_and_bound():
    g = gold("c1_tls_tanh_exact50")
    a_max = 0.5
    par = K.TanhParametrization(-a_max, a_max)
    w = W.c1_tls()
    got = S.run_param(w, [par], 5)
    assert got["info"]["block_threads"] > 32  # the warp kernel, not the one-thread kernel
    ref = S.optimize_sat(S.oracle_problem(w, [par]), 5)
    assert_parity(got, ref)
    assert np.abs(np.array(got["J_T"]) - np.array(g["J_T"])).max() <= 1e-12
    assert np.abs(got["pulses"][0] - np.array(g["pulses"])).max() <= 1e-12
    # the bound holds on every interval of every iteration; the linear run with the same lambda_a exceeds it
    for u in got["pulses_hist"]:
        assert np.abs(par.a_of_epsilon(u)).max() <= a_max
    from util import run_product

    lin = run_product(W.c1_tls(), 5)
    assert np.abs(lin["pulses"]).max() > a_max


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(5))
def test_each_kind_on_the_warp_path(i):
    par = kinds()[i][0]
    w = W.c1_tls()
    got = S.run_param(w, [par], 3)
    assert got["info"]["path"] == 1 and got["info"]["block_threads"] > 32
    ref = S.optimize_sat(S.oracle_problem(w, [par]), 3)
    assert_parity(got, ref)


@pytest.mark.gpu
def test_mixed_polynomial_and_saturating_controls():
    w, a = _ensemble()
    w.amp_poly = [[0.0, 1.0, 2.0], None]
    params = [None, K.TanhParametrization(-2 * a[1], 2 * a[1])]
    got = S.run_param(w, params, 2)
    ref = S.optimize_sat(S.oracle_problem(w, params), 2)
    assert_parity(got, ref, rtol=1e-10, atol=5e-13)


@pytest.mark.gpu
def test_ensemble_multi_cta_and_emulated_ranks():
    w, a = _ensemble()
    params = [K.LogisticParametrization(-2 * a[0], 2 * a[0]), K.TanhSqParametrization(2 * a[1])]
    got = S.run_param(w, params, 2)
    assert got["info"]["grid_blocks"] > 1
    ref = S.optimize_sat(S.oracle_problem(w, params), 2)
    assert_parity(got, ref, rtol=1e-10, atol=5e-13)
    for mode in ("shard", "replicate"):
        two = S.run_param(w, params, 2, emulate_ranks=2, multi_gpu=mode)
        assert np.abs(two["pulses"] - got["pulses"]).max() < 1e-12
        assert np.abs(np.array(two["J_T"]) - np.array(got["J_T"])).max() < 1e-12


def _block_params(w):
    a = [max(float(np.abs(np.asarray(c if not callable(c) else K.discretize(c, w.tlist))).max()), 0.1) for c in w.controls]
    return [K.TanhParametrization(-2 * a[0], 2 * a[0])] + [K.LogisticSqParametrization(2 * x) for x in a[1:]]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dense", "dense_cluster_sweep", "sparse_sweep", "sparse_stream", "reloaded_rows"])
def test_block_paths(kind, monkeypatch):
    kw = {}
    if kind == "dense":
        monkeypatch.setenv("KROTOV_NO_DSWEEP", "1")
        w = W.dummy_dense(d=40, n_traj=6, n_controls=2, n_grid=31, seed=3)
    elif kind == "dense_cluster_sweep":
        w = W.dummy_dense(d=100, n_traj=20, n_controls=1, n_grid=21, seed=101)
    elif kind == "reloaded_rows":
        monkeypatch.setenv("KROTOV_NO_PREG", "1")
        w = W.dummy_dense(d=12, n_traj=5, n_controls=2, n_grid=31, seed=4)
    else:
        if kind == "sparse_stream":
            monkeypatch.setenv("KROTOV_NO_SWEEP", "1")
        w = W.spin_chain(n_spins=6, n_traj=8, n_grid=31)
        kw = {"force_path": 3}
    params = _block_params(w)
    got = S.run_param(w, params, 2, **kw)
    assert got["info"]["path"] == {"reloaded_rows": 1, "dense": 2, "dense_cluster_sweep": 2}.get(kind, 3)
    ref = S.optimize_sat(S.oracle_problem(w, params), 2)
    assert_parity(got, ref, rtol=1e-10, atol=5e-13)


@pytest.mark.gpu
def test_block_path_graph_replay_equals_direct_launches(monkeypatch):
    monkeypatch.setenv("KROTOV_NO_DSWEEP", "1")
    w = W.dummy_dense(d=40, n_traj=6, n_controls=2, n_grid=31, seed=3)
    params = _block_params(w)
    a = S.run_param(w, params, 6)
    assert a["info"]["path"] == 2 and a["info"]["graph_replays"] >= 2
    monkeypatch.setenv("KROTOV_NO_GRAPH", "1")
    b = S.run_param(w, params, 6)
    assert b["info"]["graph_replays"] == 0
    assert np.abs(a["pulses"] - b["pulses"]).max() <= 1e-13
    assert np.abs(np.array(a["J_T"]) - np.array(b["J_T"])).max() <= 1e-14


@pytest.mark.gpu
def test_c_abi_saturation_arguments_and_resources():
    from krotov_jl_b200 import _lib as B

    live0 = B.lib().krotov_live_device_objects()
    w = W.c1_tls()
    checks = []

    def cb(wrk, it, eps_new, eps_old):
        if it != 0:
            return
        for bad in ([-1.0], [np.nan], [np.inf]):
            with pytest.raises(K.KrotovCudaError) as e:
                wrk.engine.set_amplitude_saturation(np.array(bad))
            checks.append(e.value.code == 1)
        wrk.engine.set_amplitude_saturation(np.array([1.0]))
        wrk.engine.set_amplitude_saturation(None if len(checks) == 3 else np.array([0.0]))  # NULL: back to P(u)

    def run(callback):
        H = K.hamiltonian(w.H0[0], (w.Hc[0][0], K.PolynomialAmplitude(w.controls[0], [0.0, 1.0, 0.5])))
        problem = K.ControlProblem([K.Trajectory(w.psi0[0], H, target_state=w.target[0])], w.tlist,
                                   prop_method=K.Cheby, J_T=K.J_T_sm, lambda_a=1.0, iter_stop=3, print_iters=False,
                                   callback=callback)
        return K.optimize(problem, method=K.Krotov)

    plain = run(None)
    restored = run(cb)
    assert checks == [True, True, True]
    assert np.array_equal(plain.optimized_controls[0], restored.optimized_controls[0])
    assert plain.J_T == restored.J_T
    assert B.lib().krotov_live_device_objects() == live0
