"""Saturating (bounded) control amplitudes in the test references -- TEST INFRASTRUCTURE.

A pulse parametrization (``TanhParametrization``, ``LogisticSqParametrization``, ...) enters the generator as
``a_l(u, n) = shape_l[n] * P_l(x)``, ``x = tanh(s_l u)`` for ``s_l > 0`` (else ``x = u``).  This module carries that form
through the references without touching them:

- ``SatProblemArrays``: the NumPy oracle's problem with one more field, ``amp_sat`` (per control, 0 = none), threaded
  through ``amplitude``, ``amplitude_deriv`` and the spectral-envelope corners;
- ``optimize_sat``: the oracle's loop (``optimize_krotov``, first order) on such a problem;
- ``SatOracleEngine``: the oracle-backed engine of ``oracle_engine.py`` accepting ``set_amplitude_saturation``;
- ``tls_tanh_exact``: the two-level system of ``mp_reference.tls_krotov_exact`` in 50-digit arithmetic with the exact
  propagator, the control entering through ``P(tanh(s u))`` (mpmath ``tanh``);
- ``param_problem`` / ``run_param`` / ``oracle_problem``: one Workload written with ``ParametrizedAmplitude`` for the
  product and as a ``SatProblemArrays`` for the oracle.
"""
import dataclasses
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import mpmath as mp  # noqa: E402
import numpy as np  # noqa: E402

import krotov_jl_b200 as K  # noqa: E402
import workloads as W  # noqa: E402
from krotov_jl_b200.workspace import saturated_corners  # noqa: E402
from oracle import krotov_oracle as O  # noqa: E402
from oracle_engine import OracleEngine  # noqa: E402

_JT = {"sm": K.J_T_sm, "ss": K.J_T_ss, "re": K.J_T_re}


@dataclasses.dataclass
class SatProblemArrays(O.ProblemArrays):
    amp_sat: object = None  # (L,) s_l, 0 = the polynomial is evaluated at eps itself

    def _s(self, l):
        return 0.0 if self.amp_sat is None else float(self.amp_sat[l])

    def _row(self, l):
        return [0.0, 1.0] if self.amp_poly is None or self.amp_poly[l] is None else self.amp_poly[l]

    def amplitude(self, l, n, eps):
        s = self._s(l)
        if s == 0.0:
            return super().amplitude(l, n, eps)
        x = np.tanh(s * eps)
        v = 0.0
        for c in reversed(self._row(l)):
            v = v * x + c
        return v if self.amp_shape is None else self.amp_shape[l][n] * v

    def amplitude_deriv(self, l, n, eps):
        s = self._s(l)
        if s == 0.0:
            return super().amplitude_deriv(l, n, eps)
        x = np.tanh(s * eps)
        c = self._row(l)
        v = 0.0
        for q in range(len(c) - 1, 0, -1):
            v = v * x + q * c[q]
        v = v * s * ((1.0 - x) * (1.0 + x))
        return v if self.amp_shape is None else self.amp_shape[l][n] * v

    def amplitude_corners(self, l, lo, hi):
        """Coefficients of H_l at the two sides of the control range [lo, hi] (see ``saturated_corners``)."""
        s = self._s(l)
        if s == 0.0:
            return self.amplitude_envelope(l, lo), self.amplitude_envelope(l, hi)
        return saturated_corners(self._row(l), s, lo, hi,
                                 None if self.amp_shape is None else float(np.max(np.abs(self.amp_shape[l]))))

    @property
    def nonlinear(self):
        return super().nonlinear or self.amp_sat is not None


def sat_problem(p, amp_sat):
    return SatProblemArrays(**{f.name: getattr(p, f.name) for f in dataclasses.fields(O.ProblemArrays)},
                            amp_sat=None if amp_sat is None else np.asarray(amp_sat, float))


class SatChebyPropagator(O.ChebyPropagator):
    """The oracle's Chebyshev propagator with the envelope taken at ``amplitude_corners`` (a range straddling the
    vertex of tanh**2 includes the amplitude 0)."""

    def _set_spectral_envelope(self):
        if self.explicit_specrange is not None or self.problem is None:
            return super()._set_spectral_envelope()
        corners = [self.problem.amplitude_corners(l, a, b) for l, (a, b) in enumerate(self.control_ranges)]

        def G(vals):
            out = self.H0.copy()
            for l, Hl in enumerate(self.Hc):
                if Hl is not None:
                    out = out + vals[l] * Hl
            return out

        E_min, E_max = O.specrange_diag(G([c[1] for c in corners]))
        _E_min, _E_max = O.specrange_diag(G([c[0] for c in corners]))
        E_min, E_max = min(E_min, _E_min), max(E_max, _E_max)
        Delta = E_max - E_min
        delta = self.specrange_buffer * Delta
        self.E_min = E_min - delta / 2
        self.Delta = Delta + delta
        self.dt = self.tlist[1] - self.tlist[0]
        if self.backward:
            self.dt = -self.dt
        self.coeffs = O.cheby_coeffs(self.Delta, self.dt, self.limit)


class SatOracleWrk(O.OracleWrk):
    def __init__(self, p, prop_method="cheby", store_fw=True):
        super().__init__(p, prop_method=prop_method, store_fw=store_fw)
        if prop_method != "cheby":
            return
        kw = dict(limit=p.cheby_limit, specrange_buffer=p.specrange_buffer, specrange=p.specrange, problem=p)
        self.fw_propagators, self.bw_propagators = [], []
        for k in range(p.N):
            g = p.gen_of_traj[k]
            H0, Hc = p.H0[g], p.Hc[g]
            Hca = [None if h is None else h.conj().T for h in Hc]
            self.fw_propagators.append(SatChebyPropagator(H0, Hc, self.tlist, self.pulses0, False, **kw))
            self.bw_propagators.append(SatChebyPropagator(H0.conj().T, Hca, self.tlist, self.pulses0, True, **kw))


def optimize_sat(p, iter_stop=5, prop_method="cheby"):
    """``oracle.krotov_oracle.optimize_krotov`` (first order) with ``SatOracleWrk``: per-iteration J_T, g_a_int, tau,
    the pulses of every iteration and the final pulses."""
    wrk = SatOracleWrk(p, prop_method=prop_method, store_fw=False)
    eps_i, eps_ip1 = wrk.pulses0, wrk.pulses1
    for k in range(p.N):
        O.krotov_initial_fw_prop(eps_i, p.psi0[k], k, wrk)
    O.update_result(wrk)
    hist = dict(J_T=[wrk.J_T], g_a_int=[], tau=[wrk.tau_vals.copy()], pulses_hist=[np.array(eps_i)])
    for _ in range(iter_stop):
        O.krotov_iteration(wrk, eps_i, eps_ip1)
        O.update_result(wrk)
        hist["J_T"].append(wrk.J_T)
        hist["g_a_int"].append(wrk.g_a_int.copy())
        hist["tau"].append(wrk.tau_vals.copy())
        hist["pulses_hist"].append(np.array(eps_ip1))
        eps_i, eps_ip1 = eps_ip1, eps_i
    hist["pulses"] = np.array(eps_i)
    return hist


class SatOracleEngine(OracleEngine):
    """``OracleEngine`` that also takes ``set_amplitude_saturation`` (CPU tests of the host driver)."""

    saturations = []  # every s the tests' engines were handed (to prove the call was made)

    def __init__(self, **kw):
        super().__init__(**kw)
        self.p = sat_problem(self.p, None)

    def set_amplitude_saturation(self, s=None):
        SatOracleEngine.saturations.append(None if s is None else np.array(s, float))
        self.p.amp_sat = None if s is None else np.asarray(s, float).reshape(self.L)

    def _make(self, pulses):
        self.p.pulses = np.array(pulses, float).reshape(self.L, self.N_T)
        self.wrk = SatOracleWrk(self.p, store_fw=self.store_fw)
        self._bufs = [self.wrk.pulses0, self.wrk.pulses1]


# ---- one Workload written with ParametrizedAmplitude (product) and as SatProblemArrays (oracle) ----------------------
def param_problem(w, params, **kwargs):
    """``util.to_problem`` with ``params[l]`` (a parametrization or None) wrapping control l."""
    amps = [c if params[l] is None else K.ParametrizedAmplitude(c, params[l]) for l, c in enumerate(w.controls)]
    for l, c in enumerate(w.controls):  # polynomial amplitudes of the workload on the other controls
        if params[l] is None and w.amp_poly is not None and w.amp_poly[l] is not None:
            amps[l] = K.PolynomialAmplitude(c, w.amp_poly[l])
    gens = []
    for g in range(len(w.H0)):
        terms = [w.H0[g]] + [(w.Hc[g][l], amps[l]) for l in range(len(w.controls)) if w.Hc[g][l] is not None]
        gens.append(K.hamiltonian(*terms))
    trajs = [K.Trajectory(w.psi0[k], gens[int(w.gen_of_traj[k])], target_state=w.target[k]) for k in range(w.N)]
    kw = dict(prop_method=K.Cheby, J_T=_JT[w.functional], lambda_a=w.lambda_a, update_shape=w.update_shape,
              print_iters=False)
    kw.update(kwargs)
    return K.ControlProblem(trajs, w.tlist, **kw)


def run_param(w, params, iters, **kwargs):
    """Optimise through the public API, recording per-iteration J_T, g_a_int, tau and pulses (as ``util.run_product``)."""
    hist = dict(J_T=[], g_a_int=[], tau=[], pulses_hist=[])

    def record(wrk, it, eps_new, eps_old):
        hist["J_T"].append(wrk.result.J_T)
        hist["tau"].append(np.array(wrk.result.tau_vals))
        if it > 0:
            hist["g_a_int"].append(np.array(wrk.g_a_int))
        hist["pulses"] = np.array([np.array(e) for e in eps_new])
        hist["pulses_hist"].append(hist["pulses"])
        hist["info"] = wrk.engine.info()

    res = K.optimize(param_problem(w, params, iter_stop=iters, callback=record, **kwargs), method=K.Krotov)
    hist["result"] = res
    return hist


def oracle_problem(w, params):
    p = W.to_oracle(w)
    L = len(w.controls)
    poly = list(p.amp_poly) if p.amp_poly is not None else [None] * L
    sat = np.zeros(L)
    for l, par in enumerate(params):
        if par is not None:
            poly[l], sat[l] = par.device_form()
    p.amp_poly = poly
    return sat_problem(p, sat if np.any(sat > 0) else None)


# ---- the two-level system in 50-digit arithmetic, control through P(tanh(s u)) --------------------------------------
def tls_tanh_exact(iters=5, amp_poly=(0.0, 0.5), amp_sat=1.0, dps=50, lam=1, n_grid=501):
    """``mp_reference.tls_krotov_exact`` (first order, Float64 grid and guess) with H = -sz/2 + P(tanh(s u)) sx and
    mu = P'(x) s (1 - x^2) sx at the guess value of every interval."""
    import mp_reference as M

    mp.mp.dps = dps
    lam = mp.mpf(lam)
    poly = [mp.mpf(float(c)) for c in amp_poly]
    s = mp.mpf(float(amp_sat))

    def amp(e):
        x = mp.tanh(s * e)
        return sum(c * x**q for q, c in enumerate(poly))

    def damp(e):
        x = mp.tanh(s * e)
        return sum(q * c * x ** (q - 1) for q, c in enumerate(poly) if q > 0) * s * (1 - x * x)

    tl = [mp.mpf(float(x)) for x in np.linspace(0.0, 5.0, n_grid)]
    N_T = n_grid - 1

    def guess(t):
        return mp.mpf(float(0.2 * W.flattop(float(t), T=5.0, t_rise=0.3)))

    mid = [mp.mpf(float(tl[i]) + 0.5 * (float(tl[i + 1]) - float(tl[i]))) for i in range(N_T)]
    eps = [guess(tl[0])] + [guess(mid[i]) for i in range(1, N_T - 1)] + [guess(tl[-1])]
    psi0 = (mp.mpc(1), mp.mpc(0))
    dts = [tl[n + 1] - tl[n] for n in range(N_T)]
    psi = psi0
    for n in range(N_T):
        psi = M._step(psi, amp(eps[n]), dts[n])
    tau = psi[1]
    J = [1 - abs(tau) ** 2]
    ga_hist = []
    for _ in range(iters):
        chi = (mp.mpc(0), tau)
        X = [None] * (N_T + 1)
        X[N_T] = chi
        for n in range(N_T - 1, -1, -1):
            chi = M._step(chi, amp(eps[n]), -dts[n])
            X[n] = chi
        new = list(eps)
        psi = psi0
        ga = mp.mpf(0)
        for n in range(N_T):
            c0, c1 = X[n]
            ov = mp.conj(c0) * psi[1] + mp.conj(c1) * psi[0]
            du = damp(eps[n]) * mp.im(ov)
            alpha = mp.mpf(1) / lam
            new[n] = eps[n] + alpha * du
            ga += alpha * du * du * dts[n]
            psi = M._step(psi, amp(new[n]), dts[n])
        eps = new
        tau = psi[1]
        J.append(1 - abs(tau) ** 2)
        ga_hist.append(ga)
    return dict(J_T=[float(x) for x in J], J_T_mp=J, g_a_int=[float(x) for x in ga_hist], pulses=[float(x) for x in eps])
