"""Control terms tied to one control in the test references -- TEST INFRASTRUCTURE.

A control may enter the generators through several (operator, amplitude) pairs, its TERMS; the update sums the overlaps
of all its terms (``mu = sum_t a_t' H_t``, as QuantumPropagators' ``get_control_deriv`` returns it for a generator).
This module carries that form through the references without touching them:

- ``TermCase``: one small problem written once, as a product ``ControlProblem`` (``problem``) and as the NumPy oracle's
  term-level ``ProblemArrays`` plus the control of every term (``oracle_arrays``);
- ``tie_reduce``: the oracle's ``reduce_du`` hook that sums du over the terms of a control and hands the sum back to every
  term -- with terms taken as controls and the pulse rows duplicated this is exactly the tied update, g_a included;
- ``optimize_terms``: the oracle's first-order loop with that hook;
- ``TermsOracleEngine``: the oracle-backed engine of ``oracle_engine.py`` accepting ``set_control_terms``;
- ``krotov_exact_terms``: the loop of ``mp_reference.krotov_exact_general`` with tied terms, ``mpmath.expm`` per interval;
- ``CASES``: the problems behind ``tests/golden/*_terms_exact40.json`` (``tests/golden/make_golden_terms.py``).
"""
import dataclasses
import os
import sys
from typing import Callable, List

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import mpmath as mp  # noqa: E402
import numpy as np  # noqa: E402

import krotov_jl_b200 as K  # noqa: E402
import workloads as W  # noqa: E402
from krotov_jl_b200.controls import discretize_on_midpoints  # noqa: E402
from oracle import krotov_oracle as O  # noqa: E402
from oracle_engine import OracleEngine  # noqa: E402

_JT = {"sm": K.J_T_sm, "ss": K.J_T_ss, "re": K.J_T_re}
GOLDEN = os.path.join(ROOT, "tests", "golden")


@dataclasses.dataclass
class TermCase:
    name: str
    tlist: np.ndarray
    H0: list                       # per generator
    ops: list                      # ops[g][t]: operator of term t in generator g, or None
    term_ctrl: List[int]           # control of every term (term l = control l for l < C)
    poly: list                     # per term: ascending polynomial coefficients, or None (linear)
    shape: list                    # per term: callable shape(t), or None
    gen_of_traj: np.ndarray
    psi0: np.ndarray
    target: np.ndarray
    guess: List[Callable]          # per control
    lambda_a: float
    functional: str
    iters: int = 2
    update_shape: Callable = lambda t: 1.0

    @property
    def C(self):
        return len(self.guess)

    def problem(self, **kwargs):
        """The product's ControlProblem: one control object per control, one amplitude object per term (shared by every
        generator the term appears in)."""
        controls = list(self.guess)
        amps = []
        for t, c in enumerate(self.term_ctrl):
            ctl = controls[c]
            if self.poly[t] is not None:
                amps.append(K.PolynomialAmplitude(ctl, self.poly[t], self.shape[t]))
            elif self.shape[t] is not None:
                amps.append(K.ShapedAmplitude(ctl, self.shape[t]))
            else:
                amps.append(ctl)
        gens = [K.hamiltonian(self.H0[g], *[(op, amps[t]) for t, op in enumerate(row) if op is not None])
                for g, row in enumerate(self.ops)]
        trajs = [K.Trajectory(self.psi0[k], gens[int(self.gen_of_traj[k])], target_state=self.target[k])
                 for k in range(len(self.psi0))]
        kw = dict(prop_method=K.Cheby, J_T=_JT[self.functional], lambda_a=self.lambda_a, update_shape=self.update_shape,
                  print_iters=False, iter_stop=self.iters)
        kw.update(kwargs)
        return K.ControlProblem(trajs, self.tlist, **kw)

    def oracle_arrays(self):
        """Term-level ``ProblemArrays`` (pulse rows duplicated per term) and the control of every term."""
        T, N_T = len(self.term_ctrl), len(self.tlist) - 1
        pulses = np.array([discretize_on_midpoints(self.guess[c], self.tlist) for c in self.term_ctrl])
        shape = None
        if any(s is not None for s in self.shape):
            shape = np.array([np.ones(N_T) if s is None else discretize_on_midpoints(s, self.tlist) for s in self.shape])
        poly = None if all(q is None for q in self.poly) else list(self.poly)
        dense = lambda m: None if m is None else np.asarray(m.toarray() if hasattr(m, "toarray") else m, complex)  # noqa: E731
        S = np.tile(discretize_on_midpoints(self.update_shape, self.tlist), (T, 1))
        p = O.ProblemArrays(tlist=np.asarray(self.tlist, float), H0=[dense(h) for h in self.H0],
                            Hc=[[dense(h) for h in r] for r in self.ops],
                            gen_of_traj=np.asarray(self.gen_of_traj, int), psi0=self.psi0, target=self.target,
                            pulses=pulses, S=S, lam=np.full(T, float(self.lambda_a)),
                            functional=self.functional, amp_poly=poly, amp_shape=shape)
        return p, np.asarray(self.term_ctrl, int)


def tie_reduce(term_ctrl, inner=None):
    """``reduce_du`` of ``oracle.krotov_iteration``: (after ``inner``, the cross-rank sum) du of every term -> the sum
    over its control's terms in ascending term order."""
    term_ctrl = np.asarray(term_ctrl, int)

    def reduce(du):
        du = np.asarray(du if inner is None else inner(du), float)
        out = np.empty_like(du)
        for t, c in enumerate(term_ctrl):
            out[t] = sum(du[u] for u in range(len(du)) if term_ctrl[u] == c)
        return out

    return reduce


def collapse(term_ctrl, pulses, g_a_terms):
    """Term rows -> per-control pulses (term c is control c) and per-control g_a (every tied term accumulated it)."""
    C = int(np.max(term_ctrl)) + 1
    firsts = [int(np.flatnonzero(np.asarray(term_ctrl) == c)[0]) for c in range(C)]
    return np.asarray(pulses)[:C], np.asarray(g_a_terms)[firsts]


def optimize_terms(p, term_ctrl, iter_stop=2, prop_method="cheby"):
    """The oracle's first-order loop (``optimize_krotov``) with the tie: per-iteration J_T, per-control g_a, final
    per-control pulses."""
    wrk = O.OracleWrk(p, prop_method=prop_method, store_fw=False)
    eps_i, eps_ip1 = wrk.pulses0, wrk.pulses1
    for k in range(p.N):
        O.krotov_initial_fw_prop(eps_i, p.psi0[k], k, wrk)
    O.update_result(wrk)
    hist = dict(J_T=[wrk.J_T], g_a_int=[])
    red = tie_reduce(term_ctrl)
    for _ in range(iter_stop):
        O.krotov_iteration(wrk, eps_i, eps_ip1, reduce_du=red)
        O.update_result(wrk)
        hist["J_T"].append(wrk.J_T)
        hist["g_a_int"].append(collapse(term_ctrl, eps_ip1, wrk.g_a_int)[1])
        eps_i, eps_ip1 = eps_ip1, eps_i
    hist["pulses"] = collapse(term_ctrl, eps_i, wrk.g_a_int)[0]
    return hist


class TermsOracleEngine(OracleEngine):
    """``OracleEngine`` that also takes ``set_control_terms`` (CPU tests of the host driver): the tie runs in the
    oracle's ``reduce_du`` hook after the cross-rank sum; g_a of a control is reported at its first term, as the library
    does."""

    calls = []  # every map the tests' engines were handed (to prove the call was made, or not)

    def __init__(self, **kw):
        super().__init__(**kw)
        self._tie = None

    def set_control_terms(self, control_of_term=None):
        TermsOracleEngine.calls.append(None if control_of_term is None else np.array(control_of_term))
        self._tie = None if control_of_term is None else np.asarray(control_of_term, int)

    def iterate(self, guess_pulses, out_pulses=None):
        inner = self._reduce
        if self._tie is not None:
            self._reduce = tie_reduce(self._tie, inner)
        try:
            new, ga = super().iterate(guess_pulses, out_pulses)
        finally:
            self._reduce = inner
        if self._tie is not None:
            first = np.zeros(len(ga), bool)
            for c in set(self._tie.tolist()):
                first[np.flatnonzero(self._tie == c)[0]] = True
            ga = np.where(first, ga, 0.0)
        return new, ga


# ---- 40-digit reference with tied terms ----------------------------------------------------------------------------
def krotov_exact_terms(p, term_ctrl, iters=2, dps=40):
    """``mp_reference.krotov_exact_general`` (first order, built-in functional) with tied terms: ``p`` is the term-level
    container of ``TermCase.oracle_arrays`` (Float64 inputs only; none of the oracle's code is used).  The update of
    control c at interval n is du_c = sum over its terms t of Im sum_k a_t'(eps_c[n], n) <chi_k|H_t|psi_k>; every term
    of c moves with it, H_t enters the forward step as a_t(eps_c^new[n], n) H_t.  Returns J_T per iteration, per-control
    running costs and the final per-control pulses."""
    mp.mp.dps = dps
    N, d, T, N_T = p.psi0.shape[0], p.psi0.shape[1], len(p.pulses), len(p.tlist) - 1
    ctrl = [int(c) for c in term_ctrl]
    C = max(ctrl) + 1
    first = [ctrl.index(c) for c in range(C)]
    c_ = lambda z: mp.mpc(float(z.real), float(z.imag))  # noqa: E731
    mat = lambda M: mp.matrix([[c_(M[i, j]) for j in range(d)] for i in range(d)])  # noqa: E731
    H0 = [mat(h) for h in p.H0]
    Hc = [[None if h is None else mat(h) for h in row] for row in p.Hc]
    gen = [int(g) for g in p.gen_of_traj]
    psi0 = [mp.matrix([c_(x) for x in p.psi0[k]]) for k in range(N)]
    tgt = [mp.matrix([c_(x) for x in p.target[k]]) for k in range(N)]
    dts = [mp.mpf(float(p.tlist[n + 1])) - mp.mpf(float(p.tlist[n])) for n in range(N_T)]
    eps = [[mp.mpf(float(x)) for x in p.pulses[first[c]]] for c in range(C)]
    S = [[mp.mpf(float(x)) for x in p.S[first[c]]] for c in range(C)]
    lam = [mp.mpf(float(p.lam[first[c]])) for c in range(C)]
    poly = [None] * T if p.amp_poly is None else [None if q is None else [mp.mpf(float(x)) for x in q] for q in p.amp_poly]
    ash = None if p.amp_shape is None else [[mp.mpf(float(x)) for x in row] for row in p.amp_shape]
    j = mp.mpc(0, 1)

    def amp(t, n, e):
        v = e if poly[t] is None else sum(cq * e**q for q, cq in enumerate(poly[t]))
        return v if ash is None else ash[t][n] * v

    def damp(t, n, e):
        v = mp.mpf(1) if poly[t] is None else sum(q * cq * e ** (q - 1) for q, cq in enumerate(poly[t]) if q > 0)
        return v if ash is None else ash[t][n] * v

    def H(g, n, vals):  # vals: per control
        out = H0[g].copy()
        for t in range(T):
            if Hc[g][t] is not None:
                out += amp(t, n, vals[ctrl[t]]) * Hc[g][t]
        return out

    def vdot(a, b):
        return sum(mp.conj(a[i]) * b[i] for i in range(d))

    def J_of(tau):
        if p.functional == "sm":
            return 1 - abs(sum(tau) / N) ** 2
        if p.functional == "ss":
            return 1 - sum(abs(x) ** 2 for x in tau) / N
        return 1 - mp.re(sum(tau)) / N

    def chi_of(tau):
        if p.functional == "sm":
            s = sum(tau)
            return [(s / N**2) * tgt[k] for k in range(N)]
        if p.functional == "ss":
            return [(tau[k] / N) * tgt[k] for k in range(N)]
        return [(mp.mpf(1) / (2 * N)) * tgt[k] for k in range(N)]

    gens = sorted(set(gen))
    states = list(psi0)
    for n in range(N_T):
        U = {g: mp.expm(-j * dts[n] * H(g, n, [eps[c][n] for c in range(C)])) for g in gens}
        states = [U[gen[k]] * states[k] for k in range(N)]
    tau = [vdot(tgt[k], states[k]) for k in range(N)]
    J, ga_hist = [J_of(tau)], []
    for _ in range(iters):
        chi_T = chi_of(tau)
        X = [[None] * (N_T + 1) for _ in range(N)]
        for k in range(N):
            X[k][N_T] = chi_T[k]
        for n in range(N_T - 1, -1, -1):
            Ub = {g: mp.expm(j * dts[n] * H(g, n, [eps[c][n] for c in range(C)]).H) for g in gens}
            for k in range(N):
                X[k][n] = Ub[gen[k]] * X[k][n + 1]
        new = [list(row) for row in eps]
        ga = [mp.mpf(0)] * C
        states = list(psi0)
        for n in range(N_T):
            for c in range(C):
                du = mp.mpf(0)
                for t in range(T):
                    if ctrl[t] != c:
                        continue
                    for k in range(N):
                        mu = Hc[gen[k]][t]
                        if mu is not None:
                            du += mp.im(damp(t, n, eps[c][n]) * vdot(X[k][n], mu * states[k]))
                alpha = S[c][n] / lam[c]
                new[c][n] = eps[c][n] + alpha * du
                ga[c] += alpha * du * du * dts[n]
            U = {g: mp.expm(-j * dts[n] * H(g, n, [new[c][n] for c in range(C)])) for g in gens}
            states = [U[gen[k]] * states[k] for k in range(N)]
        eps = new
        tau = [vdot(tgt[k], states[k]) for k in range(N)]
        J.append(J_of(tau))
        ga_hist.append(ga)
    return dict(J_T=[float(x) for x in J], g_a_int=[[float(x) for x in g] for g in ga_hist],
                pulses=[[float(x) for x in row] for row in eps])


# ---- the problems of the committed vectors ---------------------------------------------------------------------------
def rotating_frame_tls(n_grid=61):
    """A TLS driven in a frame that rotates at the detuning D: eps(t) (cos(D t) sx + sin(D t) sy), one control."""
    sz = np.diag([1.0, -1.0]).astype(complex)
    sx = np.array([[0, 1], [1, 0]], complex)
    sy = np.array([[0, -1j], [1j, 0]], complex)
    D = 0.7
    return TermCase(
        name="tls_rotating_frame", tlist=np.linspace(0.0, 5.0, n_grid), H0=[-0.5 * sz], ops=[[sx, sy]],
        term_ctrl=[0, 0], poly=[None, None], shape=[lambda t: np.cos(D * t), lambda t: np.sin(D * t)],
        gen_of_traj=np.zeros(1, int), psi0=np.array([[1, 0]], complex), target=np.array([[0, 1]], complex),
        guess=[lambda t: 0.2 * W.flattop(t, T=5.0, t_rise=0.3)], lambda_a=1.0, functional="sm")


def transmon_stark(n_grid=101):
    """The d = 3 transmon of C2 driven by eps, with the drive's quadratic ac-Stark shift kappa eps^2 n on the same
    control: (H_d, eps), (H_s, PolynomialAmplitude(eps, [0, 0, 1]))."""
    w = W.c2_transmon_x(n_grid=n_grid)
    Hs = np.diag([0.0, 1.0, 2.0]).astype(complex) * 0.8  # kappa = 0.8 folded into the operator
    return TermCase(
        name="transmon_stark", tlist=w.tlist, H0=list(w.H0), ops=[[w.Hc[0][0], Hs]], term_ctrl=[0, 0],
        poly=[None, [0.0, 0.0, 1.0]], shape=[None, None], gen_of_traj=w.gen_of_traj, psi0=w.psi0, target=w.target,
        guess=list(w.controls), lambda_a=w.lambda_a, functional="sm")


def two_generators_shapes(n_grid=41):
    """Two generators that see control 0 through different shapes (an ensemble member with its own distortion), and a
    second, plain control; J_T_ss."""
    w = W.dummy_dense(d=5, n_traj=4, n_controls=2, n_grid=n_grid, functional="ss", seed=31)
    rng = np.random.default_rng(32)
    A = rng.standard_normal((5, 5)) + 1j * rng.standard_normal((5, 5))
    H0 = [w.H0[0], 0.4 * (A + A.conj().T)]
    H1, H2 = w.Hc[0][0], w.Hc[0][1]
    return TermCase(
        name="two_generators_shapes", tlist=w.tlist, H0=H0, ops=[[H1, H2, None], [None, 0.6 * H2, 0.7 * H1]],
        term_ctrl=[0, 1, 0], poly=[None, None, None],
        shape=[lambda t: 0.5 + 0.25 * t, None, lambda t: 1.0 - 0.3 * t],
        gen_of_traj=np.array([0, 1, 0, 1]), psi0=w.psi0, target=w.target, guess=list(w.controls), lambda_a=0.2,
        functional="ss")


def tie_workload(w, periods=1.5):
    """Workload ``w`` (linear controls) with control 0 driven in a rotating frame: it enters every generator as the pair
    (H_0, ShapedAmplitude(eps_0, cos(D t))), (conj(H_0) / 2, ShapedAmplitude(eps_0, sin(D t))); the other controls
    stay plain.  Term order: controls 0..C-1, then the sin term of control 0."""
    T = float(w.tlist[-1] - w.tlist[0])
    D = 2 * np.pi * periods / T
    C = len(w.controls)
    ops = [[row[l] for l in range(C)] + [None if row[0] is None else 0.5 * row[0].conj()] for row in w.Hc]
    return TermCase(
        name=w.name + "-tied", tlist=w.tlist, H0=list(w.H0), ops=ops, term_ctrl=list(range(C)) + [0],
        poly=[None] * (C + 1), shape=[lambda t: np.cos(D * t)] + [None] * (C - 1) + [lambda t: np.sin(D * t)],
        gen_of_traj=w.gen_of_traj, psi0=w.psi0, target=w.target, guess=list(w.controls), lambda_a=w.lambda_a,
        functional=w.functional, update_shape=w.update_shape)


def rotating_frame_ensemble(n_samples=8, n_grid=201, periods=1.5):
    """C4's ensemble driven by ONE control in a frame rotating at the detuning D: every sample's generator is
    H0 + eps(t) (cos(D t) H_re + sin(D t) H_im) -- two shaped terms of one control, as the register-resident two-term
    instances (and their emulated-rank and replicated-forward forms) serve them."""
    w = W.c4_ensemble(n_samples=n_samples, n_grid=n_grid)
    D = 2 * np.pi * periods / float(w.tlist[-1] - w.tlist[0])
    return TermCase(
        name=f"C4-rotating-frame-{n_samples}", tlist=w.tlist, H0=list(w.H0), ops=[list(r) for r in w.Hc],
        term_ctrl=[0, 0], poly=[None, None], shape=[lambda t: np.cos(D * t), lambda t: np.sin(D * t)],
        gen_of_traj=w.gen_of_traj, psi0=w.psi0, target=w.target, guess=[w.controls[0]], lambda_a=w.lambda_a,
        functional=w.functional, update_shape=w.update_shape)


CASES = {"tls_rotating_frame": rotating_frame_tls, "transmon_stark": transmon_stark,
         "two_generators_shapes": two_generators_shapes}


def golden_path(name):
    return os.path.join(GOLDEN, f"{name}_terms_exact40.json")


def load_golden(name):
    import json

    with open(golden_path(name)) as f:
        return json.load(f)
