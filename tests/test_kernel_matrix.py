"""Every kernel family against the EXACT dynamics, on the features where kernels go wrong.

The other GPU tests compare a kernel with the NumPy or C Chebyshev oracle, which shares the kernel's Chebyshev inputs
(Bessel coefficients, dt classes, spectral window, phase): an error in those shared inputs passes them.  Here every cell
also meets the oracle run with the exact propagator of every interval (``prop_method="expm"``), which uses none of
them.  The problems combine, in few runs:

- grids with several dt classes (three segments where dt returns to an earlier value and a last step that differs), a
  jittered grid where every step has its own dt (a large coefficient table), N_T = 1 and 2;
- ensembles of generators whose spectral radii are ~1.35x apart (different term counts), their trajectories sharing a
  CTA or column block, one generator without a control term, trajectory weights, the three functionals;
- variant A: linear controls and a weakly non-Hermitian generator; variant B: Hermitian, a polynomial amplitude times a
  shape on one control and a TanhParametrization on another.

Every cell also runs with chi(T) from the host (``krotov_set_chi``, a separate code path in every kernel family): a
general observable functional, second order (sigma folded into chi(T)) and a trajectory without a target.  A sequence
test switches one handle between chi(T) from tau, ``krotov_set_chi`` and ``krotov_set_chi_coeffs``.

Each cell selects its kernel with the knobs the library reads and asserts, through ``info()``, which kernel served it.
The exact bound of every (problem, boundary condition) (BOUND) is 10x the CPU Chebyshev-oracle-vs-exact gap rounded up
to a power of ten; the CPU tests at the bottom check that the oracle meets BOUND / 10, so a GPU miss is the kernel's,
and that every host boundary condition moves the exact pulses by >= 1e4 x BOUND."""
import functools
import zlib

import numpy as np
import pytest
from scipy.linalg import expm

import krotov_jl_b200 as K
import sat_reference as S
import workloads as W
from krotov_jl_b200 import _lib as B
from oracle import krotov_oracle as O

RTOL_JT, ATOL_JT, ATOL_PULSE = 1e-10, 2e-15, 1e-9  # BASELINE.json
_JT = {"sm": K.J_T_sm, "ss": K.J_T_ss, "re": K.J_T_re}


# ---- problems ----------------------------------------------------------------------------------------------------------
def _segments(T, n):
    """~n steps in three segments, dt -> 1.25 dt -> dt, and a last step of 0.6 dt."""
    k = n // 3
    steps = [1.0] * k + [1.25] * k + [1.0] * (n - 2 * k - 1) + [0.6]
    t = np.concatenate([[0.0], np.cumsum(steps)])
    return t * (T / t[-1])


def _jittered(T, n, seed):
    """n steps, every one its own dt: dt_n = dt (1 + 1e-3 u_n)."""
    u = np.random.default_rng(seed).uniform(-1.0, 1.0, n)
    t = np.concatenate([[0.0], np.cumsum(1.0 + 1e-3 * u)])
    return t * (T / t[-1])


def _ensemble(w, n_gen, gen_of_traj, drop_term=True):
    """n_gen generators, spectral radii 1.35x apart; the last one does not depend on the last control."""
    H0, Hc = w.H0[0], w.Hc[0]
    w.H0 = [H0 * 1.35**g for g in range(n_gen)]
    w.Hc = [list(Hc) for _ in range(n_gen)]
    if drop_term and len(Hc) > 1 and n_gen > 1:
        w.Hc[-1][-1] = None
    w.gen_of_traj = np.asarray(gen_of_traj, int)
    return w


def _non_hermitian(w, seed):
    """Variant A: weak decay on every drift, a non-Hermitian admixture to the first control (as the seeded sweep), kept
    to that control's sparsity pattern so that the rows stay as narrow as the kernel family needs."""
    rng = np.random.default_rng(seed)
    d = w.d
    decay = -0.02j * np.diag(rng.uniform(0, 1, d))
    Bm = (rng.standard_normal((d, d)) + 1j * rng.standard_normal((d, d))) / np.sqrt(d)
    w.H0 = [h + decay for h in w.H0]
    w.Hc = [[row[0] + 0.05 * Bm * (row[0] != 0)] + list(row[1:]) for row in w.Hc]
    return w


def _amplitudes(w):
    """Variant B: control 0 as shape(t) * (eps + 0.8 eps^2 - 0.3 eps^3), control 1 through TanhParametrization."""
    T = float(w.tlist[-1])
    L = len(w.controls)
    w.amp_poly = [[0.0, 1.0, 0.8, -0.3]] + [None] * (L - 1)
    w.amp_shape = [lambda t: 0.6 + 0.4 * W.flattop(t, T=T, t_rise=0.3 * T)] + [None] * (L - 1)
    amax = max(abs(W.midpoint_samples(w.controls[1], w.tlist)).max(), 0.05) if L > 1 else 0.0
    params = [None] * L
    if L > 1:
        params[1] = K.TanhParametrization(-1.5 * amax, 1.5 * amax)
    return w, params


class Case:
    def __init__(self, w, params=None, weight=None):
        self.w, self.weight = w, weight
        self.params = params if params is not None else [None] * len(w.controls)

    def oracle(self):
        p = S.oracle_problem(self.w, self.params)
        if self.weight is not None:
            p.weight = np.asarray(self.weight, float)
        return p

    def problem(self, **kw):
        """The same problem through the public API (Generator objects shared by the trajectories of one generator)."""
        w = self.w
        amps = []
        for l, c in enumerate(w.controls):
            poly = None if w.amp_poly is None else w.amp_poly[l]
            shape = None if w.amp_shape is None else w.amp_shape[l]
            if self.params[l] is not None:
                amps.append(K.ParametrizedAmplitude(c, self.params[l], shape))
            elif poly is not None:
                amps.append(K.PolynomialAmplitude(c, poly, shape))
            elif shape is not None:
                amps.append(K.ShapedAmplitude(c, shape))
            else:
                amps.append(c)
        gens = [K.hamiltonian(w.H0[g], *[(w.Hc[g][l], amps[l]) for l in range(w.L) if w.Hc[g][l] is not None])
                for g in range(len(w.H0))]
        trajs = [K.Trajectory(w.psi0[k], gens[int(w.gen_of_traj[k])], target_state=w.target[k]) for k in range(w.N)]
        if self.weight is not None:
            for t, x in zip(trajs, self.weight):
                t.weight = float(x)
        args = dict(prop_method=K.Cheby, J_T=_JT[w.functional], lambda_a=w.lambda_a, update_shape=w.update_shape,
                    print_iters=False)
        if w.specrange is not None:
            args.update(prop_E_min=w.specrange[0], prop_E_max=w.specrange[1])
        args.update(kw)
        return K.ControlProblem(trajs, w.tlist, **args)


def _dummy(d, n_traj, L, n_grid, seed, functional, tlist=None, flat_shape=False):
    w = W.dummy_dense(d=d, n_traj=n_traj, n_controls=L, n_grid=n_grid, seed=seed, functional=functional)
    if tlist is not None:
        w.tlist = tlist
    if flat_shape:  # (the flattop update shape vanishes on the ends of very short grids)
        w.update_shape = lambda t: 1.0
    return w


def _weights(n, seed):
    return np.random.default_rng(seed).uniform(0.4, 1.6, n)


def _warp(L, variant, functional):
    """d = 7 (six off-diagonal slots: register-row, pair and reloaded-row instances exist for L = 1, 2, 3), three
    generators over 6 trajectories in one CTA."""
    w = _ensemble(_dummy(7, 6, L, 0, 40 + L, functional, tlist=_segments(5.0, 36)), 3, [0, 1, 2, 2, 0, 1])
    if variant == "A":
        return Case(_non_hermitian(w, 50 + L), weight=_weights(6, L))
    w, params = _amplitudes(w)
    return Case(w, params, weight=_weights(6, L))


def _pair(variant):
    """Generator-sharing pairs: trajectories 2j, 2j+1 share a generator, three generators."""
    w = _ensemble(_dummy(7, 8, 2, 0, 61, "sm", tlist=_segments(5.0, 30)), 3, [0, 0, 1, 1, 2, 2, 0, 0])
    if variant == "A":
        return Case(_non_hermitian(w, 62), weight=_weights(8, 3))
    w, params = _amplitudes(w)
    return Case(w, params, weight=_weights(8, 3))


def _c4(n_samples, levels, n_grid, T):
    w = W.c4_ensemble(n_samples=n_samples, n_grid=n_grid, levels=levels, T=T)
    w.tlist = _segments(T, n_grid - 1)
    a = 0.6 * abs(W.midpoint_samples(w.controls[0], w.tlist)).max()
    w.controls = [w.controls[0], lambda t, a=a: a * W.flattop(t, T=T, t_rise=0.2 * T)]  # (C4's second guess is 0)
    return w


def _sparse(variant):
    w = W.spin_chain(n_spins=6, n_traj=8, n_grid=2, functional="ss")
    w.tlist = _segments(4.0, 24)
    w = _ensemble(w, 2, [0, 1, 0, 1, 1, 0, 0, 1], drop_term=False)
    if variant == "A":
        w.H0 = [h - 0.02j * np.diag(np.linspace(0, 1, w.d)) for h in w.H0]  # decay: non-Hermitian
        return Case(w, weight=_weights(8, 9))
    w, params = _amplitudes(w)
    return Case(w, params, weight=_weights(8, 9))


PROBLEMS = {
    # tiny kernel: d <= 4, N <= 32, L <= 2; a jittered grid of 40 own dt (the coefficient table leaves shared memory)
    "tiny_jitter": lambda: Case(_non_hermitian(_ensemble(_dummy(4, 6, 2, 0, 11, "sm", tlist=_jittered(5.0, 40, 1)), 2,
                                                         [0, 1, 1, 0, 1, 0]), 12), weight=_weights(6, 1)),
    "tiny_nt2": lambda: Case(_dummy(3, 3, 1, 0, 13, "re", tlist=np.array([0.0, 0.3, 0.45]), flat_shape=True)),
    "warp_nt1": lambda: Case(_dummy(7, 3, 2, 2, 14, "ss", flat_shape=True), weight=_weights(3, 2)),
    "warp_L1_A": lambda: _warp(1, "A", "ss"),
    "warp_L1_B": lambda: _warp(1, "B", "re"),
    "warp_L2_A": lambda: _warp(2, "A", "re"),
    "warp_L2_B": lambda: _warp(2, "B", "sm"),
    "warp_L3_A": lambda: _warp(3, "A", "sm"),
    "warp_L3_B": lambda: _warp(3, "B", "ss"),
    "warp_L5_A": lambda: _warp(5, "A", "ss"),
    "warp_L5_B": lambda: _warp(5, "B", "sm"),
    "pair_A": lambda: _pair("A"),
    "pair_B": lambda: _pair("B"),
    # more than 7 x 148 trajectories in runs of two per generator: sequential register rows
    "seq_B": lambda: Case(*_amplitudes(_ensemble(_dummy(5, 1040, 2, 0, 71, "ss", tlist=_segments(5.0, 12)), 3,
                                                 (np.arange(1040) // 2) % 3))),
    # transmon ensembles: short times, so that the Chebyshev truncation error of the exact comparison stays small
    "wide64_A": lambda: Case(_non_hermitian(_c4(6, 7, 21, 4.0), 81), weight=_weights(24, 4)),
    "wide64_B": lambda: Case(*_amplitudes(_c4(6, 7, 21, 4.0)), weight=_weights(24, 4)),
    "wide128_B": lambda: Case(*_amplitudes(_c4(1, 10, 16, 3.0))),
    "ranks_B": lambda: Case(*_amplitudes(_c4(8, 5, 21, 4.0)), weight=_weights(32, 5)),
    "ranks_lin": lambda: Case(_c4(8, 5, 21, 4.0), weight=_weights(32, 5)),
    "dense_A": lambda: Case(_non_hermitian(_ensemble(_dummy(40, 6, 2, 0, 91, "ss", tlist=_segments(5.0, 20)), 2,
                                                     [0, 1, 1, 0, 0, 1]), 92), weight=_weights(6, 6)),
    "dense_B": lambda: Case(*_amplitudes(_ensemble(_dummy(40, 6, 2, 0, 93, "re", tlist=_segments(5.0, 20)), 2,
                                                   [0, 1, 1, 0, 0, 1])), weight=_weights(6, 7)),
    "sparse_A": lambda: _sparse("A"),
    "sparse_B": lambda: _sparse("B"),
}


def _graph_case():
    w = _ensemble(_dummy(48, 6, 2, 0, 95, "sm", tlist=_segments(5.0, 20)), 2, [0, 1, 0, 1, 1, 0])
    w.specrange = (-6.0, 6.0)  # a fixed window: the tables never change, so the settled iteration is captured
    return Case(w, weight=_weights(6, 8))


PROBLEMS["graph_A"] = _graph_case
ITERS = {"graph_A": 5}


@functools.lru_cache(maxsize=None)
def case(name):
    return PROBLEMS[name]()


# ---- boundary conditions ---------------------------------------------------------------------------------------------
# Where chi(T) comes from.  builtin: c_k |target_k>, formed on the device from tau (chi_coef_kernel); user_chi: the
# Observable functional below, chi(T) from the host (krotov_set_chi) every iteration; sigma: second order with a constant
# sigma, folded into chi(T) on the host (second_order.py); no_target: the Observable functional with no target for
# trajectory 0 (tau_0 = 0).
BOUNDARIES = ("builtin", "user_chi", "sigma", "no_target")


class Observable:
    """J_T = 1 - (1/N) sum_k w_k Re<Psi_k|O_k|Psi_k>, chi_k = -dJ_T/d<Psi_k| = (w_k / N) O_k Psi_k, with
    O_k = |tgt_k><tgt_k| + coupling R_k and R_k a seeded random Hermitian matrix of its own for every trajectory:
    trajectories that share a CTA, a pair or a column block get different chi(T), and every component of chi(T) is
    non-zero."""

    def __init__(self, target, weight, seed, coupling):
        N, d = target.shape
        g = np.random.default_rng(seed).standard_normal((2, N, d, d))
        A = g[0] + 1j * g[1]
        R =(A + A.conj().transpose(0, 2, 1)) / (2 * np.sqrt(d))
        self.O = np.einsum("ki,kj->kij", target, target.conj()) + coupling * R
        self.w = np.ones(N) if weight is None else np.asarray(weight, float)

    @staticmethod
    def _psi(states):
        return np.array([np.asarray(s) for s in states], complex)

    def chi(self, states, trajectories=None):
        return list((self.w / len(self.w))[:, None] * np.einsum("kij,kj->ki", self.O, self._psi(states)))

    def J_T(self, states, trajectories=None):
        psi = self._psi(states)
        return 1.0 - float(np.sum(self.w * np.einsum("ki,kij,kj->k", psi.conj(), self.O, psi).real)) / len(self.w)

    def mp_hooks(self):
        """(J_T, chi) of mp_reference.krotov_exact_general: the same functional on mpmath column vectors."""
        import mpmath as mp

        N, d = self.O.shape[:2]
        O = [mp.matrix([[mp.mpc(complex(self.O[k, i, j])) for j in range(d)] for i in range(d)]) for k in range(N)]
        w = [mp.mpf(float(x)) for x in self.w]

        def J_T(states):
            return 1 - sum(w[k] * mp.re((states[k].H * (O[k] * states[k]))[0, 0]) for k in range(N)) / N

        def chi(states):
            return [(w[k] / N) * (O[k] * states[k]) for k in range(N)]

        return J_T, chi


# constant sigma per Hermitian problem: moves the pulses by >= 1e-4 against first order (test_boundaries_move_the_pulses).
# Not warp_nt1: with one time interval the second-order term is <Psi^(i+1)(0) - Psi^(i)(0)|...> = 0.  The sigma term
# is summed over the trajectories without the 1/N of chi: seq_B's 1040 trajectories take a sigma ~1/200 of the others'.
SIGMA = {
    "tiny_nt2": -4.0, "warp_L1_B": -4.0, "warp_L2_B": -4.0, "warp_L3_B": -4.0, "warp_L5_B": -4.0, "pair_B": -4.0,
    "seq_B": -0.02, "wide64_B": -4.0, "wide128_B": -8.0, "ranks_B": -4.0, "ranks_lin": -4.0, "dense_B": -4.0,
    "sparse_B": -1.0, "graph_A": -4.0,
}
# problems of the no_target cells: tiny, register rows, pair, dense sweep, sparse sweep
NO_TARGET = ("tiny_nt2", "warp_L2_B", "pair_B", "dense_B", "sparse_B")


def applies(name, boundary):
    return (boundary in ("builtin", "user_chi") or (boundary == "sigma" and name in SIGMA) or
            (boundary == "no_target" and name in NO_TARGET))


@functools.lru_cache(maxsize=None)
def observable(name, boundary):
    w, c = case(name).w, case(name)
    target = np.array(w.target, complex).reshape(w.N, w.d)
    if boundary == "no_target":
        target[0] = 0.0
    # (warp_nt1: its one interval spans the whole time; with 0.3 the updated pulse widens the spectral window so far that
    # the Chebyshev oracle itself leaves the exact run by 1.7e-12)
    return Observable(target, c.weight, seed=zlib.crc32(name.encode()), coupling=0.1 if name == "warp_nt1" else 0.3)


# exact bound per (problem, boundary): 10 x the CPU Chebyshev-oracle-vs-exact gap, rounded up to a power of ten, <= 1e-11
BOUND = {
    "tiny_jitter": 1e-12, "tiny_nt2": 1e-13, "warp_nt1": 1e-12, "warp_L1_A": 1e-12, "seq_B": 1e-12, "dense_A": 1e-12,
    "dense_B": 1e-12, "sparse_B": 1e-12, "graph_A": 1e-12,
    "warp_L1_B": 1e-11, "warp_L2_A": 1e-11, "warp_L2_B": 1e-11, "warp_L3_A": 1e-11, "warp_L3_B": 1e-11,
    "warp_L5_A": 1e-11, "warp_L5_B": 1e-11, "pair_A": 1e-11, "pair_B": 1e-11, "wide64_A": 1e-11, "wide64_B": 1e-11,
    "wide128_B": 1e-11, "ranks_B": 1e-11, "ranks_lin": 1e-11, "sparse_A": 1e-11,
}
BOUND = {(name, "builtin"): b for name, b in BOUND.items()}
BOUND.update({(name, "user_chi"): 1e-11 for name in PROBLEMS})
BOUND.update({(name, "user_chi"): 1e-12 for name in ("tiny_jitter", "warp_nt1", "warp_L1_A", "seq_B", "dense_A",
                                                     "dense_B", "sparse_B", "graph_A")})
BOUND["tiny_nt2", "user_chi"] = 1e-13
BOUND.update({(name, "sigma"): 1e-11 for name in SIGMA})
BOUND.update({(name, "sigma"): 1e-12 for name in ("seq_B", "dense_B", "sparse_B", "graph_A")})
BOUND["tiny_nt2", "sigma"] = 1e-13
BOUND.update({("tiny_nt2", "no_target"): 1e-12, ("warp_L2_B", "no_target"): 1e-11, ("pair_B", "no_target"): 1e-11,
              ("dense_B", "no_target"): 1e-12, ("sparse_B", "no_target"): 1e-12})
BOUND.update({("tiny_jitter", "sequence"): 1e-12, ("warp_L2_A", "sequence"): 1e-11, ("pair_B", "sequence"): 1e-11,
              ("graph_A", "sequence"): 1e-12, ("dense_A", "sequence"): 1e-12, ("sparse_B", "sequence"): 1e-12})


# ---- references ------------------------------------------------------------------------------------------------------
class _SharedExp(O.ExpPropagator):
    """The exact propagator of one interval, computed once per (generator, direction, interval, amplitudes) and shared
    by the trajectories of that generator."""

    def __init__(self, *args, cache):
        super().__init__(*args)
        self.cache = cache

    def prop_step(self):
        ni, dt = self._interval_and_dt()
        ops, cf = self._ops_coeffs(ni)
        key = tuple(cf)
        hit = self.cache.get(ni)
        if hit is None or hit[0] != key:
            H = sum(c * op for op, c in zip(ops, cf))
            hit = (key, expm(-1j * dt * (H.toarray() if hasattr(H, "toarray") else H)))
            self.cache[ni] = hit
        self.state = hit[1] @ self.state
        self._advance()
        return self.state


def reference_run(p, iters, prop_method, chi=None, J_T=None, sigma=None):
    """The oracle's loop (``optimize_krotov``, saturating amplitudes included) recording J_T, g_a_int and tau of every
    iteration, the final pulses and states, and every slot of both storages after the last iteration.

    chi: None (the built-in chi(T) of ``p.functional``), a callable Psi(T) -> chi(T) for every iteration, or
    {iteration: callable} for the iterations (1-based) that take chi(T) from it.  J_T: a callable Psi(T) -> J_T in place
    of the built-in functional.  sigma: a constant second-order sigma, through the oracle's general formula from the
    stored previous trajectory.  With sigma there is no X: the device stores the backward-propagated boundary condition
    chi(T) - sigma/2 Psi^(i)(T) (second_order.py), whose distance from the exact one is sigma/2 times the propagation
    error of Psi^(i) -- the pulses, g_a_int and J_T test the fold."""
    wrk = S.SatOracleWrk(p, prop_method=prop_method, store_fw=True)
    if sigma is not None:
        wrk.enable_second_order()
    if prop_method == "expm":
        caches = {}
        for k in range(p.N):
            g = int(p.gen_of_traj[k])
            for q, props in enumerate((wrk.fw_propagators, wrk.bw_propagators)):
                old = props[k]
                props[k] = _SharedExp(old.H0, old.Hc, old.tlist, old.parameters, old.backward, p,
                                      cache=caches.setdefault((g, q), {}))
    eps_i, eps_ip1 = wrk.pulses0, wrk.pulses1
    for k in range(p.N):
        O.krotov_initial_fw_prop(eps_i, p.psi0[k], k, wrk)

    def result():
        states = O.update_result(wrk)
        if J_T is not None:
            wrk.J_T = J_T(states)
        return states

    result()
    out = dict(J_T=[wrk.J_T], g_a_int=[], tau=[wrk.tau_vals.copy()])
    sv = None if sigma is None else np.full(p.N_T, float(sigma))
    for i in range(1, iters + 1):
        O.krotov_iteration(wrk, eps_i, eps_ip1, chi=chi.get(i) if isinstance(chi, dict) else chi, sigma_vals=sv)
        states = result()
        out["J_T"].append(wrk.J_T)
        out["g_a_int"].append(wrk.g_a_int.copy())
        out["tau"].append(wrk.tau_vals.copy())
        eps_i, eps_ip1 = eps_ip1, eps_i
    out["pulses"] = np.array(eps_i)
    out["states"] = np.array(states)
    out["X"] = np.array(wrk.bw_storage) if sigma is None else None
    out["Phi"] = np.array(wrk.fw_storage)
    return out


def boundary_problem(name, boundary):
    """The oracle problem of `case(name)` and the keywords of reference_run for the boundary condition."""
    p = case(name).oracle()
    kw = {}
    if boundary in ("user_chi", "no_target"):
        obs = observable(name, boundary)
        kw = dict(chi=obs.chi, J_T=obs.J_T)
        if boundary == "no_target":
            p.target = np.array(p.target)
            p.target[0] = 0.0
    elif boundary == "sigma":
        kw = dict(sigma=SIGMA[name])
    return p, kw


@functools.lru_cache(maxsize=None)
def exact(name, boundary="builtin"):
    p, kw = boundary_problem(name, boundary)
    return reference_run(p, ITERS.get(name, 2), "expm", **kw)


@functools.lru_cache(maxsize=None)
def cheby(name, boundary="builtin"):
    p, kw = boundary_problem(name, boundary)
    return reference_run(p, ITERS.get(name, 2), "cheby", **kw)


def deviations(got, ref, storage=True):
    """Largest absolute deviation per quantity."""
    dev = dict(J_T=np.abs(np.asarray(got["J_T"]) - ref["J_T"]).max(),
               pulses=np.abs(np.asarray(got["pulses"]) - ref["pulses"]).max(),
               g_a_int=np.abs(np.asarray(got["g_a_int"]) - np.asarray(ref["g_a_int"])).max(),
               tau=np.abs(np.asarray(got["tau"]) - np.asarray(ref["tau"])).max(),
               states=np.abs(np.asarray(got["states"]) - ref["states"]).max())
    for key in ("X", "Phi") if storage else ():
        if ref[key] is not None:
            dev[key] = np.abs(np.asarray(got[key]) - ref[key]).max()
    return dev


# ---- cells ---------------------------------------------------------------------------------------------------------------
# name -> (problem, environment, optimize keywords, kernel, lanes per trajectory, exchange)
_PREG, _SEQ, _PAIR, _RELOAD = B.KERNEL_PREG, B.KERNEL_SEQ_PREG, B.KERNEL_PAIR, B.KERNEL_RELOAD
CELLS = {
    "tiny_jitter": ("tiny_jitter", {}, {}, B.KERNEL_TINY, 1, 0),
    "tiny_nt2": ("tiny_nt2", {}, {}, B.KERNEL_TINY, 1, 0),
    "preg_nt1": ("warp_nt1", {}, {}, _PREG, 32, 0),
    "preg_L1_A": ("warp_L1_A", {}, {}, _PREG, 32, 0),
    "preg_L1_B": ("warp_L1_B", {}, {}, _PREG, 32, 0),
    "preg_L2_A": ("warp_L2_A", {}, {}, _PREG, 32, 0),
    "preg_L2_B": ("warp_L2_B", {}, {}, _PREG, 32, 0),
    "preg_L3_A": ("warp_L3_A", {}, {}, _PREG, 32, 0),
    "preg_L3_B": ("warp_L3_B", {}, {}, _PREG, 32, 0),
    "reload_L5_A": ("warp_L5_A", {"KROTOV_NO_PREG": "1"}, {}, _RELOAD, 32, 0),
    "reload_L5_B": ("warp_L5_B", {"KROTOV_NO_PREG": "1"}, {}, _RELOAD, 32, 0),
    "pair_A": ("pair_A", {"KROTOV_FORCE_PAIR": "1"}, {}, _PAIR, 32, 0),
    "pair_B": ("pair_B", {"KROTOV_FORCE_PAIR": "1"}, {}, _PAIR, 32, 0),
    "seq_B": ("seq_B", {"KROTOV_SEQ_PREG": "1"}, {}, _SEQ, 32, 0),
    "wide64_A": ("wide64_A", {}, {}, _PREG, 64, 0),
    "wide64_B": ("wide64_B", {}, {}, _PREG, 64, 0),
    "wide128_B": ("wide128_B", {}, {}, _PREG, 128, 0),
    "ranks_hier_B": ("ranks_B", {"KROTOV_XCHG": "hier"}, dict(emulate_ranks=2, multi_gpu="shard"), _PREG, 32, 1),
    "ranks_mbox": ("ranks_lin", {"KROTOV_XCHG": "mbox"}, dict(emulate_ranks=3, multi_gpu="shard"), _PREG, 32, 3),
    "ranks_rf_B": ("ranks_B", {}, dict(emulate_ranks=2, multi_gpu="replicate"), _PREG, 32, 5),
    "dmma_A": ("dense_A", {"KROTOV_NO_DSWEEP": "1"}, {}, B.KERNEL_DMMA_STREAM, 0, 0),
    "dmma_B": ("dense_B", {"KROTOV_NO_DSWEEP": "1"}, {}, B.KERNEL_DMMA_STREAM, 0, 0),
    "dsweep_A": ("dense_A", {}, {}, B.KERNEL_DENSE_SWEEP, 0, 0),
    "dsweep_B": ("dense_B", {}, {}, B.KERNEL_DENSE_SWEEP, 0, 0),
    "sparse_sweep_A": ("sparse_A", {}, dict(force_path=3), B.KERNEL_SPARSE_SWEEP, 0, 0),
    "sparse_sweep_B": ("sparse_B", {}, dict(force_path=3), B.KERNEL_SPARSE_SWEEP, 0, 0),
    "sparse_stream_A": ("sparse_A", {"KROTOV_NO_SWEEP": "1"}, dict(force_path=3), B.KERNEL_SPARSE_STREAM, 0, 0),
    "sparse_stream_B": ("sparse_B", {"KROTOV_NO_SWEEP": "1"}, dict(force_path=3), B.KERNEL_SPARSE_STREAM, 0, 0),
    "graph_A": ("graph_A", {"KROTOV_NO_DSWEEP": "1"}, {}, B.KERNEL_DMMA_STREAM, 0, 0),
}


def run_cell(c, iters, storage, no_target=False, on_iteration=None, **kw):
    """Optimise through the public API; J_T, g_a_int, tau of every iteration, the final pulses and states, every slot of
    both storages after the last iteration (one-rank runs), ``info()`` of the last iteration, ``graph_replays`` after
    every iteration and the number of ``set_chi`` calls.  no_target: trajectory 0 has no target state.
    on_iteration(wrk, it): called at the end of the callback of iteration `it`."""
    hist = dict(J_T=[], g_a_int=[], tau=[], replays=[], set_chi=0)

    def record(wrk, it, eps_new, eps_old):
        if it == 0:
            set_chi = wrk.engine.set_chi

            def counted(chi):
                hist["set_chi"] += 1
                set_chi(chi)

            wrk.engine.set_chi = counted
        hist["J_T"].append(wrk.result.J_T)
        hist["tau"].append(np.array(wrk.result.tau_vals))
        if it > 0:
            hist["g_a_int"].append(np.array(wrk.g_a_int))
        hist["pulses"] = np.array([np.array(e) for e in eps_new])
        hist["info"] = wrk.engine.info()
        hist["replays"].append(hist["info"]["graph_replays"])
        if it == iters and storage:
            hist["X"] = np.array([np.array(wrk.bw_storage[k]) for k in range(c.w.N)])
            hist["Phi"] = np.array([np.array(wrk.fw_storage[k]) for k in range(c.w.N)])
        if on_iteration is not None:
            on_iteration(wrk, it)

    problem = c.problem(iter_stop=iters, callback=record, store_fw_states=storage, **kw)
    if no_target:
        problem.trajectories[0].target_state = None
    res = K.optimize(problem, method=K.Krotov)
    hist["states"] = np.array(res.states)
    return hist


def _boundary_keywords(name, boundary):
    """The keywords of ``optimize`` for the boundary condition."""
    if boundary in ("user_chi", "no_target"):
        obs = observable(name, boundary)
        return dict(J_T=obs.J_T, chi=obs.chi)
    if boundary == "sigma":
        return dict(sigma=SIGMA[name])
    return {}


def _cell_params():
    """(cell, boundary) for every boundary that applies to the cell's problem; the built-in cells keep their ids."""
    return [pytest.param(cell, b, id=cell if b == "builtin" else f"{cell}-{b}")
            for b in BOUNDARIES for cell in CELLS if applies(CELLS[cell][0], b)]


@pytest.mark.gpu
@pytest.mark.parametrize("cell,boundary", _cell_params())
def test_cell_against_exact_dynamics(cell, boundary, monkeypatch):
    name, env, kw, kernel, lanes, exchange = CELLS[cell]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    iters = ITERS.get(name, 2)
    storage = "emulate_ranks" not in kw
    got = run_cell(case(name), iters, storage, no_target=boundary == "no_target", **kw,
                   **_boundary_keywords(name, boundary))
    info = got["info"]
    assert (info["kernel"], info["lanes_per_traj"], info["exchange"]) == (kernel, lanes, exchange), info
    if name.startswith("tiny_jitter"):  # the coefficient table is read from global memory (coef_in_smem = 0)
        w = case(name).w
        assert len(set(np.diff(w.tlist))) == w.N_T
        assert (1 + w.L) * w.d**2 * 32 * 16 + w.N_T * (info["m_fw"] + info["m_bw"]) * 32 * 8 > 160 * 1024
    if name == "graph_A":
        assert info["graph_replays"] >= 1
    # chi(T) from the host once per iteration, and never for a built-in functional
    assert got["set_chi"] == (0 if boundary == "builtin" else iters)
    if boundary == "no_target":
        assert all(t[0] == 0 for t in got["tau"])  # krotov_get_tau: exactly 0 without a target
    ch = cheby(name, boundary)
    dj = np.abs(np.asarray(got["J_T"]) - ch["J_T"])
    assert np.all(dj <= RTOL_JT * np.abs(ch["J_T"]) + ATOL_JT), (got["J_T"], ch["J_T"])
    assert np.abs(got["pulses"] - ch["pulses"]).max() <= ATOL_PULSE
    assert np.abs(np.asarray(got["g_a_int"]) - np.asarray(ch["g_a_int"])).max() <= 1e-11
    dev = deviations(got, exact(name, boundary), storage)
    assert max(dev.values()) <= BOUND[name, boundary], dev


# ---- one handle, chi(T) from three sources in turn ----------------------------------------------------------------------
# "No krotov_set_chi* since the last sweep -> chi(T) from tau" (include/krotov_cuda.h): a built-in functional, and before
# iteration 5 krotov_set_chi (the Observable chi), before iteration 7 krotov_set_chi_coeffs; every other iteration must
# form chi(T) from tau again.
SEQ_CELLS = ("tiny_jitter", "preg_L2_A", "pair_B", "graph_A", "dsweep_A", "sparse_sweep_B", "sparse_stream_B")
SEQ_ITERS = 8


def _seq_coeffs(name):
    c = case(name).w
    g = np.random.default_rng(zlib.crc32(name.encode()) + 1).standard_normal((2, c.N))
    return (g[0] + 1j * g[1]) / c.N


def _seq_sources(name):
    """{iteration: chi(T) callable} of the sequence, for the reference."""
    target = np.array(case(name).w.target, complex).reshape(case(name).w.N, -1)
    coef = _seq_coeffs(name)
    return {5: observable(name, "user_chi").chi, 7: lambda states: list(coef[:, None] * target)}


@functools.lru_cache(maxsize=None)
def sequence_reference(name, prop_method):
    return reference_run(case(name).oracle(), SEQ_ITERS, prop_method, chi=_seq_sources(name))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", SEQ_CELLS)
def test_chi_source_sequence_on_one_handle(cell, monkeypatch):
    name, env, kw, kernel, lanes, exchange = CELLS[cell]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    sources = _seq_sources(name)

    def switch(wrk, it):
        if it == 4:
            wrk.engine.set_chi(np.array(sources[5](wrk.result.states)))
        if it == 6:
            wrk.engine.set_chi_coeffs(_seq_coeffs(name))

    got = run_cell(case(name), SEQ_ITERS, True, on_iteration=switch, **kw)
    info = got["info"]
    assert (info["kernel"], info["lanes_per_traj"], info["exchange"]) == (kernel, lanes, exchange), info
    assert got["set_chi"] == 1
    if name == "graph_A":  # iteration 4 replays the graph captured in iteration 3; iteration 5 (host chi) does not
        assert got["replays"][3:6] == [0, 1, 1], got["replays"]
    ref = sequence_reference(name, "expm")
    dev = deviations(got, ref)
    assert max(dev.values()) <= BOUND[name, "sequence"], dev
    # every iteration: J_T, tau and g_a_int are per iteration
    assert np.abs(np.asarray(got["J_T"]) - ref["J_T"]).max() <= BOUND[name, "sequence"]


# ---- CPU: the references and the bounds ----------------------------------------------------------------------------------
def _bound_params():
    return [pytest.param(name, b, id=name if b == "builtin" else f"{name}-{b}")
            for b in BOUNDARIES for name in PROBLEMS if applies(name, b)]


@pytest.mark.parametrize("name,boundary", _bound_params())
def test_chebyshev_oracle_meets_a_tenth_of_the_bound(name, boundary):
    """The bound of every (problem, boundary) is sound: the Chebyshev oracle itself stays within BOUND / 10 of the exact
    run, for every quantity the GPU cells compare (every storage slot included)."""
    assert BOUND[name, boundary] <= 1e-11
    dev = deviations(cheby(name, boundary), exact(name, boundary))
    assert max(dev.values()) <= BOUND[name, boundary] / 10, dev


@pytest.mark.parametrize("name", sorted({CELLS[c][0] for c in SEQ_CELLS}))
def test_chebyshev_oracle_meets_a_tenth_of_the_sequence_bound(name):
    assert BOUND[name, "sequence"] <= 1e-11
    dev = deviations(sequence_reference(name, "cheby"), sequence_reference(name, "expm"))
    assert max(dev.values()) <= BOUND[name, "sequence"] / 10, dev


@pytest.mark.parametrize("name,boundary", [p for p in _bound_params() if p.values[1] != "builtin"])
def test_boundaries_move_the_pulses(name, boundary):
    """Every boundary condition moves the exact pulses by >= 1e4 x BOUND against the built-in one (and sigma by >= 1e-4
    against first order): a kernel that ignored a host chi(T), or read it with the wrong stride, trajectory or pair slot,
    cannot meet the bound."""
    move = np.abs(exact(name, boundary)["pulses"] - exact(name)["pulses"]).max()
    assert move >= 1e4 * BOUND[name, boundary]
    if boundary == "sigma":
        assert move >= 1e-4


@pytest.mark.parametrize("name", sorted({CELLS[c][0] for c in SEQ_CELLS}))
def test_sequence_sources_move_the_pulses(name):
    """The host sources of the sequence change the exact pulses by >= 1e4 x BOUND against the built-in run."""
    builtin = reference_run(case(name).oracle(), SEQ_ITERS, "expm")["pulses"]
    assert np.abs(sequence_reference(name, "expm")["pulses"] - builtin).max() >= 1e4 * BOUND[name, "sequence"]


def test_exact_reference_against_40_digit_arithmetic():
    """The float64 expm reference (shared per-generator propagators) against mp_reference.krotov_exact_general."""
    _against_40_digit_arithmetic("builtin")


def test_exact_reference_with_user_chi_against_40_digit_arithmetic():
    """The same with the Observable functional (chi(T) and J_T through the hooks of krotov_exact_general)."""
    _against_40_digit_arithmetic("user_chi")


def _against_40_digit_arithmetic(boundary):
    import mp_reference as M

    name = "tiny_nt2"
    p = case(name).oracle()
    hooks = {} if boundary == "builtin" else dict(zip(("J_T", "chi"), observable(name, boundary).mp_hooks()))
    ref = M.krotov_exact_general(p, iters=2, dps=40, **hooks)
    ex = exact(name, boundary)
    assert np.abs(np.array(ref["J_T"]) - ex["J_T"]).max() < 1e-15
    assert np.abs(np.array(ref["pulses"]) - ex["pulses"]).max() < 1e-15
    assert np.abs(np.array(ref["g_a_int"]) - np.array(ex["g_a_int"])).max() < 1e-15
    assert np.abs(np.array(ref["tau"]) - ex["tau"][-1]).max() < 1e-15


def _two_corner_problem():
    """Two anti-correlated controls: lambda_max(H0 + a1 H1 + a2 H2) peaks at a MIXED corner of the control ranges."""
    w = W.dummy_dense(d=4, n_traj=2, n_controls=2, n_grid=41, seed=5)
    X = np.zeros((4, 4))
    X[0, 1] = X[1, 0] = X[2, 3] = X[3, 2] = 0.3
    H1 = np.diag([3.0, 0, 0, 0]).astype(complex) + X
    H2 = np.diag([-3.0, 0, 0, 0]).astype(complex) + X / 2
    w.H0, w.Hc = [np.diag([0.0, 0.5, 1.0, 1.5]).astype(complex)], [[H1, H2]]
    p = W.to_oracle(w)
    p.pulses[1] = p.pulses[1] - p.pulses[1].max()  # control 2 <= 0
    return p, H1, H2


def test_two_corner_spectral_envelope_misses_the_mixed_corner():
    """The spectral envelope is taken at two corners (all controls at their minimum, all at their maximum), as upstream
    does.  With anti-correlated controls the extreme eigenvalue sits at a mixed corner: the window is too narrow and the
    Chebyshev run leaves the exact dynamics by more than 1e-12; a window over all four corners brings it back."""
    p, H1, H2 = _two_corner_problem()
    ex = reference_run(p, 2, "expm")
    two = reference_run(p, 2, "cheby")
    gap = max(np.abs(np.array(two["J_T"]) - ex["J_T"]).max(), np.abs(two["states"] - ex["states"]).max())
    assert gap > 1e-12
    H0 = p.H0[0]
    lo, hi = [5 * x.min() for x in p.pulses], [5 * x.max() for x in p.pulses]  # the oracle's widened ranges
    ev = [np.linalg.eigvalsh(H0 + a * H1 + b * H2) for a in (lo[0], hi[0]) for b in (lo[1], hi[1])]
    E_lo, E_hi = min(e[0] for e in ev), max(e[-1] for e in ev)
    two_lo = min(np.linalg.eigvalsh(H0 + lo[0] * H1 + lo[1] * H2)[0], np.linalg.eigvalsh(H0 + hi[0] * H1 + hi[1] * H2)[0])
    assert E_lo < two_lo  # the mixed corner extends the window
    p4, _, _ = _two_corner_problem()
    p4.specrange = (E_lo - 0.05, E_hi + 0.05)
    four = reference_run(p4, 2, "cheby")
    gap4 = max(np.abs(np.array(four["J_T"]) - ex["J_T"]).max(), np.abs(four["states"] - ex["states"]).max())
    assert gap4 < 1e-12
