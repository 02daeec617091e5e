"""Host-side Chebyshev propagator settings: spectral envelope, control-range bookkeeping, coefficients.

This is the part of QuantumPropagators' ``init_prop`` / ``reinit_prop!`` (called by the reference at
``src/optimize.jl:251,306,324`` with Krotov's ``transform_control_ranges`` hook, ``:238-244``) that
stays on the host: it runs once per sweep, never per time step, and its product -- per generator
``E_min``, ``Delta`` and the coefficient vector -- is handed to the device through
``krotov_set_cheby``.  Semantics restated from the published algorithm (SURVEY.md Appendix A.1).
"""
from __future__ import annotations

import numpy as np
from scipy.special import jv

__all__ = ["cheby_coeffs", "specrange", "transform_control_ranges", "ChebyDirection"]


def cheby_coeffs(Delta, dt, limit=1e-12):
    """Expansion coefficients of exp(-i H dt) in Chebyshev polynomials for spectral radius ``Delta``:
    ``a_0 = J_0(alpha)``, ``a_n = 2 J_n(alpha)``, ``alpha = |Delta dt| / 2``, truncated at the first
    ``|a_n| <= limit`` beyond ``n > alpha``."""
    alpha = abs(0.5 * Delta * dt)
    out = [float(jv(0, alpha))]
    n = 1
    while abs(out[-1]) > limit or n <= alpha:
        out.append(2.0 * float(jv(n, alpha)))
        n += 1
    return np.asarray(out, np.float64)


def cheby_coeffs_table(Deltas, dt, limit=1e-12, m_hint=0):
    """`cheby_coeffs` for many spectral radii at once (one vectorised Bessel call) as a zero-padded table
    ``(a[n_gen, m_max], m[n_gen])``; every number is what the scalar function returns (same ufunc, evaluated
    elementwise).  ``m_hint``: the largest coefficient count of the previous table of this step size -- a re-derived
    envelope moves it by a term or two, so the Bessel call covers ``m_hint + 4`` orders first."""
    Deltas = np.asarray(Deltas, np.float64)
    alpha = np.abs(0.5 * Deltas * dt)
    nmax = int(np.max(alpha)) + 24  # enough for limit = 1e-12 at small alpha; doubled below when it is not
    if m_hint > 0:
        nmax = min(nmax, int(m_hint) + 4)
    while True:
        n = np.arange(nmax)
        a = jv(n[None, :], alpha[:, None])
        a[:, 1:] *= 2.0
        # length m = first n >= 1 with |a_{n-1}| <= limit and n > alpha
        stop = (np.abs(a[:, :-1]) <= limit) & (n[None, 1:] > alpha[:, None])
        if stop.any(axis=1).all():
            m = stop.argmax(axis=1) + 1
            a = a[:, : int(m.max())].copy()
            a[np.arange(a.shape[1])[None, :] >= m[:, None]] = 0.0
            return a, m.astype(np.int32)
        nmax *= 2


def cheby_coeffs_many(Deltas, dt, limit=1e-12):
    """List form of `cheby_coeffs_table`: one coefficient vector per spectral radius."""
    a, m = cheby_coeffs_table(Deltas, dt, limit)
    return [a[g, : m[g]].copy() for g in range(len(m))]


def specrange(G, method="auto"):
    """``(E_min, E_max)`` of an operator.  ``diag``: exact eigenvalues (dense).  ``auto`` uses
    ``diag`` up to dimension 512 and a Lanczos/Arnoldi estimate (scipy ``eigs``, widened by 5 %)
    beyond; pass ``prop_E_min`` / ``prop_E_max`` to bypass it."""
    sparse = hasattr(G, "tocsr")
    d = G.shape[0]
    if method == "auto":
        method = "diag" if d <= 512 else "arnoldi"
    if sparse and method == "diag":
        G = G.toarray()
    elif not sparse:
        G = np.asarray(G)
    if method == "diag":
        if np.array_equal(G, G.conj().T):  # Hermitian: symmetric solver (what Julia's `eigvals` picks)
            ev = np.linalg.eigvalsh(G)
            return float(ev[0]), float(ev[-1])
        ev = np.linalg.eigvals(G)
        return float(ev.real.min()), float(ev.real.max())
    if method == "arnoldi":
        from scipy.sparse.linalg import eigs, eigsh

        v0 = (np.arange(1, d + 1) % 7 + 1.0).astype(np.complex128)  # fixed, non-symmetric start vector
        v0 /= np.linalg.norm(v0)
        herm = (abs(G - G.conj().T).max() == 0) if sparse else np.array_equal(G, G.conj().T)
        if herm:
            hi = eigsh(G, k=1, which="LA", v0=v0, return_eigenvectors=False, tol=1e-5)[0].real
            lo = eigsh(G, k=1, which="SA", v0=v0, return_eigenvectors=False, tol=1e-5)[0].real
        else:
            hi = eigs(G, k=1, which="LR", v0=v0, return_eigenvectors=False, tol=1e-5)[0].real
            lo = eigs(G, k=1, which="SR", v0=v0, return_eigenvectors=False, tol=1e-5)[0].real
        pad = 0.05 * (hi - lo)
        return float(lo - pad), float(hi + pad)
    raise ValueError(f"unknown specrange method {method!r}")


_NATIVE_MIN_BATCH = 32  # matrices per envelope from which the library's threaded solver replaces NumPy's


def _batched(solver, stack, workers=8):
    """Apply a LAPACK-backed solver to a stack of matrices; per-matrix results are independent of the
    chunking.  Threads only pay for matrices large enough to keep LAPACK busy between GIL hand-overs
    (measured: 512 Hermitian 25x25 problems take 31 ms in one call and 38-44 ms split over 8 threads)."""
    n = stack.shape[0]
    if n < 4 * workers or stack.shape[-1] < 96:
        return solver(stack)
    from concurrent.futures import ThreadPoolExecutor

    bounds = [(i * n) // workers for i in range(workers + 1)]
    with ThreadPoolExecutor(workers) as ex:
        parts = list(ex.map(lambda ab: solver(stack[ab[0]:ab[1]]), zip(bounds[:-1], bounds[1:])))
    return np.concatenate(parts, axis=0)


def transform_control_ranges(c, eps_min, eps_max, check):
    """Krotov's range hook (``src/optimize.jl:238-244``): a propagator's spectral envelope is
    re-derived when twice the current amplitude range leaves the stored range, and then stored for
    five times the current range."""
    f = 2 if check else 5
    return (min(eps_min, f * eps_min), max(eps_max, f * eps_max))


class ChebyDirection:
    """Settings of all propagators of one direction (they see the same pulses, so their control
    ranges move in lock-step; the spectral envelope is per generator).

    ``H0[g]``, ``Hc[g][l]`` are the terms of the generator the direction propagates with: the plain
    generator forward, the ADJOINT generator backward (``src/workspace.jl:69,150-160``)."""

    def __init__(self, H0, Hc, tlist, backward, pulses, *, limit=1e-12, specrange_buffer=0.01,
                 specrange_method="auto", E_min=None, E_max=None, envelope_cache=None, amplitude=None,
                 device_envelope=None):
        self.H0, self.Hc = H0, Hc
        # `device_envelope(corners) -> (e_min, e_max)`: the engine's solver for the generators it holds (ensembles)
        self._device_envelope = device_envelope
        # non-linear amplitudes: `amplitude(l, lo, hi)` = coefficients of H_l at the two sides of the control range
        self._amplitude = amplitude
        # spectral envelopes by control ranges.  The two directions of a Hermitian problem propagate with the
        # same matrices and meet the same ranges one iteration apart (the forward check sees the pulse
        # buffer the backward check saw in the previous iteration, src/optimize.jl:305-306 vs :321-325),
        # so the workspace hands both the same dictionary and every envelope is derived once.
        self._envelopes = envelope_cache if envelope_cache is not None else {}
        # coefficient tables by (spectral radii, |dt|, limit): the two directions of a Hermitian problem meet the same
        # radii one iteration apart and a_n depends on |Delta dt| only, so the second one finds its table made
        self._tables = self._envelopes.setdefault("__tables__", {})
        self.tlist = np.asarray(tlist, np.float64)
        self.backward = bool(backward)
        self.limit = float(limit)
        self.buffer = float(specrange_buffer)
        self.method = specrange_method
        self.manual = None if (E_min is None or E_max is None) else (float(E_min), float(E_max))
        self.control_ranges = [(float(np.min(p)), float(np.max(p))) for p in pulses]
        self.n_updates = 0
        self._any_sparse = any(hasattr(m, "tocsr") for m in list(H0) + [x for row in Hc for x in row if x is not None])
        if not self._any_sparse and H0[0].shape[0] <= 512:
            self._H0s = np.stack([np.asarray(h, np.complex128) for h in H0])
            d = self._H0s.shape[1]
            self._Hcs = [np.stack([np.zeros((d, d), np.complex128) if row[l] is None else
                                   np.asarray(row[l], np.complex128) for row in Hc]) for l in range(len(pulses))]
            # Hermitian terms and real amplitudes: every evaluated generator is Hermitian (checked once, not per event)
            self._herm = all(np.array_equal(a, a.conj().transpose(0, 2, 1)) for a in [self._H0s] + self._Hcs)
            self._Hcs_stack = np.stack(self._Hcs) if self._Hcs else np.zeros((0,) + self._H0s.shape, np.complex128)
        self._classify_steps()
        self._derive()

    # -- spectral envelope (cheby_get_spectral_envelope + specrange_buffer) ----------------
    def _evaluate(self, g, vals):
        G = self.H0[g].copy() if hasattr(self.H0[g], "tocsr") else np.array(self.H0[g], np.complex128)
        for l, Hl in enumerate(self.Hc[g]):
            if Hl is not None:
                G = G + vals[l] * Hl
        return G

    def _derive(self):
        n_gen = len(self.H0)
        lo = [r[0] for r in self.control_ranges]
        hi = [r[1] for r in self.control_ranges]
        if self._amplitude is not None:  # the generator at the range corners carries a_l(corner), not the corner itself
            corners = [self._amplitude(l, a, b) for l, (a, b) in enumerate(zip(lo, hi))]
            lo = [c[0] for c in corners]
            hi = [c[1] for c in corners]
        key = tuple(self.control_ranges)
        if self.manual is not None:
            e_min = np.full(n_gen, self.manual[0])
            e_max = np.full(n_gen, self.manual[1])
        elif key in self._envelopes:
            e_min, e_max = self._envelopes[key]
        elif self.method in ("auto", "diag") and self.H0[0].shape[0] <= 512 and not self._any_sparse:
            # all generators in two batched LAPACK calls (numpy loops over the stack in C and calls the same
            # zgeev per matrix, so every number is what `specrange` returns for the single matrix)
            # (the Hermitian solver when every evaluated generator is Hermitian, like `specrange`)
            if self._herm and 2 * n_gen >= _NATIVE_MIN_BATCH and self._H0s.shape[-1] <= 64:
                # ensembles: the library's threaded host solver (forms the corner generators and finds their extreme
                # eigenvalues only); agrees with LAPACK to a few ulp of the matrix norm, far below what the
                # Chebyshev expansion resolves
                if self._device_envelope is not None:
                    # ... or, on the persistent-kernel path, the device (one warp per corner generator, Jacobi rotations)
                    e_min, e_max = self._device_envelope(np.array([hi, lo], np.float64))
                else:
                    from ._lib import envelope_extremes

                    e_min, e_max = envelope_extremes(self._H0s, self._Hcs_stack, np.array([hi, lo], np.float64))
            else:
                G_hi, G_lo = self._H0s.copy(), self._H0s.copy()  # same elementwise sums as `_evaluate`, for all g at once
                for l in range(len(hi)):
                    G_hi = G_hi + hi[l] * self._Hcs[l]
                    G_lo = G_lo + lo[l] * self._Hcs[l]
                herm = self._herm or (np.array_equal(G_hi, G_hi.conj().transpose(0, 2, 1)) and np.array_equal(
                    G_lo, G_lo.conj().transpose(0, 2, 1)))
                solver = np.linalg.eigvalsh if herm else (lambda a: np.linalg.eigvals(a).real)
                ev = _batched(solver, np.concatenate([G_hi, G_lo]))
                ev_hi, ev_lo = ev[:n_gen], ev[n_gen:]
                e_min = np.minimum(ev_hi.min(axis=1), ev_lo.min(axis=1))
                e_max = np.maximum(ev_hi.max(axis=1), ev_lo.max(axis=1))
        else:
            e_min, e_max = np.empty(n_gen), np.empty(n_gen)
            for g in range(n_gen):
                a0, b0 = specrange(self._evaluate(g, hi), self.method)
                a1, b1 = specrange(self._evaluate(g, lo), self.method)
                e_min[g], e_max[g] = min(a0, a1), max(b0, b1)
        if self.manual is None:
            env_keys = [k for k in self._envelopes if k != "__tables__"]
            if len(env_keys) >= 8:
                self._envelopes.pop(env_keys[0])
            self._envelopes[key] = (e_min, e_max)
        Delta = e_max - e_min
        delta = self.buffer * Delta
        self.E_min = e_min - delta / 2
        self.Delta = Delta + delta
        self._tabulate()

    def _classify_steps(self):
        """dt classes, walking the grid in propagation order with the propagator's rule: coefficients are
        re-derived only when the step differs from the one they were derived for.  A class is a (exact step,
        step the coefficients belong to) pair: the final phase e^{-i beta dt} uses the exact step.  Depends on
        the time grid only, so it is done once."""
        t = self.tlist
        N_T = len(t) - 1
        sign = -1.0 if self.backward else 1.0
        cur = sign * (t[1] - t[0])
        order = range(N_T - 1, -1, -1) if self.backward else range(N_T)
        classes, key_to_class = [], {}
        self.dt_class_of_step = np.zeros(N_T, np.int32)
        for n in order:
            dt = sign * (t[n + 1] - t[n])
            if abs(dt - cur) > 1e-12 * max(1.0, abs(cur)):
                cur = dt
            key = (dt, cur)
            if key not in key_to_class:
                key_to_class[key] = len(classes)
                classes.append(key)
            self.dt_class_of_step[n] = key_to_class[key]
        self.dt_of_class = np.array([k[0] for k in classes], np.float64)
        self._classes = classes

    def _tabulate(self):
        """Per-class coefficients for the current spectral radii."""
        classes = self._classes
        reps = []
        for (_, rep) in classes:
            if rep not in reps:
                reps.append(rep)
        hints = getattr(self, "_m_hint", {})
        per_rep = {}
        for rep in reps:
            key = (np.ascontiguousarray(self.Delta, np.float64).tobytes(), abs(float(rep)), self.limit)
            hit = self._tables.get(key)
            if hit is None:
                hit = cheby_coeffs_table(self.Delta, rep, self.limit, hints.get(rep, 0))
                while len(self._tables) >= 8:
                    self._tables.pop(next(iter(self._tables)))
                self._tables[key] = hit
            per_rep[rep] = hit
        self._m_hint = {rep: int(per_rep[rep][1].max()) for rep in reps}
        n_gen = len(self.H0)
        m_max = max(int(a.shape[1]) for a, _ in per_rep.values())
        self.coeff_table = np.zeros((n_gen, len(classes), m_max), np.float64)  # [g][class][j], zero-padded
        self.coeff_count = np.zeros((n_gen, len(classes)), np.int32)
        for c, (_, rep) in enumerate(classes):
            a, m = per_rep[rep]
            self.coeff_table[:, c, : a.shape[1]] = a
            self.coeff_count[:, c] = m

    @property
    def coeffs(self):
        """``coeffs[g][class]``: the coefficient vector of generator g for a dt class."""
        return [[self.coeff_table[g, c, : self.coeff_count[g, c]] for c in range(self.coeff_table.shape[1])]
                for g in range(self.coeff_table.shape[0])]

    # -- reinit_prop! ------------------------------------------------------------------------
    def reinit(self, pulses, transform=transform_control_ranges):
        """Range check of ``reinit_prop!``; returns True when the envelope (hence the device tables)
        changed."""
        need = False
        for l, p in enumerate(pulses):
            lo, hi = float(np.min(p)), float(np.max(p))
            c_lo, c_hi = transform(l, lo, hi, True)
            o_lo, o_hi = self.control_ranges[l]
            if c_lo < o_lo or c_hi > o_hi:
                need = True
        if need:
            self.control_ranges = [transform(l, float(np.min(p)), float(np.max(p)), False)
                                   for l, p in enumerate(pulses)]
            self._derive()
            self.n_updates += 1
        return need

    def push(self, engine, direction):
        engine.set_cheby(direction, self.dt_class_of_step, self.dt_of_class, self.E_min, self.Delta,
                         self.coeff_count, self.coeff_table)
