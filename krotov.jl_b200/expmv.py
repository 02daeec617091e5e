"""Host-side settings of the truncated-Taylor propagator (``prop_method=Expmv``): shift, row scale, 1-norm bound and
the (m, s) choice of Al-Mohy & Higham, "Computing the action of the matrix exponential" (SIAM J. Sci. Comput. 33,
2011), the algorithm behind ``scipy.sparse.linalg.expm_multiply``.

One interval of generator g applies ``psi <- [e^{-i mu dt/s} sum_{j<m} B^j / j!]^s psi`` with
``B = -i dt/s (H(eps) - mu)``: only matrix-vector products, exact to double-precision backward error for any generator,
Hermitian or not (Liouvillians with strong dissipation, where the Chebyshev window built from the real parts of the
eigenvalues loses accuracy).  The device holds the rows ``R = -i scale (H(eps) - mu)``; ``coeffs[j] = (dt / (scale
s))^j / j!``.  Like the Chebyshev settings (``cheby.ChebyDirection``) this runs once per sweep on the host and is
re-derived on the same control-range events (``transform_control_ranges``, factors 2 and 5)."""
from __future__ import annotations

import math

import numpy as np

from .cheby import ChebyDirection

__all__ = ["THETA", "THETA_CAP", "M_MAX", "taylor_params", "taylor_coeffs", "generator_shift", "TaylorDirection"]

# theta_p (double precision): the largest ||B||_1 for which the degree-p truncation of exp(B) meets the unit roundoff
# as a backward error (Al-Mohy & Higham 2011, Table 3.1; the values scipy's expm_multiply uses)
THETA = {1: 2.29e-16, 2: 2.58e-8, 3: 1.39e-5, 4: 3.40e-4, 5: 2.40e-3, 6: 9.07e-3, 7: 2.38e-2, 8: 5.00e-2, 9: 8.96e-2,
         10: 1.44e-1, 11: 2.14e-1, 12: 3.00e-1, 13: 4.00e-1, 14: 5.14e-1, 15: 6.41e-1, 16: 7.81e-1, 17: 9.31e-1,
         18: 1.09, 19: 1.26, 20: 1.44, 21: 1.62, 22: 1.82, 23: 2.01, 24: 2.22, 25: 2.43, 26: 2.64, 27: 2.86, 28: 3.08,
         29: 3.31, 30: 3.54, 35: 4.7, 40: 6.0, 45: 7.2, 50: 8.5, 55: 9.9}
M_MAX = 55  # largest degree of the table
# Largest ||B||_1 of one repeat.  The partial sums of exp(B) pass through terms of size up to ~e^{||B||} before they
# cancel, so the rounding error of the sum grows with ||B|| even where the truncation error is below the unit roundoff;
# DESIGN.md 4.7 records the measurement this value comes from.
THETA_CAP = 2.0


def taylor_params(norm, theta_cap=THETA_CAP, m_max=M_MAX):
    """``(m, s)`` for ``||A||_1 <= norm`` (A = -i dt (H - mu)): s repeats of the first m terms (degree m - 1) of the
    series, the least number of products (m - 1) s with ``norm / s <= theta_{m-1}`` and ``norm / s <= theta_cap``."""
    norm = float(norm)
    if not np.isfinite(norm):
        raise ValueError(f"norm bound {norm!r} is not finite")
    if norm == 0.0:
        return 1, 1
    best = None
    for p, th in THETA.items():
        if p > m_max:
            break
        s = max(1, math.ceil(norm / min(th, theta_cap)))
        if best is None or p * s < best[0] * best[1]:
            best = (p, s)
    return best[0] + 1, best[1]


def taylor_coeffs(x, m):
    """``[x^j / j! for j < m]`` by the recurrence c_j = c_{j-1} x / j."""
    out = np.empty(m, np.float64)
    c = 1.0
    for j in range(m):
        if j > 0:
            c = c * x / j
        out[j] = c
    return out


def generator_shift(H0):
    """The shift mu = Re tr(H0) / d of Al-Mohy & Higham (the real part: mu enters as the phase e^{-i mu dt})."""
    H0 = np.asarray(H0.toarray() if hasattr(H0, "toarray") else H0, np.complex128)
    return float(np.trace(H0).real / H0.shape[0])


def _norm1(M):
    """Induced 1-norm (largest column sum of |M|)."""
    M = np.asarray(M.toarray() if hasattr(M, "toarray") else M, np.complex128)
    return float(np.abs(M).sum(axis=0).max())


class TaylorDirection:
    """Taylor settings of all propagators of one direction: the counterpart of ``ChebyDirection`` (same ``reinit`` /
    ``push`` hooks, same dt classes).  ``H0[g]``, ``Hc[g][l]``: the terms the direction propagates with (the ADJOINT
    generator backward).  ``amplitude_max(l, lo, hi)``: the largest |coefficient| of H_l over the control range [lo, hi]
    (None: linear controls, max(|lo|, |hi|))."""

    def __init__(self, H0, Hc, tlist, backward, pulses, *, theta_cap=THETA_CAP, amplitude_max=None):
        self.tlist = np.asarray(tlist, np.float64)
        self.backward = bool(backward)
        self.theta_cap = float(theta_cap)
        self._amplitude_max = amplitude_max
        self.control_ranges = [(float(np.min(p)), float(np.max(p))) for p in pulses]
        self.n_updates = 0
        n_gen, L = len(H0), len(pulses)
        self.mu = np.array([generator_shift(h) for h in H0], np.float64)
        d = H0[0].shape[0]
        self._h0_norm = np.array([_norm1(np.asarray(H0[g].toarray() if hasattr(H0[g], "toarray") else H0[g]) -
                                         self.mu[g] * np.eye(d)) for g in range(n_gen)])
        self._hc_norm = np.array([[0.0 if Hc[g][l] is None else _norm1(Hc[g][l]) for l in range(L)] for g in range(n_gen)])
        # dt classes: the distinct signed steps of the grid (the coefficients depend on the exact step)
        sign = -1.0 if self.backward else 1.0
        dts = sign * np.diff(self.tlist)
        self.dt_of_class, inv = np.unique(dts, return_inverse=True)
        self.dt_class_of_step = inv.astype(np.int32)
        self._derive()

    def norm_rate(self):
        """Per generator the bound nu_g >= ||H_g(eps) - mu_g||_1 over the current control ranges."""
        amax = np.empty(len(self.control_ranges))
        for l, (lo, hi) in enumerate(self.control_ranges):
            amax[l] = max(abs(lo), abs(hi)) if self._amplitude_max is None else self._amplitude_max(l, lo, hi)
        return self._h0_norm + self._hc_norm @ amax

    def _derive(self):
        nu = self.norm_rate()
        # rows R = -i scale (H - mu) with ||R||_1 <= 1: the powers R^j v stay of the size of v
        self.scale = np.where(nu > 0, 1.0 / np.where(nu > 0, nu, 1.0), 1.0)
        n_gen, n_cls = len(nu), len(self.dt_of_class)
        self.m = np.ones((n_gen, n_cls), np.int32)
        self.s = np.ones((n_gen, n_cls), np.int32)
        for g in range(n_gen):
            for c, dt in enumerate(self.dt_of_class):
                self.m[g, c], self.s[g, c] = taylor_params(abs(dt) * nu[g], self.theta_cap)
        self.coeff_table = np.zeros((n_gen, n_cls, int(self.m.max())), np.float64)
        for g in range(n_gen):
            for c, dt in enumerate(self.dt_of_class):
                m, s = int(self.m[g, c]), int(self.s[g, c])
                self.coeff_table[g, c, :m] = taylor_coeffs(dt / (self.scale[g] * s), m)

    @property
    def coeffs(self):
        """``coeffs[g][class]``: the Taylor coefficients of one repeat (as ``ChebyDirection.coeffs``)."""
        return [[self.coeff_table[g, c, : self.m[g, c]] for c in range(self.m.shape[1])] for g in range(self.m.shape[0])]

    # the range check of reinit_prop!: the same rule as the Chebyshev settings
    reinit = ChebyDirection.reinit

    def push(self, engine, direction):
        engine.set_taylor(direction, self.dt_class_of_step, self.dt_of_class, self.mu, self.scale, self.s, self.m,
                          self.coeff_table)

