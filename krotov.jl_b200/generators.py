"""Generators: ``hamiltonian(H0, (H1, eps1), ...)`` as in QuantumControl (used by the reference's tests,
``test/test_tls_optimization.jl:16-28``)."""
from __future__ import annotations

import numpy as np

__all__ = ["Generator", "hamiltonian", "ShapedAmplitude", "PolynomialAmplitude", "ParametrizedAmplitude",
           "SquareParametrization", "TanhParametrization", "TanhSqParametrization", "LogisticParametrization",
           "LogisticSqParametrization"]


class ControlAmplitude:
    """A control term's amplitude ``a(eps, n) = shape[n] * P(x)`` with the polynomial ``P`` (``coeffs`` ascending,
    degree 1..4) evaluated at ``x = tanh(saturation * eps)`` when ``saturation > 0`` and at ``x = eps`` otherwise.
    This is what the device evaluates (``krotov_set_amplitudes``, ``krotov_set_amplitude_saturation``); the subclasses
    are the user-facing forms."""

    saturation = 0.0

    def __init__(self, control, coeffs, shape=None):
        coeffs = [float(c) for c in coeffs]
        if not 2 <= len(coeffs) <= 5:
            raise ValueError(f"{type(self).__name__}: 2 to 5 coefficients (degree 1 to 4)")
        self.control, self.coeffs, self.shape = control, coeffs, shape

    def key(self):
        """What makes two amplitudes of one control the same function of the control (shape aside)."""
        return (tuple(self.coeffs), self.saturation)

    def _poly(self, x):
        v = 0.0
        for c in reversed(self.coeffs):
            v = v * x + c
        return v

    def __call__(self, eps, t=None):
        v = self._poly(np.tanh(self.saturation * eps) if self.saturation > 0 else eps)
        if self.shape is not None and t is not None and callable(self.shape):
            v = self.shape(t) * v
        return v


class PolynomialAmplitude(ControlAmplitude):
    """A control amplitude that is a NON-LINEAR function of its control: the term enters the generator as
    ``a(eps(t), t) * op`` with ``a(eps, t) = shape(t) * sum_p coeffs[p] * eps**p`` (``coeffs`` ascending, degree
    1..4; ``shape`` a callable or a vector on the intervals of the time grid, default 1).

    The reference handles such terms through ``get_control_derivs`` / ``evaluate`` (``src/optimize.jl:268-272``):
    the derivative ``mu = a'(eps, t) op`` is evaluated at the GUESS pulse of every interval (``:337``).  Here the
    amplitude is handed to the device as its polynomial (``krotov_set_amplitudes``)."""

    def __call__(self, eps, t=None):
        v = self._poly(eps)
        if self.shape is not None and t is not None and callable(self.shape):
            v = self.shape(t) * v
        return v


class ShapedAmplitude(PolynomialAmplitude):
    """``a(t) = shape(t) * eps(t)``: QuantumPropagators' ``ShapedAmplitude`` -- linear in the control, but the
    derivative ``mu = shape(t) op`` depends on time."""

    def __init__(self, control, shape):
        super().__init__(control, [0.0, 1.0], shape)


# ---- pulse parametrizations: bounded amplitudes a(u) of an unbounded control u --------------------------------------
# QuantumControl.jl's `ParametrizedAmplitude` with `SquareParametrization`, `TanhParametrization`, `TanhSqParametrization`,
# `LogisticParametrization`, `LogisticSqParametrization` (the `krotov` Python package has the same set; the formulas are
# recalled from both, see DESIGN 4.5).  Every one of them is a polynomial of degree <= 2 in x = tanh(s u):
# `device_form()` returns (P ascending, s), s = 0 meaning x = u.  The logistic forms use 1/(1+e^-y) = (1 + tanh(y/2))/2.
_EDGE = 1e-15  # epsilon_of_a clamps into the open range by this fraction, so that the inverse stays finite


def _clamp_unit(y):
    return np.clip(y, -1.0 + _EDGE, 1.0 - _EDGE)


class _Parametrization:
    def key(self):
        return (type(self).__name__,) + tuple(float(v) for v in self._params)

    def __repr__(self):
        return f"{type(self).__name__}{tuple(float(v) for v in self._params)}"


class SquareParametrization(_Parametrization):
    """``a(u) = u**2``: a non-negative amplitude (a detuning that may only be positive)."""

    _params = ()

    def a_of_epsilon(self, u):
        return np.square(u)

    def epsilon_of_a(self, a):
        return np.sqrt(np.maximum(a, 0.0))

    def da_deps_derivative(self, u):
        return 2.0 * np.asarray(u, float)

    def device_form(self):
        return [0.0, 0.0, 1.0], 0.0


class TanhParametrization(_Parametrization):
    """``a(u) = (a_max + a_min)/2 + (a_max - a_min)/2 * tanh(u)``: a_min < a(u) < a_max."""

    def __init__(self, a_min, a_max):
        a_min, a_max = float(a_min), float(a_max)
        if not (np.isfinite(a_min) and np.isfinite(a_max)) or a_min >= a_max:
            raise ValueError(f"TanhParametrization: need finite a_min < a_max, got a_min={a_min}, a_max={a_max}")
        self.a_min, self.a_max = a_min, a_max
        self._params = (a_min, a_max)

    def a_of_epsilon(self, u):
        return (self.a_max + self.a_min) / 2 + (self.a_max - self.a_min) / 2 * np.tanh(u)

    def epsilon_of_a(self, a):
        y = (2 * np.asarray(a, float) - self.a_max - self.a_min) / (self.a_max - self.a_min)
        return np.arctanh(_clamp_unit(y))

    def da_deps_derivative(self, u):
        return (self.a_max - self.a_min) / 2 / np.cosh(u) ** 2

    def device_form(self):
        return [(self.a_max + self.a_min) / 2, (self.a_max - self.a_min) / 2], 1.0


class TanhSqParametrization(_Parametrization):
    """``a(u) = a_max * tanh(u)**2``: 0 <= a(u) < a_max."""

    def __init__(self, a_max):
        a_max = float(a_max)
        if not np.isfinite(a_max) or a_max <= 0:
            raise ValueError(f"TanhSqParametrization: need a finite a_max > 0, got {a_max}")
        self.a_max = a_max
        self._params = (a_max,)

    def a_of_epsilon(self, u):
        return self.a_max * np.tanh(u) ** 2

    def epsilon_of_a(self, a):
        return np.arctanh(np.sqrt(np.clip(np.asarray(a, float) / self.a_max, 0.0, 1.0 - _EDGE)))

    def da_deps_derivative(self, u):
        return 2 * self.a_max * np.tanh(u) / np.cosh(u) ** 2

    def device_form(self):
        return [0.0, 0.0, self.a_max], 1.0


class LogisticParametrization(_Parametrization):
    """``a(u) = a_min + (a_max - a_min) / (1 + exp(-k u))``: a_min < a(u) < a_max."""

    def __init__(self, a_min, a_max, k=1.0):
        a_min, a_max, k = float(a_min), float(a_max), float(k)
        if not (np.isfinite(a_min) and np.isfinite(a_max)) or a_min >= a_max:
            raise ValueError(f"LogisticParametrization: need finite a_min < a_max, got a_min={a_min}, a_max={a_max}")
        if not np.isfinite(k) or k <= 0:
            raise ValueError(f"LogisticParametrization: need a finite k > 0, got {k}")
        self.a_min, self.a_max, self.k = a_min, a_max, k
        self._params = (a_min, a_max, k)

    def a_of_epsilon(self, u):
        return self.a_min + (self.a_max - self.a_min) / (1 + np.exp(-self.k * np.asarray(u, float)))

    def epsilon_of_a(self, a):
        y = (np.asarray(a, float) - self.a_min) / (self.a_max - self.a_min)  # in (0, 1)
        y = np.clip(y, _EDGE, 1.0 - _EDGE)
        return -np.log(1.0 / y - 1.0) / self.k

    def da_deps_derivative(self, u):
        e = np.exp(-self.k * np.asarray(u, float))
        return self.k * (self.a_max - self.a_min) * e / (1 + e) ** 2

    def device_form(self):
        return [(self.a_max + self.a_min) / 2, (self.a_max - self.a_min) / 2], self.k / 2


class LogisticSqParametrization(_Parametrization):
    """``a(u) = a_max * (2 / (1 + exp(-k u)) - 1)**2``: 0 <= a(u) < a_max."""

    def __init__(self, a_max, k=1.0):
        a_max, k = float(a_max), float(k)
        if not np.isfinite(a_max) or a_max <= 0:
            raise ValueError(f"LogisticSqParametrization: need a finite a_max > 0, got {a_max}")
        if not np.isfinite(k) or k <= 0:
            raise ValueError(f"LogisticSqParametrization: need a finite k > 0, got {k}")
        self.a_max, self.k = a_max, k
        self._params = (a_max, k)

    def a_of_epsilon(self, u):
        return self.a_max * (2 / (1 + np.exp(-self.k * np.asarray(u, float))) - 1) ** 2

    def epsilon_of_a(self, a):
        r = np.sqrt(np.clip(np.asarray(a, float) / self.a_max, 0.0, 1.0 - _EDGE))  # r = 2/(1+e^-ku) - 1 in [0, 1)
        return -np.log(2.0 / (r + 1.0) - 1.0) / self.k

    def da_deps_derivative(self, u):
        e = np.exp(-self.k * np.asarray(u, float))
        return self.a_max * 2 * (2 / (1 + e) - 1) * 2 * self.k * e / (1 + e) ** 2

    def device_form(self):
        return [0.0, 0.0, self.a_max], self.k / 2


class ParametrizedAmplitude(ControlAmplitude):
    """``a(u, t) = shape(t) * parametrization.a_of_epsilon(u)``: QuantumControl's ``ParametrizedAmplitude``.  The control
    ``u`` is what Krotov optimises (``result.optimized_controls`` hold u); ``parametrization.epsilon_of_a`` turns a
    physical guess pulse into u.  On the device the amplitude is the polynomial of ``device_form()`` evaluated at
    ``tanh(s u)``; ``mu = a'(u_guess) H`` as for every non-linear amplitude."""

    def __init__(self, control, parametrization, shape=None):
        if not isinstance(parametrization, _Parametrization):
            raise TypeError("ParametrizedAmplitude: parametrization must be one of SquareParametrization, "
                            "TanhParametrization, TanhSqParametrization, LogisticParametrization, "
                            "LogisticSqParametrization")
        coeffs, s = parametrization.device_form()
        super().__init__(control, coeffs, shape)
        self.parametrization, self.saturation = parametrization, float(s)

    def key(self):
        return super().key() + self.parametrization.key()

    def __call__(self, eps, t=None):
        v = self.parametrization.a_of_epsilon(eps)
        if self.shape is not None and t is not None and callable(self.shape):
            v = self.shape(t) * v
        return v


def _is_sparse(op):
    return hasattr(op, "tocsr") and hasattr(op, "nnz")


def _as_matrix(op):
    if _is_sparse(op):  # scipy.sparse operators stay sparse: large spin chains are never densified
        m = op.tocsr().astype(np.complex128)
        if m.shape[0] != m.shape[1]:
            raise ValueError("operators must be square matrices")
        return m
    m = np.asarray(op, dtype=np.complex128)
    if m.ndim != 2 or m.shape[0] != m.shape[1]:
        raise ValueError("operators must be square matrices")
    return m


class Generator:
    """``G(t) = sum(drift ops) + sum_i amplitudes[i](t) * control_ops[i]`` with linear controls."""

    def __init__(self, drift_ops, control_ops, amplitudes):
        self.drift_ops = [_as_matrix(o) for o in drift_ops]
        self.control_ops = [_as_matrix(o) for o in control_ops]
        self.amplitudes = list(amplitudes)
        if len(self.control_ops) != len(self.amplitudes):
            raise ValueError("one amplitude per control operator")

    @property
    def ops(self):
        return self.drift_ops + self.control_ops

    @property
    def dim(self):
        return self.ops[0].shape[0]

    def drift(self):
        out = self.drift_ops[0]
        for o in self.drift_ops[1:]:
            out = out + o
        return out.copy()

    def adjoint(self):
        adj = lambda o: o.conj().T.tocsr() if _is_sparse(o) else o.conj().T  # noqa: E731
        return Generator([adj(o) for o in self.drift_ops], [adj(o) for o in self.control_ops], self.amplitudes)

    def __repr__(self):
        return f"Generator(dim={self.dim}, drift terms={len(self.drift_ops)}, controls={len(self.amplitudes)})"


def hamiltonian(*terms):
    """``hamiltonian(H0, (H1, eps1), (H2, eps2))``: bare operators are drift terms, ``(op, control)``
    pairs are control terms.  Without any control term the plain (summed) matrix is returned, as in
    ``test/test_empty_optimization.jl:16-29``."""
    drift, cops, amps = [], [], []
    for term in terms:
        if isinstance(term, (tuple, list)) and len(term) == 2 and not np.isscalar(term[0]) and (
                callable(term[1]) or isinstance(term[1], ControlAmplitude) or np.ndim(term[1]) == 1) and (
                _is_sparse(term[0]) or np.ndim(term[0]) == 2):
            cops.append(term[0])
            amps.append(term[1])
        else:
            drift.append(term)
    if not cops:
        out = _as_matrix(drift[0])
        for o in drift[1:]:
            out = out + _as_matrix(o)
        return out
    if not drift:
        first = _as_matrix(cops[0])
        drift = [first * 0.0 if _is_sparse(first) else np.zeros(first.shape, np.complex128)]
    return Generator(drift, cops, amps)
