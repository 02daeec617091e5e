"""Control discretisation and bookkeeping (the pieces of ``QuantumPropagators.Controls`` that
``KrotovWrk`` / ``KrotovResult`` call: ``src/workspace.jl:70,74,102,119,123``; ``src/result.jl:55,61``;
``src/optimize.jl:404``)."""
from __future__ import annotations

import numpy as np

__all__ = ["discretize", "discretize_on_midpoints", "get_controls", "get_control_derivs", "control_of", "get_amplitudes",
           "get_control_terms"]


def control_of(amplitude):
    """The control object behind an amplitude (the amplitude itself for a plain control function / vector)."""
    from .generators import ControlAmplitude

    return amplitude.control if isinstance(amplitude, ControlAmplitude) else amplitude


def _as_grid(tlist):
    return np.asarray(tlist, dtype=np.float64)


def discretize(control, tlist):
    """Values of ``control`` ON the points of ``tlist`` (length ``len(tlist)``).

    A callable is sampled; an array on the grid is copied; an array on the intervals
    (``len(tlist)-1`` values) is converted: end points kept, interior points averaged."""
    t = _as_grid(tlist)
    if callable(control):
        return np.fromiter((float(control(x)) for x in t), dtype=np.float64, count=len(t))
    v = np.asarray(control, dtype=np.float64)
    if v.ndim != 1:
        raise ValueError("control must be a callable or a vector")
    if v.size == t.size:
        return v.copy()
    if v.size == t.size - 1:
        out = np.empty(t.size)
        out[0], out[-1] = v[0], v[-1]
        out[1:-1] = 0.5 * (v[:-1] + v[1:])
        return out
    raise ValueError("control array must have len(tlist) or len(tlist)-1 values")


def discretize_on_midpoints(control, tlist):
    """Values of ``control`` on the intervals of ``tlist`` (length ``len(tlist)-1``).

    The first / last value sit on the first / last grid point, the others on interval
    midpoints.  A vector that already has ``len(tlist)-1`` values is COPIED, never aliased
    (``test/test_pulse_optimization.jl:42``).  A vector ON the grid is mapped back by the exact inverse of
    :func:`discretize`, so that continuing from ``result.optimized_controls`` restarts from the very
    same pulse (``test/test_tls_optimization.jl:126,160`` demand the same J_T to 1e-14)."""
    t = _as_grid(tlist)
    if callable(control):
        mid = np.empty(t.size - 1)
        mid[0], mid[-1] = t[0], t[-1]
        mid[1:-1] = t[1:-2] + 0.5 * (t[2:-1] - t[1:-2])
        return np.fromiter((float(control(x)) for x in mid), dtype=np.float64, count=mid.size)
    v = np.asarray(control, dtype=np.float64)
    if v.size == t.size - 1:
        return v.copy()
    if v.size == t.size:
        out = np.empty(t.size - 1)
        out[0], out[-1] = v[0], v[-1]
        for i in range(1, t.size - 2):  # exact inverse of `discretize`: v[i] = (out[i-1] + out[i]) / 2
            out[i] = 2.0 * v[i] - out[i - 1]
        return out
    raise ValueError("control array must have len(tlist) or len(tlist)-1 values")


def get_controls(obj):
    """Tuple of the unique control objects (by identity) of a generator, a trajectory or a list of
    trajectories.  Identity is what lets an ensemble share its controls."""
    from .generators import Generator
    from .problem import Trajectory

    seen, out = set(), []

    def visit(x):
        if isinstance(x, Trajectory):
            visit(x.generator)
        elif isinstance(x, Generator):
            for a in x.amplitudes:
                a = control_of(a)
                if id(a) not in seen:
                    seen.add(id(a))
                    out.append(a)
        elif isinstance(x, (list, tuple)):
            for y in x:
                visit(y)
        # a bare matrix has no controls

    visit(obj)
    return tuple(out)


def get_control_derivs(generator, controls):
    """``[dG/d(control) for control in controls]``: the static operator for a linear control, ``None``
    when the generator does not depend on that control (``src/optimize.jl:344``)."""
    from .generators import Generator

    derivs = []
    for c in controls:
        mu = None
        if isinstance(generator, Generator):
            for op, a in zip(generator.control_ops, generator.amplitudes):
                if control_of(a) is c:
                    mu = op if mu is None else mu + op
        derivs.append(mu)
    return derivs


def get_amplitudes(generator, controls):
    """``[amplitude object of control c or None]``: the non-linear / shaped amplitude through which each control enters
    ``generator`` (None = the control itself multiplies its operator).  One amplitude per control and generator."""
    from .generators import ControlAmplitude, Generator

    out = []
    for c in controls:
        found = None
        if isinstance(generator, Generator):
            for a in generator.amplitudes:
                if control_of(a) is c and isinstance(a, ControlAmplitude):
                    if found is not None and found is not a:
                        raise ValueError("a control enters one generator through two different amplitudes: unsupported")
                    found = a
                elif control_of(a) is c and found is not None:
                    raise ValueError("a control enters one generator both directly and through an amplitude: unsupported")
        out.append(found)
    return out


def _amplitude_key(a):
    """What makes two amplitudes of one control the same term: the same function of the control and the same shape
    object.  None for the control itself."""
    from .generators import ControlAmplitude

    if not isinstance(a, ControlAmplitude):
        return None
    return (a.key(), id(a.shape) if a.shape is not None else None)


def get_control_terms(generators, controls):
    """The control terms of ``generators``: every (operator, amplitude) pair through which a control enters them.

    Operators of one generator that depend on one control through the same amplitude (same ``key()`` and the same shape
    object, or the control itself) are summed into one operator; different amplitudes make separate terms.  Term l is
    control l for l < L (the control's first amplitude, in order of appearance); the further terms of controls that
    enter through several amplitudes follow.  Returns ``(terms, ops)``: ``terms[t] = (l, amplitude or None)`` and
    ``ops[g][t]`` the operator of term t in ``generators[g]`` (None where the generator lacks the term)."""
    from .generators import ControlAmplitude, Generator

    index = {id(c): l for l, c in enumerate(controls)}
    seen = [[] for _ in controls]  # per control: (key, amplitude) in order of appearance
    per_gen = []
    for gen in generators:
        ops = {}
        if isinstance(gen, Generator):
            for op, a in zip(gen.control_ops, gen.amplitudes):
                l = index[id(control_of(a))]
                k = _amplitude_key(a)
                ops[(l, k)] = op if (l, k) not in ops else ops[(l, k)] + op
                if all(k != kk for kk, _ in seen[l]):
                    seen[l].append((k, a if isinstance(a, ControlAmplitude) else None))
        per_gen.append(ops)
    order = [(l, seen[l][0]) for l in range(len(controls)) if seen[l]]
    order += [(l, ka) for l in range(len(controls)) for ka in seen[l][1:]]
    terms = [(l, a) for l, (_, a) in order]
    return terms, [[ops.get((l, k)) for l, (k, _) in order] for ops in per_gen]
