"""``optimize(problem; method=Krotov)``: the driver of ``src/optimize.jl:155-235`` around the device
hot path.

The two functions that ARE the hot path in the reference -- ``krotov_initial_fw_prop!``
(``src/optimize.jl:247-265``) and ``krotov_iteration`` (``:279-371``) -- keep their names here and are
each one call into ``libkrotov_cuda`` (``krotov_forward`` / ``krotov_iterate``).  Everything else is the
reference's host-side bookkeeping: result updates (``:374-406``), callbacks, convergence, the
iteration table (``:413-496``).
"""
from __future__ import annotations

import atexit
import datetime as _dt
import logging
import pickle
import sys

import numpy as np

from . import _lib as B
from .cheby import transform_control_ranges
from .controls import discretize
from .errors import ArgumentError
from .functionals import chi_coefficients
from .second_order import sigma_value
from .workspace import KrotovWrk

log = logging.getLogger("krotov_jl_b200")

__all__ = ["optimize", "optimize_krotov", "krotov_initial_fw_prop", "krotov_iteration", "update_result", "update_sigma",
           "finalize_result", "detached_result", "make_krotov_print_iters", "make_print_iters", "Krotov", "Cheby", "Expmv"]


class _Method:
    def __init__(self, name):
        self.__name__ = name

    def __repr__(self):
        return self.__name__


Krotov = _Method("Krotov")  # `optimize(problem; method=Krotov)`
Cheby = _Method("Cheby")  # `prop_method=Cheby`
Expmv = _Method("Expmv")  # `prop_method=Expmv`: truncated Taylor series with scaling (expmv.py), any generator


# --------------------------------------------------------------------------------------------
# hot path: one C-ABI call each
# --------------------------------------------------------------------------------------------
def _stack(pulses):
    return np.ascontiguousarray(np.stack([np.asarray(p, np.float64) for p in pulses]))


def krotov_initial_fw_prop(eps0, wrk):
    """All trajectories at once (the reference loops k over ``krotov_initial_fw_prop!``,
    ``src/optimize.jl:182-184``): range check of ``reinit_prop!`` (``:251``), then one device sweep."""
    for view in wrk.fw_propagators:
        view.parameters = eps0
    if wrk.fw_settings.reinit(wrk._term_rows(eps0), transform_control_ranges):
        wrk.fw_settings.push(wrk.engine, B.FORWARD)
    wrk.engine.forward(_stack(wrk._term_rows(eps0)))
    wrk._states.invalidate()


def krotov_iteration(wrk, eps_i, eps_ip1):
    """One Krotov iteration (``src/optimize.jl:279-371``): chi boundary condition, then
    ``krotov_iterate`` = backward sweep + sequential update + forward sweep on the device."""
    # chi_k(T)  (:297-302)
    if wrk.functional == B.CHI_HOST or wrk.sigma is not None:
        lo, hi = wrk._shard
        Psi = wrk.result.states
        if wrk.functional == B.CHI_HOST:
            chi_fn = wrk.kwargs["chi"]
            if wrk.chi_takes_tau:
                chi = chi_fn(Psi, wrk.trajectories, tau=wrk.result.tau_vals)
            else:
                chi = chi_fn(Psi, wrk.trajectories)
            chi = np.array([np.asarray(c) for c in chi], np.complex128)
        else:  # (second order with a built-in functional: chi = c_k |target_k>, all trajectories at once)
            kind = {B.CHI_SM: "sm", B.CHI_SS: "ss", B.CHI_RE: "re"}[wrk.functional]
            chi = chi_coefficients(kind, wrk.result.tau_vals, wrk._weight)[:, None] * wrk._target
        chi_T = chi[lo:hi]
        if wrk.sigma is not None:
            # second order (the TODO at :350): for Hermitian generators and a sigma that is constant over the time
            # grid, chi(t_n) + sigma/2 (Psi^(i+1)(t_n) - Psi^(i)(t_n)) acts in the update like the backward-propagated
            # chi(T) - sigma/2 Psi^(i)(T)  (second_order.py)
            sig = sigma_value(wrk.sigma, wrk.result.tlist, full=False)
            psi_T = np.array(Psi._get() if hasattr(Psi, "_get") else [np.asarray(s) for s in Psi], np.complex128)
            wrk._sigma_info = dict(forward_states0=psi_T, chi_states=chi)
            chi_T = chi_T - (0.5 * sig) * psi_T[lo:hi]
        wrk.engine.set_chi(np.ascontiguousarray(chi_T))
    elif wrk._n_ranks > 1 and wrk.functional == B.CHI_SM:
        # the only functional whose chi needs a sum over ALL ranks' tau: done here from the gathered tau
        tau, w, n = wrk.result.tau_vals, wrk._weight, wrk.N
        s = np.sum(w * tau)
        lo, hi = wrk._shard
        wrk.engine.set_chi_coeffs((w[lo:hi] / n**2) * s)
    # reinit_prop! of the backward propagators under the guess pulses (:305-306)
    for view in wrk.bw_propagators:
        view.parameters = eps_i
    if wrk.bw_settings.reinit(wrk._term_rows(eps_i), transform_control_ranges):
        wrk.bw_settings.push(wrk.engine, B.BACKWARD)
    # reinit_prop! of the forward propagators (:321-325): the check sees the eps^(i+1) buffers as they
    # are NOW (stale content), exactly like the reference's aliased arrays
    for view in wrk.fw_propagators:
        view.parameters = eps_ip1
    if wrk.fw_settings.reinit(wrk._term_rows(eps_ip1), transform_control_ranges):
        wrk.fw_settings.push(wrk.engine, B.FORWARD)
    new, ga = wrk.engine.iterate(_stack(wrk._term_rows(eps_i)))
    if wrk._term_ctrl is not None:  # control terms -> controls: term l < L is control l, g_a sits at a control's first term
        ga = np.bincount(wrk._term_ctrl, weights=ga, minlength=len(eps_ip1))
    for l in range(len(eps_ip1)):
        eps_ip1[l][:] = new[l]  # in place: callbacks hold references to these arrays
    wrk.g_a_int[:] = ga
    wrk._states.invalidate()


# --------------------------------------------------------------------------------------------
# host-side bookkeeping
# --------------------------------------------------------------------------------------------
def update_result(wrk, i):
    """``update_result!`` (``src/optimize.jl:374-397``)."""
    res = wrk.result
    J_T = wrk.kwargs["J_T"]
    res.J_T_prev = res.J_T
    res.states = wrk._states  # aliases the live propagator states (:378-380)
    res.tau_vals = wrk._fetch_tau()  # taus! on the device (zero where no target)
    if wrk.J_T_takes_tau:
        res.J_T = float(J_T(res.states, wrk.trajectories, tau=res.tau_vals))
    else:
        res.J_T = float(J_T(res.states, wrk.trajectories))
    if i > 0:
        res.iter = i
    if i >= res.iter_stop:
        res.converged = True
        res.message = "Reached maximum number of iterations"
    prev = res.end_local_time
    res.end_local_time = _dt.datetime.now()
    res.secs = (res.end_local_time - prev).total_seconds()


def update_sigma(wrk, eps_ip1, eps_i):
    """The "update sigma" step (TODO at ``src/optimize.jl:369``), run once the iteration's J_T is known:
    ``sigma.refresh(**info)`` with the final-time states of this and of the previous iteration, chi(T), J_T."""
    refresh = getattr(wrk.sigma, "refresh", None)
    if refresh is None:
        return
    res = wrk.result
    Psi = res.states
    new = np.array(Psi._get() if hasattr(Psi, "_get") else [np.asarray(s) for s in Psi], np.complex128)
    refresh(forward_states=new, J_T=res.J_T, J_T_prev=res.J_T_prev,
            optimized_pulses=eps_ip1, guess_pulses=eps_i, trajectories=wrk.trajectories, result=res,
            **wrk._sigma_info)


def detached_result(res):
    """Copy of a result that holds plain arrays only (no view of device memory, no engine handle): what
    ``atexit_filename`` and user callbacks may pickle."""
    import dataclasses

    states = res.states
    if not isinstance(states, list) or any(not isinstance(s, np.ndarray) for s in states):
        try:
            states = states.snapshot() if hasattr(states, "snapshot") else [np.array(s) for s in states]
        except Exception:  # the device is gone (interpreter shutdown after a fault): keep the rest of the result
            states = []
    return dataclasses.replace(res, states=states, records=list(res.records),
                               optimized_controls=[np.array(c) for c in res.optimized_controls],
                               guess_controls=[np.array(c) for c in res.guess_controls])


def _dump_result(res, filename):
    import os
    import tempfile

    folder = os.path.dirname(os.path.abspath(filename))
    fd, tmp = tempfile.mkstemp(prefix=".krotov_atexit_", dir=folder)
    try:
        with os.fdopen(fd, "wb") as fh:
            pickle.dump(res, fh)
        os.replace(tmp, filename)
    except BaseException:
        try:
            os.unlink(tmp)
        except OSError:
            pass
        raise


def finalize_result(eps_opt, wrk):
    """``finalize_result!`` (``src/optimize.jl:400-406``)."""
    res = wrk.result
    res.end_local_time = _dt.datetime.now()
    for l in range(len(eps_opt)):
        res.optimized_controls[l] = discretize(eps_opt[l], res.tlist)
    res.states = [np.array(s) for s in wrk._states]  # detach from the device before the handle goes away


_HEADER = ["iter.", "J_T", "∫gₐ(t)dt", "J", "ΔJ_T", "ΔJ", "secs"]


def make_krotov_print_iters(store_iter_info=(), **_):
    """The iteration-table callback (``src/optimize.jl:413-496``): same columns, widths and formats;
    returns the values listed in ``store_iter_info`` in header order."""
    wanted = set(store_iter_info)
    for item in wanted:
        if item not in _HEADER:
            raise ArgumentError(f"Item {item!r} in `store_iter_info` is not one of {_HEADER!r})")
    keep = [h in wanted for h in _HEADER]

    def print_table(wrk, iteration, *args):
        J_T = wrk.result.J_T
        g_a_int = float(np.sum(wrk.g_a_int))
        J = J_T + g_a_int
        dJ_T = J_T - wrk.result.J_T_prev
        dJ = dJ_T + g_a_int
        secs = wrk.result.secs
        values = [iteration, J_T, g_a_int, J, dJ_T, dJ, secs]
        iter_stop = str(wrk.kwargs.get("iter_stop", 5000))
        widths = [max(len(iter_stop), 6), 11, 11, 11, 11, 11, 8]
        out = sys.stdout
        if iteration == 0:
            out.write("".join(h.rjust(w) for h, w in zip(_HEADER, widths)) + "\n")
        cells = [str(iteration), f"{J_T:.2e}", f"{g_a_int:.2e}", f"{J:.2e}",
                 f"{dJ_T:.2e}" if iteration > 0 else "n/a", f"{dJ:.2e}" if iteration > 0 else "n/a", f"{secs:.1f}"]
        out.write("".join(c.rjust(w) for c, w in zip(cells, widths)) + "\n")
        out.flush()
        return tuple(v for v, k in zip(values, keep) if k)

    return print_table


make_print_iters = make_krotov_print_iters


def _chain(callbacks):
    """Run callbacks in order; concatenate the tuples they return (QuantumControl's chaining)."""
    callbacks = [c for c in callbacks if c is not None]

    def chained(*args):
        rec = ()
        for cb in callbacks:
            r = cb(*args)
            if r is not None:
                rec = rec + tuple(r)
        return rec

    return chained


def optimize(problem, method=Krotov, *, comm=None, **kwargs):
    """``optimize(problem; method=Krotov, kwargs...)``.  Keyword arguments override those of the problem
    (``src/optimize.jl:60-62``); ``print_iters=True`` appends the table callback after user callbacks."""
    name = method if isinstance(method, str) else getattr(method, "__name__", str(method))
    if name.split(".")[-1].lower().lstrip(":") != "krotov":
        raise ArgumentError(f"method={method!r}: only Krotov is implemented here")
    from .problem import ControlProblem

    merged = dict(problem.kwargs)
    merged.update(kwargs)
    cb = merged.get("callback", None)
    cbs = list(cb) if isinstance(cb, (tuple, list)) else [cb]
    if merged.get("print_iters", True):
        cbs.append(make_krotov_print_iters(store_iter_info=merged.get("store_iter_info", ())))
    merged["callback"] = _chain(cbs)
    return optimize_krotov(ControlProblem(problem.trajectories, problem.tlist, **merged), comm=comm)


def optimize_krotov(problem, comm=None):
    """``optimize_krotov`` (``src/optimize.jl:161-235``)."""
    kw = problem.kwargs
    callback = kw.get("callback", lambda *a: None)
    if "update_hook" in kw or "info_hook" in kw:
        raise ArgumentError("The `update_hook` and `info_hook` arguments have been superseded by the `callback` argument")
    check_convergence = kw.get("check_convergence", lambda res: res)
    verbose = kw.get("verbose", False)
    skip_initial = kw.get("skip_initial_forward_propagation", False)

    wrk = KrotovWrk(problem, verbose=verbose, comm=comm)
    try:
        eps_i, eps_ip1 = wrk.pulses0, wrk.pulses1
        if skip_initial:
            log.info("Skipping initial forward propagation")
        else:
            krotov_initial_fw_prop(eps_i, wrk)
        update_result(wrk, 0)
        info = callback(wrk, 0, eps_ip1, eps_i)
        if info:
            wrk.result.records.append(tuple(info))
        i = wrk.result.iter  # = 0 unless continuing
        atexit_filename = kw.get("atexit_filename", None)
        hook = None
        if atexit_filename is not None:
            # set_atexit_save_optimization (src/optimize.jl:195-205): dump the result if the process dies mid-run.
            # The live result aliases device-backed views, so a detached copy is written (to a temporary file that
            # is renamed into place: a crash while dumping never leaves a truncated checkpoint behind).
            def hook(wrk=wrk, fn=atexit_filename):
                _dump_result(detached_result(wrk.result), fn)
            atexit.register(hook)
        try:
            while not wrk.result.converged:
                i += 1
                krotov_iteration(wrk, eps_i, eps_ip1)
                update_result(wrk, i)
                if wrk.sigma is not None:
                    update_sigma(wrk, eps_ip1, eps_i)
                info = callback(wrk, i, eps_ip1, eps_i)
                if info:
                    wrk.result.records.append(tuple(info))
                check_convergence(wrk.result)
                eps_i, eps_ip1 = eps_ip1, eps_i
        except BaseException as exc:  # incl. KeyboardInterrupt, like InterruptException in the reference
            if kw.get("rethrow_exceptions", False):
                raise
            wrk.result.message = f"Exception: {exc}"
        finalize_result(eps_i, wrk)
        if hook is not None:
            atexit.unregister(hook)
        return wrk.result
    finally:
        wrk.close()
