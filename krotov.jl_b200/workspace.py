"""``KrotovWrk``: the workspace of ``src/workspace.jl:30-200`` with the device as owner of the heavy
fields.  Field names follow the reference so that callbacks written for it keep working:
``trajectories, adjoint_trajectories, kwargs, controls, pulses0, pulses1, g_a_int, update_shapes,
lambda_vals, J_T_takes_tau, chi_takes_tau, result, control_derivs, fw_prop_kwargs, bw_prop_kwargs,
fw_storage, fw_storage2, bw_storage, fw_propagators, bw_propagators, use_threads``.

What lives where: pulses, S_l, lambda_l, g_a_int and the result are host NumPy arrays (the host copy
of the pulses is authoritative between iterations -- callbacks may edit it); states, the chi
trajectory (``bw_storage``) and the optional forward storage live in HBM behind a ``KrotovCuda``
handle and are fetched lazily when a callback touches them.
"""
from __future__ import annotations

import datetime as _dt
import inspect
import logging
import warnings

import numpy as np

from . import _lib as B
from .cheby import ChebyDirection
from .expmv import TaylorDirection
from .controls import discretize_on_midpoints, get_control_derivs, get_control_terms, get_controls
from .engine import KrotovCuda
from .errors import ArgumentError, ErrorException
from .functionals import make_chi
from .generators import Generator
from .result import KrotovResult, convert_result
from .second_order import sigma_value

log = logging.getLogger("krotov_jl_b200")

__all__ = ["KrotovWrk", "IdDict", "saturated_corners"]


def saturated_corners(poly, s, lo, hi, shape_max=None):
    """Range of ``shape_max * P(tanh(s eps))`` over eps in [lo, hi] for a polynomial P of degree <= 2 (ascending
    ``poly``): ``(P(x_lo), P(x_hi))`` when P is monotone on [x_lo, x_hi], else ``(min, max)`` including the vertex."""
    c = [float(v) for v in poly] + [0.0] * 3
    if any(v != 0.0 for v in c[3:]):
        raise ArgumentError("a saturating amplitude takes a polynomial of degree <= 2")
    P = lambda x: (c[2] * x + c[1]) * x + c[0]  # noqa: E731
    x_lo, x_hi = float(np.tanh(s * lo)), float(np.tanh(s * hi))
    v_lo, v_hi = P(x_lo), P(x_hi)
    if c[2] != 0.0:
        x_v = -c[1] / (2.0 * c[2])
        if x_lo < x_v < x_hi:
            vals = (v_lo, v_hi, P(x_v))
            v_lo, v_hi = min(vals), max(vals)
    if shape_max is not None:
        v_lo, v_hi = shape_max * v_lo, shape_max * v_hi
    return v_lo, v_hi


class IdDict:
    """Mapping keyed by object identity (controls may be unhashable arrays)."""

    def __init__(self, pairs=()):
        self._items = [(k, v) for k, v in (pairs.items() if hasattr(pairs, "items") else pairs)]

    def __contains__(self, key):
        return any(k is key for k, _ in self._items)

    def __getitem__(self, key):
        for k, v in self._items:
            if k is key:
                return v
        raise KeyError(key)

    def __setitem__(self, key, value):
        for i, (k, _) in enumerate(self._items):
            if k is key:
                self._items[i] = (key, value)
                return
        self._items.append((key, value))

    def keys(self):
        return [k for k, _ in self._items]

    def items(self):
        return list(self._items)

    def __len__(self):
        return len(self._items)


def _lookup(options, control):
    if isinstance(options, IdDict):
        return options[control]
    for k, v in options.items():
        if k is control:
            return v
    raise KeyError


def _has(options, control):
    try:
        _lookup(options, control)
        return True
    except KeyError:
        return False


def _takes_tau(fn):
    try:
        return "tau" in inspect.signature(fn).parameters
    except (TypeError, ValueError):
        return False


_CHEBY_NAMES = {"cheby", "Cheby", ":Cheby", ":cheby"}
_EXPMV_NAMES = {"expmv", "Expmv", ":Expmv", ":expmv"}


def _is_cheby(method):
    if method is None:
        return False
    if isinstance(method, str):
        return method in _CHEBY_NAMES
    return getattr(method, "__name__", "").split(".")[-1] in _CHEBY_NAMES


def _is_expmv(method):
    if method is None:
        return False
    name = method if isinstance(method, str) else getattr(method, "__name__", "").split(".")[-1]
    return name in _EXPMV_NAMES


def _prop_kwargs(traj, kwargs, prefixes):
    """``init_prop_trajectory``'s harvesting rule: problem kwargs first, trajectory properties
    override; later prefixes override earlier ones (``src/workspace.jl:133,148``)."""
    out = {}
    for source in (kwargs, getattr(traj, "kwargs", {})):
        for prefix in prefixes:
            for key, val in source.items():
                if key.startswith(prefix):
                    out[key[len(prefix):]] = val
    return out


def _comparable(pk):
    return {k: (getattr(v, "__name__", None) or repr(v)) for k, v in pk.items()}


class _LazyStates:
    """List-like view of Psi_k(T) on the device; fetched once per sweep on first access."""

    def __init__(self, wrk):
        self._wrk = wrk
        self._cache = None

    def invalidate(self):
        self._cache = None

    def _get(self):
        if self._cache is None:
            self._cache = self._wrk._fetch_states()
        return self._cache

    def __len__(self):
        return self._wrk.N

    def __getitem__(self, k):
        return self._get()[k]

    def __iter__(self):
        return iter(self._get())

    def __setitem__(self, k, v):  # `res.states[k] = propagator.state` (src/optimize.jl:379) is a no-op alias
        pass

    def snapshot(self):
        """Plain copies of the states WITHOUT a collective: the cached gather when there is one, a local fetch on a
        single rank, else only what this rank can see without its peers (an exit hook must never wait for them)."""
        if self._cache is not None:
            return [np.array(s) for s in self._cache]
        wrk = self._wrk
        if wrk.comm is None or wrk.comm.world == 1:
            return [np.array(s) for s in self._get()]
        return [np.array(s) for s in wrk.engine.states()]  # this rank's shard only

    def __reduce__(self):
        # pickling (a callback that checkpoints `wrk.result`, the atexit hook) stores the plain state vectors, as
        # the reference's `result.states` are; the view itself holds the engine handle and cannot be pickled
        return (list, (self.snapshot(),))


class _PropagatorView:
    """What callbacks see as ``wrk.fw_propagators[k]`` / ``wrk.bw_propagators[k]``."""

    def __init__(self, wrk, k, backward):
        self._wrk, self._k, self.backward = wrk, k, backward
        self.parameters = None

    @property
    def state(self):
        if self.backward:
            return self._wrk.bw_storage[self._k][:, 0]
        return self._wrk.result.states[self._k]

    @property
    def tlist(self):
        return self._wrk.result.tlist


class _Storage:
    """``storage[k]`` -> (d, N_T+1) array, column n = time-grid point n, fetched from HBM on demand."""

    def __init__(self, wrk, which):
        self._wrk, self._which = wrk, which

    def __len__(self):
        return self._wrk.N

    def __getitem__(self, k):
        wrk = self._wrk
        if self._which == B.FORWARD and not wrk.store_fw:
            raise ErrorException("forward storage is off; pass `store_fw_states=True` to `optimize`")
        lo, hi = wrk._shard
        if not (lo <= k < hi):
            raise ErrorException(f"trajectory {k} lives on another rank (this rank holds {lo}:{hi})")
        return wrk.engine.storage(self._which, k - lo).T.copy()


class KrotovWrk:
    def __init__(self, problem, *, verbose=False, comm=None):
        kwargs_in = problem.kwargs
        self.use_threads = bool(kwargs_in.get("use_threads", False))  # accepted, ignored: the GPU batches
        self.trajectories = list(problem.trajectories)
        N = len(self.trajectories)
        self.adjoint_trajectories = [t.adjoint() for t in self.trajectories]
        self.controls = get_controls(self.trajectories)
        if len(self.controls) == 0:
            raise ErrorException("no controls in trajectories: cannot optimize")
        # control_derivs[k][l]: the sum of the operators through which control l enters generator k (None: it does not),
        # whatever their amplitudes -- for a control with several terms this is not mu = sum_t a_t' H_t; the device
        # evaluates mu per term (see _terms)
        self.control_derivs = [get_control_derivs(t.generator, self.controls) for t in self.trajectories]
        tlist = np.asarray(problem.tlist, np.float64)
        # control terms: (control, amplitude) pairs, term l = control l for l < L, further terms of controls that enter
        # through several amplitudes after them; _term_ops[g][t] per distinct generator (by identity, first appearance)
        gens = list({id(t.generator): t.generator for t in self.trajectories}.values())
        self._terms, self._term_ops = get_control_terms(gens, self.controls)
        self._term_ctrl = (None if len(self._terms) == len(self.controls) else
                           np.array([l for l, _ in self._terms], np.int32))
        self._check_term_functions()
        self._amp_poly, self._amp_shape, self._amp_sat = self._collect_amplitudes(tlist)
        kwargs = dict(kwargs_in)  # shallow copy; ok to modify
        default_shape = kwargs_in.get("update_shape", lambda t: 1.0)
        default_lambda = float(kwargs_in.get("lambda_a", 1.0))
        default_options = IdDict(
            [(c, {"lambda_a": default_lambda, "update_shape": default_shape}) for c in self.controls])
        if "pulse_options" in kwargs:
            if "update_shape" in kwargs:
                warnings.warn("`update_shape` is ignored due to given `pulse_options`")
            if "lambda_a" in kwargs:
                warnings.warn(f"`lambda_a={kwargs['lambda_a']}` is ignored due to given `pulse_options`")
        elif "update_shape" not in kwargs and "lambda_a" not in kwargs:
            warnings.warn("Using default pulse_options: (:lambda_a => 1.0, :update_shape => (t -> 1.0))")
        pulse_options = kwargs.get("pulse_options", default_options)
        for c in self.controls:
            if not _has(pulse_options, c):
                raise ErrorException("pulse_options must be defined for all controls")

        def opt(c, name):
            o = _lookup(pulse_options, c)
            return o[name] if name in o else o[":" + name]

        self.update_shapes = [discretize_on_midpoints(opt(c, "update_shape"), tlist) for c in self.controls]
        self.lambda_vals = np.array([float(opt(c, "lambda_a")) for c in self.controls], np.float64)
        if "continue_from" in kwargs:
            log.info("Continuing previous optimization")
            result = convert_result(kwargs["continue_from"])
            result.iter_stop = int(kwargs.get("iter_stop", 5000))
            result.converged = False
            result.start_local_time = _dt.datetime.now()
            result.message = "in progress"
            pulses0 = [discretize_on_midpoints(c, tlist) for c in result.optimized_controls]
        else:
            result = KrotovResult.from_problem(problem)
            pulses0 = [discretize_on_midpoints(c, tlist) for c in self.controls]
        self.result = result
        self.pulses0 = pulses0
        # init_prop_trajectory (src/workspace.jl:136-161) sees the generator's ORIGINAL controls: their ranges seed the
        # propagators' control ranges (differs from pulses0 only under `continue_from`)
        self._init_pulses = pulses0 if "continue_from" not in kwargs else [
            discretize_on_midpoints(c, tlist) for c in self.controls]
        self.pulses1 = [p.copy() for p in pulses0]
        self.g_a_int = np.zeros(len(pulses0))
        kwargs["piecewise"] = True  # only piecewise propagators
        self.fw_prop_kwargs = [_prop_kwargs(t, kwargs, ["prop_", "fw_prop_"]) for t in self.trajectories]
        self.bw_prop_kwargs = [_prop_kwargs(t, kwargs, ["prop_", "bw_prop_"]) for t in self.adjoint_trajectories]
        for k in range(N):
            self.bw_prop_kwargs[k]["backward"] = True
        for pk in self.fw_prop_kwargs + self.bw_prop_kwargs:
            if "method" not in pk:
                raise ArgumentError("The propagation method must be specified (`prop_method=Cheby`)")
            if not (_is_cheby(pk["method"]) or _is_expmv(pk["method"])):
                raise ArgumentError(
                    f"prop_method={pk['method']!r}: libkrotov_cuda serves the `Cheby` propagator and `Expmv` (truncated "
                    "Taylor series, exact for non-Hermitian generators such as Liouvillians) only; there is no CPU "
                    "fallback for other methods")
            if "callback" in pk:
                raise ArgumentError("per-step propagation callbacks cannot run inside the device sweep")
        for name, pks in (("fw", self.fw_prop_kwargs), ("bw", self.bw_prop_kwargs)):
            # one set of propagator settings serves the whole batch: per-trajectory overrides that differ would be
            # silently lost, so they are refused
            for pk in pks[1:]:
                if _comparable(pk) != _comparable(pks[0]):
                    raise ArgumentError(f"{name}_prop_kwargs differ between trajectories; the batched device "
                                        "propagator needs the same propagator settings for all of them")
        # both directions run in one persistent kernel, which carries one propagator
        self._expmv = _is_expmv(self.fw_prop_kwargs[0]["method"])
        if self._expmv != _is_expmv(self.bw_prop_kwargs[0]["method"]):
            raise ArgumentError("the forward and backward propagators must use the same method (`Cheby` or `Expmv`): "
                                f"got fw {self.fw_prop_kwargs[0]['method']!r}, bw {self.bw_prop_kwargs[0]['method']!r}")
        if "J_T" not in kwargs:
            raise ArgumentError("`optimize` for `method=Krotov` must be passed the functional `J_T`.")
        J_T = kwargs["J_T"]
        self.J_T_takes_tau = _takes_tau(J_T)
        if "chi" not in kwargs:
            kwargs["chi"] = make_chi(J_T, self.trajectories)
        self.chi_takes_tau = _takes_tau(kwargs["chi"])
        self.kwargs = kwargs
        self.N = N
        self.verbose = verbose
        self.store_fw = bool(kwargs.get("store_fw_states", False))
        self.fw_storage2 = None  # never read or written by the reference (src/workspace.jl:129-130)
        # second order (`sigma`, src/optimize.jl:104-105; TODOs :187, :350, :369): see second_order.py
        self.sigma = kwargs.get("sigma", None)
        if self.sigma is not None:
            if kwargs.get("skip_initial_forward_propagation", False):
                raise ArgumentError("`sigma` needs the forward states of the guess pulses: it cannot be combined with "
                                    "`skip_initial_forward_propagation`")
            sigma_value(self.sigma, tlist)  # (raises for a sigma that varies over the time grid)
        self._build_device_side(tlist, comm)
        if self.sigma is not None and not self._hermitian:
            self.engine.close()
            raise ArgumentError("`sigma` (second-order Krotov) needs Hermitian generators and control operators: "
                                "the device path folds the second-order term into the boundary condition chi(T)")
        self.fw_storage = _Storage(self, B.FORWARD)
        self.bw_storage = _Storage(self, B.BACKWARD)
        self.fw_propagators = [_PropagatorView(self, k, False) for k in range(N)]
        self.bw_propagators = [_PropagatorView(self, k, True) for k in range(N)]
        self._states = _LazyStates(self)
        if not isinstance(self.result.states, _LazyStates):
            self.result.states = self._states

    # -------------------------------------------------------------------------------------
    def _collect_amplitudes(self, tlist):
        """Non-linear / shaped amplitudes (``src/optimize.jl:268-272``): per control TERM the polynomial, the per-interval
        shape and the saturation ``s`` (a parametrization's ``tanh(s u)``, 0 = none) through which it enters the
        generators.  ``(None, None, None)`` when every term is its control itself."""
        amps = [a for _, a in self._terms]
        T = len(amps)
        if all(a is None for a in amps):
            return None, None, None
        deg = max(len(a.coeffs) - 1 for a in amps if a is not None)
        poly = np.zeros((T, deg + 1))
        shape = None
        for l, a in enumerate(amps):
            if a is None:
                poly[l, 1] = 1.0
                continue
            poly[l, : len(a.coeffs)] = a.coeffs
            if a.shape is not None:
                if shape is None:
                    shape = np.ones((T, len(tlist) - 1))
                shape[l] = discretize_on_midpoints(a.shape, tlist)
        if all(np.array_equal(poly[l], np.eye(deg + 1)[1]) for l in range(T)):
            poly = None  # only shapes: a(eps, n) = shape[n] * eps
        sat = np.array([0.0 if a is None else a.saturation for a in amps])
        return poly, shape, (sat if np.any(sat > 0) else None)

    def _check_term_functions(self):
        """Every generator that depends on a control must see it through the same amplitude FUNCTIONS (``key()``): the
        terms of a control may differ between generators in their shapes only (an ensemble member with its own
        distortion of the pulse envelope), not in the polynomial or parametrization that maps the control value."""
        fn = lambda a: None if a is None else a.key()  # noqa: E731
        for l in range(len(self.controls)):
            seen = {frozenset(fn(a) for (c, a), op in zip(self._terms, row) if c == l and op is not None)
                    for row in self._term_ops}
            seen.discard(frozenset())
            if len(seen) > 1:
                raise ArgumentError("a control must enter all generators through the same amplitudes (their shapes may "
                                    "differ between generators)")

    def _term_rows(self, rows):
        """Per-control rows (pulses, update shapes, lambda) -> one row per control term: term t carries its control's."""
        return rows if self._term_ctrl is None else [rows[l] for l in self._term_ctrl]

    def _amp_envelope(self, l, eps):
        """Coefficient of H_l at a corner ``eps`` of the control range, for the spectral envelope: the polynomial at
        the corner times the largest |shape| (unpinned convention, see oracle ``amplitude_envelope``)."""
        v = eps
        if self._amp_poly is not None:
            v = 0.0
            for c in self._amp_poly[l][::-1]:
                v = v * eps + c
        if self._amp_shape is not None:
            v = float(np.max(np.abs(self._amp_shape[l]))) * v
        return v

    def _amp_envelope_corners(self, l, lo, hi):
        """Coefficients of H_l for the spectral envelope over the control range [lo, hi]: ``(value at the lo side,
        value at the hi side)``.  A saturating control (s_l > 0) takes the range of its polynomial P (degree <= 2) over
        [tanh(s lo), tanh(s hi)] -- the end values, plus P at its vertex when the vertex lies inside, in which case the
        pair is (min, max): tanh**2 over a range that straddles 0 must include the amplitude 0.  Every other control keeps
        the corners of ``_amp_envelope``."""
        s = 0.0 if self._amp_sat is None else float(self._amp_sat[l])
        if s == 0.0:
            return self._amp_envelope(l, lo), self._amp_envelope(l, hi)
        return saturated_corners(self._amp_poly[l] if self._amp_poly is not None else [0.0, 1.0], s, lo, hi,
                                 None if self._amp_shape is None else float(np.max(np.abs(self._amp_shape[l]))))

    def _amp_abs_max(self, l, lo, hi):
        """Largest |coefficient of H_l| over the control range [lo, hi] (the Taylor norm bound): the corners of
        ``_amp_envelope_corners`` and, for a polynomial amplitude, its value at every critical point inside the range."""
        v = max(abs(c) for c in self._amp_envelope_corners(l, lo, hi))
        if self._amp_poly is not None and (self._amp_sat is None or self._amp_sat[l] == 0.0):
            q = np.polynomial.Polynomial(self._amp_poly[l])
            shp = 1.0 if self._amp_shape is None else float(np.max(np.abs(self._amp_shape[l])))
            for x in q.deriv().roots():
                if abs(x.imag) < 1e-12 and lo <= x.real <= hi:
                    v = max(v, shp * abs(q(x.real)))
        return v

    def _build_device_side(self, tlist, comm):
        trajs = self.trajectories
        N, L = self.N, len(self._terms)  # (the device counts control terms)
        d = trajs[0].initial_state.shape[0]
        if self._expmv and d > 32:
            raise ArgumentError(f"prop_method=Expmv runs on the one-warp-per-trajectory kernel, d <= 32 (got d = {d})")
        # distinct generators by identity: ensemble members sharing a Hamiltonian share its storage
        gen_ids, gens, gen_of_traj = {}, [], np.zeros(N, np.int32)
        for k, t in enumerate(trajs):
            key = id(t.generator)
            if key not in gen_ids:
                gen_ids[key] = len(gens)
                gens.append((t.generator, self._term_ops[len(gens)]))
            gen_of_traj[k] = gen_ids[key]
        H0, Hc = [], []
        for gen, derivs in gens:
            keep = lambda m: m if hasattr(m, "tocsr") else np.asarray(m, np.complex128)  # noqa: E731
            H0.append(keep(gen.drift()) if isinstance(gen, Generator) else keep(gen))
            Hc.append([None if mu is None else keep(mu) for mu in derivs])
        psi0 = np.array([t.initial_state for t in trajs], np.complex128).reshape(N, d)
        has_all_targets = all(t.target_state is not None for t in trajs)
        has_any_target = any(t.target_state is not None for t in trajs)
        target = None
        if has_any_target:
            target = np.zeros((N, d), np.complex128)
            for k, t in enumerate(trajs):
                if t.target_state is not None:
                    target[k] = t.target_state
        weight = np.array([t.weight for t in trajs], np.float64)
        builtin = getattr(self.kwargs["chi"], "krotov_builtin", None)
        functional = {"sm": B.CHI_SM, "ss": B.CHI_SS, "re": B.CHI_RE}.get(builtin, B.CHI_HOST)
        if functional != B.CHI_HOST and not has_all_targets:
            functional = B.CHI_HOST
        self.functional = functional
        # ---- sharding over ranks (contiguous blocks of trajectories, aligned to generators when possible)
        self.comm = comm
        rank, world = (comm.rank, comm.world) if comm is not None else (0, 1)
        from .distributed import shard_bounds

        S = np.array(self._term_rows(self.update_shapes), np.float64).reshape(L, -1)
        lam = np.array(self._term_rows(self.lambda_vals), np.float64)
        pk = self.fw_prop_kwargs[0]
        device = int(self.kwargs.get("device", comm.device if comm is not None else 0))

        # several ranks: "shard" = every rank holds its block of trajectories, the overlap sums cross the ranks at every
        # time step; "replicate" = every rank holds ALL trajectories, the backward sweep is sharded and writes chi to
        # every rank, the time-serial forward sweep runs everywhere (no per-step exchange; replicas identical by
        # construction).  "auto": replicate where the persistent one-warp-per-trajectory kernel serves the problem.
        mode = str(self.kwargs.get("multi_gpu", "auto"))
        n_ranks_wanted = max(world, int(self.kwargs.get("emulate_ranks", 0) or 0))
        any_sparse = any(hasattr(m, "tocsr") for m in H0)
        if mode == "auto":
            mode = "replicate" if (n_ranks_wanted > 1 and d <= 32 and N <= 7 * 148 and not any_sparse and not self._expmv
                                   and int(self.kwargs.get("force_path", 0)) in (0, 1)) else "shard"
        if mode not in ("shard", "replicate"):
            raise ArgumentError(f"multi_gpu={mode!r}: expected 'auto', 'shard' or 'replicate'")
        if self._expmv and mode == "replicate":
            raise ArgumentError("prop_method=Expmv has no replicated forward sweep: use multi_gpu='shard' (or 'auto')")
        self._replicated = mode == "replicate" and n_ranks_wanted > 1

        def make_engine(lo, hi):
            local_gens = sorted(set(int(g) for g in gen_of_traj[lo:hi]))
            remap = {g: i for i, g in enumerate(local_gens)}
            eng = KrotovCuda(
                tlist=tlist, H0=[H0[g] for g in local_gens], Hc=[Hc[g] for g in local_gens],
                gen_of_traj=np.array([remap[int(g)] for g in gen_of_traj[lo:hi]], np.int32),
                psi0=psi0[lo:hi], target=None if target is None else target[lo:hi], weight=weight[lo:hi],
                update_shape=S, lambda_a=lam, functional=functional, n_traj_global=N,
                store_fw=self.store_fw, device=device, force_path=int(self.kwargs.get("force_path", 0)),
                csr=bool(self.kwargs.get("csr_generators", False)), replicated_forward=self._replicated,
                propagator=B.PROP_EXPMV if self._expmv else B.PROP_CHEBY)
            return eng, local_gens

        emulate = int(self.kwargs.get("emulate_ranks", 0) or 0)
        if emulate > 1:
            # several ranks emulated on ONE device (tests / diagnostics): one handle per shard, one cooperative launch
            if comm is not None and world > 1:
                raise ArgumentError("`emulate_ranks` and a multi-rank `comm` exclude each other")
            from .engine import KrotovCudaGroup

            bounds = [(0, N)] * emulate if self._replicated else [shard_bounds(gen_of_traj, r, emulate) for r in range(emulate)]
            made = [make_engine(lo, hi) for lo, hi in bounds]
            self.engine = KrotovCudaGroup([m[0] for m in made], bounds, [m[1] for m in made], replicated=self._replicated)
            self._shard = (0, N)
            self._n_ranks = 1 if self._replicated else emulate
            self._H0, self._Hc = H0, Hc
        else:
            lo, hi = (0, N) if self._replicated else shard_bounds(gen_of_traj, rank, world)
            self._shard = (lo, hi)
            self._n_ranks = 1 if self._replicated else world
            self.engine, local_gens = make_engine(lo, hi)
            self._H0 = [H0[g] for g in local_gens]
            self._Hc = [Hc[g] for g in local_gens]
        if comm is not None and world > 1:
            comm.connect(self.engine)
        if self._term_ctrl is not None:
            self.engine.set_control_terms(self._term_ctrl)
        nonlinear = self._amp_poly is not None or self._amp_shape is not None or self._amp_sat is not None
        if nonlinear:
            self.engine.set_amplitudes(self._amp_poly, self._amp_shape)
        if self._amp_sat is not None:
            self.engine.set_amplitude_saturation(self._amp_sat)
        # ---- propagator settings of both directions (Chebyshev or Taylor) (init_prop: un-widened ranges of the guess pulses)
        adj = lambda m: m.conj().T.tocsr() if hasattr(m, "tocsr") else m.conj().T  # noqa: E731
        same = lambda a, b: (abs(a - b).max() == 0) if hasattr(a, "tocsr") else np.array_equal(a, b)  # noqa: E731
        terms = list(self._H0) + [h for row in self._Hc for h in row if h is not None]
        # Hermitian generators: both directions propagate with the same matrices, so they share their
        # spectral envelopes (see ChebyDirection)
        shared = {} if all(same(m, adj(m)) for m in terms) else None
        self._hermitian = shared is not None

        # ensembles on the persistent-kernel path: the spectral envelopes behind `reinit_prop!` are solved on the device
        # from the generator terms the handle holds (ChebyDirection uses it for Hermitian generators only, where both
        # directions propagate with the same matrices); KROTOV_HOST_ENVELOPE=1 keeps the threaded host solver
        device_envelope = None
        import os as _os
        if (hasattr(self.engine, "envelope_extremes") and d <= 32 and not _os.environ.get("KROTOV_HOST_ENVELOPE")
                and self.engine.info()["path"] == 1):
            device_envelope = self.engine.envelope_extremes

        def settings(pk, backward):
            H0s = [adj(h) for h in self._H0] if backward else self._H0
            Hcs = [[None if h is None else adj(h) for h in row] for row in self._Hc] if backward else self._Hc
            if self._expmv:
                return TaylorDirection(H0s, Hcs, tlist, backward, self._term_rows(self._init_pulses),
                                       amplitude_max=self._amp_abs_max if nonlinear else None)
            return ChebyDirection(
                H0s, Hcs, tlist, backward, self._term_rows(self._init_pulses),
                limit=pk.get("cheby_coeffs_limit", 1e-12), specrange_buffer=pk.get("specrange_buffer", 0.01),
                specrange_method=pk.get("specrange_method", "auto"), E_min=pk.get("E_min"), E_max=pk.get("E_max"),
                envelope_cache=shared if self._shared_envelope_ok(pk) else None,
                amplitude=self._amp_envelope_corners if nonlinear else None, device_envelope=device_envelope)

        self.fw_settings = settings(self.fw_prop_kwargs[0], False)
        self.bw_settings = settings(self.bw_prop_kwargs[0], True)
        self.fw_settings.push(self.engine, B.FORWARD)
        self.bw_settings.push(self.engine, B.BACKWARD)
        self._weight = weight
        self._target = target

    def _shared_envelope_ok(self, pk):
        """The shared cache is keyed by control ranges only, so both directions must also agree on how the
        envelope is computed."""
        other = self.bw_prop_kwargs[0] if pk is self.fw_prop_kwargs[0] else self.fw_prop_kwargs[0]
        return all(pk.get(k) == other.get(k) for k in ("specrange_method", "E_min", "E_max"))

    def _fetch_states(self):
        local = self.engine.states()
        if self.comm is not None and self.comm.world > 1 and not self._replicated:
            return self.comm.all_gather_rows(local, self.N)
        return local

    def _fetch_tau(self):
        local = self.engine.tau()
        if self.comm is not None and self.comm.world > 1 and not self._replicated:
            return self.comm.all_gather_rows(local, self.N)
        return local

    def close(self):
        self.engine.close()
