"""NumPy restatement of the device's truncated-Taylor step (``taylor_step`` in warp_kernel.cuh, ``prop_method=Expmv``)
and an oracle-backed engine that propagates with it -- TEST INFRASTRUCTURE.

``ExpmvOracleEngine`` is the oracle engine of tied control terms (``terms_reference.TermsOracleEngine``) with
``set_taylor`` and ``set_amplitude_saturation``: the settings the host driver pushes (``expmv.py``'s
``TaylorDirection``: shift, row scale, (m, s), coefficients, dt classes) are the ones the propagators USE, so the CPU
tests exercise the host's parameter choice and its re-derivation on control-range events."""
import numpy as np

from oracle import krotov_oracle as O
from terms_reference import TermsOracleEngine


def liouvillian(H, cops):
    """G with d vec(rho)/dt = -i G vec(rho) (column-stacked vec): G = L_H + i D for the Lindblad equation."""
    d = H.shape[0]
    I = np.eye(d)
    G = np.kron(I, H) - np.kron(H.T, I)
    for c in cops:
        cd = c.conj().T
        G = G + 1j * (np.kron(c.conj(), c) - 0.5 * np.kron(I, cd @ c) - 0.5 * np.kron((cd @ c).T, I))
    return G


def taylor_step(Hmat, v, dt, mu, scale, m, s, coeffs):
    """One interval as the device computes it: rows R = -i scale (H - mu), s repeats of e^{-i mu dt/s} sum_j c_j R^j v."""
    R = -1j * scale * (Hmat - mu * np.eye(Hmat.shape[0]))
    ph = np.exp(-1j * mu * dt / s)
    for _ in range(s):
        out = coeffs[0] * v
        vj = v
        for j in range(1, m):
            vj = R @ vj
            out = out + coeffs[j] * vj
        v = ph * out
    return v


def step_with_host_params(Hmat, v, dt, nu=None, theta_cap=None):
    """`taylor_step` with the parameters TaylorDirection chooses for a generator whose norm rate is nu (default: the
    1-norm of H - mu itself)."""
    from krotov_jl_b200 import expmv as E

    mu = E.generator_shift(Hmat)
    if nu is None:
        nu = E._norm1(Hmat - mu * np.eye(Hmat.shape[0]))
    scale = 1.0 / nu if nu > 0 else 1.0
    kw = {} if theta_cap is None else dict(theta_cap=theta_cap)
    m, s = E.taylor_params(abs(dt) * nu, **kw)
    return taylor_step(Hmat, v, dt, mu, scale, m, s, E.taylor_coeffs(dt / (scale * s), m)), (m, s)


class ExpmvPropagator(O._PWCPropagator):
    """Piecewise propagator of the oracle that steps with `taylor_step` and the tables last pushed for its direction."""

    def __init__(self, H0, Hc, tlist, parameters, backward, problem, tables, g):
        super().__init__(H0, Hc, tlist, parameters, backward, problem)
        self.tables, self.g = tables, g

    def reinit_prop(self, state, transform=None):
        self.state = np.array(state, dtype=complex)
        self._reset_time()

    def prop_step(self):
        ni, dt = self._interval_and_dt()
        t = self.tables
        c = int(t["dtc"][ni])
        assert t["dts"][c] == dt
        ops, cf = self._ops_coeffs(ni)
        Hmat = sum(co * op for op, co in zip(ops, cf))
        m, s = int(t["m"][self.g, c]), int(t["s"][self.g, c])
        self.state = taylor_step(Hmat, self.state, dt, t["mu"][self.g], t["scale"][self.g], m, s, t["tab"][self.g, c])
        self._advance()
        return self.state


class ExpmvOracleEngine(TermsOracleEngine):
    """Oracle engine whose propagators use the Taylor settings pushed through ``set_taylor`` (tied terms, non-linear and
    saturating amplitudes as in the Chebyshev test engines)."""

    pushed = []  # (direction, m * s per generator and class) of every push the tests' engines received

    def __init__(self, **kw):
        super().__init__(**kw)
        self.tables = [None, None]

    def set_taylor(self, direction, dtc, dts, mu, scale, s, m, tab):
        self.tables[int(direction)] = dict(dtc=np.asarray(dtc), dts=np.asarray(dts), mu=np.asarray(mu),
                                           scale=np.asarray(scale), s=np.asarray(s), m=np.asarray(m), tab=np.asarray(tab))
        ExpmvOracleEngine.pushed.append((int(direction), np.asarray(m) * np.asarray(s)))

    def set_amplitude_saturation(self, s=None):
        from sat_reference import sat_problem

        self.p = sat_problem(self.p, s)

    def _make(self, pulses):
        self.p.pulses = np.array(pulses, float).reshape(self.L, self.N_T)
        self.wrk = O.OracleWrk(self.p, prop_method="expm", store_fw=self.store_fw)
        p, w = self.p, self.wrk
        w.fw_propagators, w.bw_propagators = [], []
        for k in range(p.N):
            g = int(p.gen_of_traj[k])
            H0, Hc = p.H0[g], p.Hc[g]
            Hca = [None if h is None else h.conj().T for h in Hc]
            w.fw_propagators.append(ExpmvPropagator(H0, Hc, w.tlist, w.pulses0, False, p, self.tables[0], g))
            w.bw_propagators.append(ExpmvPropagator(H0.conj().T, Hca, w.tlist, w.pulses0, True, p, self.tables[1], g))
        self._bufs = [w.pulses0, w.pulses1]

    def iterate(self, guess_pulses, out_pulses=None):
        # the propagators hold the tables of the sweep they were made for: refresh them with the latest pushes
        if self.wrk is not None:
            for props, t in ((self.wrk.fw_propagators, self.tables[0]), (self.wrk.bw_propagators, self.tables[1])):
                for pr in props:
                    pr.tables = t
        return super().iterate(guess_pulses, out_pulses)


def damped_qubit(gammas=(1.0, 2.0), n_grid=41, T=4.0):
    """Driven qubit with amplitude damping in Liouville space (d = 4): H = -sz/2 + eps(t) sx, L = sqrt(gamma) s_-, one
    generator per gamma and one density-matrix trajectory per generator (|0><0| -> |1><1| and |+><+| -> |-><-|), J_T_re."""
    import workloads as W

    sx = np.array([[0, 1], [1, 0]], complex)
    sz = np.diag([1.0, -1.0]).astype(complex)
    sm = np.array([[0, 1], [0, 0]], complex)
    I2 = np.eye(2)
    ctrl = np.kron(I2, sx) - np.kron(sx.T, I2)  # the drive's Liouvillian (Hermitian)
    vec = lambda r: r.reshape(-1, order="F")  # noqa: E731  (column-stacked)
    plus, minus = np.array([1, 1]) / np.sqrt(2), np.array([1, -1]) / np.sqrt(2)
    rhos = [(np.diag([1.0, 0.0]), np.diag([0.0, 1.0])), (np.outer(plus, plus), np.outer(minus, minus))]
    n = len(gammas)
    return W.Workload(
        name="damped-qubit", tlist=np.linspace(0.0, T, n_grid),
        H0=[liouvillian(-0.5 * sz, [np.sqrt(g) * sm]) for g in gammas], Hc=[[ctrl] for _ in gammas],
        gen_of_traj=np.arange(n), psi0=np.array([vec(rhos[k % 2][0]) for k in range(n)], complex),
        target=np.array([vec(rhos[k % 2][1]) for k in range(n)], complex),
        controls=[lambda t: 0.3 * W.flattop(t, T=T, t_rise=0.3 * T)], update_shape=lambda t: W.flattop(t, T=T, t_rise=0.3 * T),
        lambda_a=2.0, functional="re")


def damped_ensemble(n_samples=300, n_grid=51, T=4.0, seed=5):
    """`damped_qubit` over a spread of decay rates (one generator per sample): enough trajectories for several CTAs."""
    gammas = np.random.default_rng(seed).uniform(0.2, 2.0, n_samples)
    return damped_qubit(tuple(gammas), n_grid=n_grid, T=T)
