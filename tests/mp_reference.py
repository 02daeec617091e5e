"""An oracle-INDEPENDENT check of the Krotov loop: the two-level system of ``test/test_tls_optimization.jl:12-63``
optimised in 50-digit arithmetic (mpmath) with the EXACT propagator of every interval,

    exp(-i H dt) = cos(w dt) 1 - i sin(w dt) H / w,     H = -sz/2 + eps sx,  w = sqrt(1/4 + eps^2),

so that nothing of the recalled QuantumPropagators conventions of SURVEY.md Appendix A.1 (Chebyshev coefficients,
truncation rule, spectral range, buffer) enters.  What it does share with the oracles -- deliberately, these are the
lines of the reference under test -- is the loop of ``src/optimize.jl:279-371``: chi(T) = -dJ_T/d<psi| for J_T_sm,
backward propagation with the guess pulse storing chi(t_n), the sequential update
eps_new[n] = eps_old[n] + S[n]/lambda * Im<chi(t_n)|sx|psi(t_n)>, the running cost, the forward step with the updated
value; and the midpoint discretisation (first / last sample ON the grid ends).

Test infrastructure only.  Written without looking at oracle/krotov_oracle.py's propagators: a different number type,
a different propagator, a different code path."""
import mpmath as mp


def _blackman(t, t0, T, a=mp.mpf("0.16")):
    if t < t0 or t > T:
        return mp.mpf(0)
    x = (t - t0) / (T - t0)
    return (1 - a - mp.cos(2 * mp.pi * x) + a * mp.cos(4 * mp.pi * x)) / 2


def _flattop(t, T, t_rise):
    if t <= 0 or t >= T:
        return mp.mpf(0)
    if t <= t_rise:
        return _blackman(t, mp.mpf(0), 2 * t_rise)
    if t >= T - t_rise:
        return _blackman(t, T - 2 * t_rise, T)
    return mp.mpf(1)


def _step(psi, eps, dt):
    """psi <- exp(-i H dt) psi for H = -sz/2 + eps sx (closed form)."""
    w = mp.sqrt(mp.mpf(1) / 4 + eps * eps)
    c, s = mp.cos(w * dt), mp.sin(w * dt) / w
    a, b = psi
    # H psi = (-a/2 + eps b, eps a + b/2)
    return (c * a - 1j * s * (-a / 2 + eps * b), c * b - 1j * s * (eps * a + b / 2))


def tls_krotov_exact(iters=5, n_grid=501, dps=50, float_grid=True, amp_poly=None, amp_shape=None, lam=1, sigma=None):
    """J_T history, running costs and final pulses of the TLS optimisation in `dps`-digit arithmetic.

    float_grid: take the time grid and the guess pulse samples from their Float64 values (what both the reference
    and the oracles start from) so that the comparison isolates the arithmetic of the loop.

    sigma: None (first order) | a number | one number per time interval -- the second-order update of Reich, Ndong, Koch,
    J. Chem. Phys. 136, 104103 (2012): the overlap gains (sigma_n / 2) <psi_new(t_n) - psi_old(t_n)| mu |psi_new(t_n)>."""
    mp.mp.dps = dps
    T, t_rise, lam = mp.mpf(5), mp.mpf("0.3"), mp.mpf(lam)
    # non-linear amplitude: H = -sz/2 + a(eps, n) sx,  a = shape[n] * sum_p c_p eps^p;  mu = dH/d eps = a'(eps, n) sx is
    # evaluated at the GUESS value of the interval (src/optimize.jl:337)
    poly = None if amp_poly is None else [mp.mpf(float(c)) for c in amp_poly]
    shape = None if amp_shape is None else [mp.mpf(float(x)) for x in amp_shape]

    def amp(e, n):
        v = e if poly is None else sum(c * e**q for q, c in enumerate(poly))
        return v if shape is None else shape[n] * v

    def damp(e, n):
        v = mp.mpf(1) if poly is None else sum(q * c * e ** (q - 1) for q, c in enumerate(poly) if q > 0)
        return v if shape is None else shape[n] * v

    if float_grid:
        import numpy as np

        tl = [mp.mpf(float(x)) for x in np.linspace(0.0, 5.0, n_grid)]
    else:
        tl = [T * i / (n_grid - 1) for i in range(n_grid)]
    N_T = n_grid - 1

    def guess(t):
        if float_grid:
            import workloads as W

            return mp.mpf(float(0.2 * W.flattop(float(t), T=5.0, t_rise=0.3)))
        return mp.mpf("0.2") * _flattop(t, T, t_rise)

    # discretize_on_midpoints: first / last sample on the grid ends, interior on the interval midpoints
    def mid(i):
        if float_grid:
            return mp.mpf(float(tl[i]) + 0.5 * (float(tl[i + 1]) - float(tl[i])))
        return (tl[i] + tl[i + 1]) / 2

    eps = [guess(tl[0])] + [guess(mid(i)) for i in range(1, N_T - 1)] + [guess(tl[-1])]
    psi0 = (mp.mpc(1), mp.mpc(0))
    dts = [tl[n + 1] - tl[n] for n in range(N_T)]

    if sigma is not None:
        sig = [mp.mpf(float(x)) for x in sigma] if hasattr(sigma, "__len__") else [mp.mpf(float(sigma))] * N_T
    old_traj = []

    def forward(e):
        psi = psi0
        for n in range(N_T):
            old_traj.append(psi)
            psi = _step(psi, amp(e[n], n), dts[n])
        old_traj.append(psi)
        return psi

    psi = forward(eps)
    tau = psi[1]  # <target|psi>, target = (0, 1)
    J = [1 - abs(tau) ** 2]
    ga_hist = []
    for _ in range(iters):
        chi = (mp.mpc(0), tau)  # chi = (1/N^2)(sum tau) |tgt>, N = 1
        X = [None] * (N_T + 1)
        X[N_T] = chi
        for n in range(N_T - 1, -1, -1):  # exp(+i H^dagger dt) with the GUESS pulse
            chi = _step(chi, amp(eps[n], n), -dts[n])
            X[n] = chi
        new = list(eps)
        psi = psi0
        ga = mp.mpf(0)
        for n in range(N_T):
            c0, c1 = X[n]
            # <chi| sx |psi> = conj(c0) psi1 + conj(c1) psi0
            ov = mp.conj(c0) * psi[1] + mp.conj(c1) * psi[0]
            if sigma is not None:
                d0, d1 = psi[0] - old_traj[n][0], psi[1] - old_traj[n][1]
                ov += sig[n] / 2 * (mp.conj(d0) * psi[1] + mp.conj(d1) * psi[0])
                old_traj[n] = psi  # (slot n is not read again in this iteration)
            du = damp(eps[n], n) * mp.im(ov)
            alpha = mp.mpf(1) / lam  # S = 1
            new[n] = eps[n] + alpha * du
            ga += alpha * du * du * dts[n]
            psi = _step(psi, amp(new[n], n), dts[n])
        eps = new
        old_traj[N_T] = psi
        tau = psi[1]
        J.append(1 - abs(tau) ** 2)
        ga_hist.append(ga)
    return dict(J_T=[float(x) for x in J], J_T_mp=J, g_a_int=[float(x) for x in ga_hist], pulses=[float(x) for x in eps])


def krotov_exact_general(p, iters=2, dps=40, sigma=None, chi=None, J_T=None):
    """The Krotov loop of ``src/optimize.jl:279-371`` for ANY small problem in `dps`-digit arithmetic with the exact
    propagator of every interval (``mpmath.expm``): several trajectories and generators, several controls, complex /
    missing control operators, weights, non-uniform grids, non-Hermitian generators (the backward sweep uses the adjoint
    generator), all three built-in functionals.  `p` is only the CONTAINER of the Float64 inputs (``W.to_oracle(w)``:
    time grid, midpoint pulses, update shapes, lambda_a, matrices, states); none of its methods or of the oracle's code is
    used.  Returns J_T per iteration, the running costs and the final pulses as floats.

    sigma: None | one number per time interval -- second-order update, the overlap of interval n gains
    (sigma_n / 2) <psi_new(t_n) - psi_old(t_n)| mu |psi_new(t_n)> (any generator, any sigma(t): the general formula).

    chi, J_T: None (the built-in functional of ``p.functional``) or callables of the final-time states (`dps`-digit
    column vectors, one per trajectory) returning chi(T) (one column vector per trajectory) and J_T: a general
    boundary condition.  tau stays the overlap with the targets."""
    mp.mp.dps = dps
    N, d, L, N_T = p.psi0.shape[0], p.psi0.shape[1], len(p.pulses), len(p.tlist) - 1
    c = lambda z: mp.mpc(float(z.real), float(z.imag))  # noqa: E731
    mat = lambda M: mp.matrix([[c(M[i, j]) for j in range(d)] for i in range(d)])  # noqa: E731
    H0 = [mat(h) for h in p.H0]
    Hc = [[None if h is None else mat(h) for h in row] for row in p.Hc]
    gen = [int(g) for g in p.gen_of_traj]
    psi0 = [mp.matrix([c(x) for x in p.psi0[k]]) for k in range(N)]
    tgt = [mp.matrix([c(x) for x in p.target[k]]) for k in range(N)]
    w = [mp.mpf(1)] * N if p.weight is None else [mp.mpf(float(x)) for x in p.weight]
    dts = [mp.mpf(float(p.tlist[n + 1])) - mp.mpf(float(p.tlist[n])) for n in range(N_T)]
    eps = [[mp.mpf(float(x)) for x in row] for row in p.pulses]
    S = [[mp.mpf(float(x)) for x in row] for row in p.S]
    lam = [mp.mpf(float(x)) for x in p.lam]
    j = mp.mpc(0, 1)

    def H(g, vals):
        out = H0[g].copy()
        for l in range(L):
            if Hc[g][l] is not None:
                out += vals[l] * Hc[g][l]
        return out

    def vdot(a, b):
        return sum(mp.conj(a[i]) * b[i] for i in range(d))

    def taus(states):
        return [vdot(tgt[k], states[k]) for k in range(N)]

    def J_of(tau):
        if p.functional == "sm":
            return 1 - abs(sum(w[k] * tau[k] for k in range(N)) / N) ** 2
        if p.functional == "ss":
            return 1 - sum(w[k] * abs(tau[k]) ** 2 for k in range(N)) / N
        return 1 - mp.re(sum(w[k] * tau[k] for k in range(N))) / N

    def chi_of(tau):  # chi_k = -dJ_T/d<psi_k|
        if p.functional == "sm":
            s = sum(w[k] * tau[k] for k in range(N))
            return [(w[k] / N**2) * s * tgt[k] for k in range(N)]
        if p.functional == "ss":
            return [(w[k] / N) * tau[k] * tgt[k] for k in range(N)]
        return [(w[k] / (2 * N)) * tgt[k] for k in range(N)]

    gens = sorted(set(gen))
    sig = None if sigma is None else [mp.mpf(float(x)) for x in sigma]
    # non-linear amplitudes (data fields of the container only): control l enters as shape_l[n] * sum_q c_lq eps^q;
    # mu_l = dH/d eps_l is taken at the GUESS value of the interval (src/optimize.jl:337)
    poly = None if p.amp_poly is None else [None if c is None else [mp.mpf(float(x)) for x in c] for c in p.amp_poly]
    ashape = None if p.amp_shape is None else [[mp.mpf(float(x)) for x in row] for row in p.amp_shape]

    def amp(l, n, e):
        v = e if poly is None or poly[l] is None else sum(cq * e**q for q, cq in enumerate(poly[l]))
        return v if ashape is None else ashape[l][n] * v

    def damp(l, n, e):
        v = mp.mpf(1) if poly is None or poly[l] is None else sum(q * cq * e ** (q - 1) for q, cq in enumerate(poly[l]) if q > 0)
        return v if ashape is None else ashape[l][n] * v

    states = list(psi0)
    old = [[None] * (N_T + 1) for _ in range(N)]  # psi_k^(i)(t_n): the previous iteration's forward trajectory
    for n in range(N_T):
        for k in range(N):
            old[k][n] = states[k]
        U = {g: mp.expm(-j * dts[n] * H(g, [amp(l, n, eps[l][n]) for l in range(L)])) for g in gens}
        states = [U[gen[k]] * states[k] for k in range(N)]
    for k in range(N):
        old[k][N_T] = states[k]
    tau = taus(states)
    J, ga_hist = [J_of(tau) if J_T is None else J_T(states)], []
    for _ in range(iters):
        chi_T = chi_of(tau) if chi is None else chi(states)
        X = [[None] * (N_T + 1) for _ in range(N)]
        for k in range(N):
            X[k][N_T] = chi_T[k]
        for n in range(N_T - 1, -1, -1):  # backward with the adjoint generator under the GUESS pulses
            Ub = {g: mp.expm(j * dts[n] * H(g, [amp(l, n, eps[l][n]) for l in range(L)]).H) for g in gens}
            for k in range(N):
                X[k][n] = Ub[gen[k]] * X[k][n + 1]
        new = [list(row) for row in eps]
        ga = [mp.mpf(0)] * L
        states = list(psi0)
        for n in range(N_T):
            for l in range(L):
                du = mp.mpf(0)
                for k in range(N):
                    mu = Hc[gen[k]][l]
                    if mu is not None:
                        ov = vdot(X[k][n], mu * states[k])
                        if sig is not None:
                            ov += sig[n] / 2 * vdot(states[k] - old[k][n], mu * states[k])
                        du += mp.im(damp(l, n, eps[l][n]) * ov)
                alpha = S[l][n] / lam[l]
                new[l][n] = eps[l][n] + alpha * du
                ga[l] += alpha * du * du * dts[n]
            for k in range(N):
                old[k][n] = states[k]  # (slot n is not read again in this iteration)
            U = {g: mp.expm(-j * dts[n] * H(g, [amp(l, n, new[l][n]) for l in range(L)])) for g in gens}
            states = [U[gen[k]] * states[k] for k in range(N)]
        for k in range(N):
            old[k][N_T] = states[k]
        eps = new
        tau = taus(states)
        J.append(J_of(tau) if J_T is None else J_T(states))
        ga_hist.append(ga)
    return dict(J_T=[float(x) for x in J], g_a_int=[[float(x) for x in g] for g in ga_hist],
                pulses=[[float(x) for x in row] for row in eps],
                tau=[complex(float(mp.re(t)), float(mp.im(t))) for t in tau])


def exact_cases():
    """Small problems for ``krotov_exact_general``: name -> (workload factory, iterations).  Between them: several
    trajectories, two generators, a control one generator does not depend on, complex control operators, two controls,
    the three functionals, a non-Hermitian generator."""
    import numpy as np

    import workloads as W

    def two_generators():
        w = W.dummy_dense(d=5, n_traj=4, n_controls=2, n_grid=41, functional="ss", seed=31)
        rng = np.random.default_rng(32)
        A = rng.standard_normal((5, 5)) + 1j * rng.standard_normal((5, 5))
        w.H0 = [w.H0[0], 0.4 * (A + A.conj().T)]
        w.Hc = [w.Hc[0], [w.Hc[0][0] * 0.7, None]]
        w.gen_of_traj = np.array([0, 1, 0, 1])
        w.lambda_a = 0.2
        return w

    def non_hermitian():
        w = W.dummy_dense(d=4, n_traj=3, n_controls=1, n_grid=41, functional="re", seed=33)
        w.H0 = [w.H0[0] - 0.05j * np.diag(np.arange(4.0))]
        w.lambda_a = 0.3
        return w

    def nonlinear():
        w = two_generators()
        w.amp_poly = [[0.0, 1.0, 0.4], None]  # control 0 enters as eps + 0.4 eps^2
        w.amp_shape = [None, lambda t: 0.5 + 0.25 * t]  # control 1 as shape(t) * eps
        return w

    return {"c2_transmon_x_g101": (lambda: W.c2_transmon_x(n_grid=101), 3),
            "nonlinear_two_generators_d5": (nonlinear, 2),
            "two_generators_d5": (two_generators, 2),
            "non_hermitian_d4": (non_hermitian, 2)}
