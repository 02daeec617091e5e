"""`KrotovCuda`: thin object wrapper over one ``krotov_handle`` (one GPU, one shard of trajectories).

Everything numeric happens in ``libkrotov_cuda``; this class only marshals NumPy arrays to
the C ABI.  It is what the Julia shim's ``ccall`` layer would be (INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as B


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class KrotovCuda:
    def __init__(self, *, tlist, H0, Hc, gen_of_traj, psi0, target=None, weight=None, update_shape, lambda_a,
                 functional=B.CHI_HOST, n_traj_global=0, store_fw=False, device=0, force_path=0, csr=False,
                 replicated_forward=False, propagator=B.PROP_CHEBY):
        """H0: (n_gen, d, d) complex, Hc: (n_gen, L, d, d) complex with ``None`` entries allowed
        (as zeros + term_present=0); psi0/target: (N, d); update_shape: (L, N_T); lambda_a: (L,)."""
        lib = B.lib()
        self._lib = lib
        self._h = C.c_void_p()
        tlist = np.ascontiguousarray(tlist, np.float64)
        psi0 = np.ascontiguousarray(psi0, np.complex128)
        N, d = psi0.shape
        n_gen = len(H0)
        L = len(Hc[0])
        N_T = len(tlist) - 1
        present = np.ones((n_gen, 1 + L), np.uint8)
        for g in range(n_gen):
            for l in range(L):
                if Hc[g][l] is None:
                    present[g, 1 + l] = 0
        any_sparse = any(hasattr(m, "tocsr") for m in list(H0) + [x for row in Hc for x in row if x is not None])
        self.N, self.d, self.L, self.N_T, self.n_gen = N, d, L, N_T, n_gen
        rowptr = colind = None
        nnz = 0
        if any_sparse or csr:
            # KROTOV_GEN_CSR: one shared (union) pattern, values [n_gen][1+L][nnz]; nothing is densified
            import scipy.sparse as sp

            terms = [[sp.csr_matrix(H0[g], dtype=np.complex128)] +
                     [None if Hc[g][l] is None else sp.csr_matrix(Hc[g][l], dtype=np.complex128) for l in range(L)]
                     for g in range(n_gen)]
            keys = []
            for row in terms:
                for m in row:
                    if m is not None:
                        c = m.tocoo()
                        nz = c.data != 0
                        keys.append(c.row[nz].astype(np.int64) * d + c.col[nz])
            union = np.unique(np.concatenate(keys)) if keys else np.zeros(0, np.int64)
            rows, cols = union // d, union % d
            rowptr = np.zeros(d + 1, np.int64)
            np.add.at(rowptr, rows + 1, 1)
            rowptr = np.cumsum(rowptr).astype(np.int32)
            colind = cols.astype(np.int32)
            nnz = len(colind)
            vals = np.zeros((n_gen, 1 + L, nnz), np.complex128)
            for g, row in enumerate(terms):
                for t, m in enumerate(row):
                    if m is not None:
                        c = m.tocoo()
                        pos = np.searchsorted(union, c.row.astype(np.int64) * d + c.col)
                        ok = c.data != 0
                        np.add.at(vals[g, t], pos[ok], c.data[ok])
        else:
            vals = np.zeros((n_gen, 1 + L, d, d), np.complex128)
            for g in range(n_gen):
                vals[g, 0] = np.asarray(H0[g]).T  # column-major on the wire (Julia Matrix layout)
                for l in range(L):
                    if Hc[g][l] is not None:
                        vals[g, 1 + l] = np.asarray(Hc[g][l]).T
        gen = np.ascontiguousarray(gen_of_traj, np.int32)
        S = np.ascontiguousarray(update_shape, np.float64).reshape(L, N_T)
        lam = np.ascontiguousarray(lambda_a, np.float64).reshape(L)
        tgt = None if target is None else np.ascontiguousarray(target, np.complex128).reshape(N, d)
        w = None if weight is None else np.ascontiguousarray(weight, np.float64).reshape(N)
        p = B.Problem()
        p.struct_size = C.sizeof(B.Problem)
        p.d, p.n_traj, p.n_ctrl, p.n_steps, p.n_gen = d, N, L, N_T, n_gen
        p.gen_format, p.nnz = (B.GEN_CSR, nnz) if rowptr is not None else (B.GEN_DENSE_COLMAJOR, 0)
        p.csr_rowptr, p.csr_colind = _ptr(rowptr), _ptr(colind)
        p.tlist, p.gen_of_traj = _ptr(tlist), _ptr(gen)
        p.gen_values, p.term_present = _ptr(vals), _ptr(present)
        p.psi0, p.target, p.weight = _ptr(psi0), _ptr(tgt), _ptr(w)
        p.update_shape, p.lambda_a = _ptr(S), _ptr(lam)
        p.functional, p.n_traj_global = int(functional), int(n_traj_global)
        p.store_fw, p.device, p.force_path = int(bool(store_fw)), int(device), int(force_path)
        p.replicated_forward = int(bool(replicated_forward))
        p.propagator = int(propagator)
        rc = lib.krotov_create(C.byref(p), C.byref(self._h))
        if rc != B.KROTOV_OK:
            msg = lib.krotov_last_error(None).decode()
            self._h = C.c_void_p()
            raise B.KrotovCudaError(rc, msg)

    # -- plumbing -------------------------------------------------------------------------
    def _check(self, rc):
        if rc != B.KROTOV_OK:
            raise B.KrotovCudaError(rc, self._lib.krotov_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.krotov_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        i = B.Info()
        self._check(self._lib.krotov_get_info(self._h, C.byref(i)))
        return {k: getattr(i, k) for k, _ in B.Info._fields_ if not k.startswith("reserved")}

    # -- propagator settings --------------------------------------------------------------
    def set_cheby(self, direction, dt_class_of_step, dt_of_class, E_min, Delta, m, tab):
        """m: (n_gen, n_dt_class) coefficient counts; tab: (n_gen, n_dt_class, m_max) zero-padded coefficients."""
        n_gen, ndtc = self.n_gen, len(dt_of_class)
        m = np.ascontiguousarray(m, np.int32).reshape(n_gen, ndtc)
        tab = np.ascontiguousarray(tab, np.float64).reshape(n_gen, ndtc, -1)
        m_max = int(tab.shape[2])
        dtc = np.ascontiguousarray(dt_class_of_step, np.int32)
        dts = np.ascontiguousarray(dt_of_class, np.float64)
        Emin = np.ascontiguousarray(E_min, np.float64).reshape(n_gen)
        Dl = np.ascontiguousarray(Delta, np.float64).reshape(n_gen)
        self._check(self._lib.krotov_set_cheby(self._h, int(direction), ndtc, _ptr(dtc), _ptr(dts), _ptr(Emin),
                                               _ptr(Dl), _ptr(m), _ptr(tab), m_max))

    def set_taylor(self, direction, dt_class_of_step, dt_of_class, mu, scale, s, m, tab):
        """Taylor settings of a ``propagator=PROP_EXPMV`` handle (``krotov_set_taylor``): mu, scale: (n_gen,); s, m:
        (n_gen, n_dt_class) repeats and terms; tab: (n_gen, n_dt_class, m_max) zero-padded coefficients."""
        n_gen, ndtc = self.n_gen, len(dt_of_class)
        s = np.ascontiguousarray(s, np.int32).reshape(n_gen, ndtc)
        m = np.ascontiguousarray(m, np.int32).reshape(n_gen, ndtc)
        tab = np.ascontiguousarray(tab, np.float64).reshape(n_gen, ndtc, -1)
        dtc = np.ascontiguousarray(dt_class_of_step, np.int32)
        dts = np.ascontiguousarray(dt_of_class, np.float64)
        mu = np.ascontiguousarray(mu, np.float64).reshape(n_gen)
        sc = np.ascontiguousarray(scale, np.float64).reshape(n_gen)
        self._check(self._lib.krotov_set_taylor(self._h, int(direction), ndtc, _ptr(dtc), _ptr(dts), _ptr(mu), _ptr(sc),
                                                _ptr(s), _ptr(m), _ptr(tab), int(tab.shape[2])))

    def set_amplitudes(self, poly=None, shape=None):
        """Non-linear amplitudes ``a_l(eps, n) = shape[l][n] * sum_p poly[l][p] eps^p`` (``krotov_set_amplitudes``);
        ``poly``: (L, degree+1) or None, ``shape``: (L, N_T) or None."""
        deg = 1
        if poly is not None:
            poly = np.ascontiguousarray(poly, np.float64).reshape(self.L, -1)
            deg = poly.shape[1] - 1
        if shape is not None:
            shape = np.ascontiguousarray(shape, np.float64).reshape(self.L, self.N_T)
        self._check(self._lib.krotov_set_amplitudes(self._h, int(deg), _ptr(poly), _ptr(shape)))

    def set_amplitude_saturation(self, s=None):
        """Saturating amplitudes (``krotov_set_amplitude_saturation``): ``s``: (L,) or None.  Where ``s[l] > 0`` the
        amplitude polynomial of control l is evaluated at ``tanh(s[l] * eps)``; None restores s = 0 everywhere."""
        if s is not None:
            s = np.ascontiguousarray(s, np.float64).reshape(self.L)
        self._check(self._lib.krotov_set_amplitude_saturation(self._h, _ptr(s)))

    def set_control_terms(self, control_of_term=None):
        """Tie control terms to controls (``krotov_set_control_terms``): ``control_of_term``: (L,) control id of every
        term, numbered in order of first appearance; None = every term is its own control."""
        if control_of_term is not None:
            control_of_term = np.ascontiguousarray(control_of_term, np.int32).reshape(self.L)
        self._check(self._lib.krotov_set_control_terms(self._h, _ptr(control_of_term)))

    # -- hot path -------------------------------------------------------------------------
    def forward(self, pulses):
        p = np.ascontiguousarray(pulses, np.float64).reshape(self.L, self.N_T)
        self._check(self._lib.krotov_forward(self._h, _ptr(p)))

    def set_chi(self, chi):
        c = np.ascontiguousarray(chi, np.complex128).reshape(self.N, self.d)
        self._check(self._lib.krotov_set_chi(self._h, _ptr(c)))

    def set_chi_coeffs(self, coef):
        c = np.ascontiguousarray(coef, np.complex128).reshape(self.N)
        self._check(self._lib.krotov_set_chi_coeffs(self._h, _ptr(c)))

    def iterate(self, guess_pulses, out_pulses=None):
        g = np.ascontiguousarray(guess_pulses, np.float64).reshape(self.L, self.N_T)
        out = np.empty((self.L, self.N_T), np.float64) if out_pulses is None else out_pulses
        ga = np.empty(self.L, np.float64)
        self._check(self._lib.krotov_iterate(self._h, _ptr(g), _ptr(out), _ptr(ga)))
        return out, ga

    # -- results --------------------------------------------------------------------------
    def states(self):
        out = np.empty((self.N, self.d), np.complex128)
        self._check(self._lib.krotov_get_states(self._h, _ptr(out)))
        return out

    def tau(self):
        out = np.empty(self.N, np.complex128)
        self._check(self._lib.krotov_get_tau(self._h, _ptr(out)))
        return out

    def storage(self, which, k, n0=0, n1=None):
        n1 = self.N_T + 1 if n1 is None else n1
        out = np.empty((n1 - n0, self.d), np.complex128)
        self._check(self._lib.krotov_get_storage(self._h, int(which), int(k), int(n0), int(n1), _ptr(out)))
        return out

    def envelope_extremes(self, corners):
        """``(e_min, e_max)`` per generator over the amplitude corners ``(n_corner, L)``, solved on the device from the
        generator terms the handle holds (``krotov_envelope_extremes_device``); raises where the path has no device
        solver."""
        amps = np.ascontiguousarray(corners, np.float64).reshape(-1, self.L)
        lo, hi = np.empty(self.n_gen, np.float64), np.empty(self.n_gen, np.float64)
        self._check(self._lib.krotov_envelope_extremes_device(self._h, amps.shape[0], _ptr(amps), _ptr(lo), _ptr(hi)))
        return lo, hi

    def profile(self, cta=-1):
        out = np.zeros(8, np.int64)
        self._check(self._lib.krotov_get_profile(self._h, int(cta), _ptr(out)))
        names = ["backward", "forward", "wait_pulse", "comm_wait_partials", "comm_reduce", "comm_gather", "overlap", "fw_step_total"]
        return dict(zip(names, out.tolist()))

    # -- multi-GPU ------------------------------------------------------------------------
    def comm_export(self):
        buf = (C.c_ubyte * B.COMM_DESC_BYTES)()
        self._check(self._lib.krotov_comm_export(self._h, buf))
        return bytes(buf)

    def comm_connect(self, rank, world, descs):
        blob = b"".join(descs)
        assert len(blob) == world * B.COMM_DESC_BYTES
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._check(self._lib.krotov_comm_connect(self._h, int(rank), int(world), buf))


class KrotovCudaGroup:
    """Several ranks EMULATED on one device behind the interface of one :class:`KrotovCuda` (tests and diagnostics).

    Every rank is a real handle holding its shard of the trajectories; ``krotov_group_connect`` wires their mailboxes
    and cross-rank accumulators together in-process and ``krotov_group_iterate`` runs all ranks' CTAs in ONE
    cooperative launch, so the multi-rank exchange protocols of the persistent kernel can be exercised (and compared
    with a one-rank run) on a single-GPU box.  ``bounds[r] = (lo, hi)``: trajectories of rank r; ``gens[r]``: indices
    (into the caller's generator list) of the generators rank r holds, in the rank's local order."""

    def __init__(self, engines, bounds, gens, replicated=False):
        """replicated: every engine holds ALL trajectories (replicated forward sweep, sharded backward sweep): arrays are
        passed whole to every rank and read back from rank 0."""
        self.engines, self.bounds, self.gens = list(engines), list(bounds), [np.asarray(g, int) for g in gens]
        self.replicated = bool(replicated)
        e0 = self.engines[0]
        self._lib = e0._lib
        self.N = e0.N if replicated else sum(e.N for e in self.engines)
        self.d, self.L, self.N_T = e0.d, e0.L, e0.N_T
        self.n_gen = len(self.gens[0]) if replicated else sum(len(g) for g in self.gens)
        self.world = len(self.engines)
        self.pulses_all = None  # every rank's copy of the last new pulses: (world, L, N_T)
        arr = (C.c_void_p * self.world)(*[e._h for e in self.engines])
        self._handles = arr
        rc = self._lib.krotov_group_connect(arr, self.world)
        if rc != B.KROTOV_OK:
            raise B.KrotovCudaError(rc, "; ".join(self._lib.krotov_last_error(e._h).decode() for e in self.engines))

    def close(self):
        for e in self.engines:
            e.close()

    def info(self):
        out = self.engines[0].info()
        out["grid_blocks"] = sum(e.info()["grid_blocks"] for e in self.engines)
        out["fallback_steps"] = max(e.info()["fallback_steps"] for e in self.engines)
        out["ranks"] = self.world
        return out

    def set_cheby(self, direction, dt_class_of_step, dt_of_class, E_min, Delta, m, tab):
        E_min, Delta = np.asarray(E_min), np.asarray(Delta)
        m, tab = np.asarray(m), np.asarray(tab)
        for e, g in zip(self.engines, self.gens):
            e.set_cheby(direction, dt_class_of_step, dt_of_class, E_min[g], Delta[g], m[g], tab[g])  # (replicated: g = all)

    def set_taylor(self, direction, dt_class_of_step, dt_of_class, mu, scale, s, m, tab):
        mu, scale, s, m, tab = (np.asarray(a) for a in (mu, scale, s, m, tab))
        for e, g in zip(self.engines, self.gens):
            e.set_taylor(direction, dt_class_of_step, dt_of_class, mu[g], scale[g], s[g], m[g], tab[g])

    def set_amplitudes(self, poly=None, shape=None):
        for e in self.engines:
            e.set_amplitudes(poly, shape)

    def set_amplitude_saturation(self, s=None):
        for e in self.engines:
            e.set_amplitude_saturation(s)

    def set_control_terms(self, control_of_term=None):
        for e in self.engines:
            e.set_control_terms(control_of_term)

    def forward(self, pulses):
        for e in self.engines:  # no cross-rank dependency in a plain forward sweep
            e.forward(pulses)

    def set_chi(self, chi):
        chi = np.asarray(chi)
        for e, (lo, hi) in zip(self.engines, self.bounds):
            e.set_chi(chi[lo:hi])

    def set_chi_coeffs(self, coef):
        coef = np.asarray(coef)
        for e, (lo, hi) in zip(self.engines, self.bounds):
            e.set_chi_coeffs(coef[lo:hi])

    def iterate(self, guess_pulses, out_pulses=None):
        g = np.ascontiguousarray(guess_pulses, np.float64).reshape(self.L, self.N_T)
        allp = np.empty((self.world, self.L, self.N_T), np.float64)
        ga = np.empty((self.world, self.L), np.float64)
        rc = self._lib.krotov_group_iterate(self._handles, self.world, _ptr(g), _ptr(allp), _ptr(ga))
        if rc != B.KROTOV_OK:
            raise B.KrotovCudaError(rc, "; ".join(self._lib.krotov_last_error(e._h).decode() for e in self.engines))
        self.pulses_all, self.g_a_all = allp, ga
        if out_pulses is not None:
            out_pulses[...] = allp[0]
            return out_pulses, ga[0]
        return allp[0].copy(), ga[0].copy()

    def states(self):
        if self.replicated:
            return self.engines[0].states()
        return np.concatenate([e.states() for e in self.engines], axis=0)

    def tau(self):
        if self.replicated:
            return self.engines[0].tau()
        return np.concatenate([e.tau() for e in self.engines], axis=0)

    def envelope_extremes(self, corners):
        """Device-side spectral envelopes of all generators of the group (every rank solves the ones it holds)."""
        if self.replicated:
            return self.engines[0].envelope_extremes(corners)
        lo, hi = np.empty(self.n_gen, np.float64), np.empty(self.n_gen, np.float64)
        for e, g in zip(self.engines, self.gens):
            lo[g], hi[g] = e.envelope_extremes(corners)
        return lo, hi

    def states_all(self):
        """Final states of EVERY rank (replicated mode: they must be identical)."""
        return [e.states() for e in self.engines]

    def storage(self, which, k, n0=0, n1=None):
        for e, (lo, hi) in zip(self.engines, self.bounds):
            if lo <= k < hi:
                return e.storage(which, k - lo, n0, n1)
        raise IndexError(k)

    def profile(self, cta=-1):
        return self.engines[0].profile(cta)
