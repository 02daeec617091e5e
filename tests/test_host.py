"""Host-side logic of the product, without a GPU: the reference's API semantics, error behaviour,
the C-ABI export surface, sharding, and a world_size=2 gloo run of the plumbing."""
import ctypes
import io
import os
import re
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

import krotov_jl_b200 as K
import workloads as W
from util import to_problem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- C ABI surface -----------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "krotov_cuda.h")).read()
    declared = set(re.findall(r"^(?:int|const char \*)\s*(krotov_\w+)\(", hdr, flags=re.M))
    assert len(declared) >= 15
    lib = ctypes.CDLL(K._lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/krotov_cuda.h but not exported"
    assert declared == set(K._lib.EXPORTS)
    assert lib.krotov_abi_version() == 1


def test_problem_struct_layout_matches_header():
    # krotov_create rejects a struct of the wrong size: proves the ctypes mirror and the header agree
    lib = K._lib.lib()
    p = K._lib.Problem()
    p.struct_size = ctypes.sizeof(K._lib.Problem) - 4
    h = ctypes.c_void_p()
    assert lib.krotov_create(ctypes.byref(p), ctypes.byref(h)) == 1
    assert b"struct_size" in lib.krotov_last_error(None)


def test_create_without_gpu_fails_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    w = W.c1_tls()
    with pytest.raises(K.KrotovCudaError) as ei:
        K.optimize(to_problem(w, iter_stop=1), method=K.Krotov)
    assert "KROTOV_ERR_CUDA" in str(ei.value)  # no silent CPU fallback


# ---- reference error behaviour -------------------------------------------------------------------
def test_no_controls_error_message():
    """test/test_empty_optimization.jl:31-32."""
    rng = np.random.default_rng(1)
    H = rng.standard_normal((10, 10))
    H = H + H.T
    traj = [K.Trajectory(np.ones(10) / np.sqrt(10), K.hamiltonian(H), target_state=np.eye(10)[0])]
    assert len(K.get_controls(traj)) == 0
    problem = K.ControlProblem(traj, np.arange(1001.0), pulse_options={})
    with pytest.raises(K.ErrorException, match="no controls in trajectories: cannot optimize"):
        K.optimize(problem, method=K.Krotov)


def test_argument_errors():
    w = W.c1_tls()
    with pytest.raises(K.ArgumentError, match="must be passed the functional `J_T`"):
        K.optimize(to_problem(w, J_T=None, iter_stop=1).__class__(to_problem(w).trajectories, w.tlist,
                                                                   prop_method=K.Cheby, lambda_a=1.0), method=K.Krotov)
    with pytest.raises(K.ArgumentError, match="superseded by the `callback` argument"):
        K.optimize(to_problem(w, update_hook=lambda *a: None), method=K.Krotov)
    with pytest.raises(K.ArgumentError, match="Cheby"):
        K.optimize(to_problem(w, prop_method="ExpProp"), method=K.Krotov)
    with pytest.raises(K.ArgumentError, match="propagation method must be specified"):
        p = to_problem(w)
        del p.kwargs["prop_method"]
        K.optimize(p, method=K.Krotov)
    with pytest.raises(K.ErrorException, match="pulse_options must be defined for all controls"):
        K.optimize(to_problem(w, pulse_options=K.IdDict()), method=K.Krotov)
    with pytest.raises(K.ArgumentError, match="store_iter_info"):
        K.optimize(to_problem(w, print_iters=True, store_iter_info=["nope"]), method=K.Krotov)


# ---- controls / shapes ---------------------------------------------------------------------------
def test_discretize_semantics():
    t = np.linspace(0, 5, 501)
    eps = lambda x: 0.2 * K.flattop(x, T=5, t_rise=0.3, func="blackman")  # noqa: E731
    mid = K.discretize_on_midpoints(eps, t)
    assert len(mid) == 500 and mid[0] == 0.0 and mid[-1] == 0.0
    assert mid[10] == eps(t[10] + 0.5 * (t[11] - t[10]))
    v = np.arange(500.0)
    c = K.discretize_on_midpoints(v, t)
    assert c is not v and np.array_equal(c, v)  # must copy (test_pulse_optimization.jl:42)
    g = K.discretize(v, t)
    assert len(g) == 501 and g[0] == v[0] and g[-1] == v[-1] and g[7] == 0.5 * (v[6] + v[7])
    back = K.discretize_on_midpoints(g, t)
    assert len(back) == 500 and np.abs(back - v).max() < 1e-9  # exact inverse of `discretize`
    # same numbers as the oracle's independent restatement
    from oracle import krotov_oracle as O

    ref = O.discretize_on_midpoints(lambda x: 0.2 * O.flattop(x, T=5, t_rise=0.3), t)
    assert np.abs(mid - ref).max() < 1e-15  # (the two Blackman formulas round differently in the last bit)


def test_get_controls_by_identity_and_derivs():
    f = lambda t: 1.0  # noqa: E731
    g = lambda t: 1.0  # noqa: E731
    sx = np.array([[0, 1], [1, 0]], complex)
    sz = np.diag([1.0, -1.0]).astype(complex)
    H1 = K.hamiltonian(sz, (sx, f))
    H2 = K.hamiltonian(sz, (sx, f), (sz, g))
    trajs = [K.Trajectory([1, 0], H1), K.Trajectory([1, 0], H2)]
    ctr = K.get_controls(trajs)
    assert len(ctr) == 2 and ctr[0] is f and ctr[1] is g
    d1 = K.get_control_derivs(H1, ctr)
    assert np.array_equal(d1[0], sx) and d1[1] is None  # `nothing` for a control the generator lacks
    assert isinstance(K.hamiltonian(sz), np.ndarray)  # no controls -> bare matrix


def test_cheby_settings_match_oracle_bits():
    from oracle import krotov_oracle as O

    w = W.c3_two_transmon(n_grid=101)
    p = W.to_oracle(w)
    pulses = [p.pulses[0].copy(), p.pulses[1].copy()]
    for backward in (False, True):
        H0 = [h.conj().T for h in p.H0] if backward else p.H0
        Hc = [[h.conj().T for h in row] for row in p.Hc] if backward else p.Hc
        mine = K.cheby.ChebyDirection(H0, Hc, p.tlist, backward, pulses)
        ref = O.ChebyPropagator(H0[0], Hc[0], p.tlist, pulses, backward)
        assert mine.E_min[0] == ref.E_min and mine.Delta[0] == ref.Delta
        assert np.array_equal(mine.coeffs[0][0], ref.coeffs)
        assert mine.reinit(pulses) is True  # first reinit widens to 5x
        ref.reinit_prop(p.psi0[0], O.transform_control_ranges)
        assert mine.Delta[0] == ref.Delta and np.array_equal(mine.coeffs[0][0], ref.coeffs)
        assert mine.reinit(pulses) is False
        assert mine.reinit([3.0 * pulses[0], pulses[1]]) is True  # 2 x 3 > 5: leaves the stored range
        assert len(mine.dt_of_class) >= 1 and (np.sign(mine.dt_of_class) == (-1 if backward else 1)).all()
    assert K.transform_control_ranges(None, -1.0, 2.0, True) == (-2.0, 4.0)


def test_coefficient_tables_with_hint_and_shared_between_directions():
    """The Bessel table sized from the previous coefficient count holds the numbers of the scalar function (and grows when
    the hint is too small); the two directions of a Hermitian problem share one table per (radii, |dt|)."""
    Deltas = np.array([3.1, 7.7, 12.9, 0.4])
    full, m_full = K.cheby.cheby_coeffs_table(Deltas, 0.37)
    for hint in (1, 3, int(m_full.max()), 40):
        a, m = K.cheby.cheby_coeffs_table(Deltas, 0.37, m_hint=hint)
        assert np.array_equal(m, m_full) and np.array_equal(a, full)
    for g, D in enumerate(Deltas):
        assert np.array_equal(full[g, : m_full[g]], K.cheby.cheby_coeffs(D, 0.37))
    w = W.c3_two_transmon(n_grid=41)
    p = W.to_oracle(w)
    shared = {}
    fw = K.cheby.ChebyDirection(p.H0, p.Hc, p.tlist, False, p.pulses, envelope_cache=shared)
    bw = K.cheby.ChebyDirection(p.H0, p.Hc, p.tlist, True, p.pulses, envelope_cache=shared)
    assert fw._tables is bw._tables and len(fw._tables) == 1  # the backward direction found the forward one's table
    assert np.array_equal(fw.coeff_table, bw.coeff_table)
    alone = K.cheby.ChebyDirection(p.H0, p.Hc, p.tlist, True, p.pulses)
    assert np.array_equal(alone.coeff_table, bw.coeff_table) and np.array_equal(alone.coeff_count, bw.coeff_count)


def test_result_layout():
    names = [f.name for f in K.KrotovResult.__dataclass_fields__.values()]
    assert names == ["tlist", "iter_start", "iter_stop", "iter", "secs", "tau_vals", "J_T", "J_T_prev",
                     "guess_controls", "optimized_controls", "states", "start_local_time", "end_local_time",
                     "records", "converged", "message"]  # src/result.jl:34-51
    r = K.KrotovResult.from_problem(to_problem(W.c1_tls(), iter_start=10, iter_stop=12))
    assert (r.iter_start, r.iter_stop, r.iter, r.message, r.converged) == (10, 12, 10, "in progress", False)
    assert len(r.guess_controls[0]) == 501 and r.optimized_controls[0] is not r.guess_controls[0]
    assert repr(r) == "KrotovResult<in progress>" and "Number of trajectories: 1" in str(r)


def test_iteration_table_format():
    """Header string and column formats of src/optimize.jl:448-492 (pinned by test_iterations.jl:71-74)."""

    class R:
        J_T, J_T_prev, secs = 0.9514, 0.0, 0.21

    class Wk:
        result, g_a_int, kwargs = R(), np.array([0.0]), {"iter_stop": 5}

    pr = K.make_krotov_print_iters(store_iter_info=["iter.", "J_T"])
    buf = io.StringIO()
    with redirect_stdout(buf):
        rec0 = pr(Wk(), 0)
        Wk.result.J_T, Wk.result.J_T_prev, Wk.g_a_int = 0.7236, 0.9514, np.array([0.0671])
        rec1 = pr(Wk(), 1)
    lines = buf.getvalue().splitlines()
    assert lines[0] == " iter.        J_T   ∫gₐ(t)dt          J       ΔJ_T         ΔJ    secs"
    assert lines[1] == "     0   9.51e-01   0.00e+00   9.51e-01        n/a        n/a     0.2"
    assert lines[2] == "     1   7.24e-01   6.71e-02   7.91e-01  -2.28e-01  -1.61e-01     0.2"
    assert rec0 == (0, 0.9514) and rec1 == (1, 0.7236)


def test_sharding():
    from krotov_jl_b200.distributed import shard_bounds

    gen = np.repeat(np.arange(256), 4)
    for world in (1, 2, 4, 8):
        b = [shard_bounds(gen, r, world) for r in range(world)]
        assert b[0][0] == 0 and b[-1][1] == 1024
        assert all(b[r][1] == b[r + 1][0] for r in range(world - 1))
        assert all((hi - lo) == 1024 // world and lo % 4 == 0 for lo, hi in b)  # whole samples per GPU
    assert shard_bounds(np.zeros(10, int), 1, 3) == (3, 6)
    gen = np.repeat(np.arange(3), [5, 1, 6])  # uneven groups: cut at generator boundaries
    b = [shard_bounds(gen, r, 2) for r in range(2)]
    assert b == [(0, 6), (6, 12)]
    # degenerate cut-aligned split (runs of 1, 1, 98 over 3 ranks): falls back to equal counts, nobody gets an
    # empty shard; more ranks than trajectories: every rank raises the same error (no rank left waiting)
    gen = np.repeat(np.arange(3), [1, 1, 98])
    b = [shard_bounds(gen, r, 3) for r in range(3)]
    assert b[0][0] == 0 and b[-1][1] == 100 and all(hi > lo for lo, hi in b)
    assert all(b[r][1] == b[r + 1][0] for r in range(2))
    for r in range(4):
        with pytest.raises(ValueError):
            shard_bounds(np.zeros(3, int), r, 4)


def test_reference_arm_uses_all_cores_even_under_torchrun_env():
    """bench.py --impl reference must not inherit OMP_NUM_THREADS=1 from torch.distributed.run (round-1 SCALE bug)."""
    import json
    import subprocess

    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--ref-samples", "2", "--n-grid", "101"], env=env, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    cores = len(os.sched_getaffinity(0))
    assert line["impl"] == "reference" and line["cpu_baseline"]["cores"] == cores
    # a non-zero rank of the reference arm does no work and prints nothing
    env["RANK"] = "1"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_dump_outputs_float64_within_budget(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: every array as float64 .npy, complex ones with a trailing [re, im] axis; beyond the
    byte budget tau and the states are cut to the same seeded sample of trajectories on every run."""
    import types

    import bench

    rng = np.random.default_rng(3)
    n, d = 64, 5
    states = rng.standard_normal((n, d)) + 1j * rng.standard_normal((n, d))
    res = types.SimpleNamespace(tau_vals=states[:, 0].copy(), states=list(states), J_T=0.25)
    pulses, ga = rng.standard_normal((2, 30)), rng.standard_normal(2)
    bench.dump_outputs(str(tmp_path / "full"), pulses, ga, res)
    got = {f[:-4]: np.load(tmp_path / "full" / f) for f in os.listdir(tmp_path / "full")}
    assert set(got) == {"pulses", "g_a_int", "tau", "states", "J_T"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert np.array_equal(got["pulses"], pulses) and np.array_equal(got["g_a_int"], ga) and got["J_T"].tolist() == [0.25]
    assert np.array_equal(got["states"][..., 0] + 1j * got["states"][..., 1], states)
    assert np.array_equal(got["tau"][:, 0] + 1j * got["tau"][:, 1], states[:, 0])

    monkeypatch.setattr(bench, "DUMP_BYTES", pulses.nbytes + 4096 + 20 * (d * 16 + 16 + 8))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), pulses, ga, res)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_BYTES
    rows = np.load(tmp_path / "a" / "trajectory_index.npy").astype(int)
    assert len(rows) == 20 and np.array_equal(rows, np.load(tmp_path / "b" / "trajectory_index.npy"))
    sampled = np.load(tmp_path / "a" / "states.npy")
    assert np.array_equal(sampled[..., 0] + 1j * sampled[..., 1], states[rows])


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from krotov_jl_b200.distributed import Comm, shard_bounds

        comm = Comm(device=0)
        gen = np.repeat(np.arange(8), 4)
        lo, hi = shard_bounds(gen, rank, world)
        local_tau = (np.arange(lo, hi) + 1j * rank).astype(complex)
        tau = comm.all_gather_rows(local_tau, len(gen))
        descs = comm.all_gather_object(bytes([rank]) * 256)
        # J_T_sm chi coefficients from the gathered tau: identical on all ranks
        coef = (1.0 / len(gen) ** 2) * np.sum(tau)
        out.put((rank, lo, hi, tau.real.tolist(), [d[0] for d in descs], complex(coef)))
    finally:
        dist.destroy_process_group()


def test_gloo_world2_plumbing():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert [(r[1], r[2]) for r in res] == [(0, 16), (16, 32)]
    assert res[0][3] == res[1][3] == list(map(float, range(32)))
    assert res[0][4] == res[1][4] == [0, 1]
    assert res[0][5] == res[1][5]


def test_hermitian_extremes_matches_lapack():
    """krotov_hermitian_extremes (threaded Householder + Sturm multi-section) against numpy's eigvalsh: the
    spectral envelopes of an ensemble differ from LAPACK's by a few ulp of the matrix norm at most."""
    from krotov_jl_b200._lib import hermitian_extremes

    rng = np.random.default_rng(3)
    for d in (1, 2, 3, 7, 25, 32, 48):
        A = rng.normal(size=(40, d, d)) + 1j * rng.normal(size=(40, d, d))
        A = A + A.conj().transpose(0, 2, 1)
        A[0] = np.diag(np.arange(d)).astype(complex)  # already diagonal
        A[1] = np.eye(d)  # fully degenerate
        A[2] = 0.0
        if d >= 3:
            A[3] = np.diag(np.ones(d)) + 1e-9 * (np.eye(d, k=1) + np.eye(d, k=-1))  # near-degenerate
        ev = np.linalg.eigvalsh(A)
        lo, hi = hermitian_extremes(A)
        lo1, hi1 = hermitian_extremes(A, n_threads=1)
        assert np.array_equal(lo, lo1) and np.array_equal(hi, hi1)  # independent of the thread count
        nrm = np.abs(ev).max(axis=1)
        assert np.all(np.abs(lo - ev[:, 0]) <= 8e-15 * nrm + 1e-300)
        assert np.all(np.abs(hi - ev[:, -1]) <= 8e-15 * nrm + 1e-300)
    # the ensemble path of ChebyDirection uses it and agrees with the per-matrix LAPACK path
    w = W.c4_ensemble(n_samples=20, n_grid=21)
    p = W.to_oracle(w)
    pulses = [q.copy() for q in p.pulses]
    many = K.cheby.ChebyDirection(p.H0, p.Hc, p.tlist, False, pulses)
    for g in (0, 7, 19):
        one = K.cheby.ChebyDirection([p.H0[g]], [p.Hc[g]], p.tlist, False, pulses)
        assert abs(many.Delta[g] - one.Delta[0]) <= 1e-14 * one.Delta[0]
        assert abs(many.E_min[g] - one.E_min[0]) <= 1e-14 * one.Delta[0]
        assert len(many.coeffs[g][0]) == len(one.coeffs[0][0])
        assert np.abs(many.coeffs[g][0] - one.coeffs[0][0]).max() < 1e-12  # alpha ~ 200 on this coarse grid


def test_cross_rank_fixed_point_word_format():
    """Bit budget of the one-hop cross-rank sum (`xrank_atomic_sum`, csrc/warp_kernel.cuh), modelled with Python
    integers: 117-bit biased numbers (unit 2^-88, bias 2^116) in four 30-bit limbs; word = limb sum (41 bits) |
    misfit count (11 bits) | arrival count (12 bits).  With the largest number of arrivals no field carries into
    its neighbour, the total stays below 2^128, and the reconstruction is the exact sum rounded once."""
    import math
    from fractions import Fraction

    FRAC, LIMB, LIMBS, BIAS, MIS, CNT, MAXARR = 88, 30, 4, 116, 41, 52, 2047
    assert LIMB * LIMBS >= BIAS + 1 and MIS == LIMB + 11 and CNT == MIS + 11 and CNT + 12 == 64

    def to_fixed(x):
        assert abs(x) < 2.0 ** (BIAS - FRAC)
        mag = int(Fraction(abs(x)) * 2**FRAC)  # truncation below 2^-88, like the kernel
        return (1 << BIAS) - mag if x < 0 else (1 << BIAS) + mag

    rng = np.random.default_rng(3)
    for n in (2, 256, MAXARR):
        xs = rng.standard_normal(n) * 10.0 ** rng.integers(-12, 8, n)
        xs[0] = -(2.0**28) * (1 - 2.0**-53)  # extremes of the range
        xs[1] = 2.0**28 * (1 - 2.0**-53)
        words = [0] * LIMBS
        for x in xs:
            v = to_fixed(float(x))
            assert 0 < v < (1 << (BIAS + 1))
            for j in range(LIMBS):
                words[j] += (1 << CNT) + ((v >> (j * LIMB)) & ((1 << LIMB) - 1))
        for wd in words:
            assert wd < (1 << 64) and (wd >> CNT) == n and ((wd >> MIS) & 0x7FF) == 0
        total = sum((wd & ((1 << MIS) - 1)) << (j * LIMB) for j, wd in enumerate(words))
        assert total < (1 << 128)
        exact = Fraction(total - (n << BIAS), 2**FRAC)
        truncated = sum(Fraction(int(Fraction(abs(float(x))) * 2**FRAC), 2**FRAC) * (1 if x >= 0 else -1) for x in xs)
        assert exact == truncated
        assert abs(float(exact) - math.fsum(float(x) for x in xs)) <= n * 2.0**-FRAC
    # all arrivals misfit: the misfit field holds them without touching the arrival count
    wd = MAXARR * ((1 << CNT) + (1 << MIS))
    assert (wd >> CNT) == MAXARR and ((wd >> MIS) & 0x7FF) == MAXARR and wd < (1 << 64)


# ---- the Julia module (julia/Krotov) cannot run here: keep its bindings in step with the header mechanically ---------------
_C2JL = {"int32_t": "Int32", "int64_t": "Int64", "double": "Float64", "int": "Cint", "const double *": "Ptr{Float64}",
         "double *": "Ptr{Float64}", "const int32_t *": "Ptr{Int32}", "const uint8_t *": "Ptr{UInt8}",
         "int64_t *": "Ptr{Int64}", "krotov_handle": "Ptr{Cvoid}", "void *": "Ptr{Cvoid}", "const void *": "Ptr{Cvoid}",
         "const krotov_problem *": "Ref{Problem}", "krotov_info *": "Ref{Info}"}
_HANDLE_OUT = {"Ref{Ptr{Cvoid}}", "Ptr{Ptr{Cvoid}}"}


def _c_struct_fields(hdr, name):
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\}\s*" + name + ";", hdr, flags=re.S).group(1)
    out = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.match(r"(.*?)(\w+)(\[(\d+)\])?$", decl)
        ctype, fname, arr = m.group(1).strip(), m.group(2), m.group(4)
        ctype = ctype.replace(" *", " *").strip()
        jl = _C2JL[ctype if ctype.endswith("*") else ctype]
        out.append((fname, f"NTuple{{{arr},{jl}}}" if arr else jl))
    return out


def _jl_struct_fields(src, name):
    body = re.search(r"^struct " + name + r"\n(.*?)^end", src, flags=re.S | re.M).group(1)
    return [(m.group(1), m.group(2)) for m in re.finditer(r"^\s*(\w+)::([\w{},]+)", body, flags=re.M)]


def test_julia_bindings_match_the_header():
    hdr = open(os.path.join(ROOT, "include", "krotov_cuda.h")).read()
    src = open(os.path.join(ROOT, "julia", "Krotov", "src", "LibKrotovCuda.jl")).read()
    # struct layouts, field by field
    assert _jl_struct_fields(src, "Problem") == _c_struct_fields(hdr, "krotov_problem")
    assert _jl_struct_fields(src, "Info") == _c_struct_fields(hdr, "krotov_info")
    # every C entry point is bound, with the header's argument types
    protos = {}
    clean = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for m in re.finditer(r"^(int|const char \*)\s*(krotov_\w+)\((.*?)\);", clean, flags=re.S | re.M):
        args = [] if m.group(3).strip() == "void" else [" ".join(a.split()) for a in m.group(3).split(",")]
        types = []
        for a in args:
            t = re.match(r"(.*?)(\w+)$", a).group(1).strip()
            types.append(t)
        protos[m.group(2)] = (m.group(1), types)
    calls = {}
    for m in re.finditer(r"ccall\(\(:(krotov_\w+), lib\),\s*(\w+),\s*\((.*?)\)\s*(?:,|\))", src, flags=re.S):
        calls[m.group(1)] = (m.group(2), [t.strip() for t in m.group(3).split(",") if t.strip()])
    assert set(calls) == set(protos), (sorted(set(protos) - set(calls)), sorted(set(calls) - set(protos)))
    for name, (ret, ctypes_) in protos.items():
        jret, jtypes = calls[name]
        assert jret == ("Cstring" if ret.startswith("const char") else "Cint"), name
        assert len(jtypes) == len(ctypes_), (name, jtypes, ctypes_)
        for jt, ct in zip(jtypes, ctypes_):
            if ct == "krotov_handle *":
                assert jt in _HANDLE_OUT, (name, jt)
            else:
                assert jt == _C2JL[ct], (name, jt, ct)
    # enum values used by the module
    for cname, val in re.findall(r"(KROTOV_[A-Z_]+) = (\d+)", clean):
        m = re.search(r"\b" + cname + r"\b[^\n]*", src)
        if m and "=" in m.group(0):
            names = [n.strip() for n in m.group(0).split("=")[0].replace("const", "").split(",")]
            vals = re.findall(r"Cint\((\d+)\)", m.group(0))
            if cname in names and len(vals) == len(names):
                assert int(vals[names.index(cname)]) == int(val), cname
    # the driver calls only bindings that exist
    drv = open(os.path.join(ROOT, "julia", "Krotov", "src", "optimize.jl")).read() + open(
        os.path.join(ROOT, "julia", "Krotov", "src", "workspace.jl")).read()
    defined = set(re.findall(r"^(?:function\s+)?(\w+!?)\(", src, flags=re.M))
    for fn in set(re.findall(r"LibKrotovCuda\.(\w+!?)\(", drv)):
        assert fn in defined or fn in ("Problem", "Handle"), fn


def _jl_strip(src):
    """Julia source without comments, strings (incl. interpolations) and character literals."""
    out, i, n = [], 0, len(src)
    while i < n:
        if src.startswith('"""', i):
            i = src.find('"""', i + 3) + 3
            out.append('""')
            continue
        c = src[i]
        if c == '"':
            j = i + 1
            while j < n and src[j] != '"':
                if src[j] == "\\":
                    j += 1
                elif src[j] == "$" and j + 1 < n and src[j + 1] == "(":
                    depth, k = 0, j + 1
                    while k < n:
                        depth += (src[k] == "(") - (src[k] == ")")
                        if depth == 0:
                            break
                        k += 1
                    j = k
                j += 1
            i = j + 1
            out.append('""')
            continue
        if c == "#":
            j = src.find("\n", i)
            i = n if j < 0 else j
            continue
        if c == "'" and i + 2 < n and (src[i + 2] == "'" or (src[i + 1] == "\\" and i + 3 < n and src[i + 3] == "'")):
            i += 3 if src[i + 2] == "'" else 4
            out.append("' '")
            continue
        out.append(c)
        i += 1
    return "".join(out)


def test_julia_sources_have_balanced_blocks():
    """Julia cannot run here, so the module cannot even be parsed by its own compiler; this catches the crudest class of
    slip in an edit: every block opener (function / if / for / while / begin / let / try / struct / module / do) outside
    brackets has its `end`, brackets balance, and `end` inside an index expression is not counted."""
    openers = {"function", "if", "for", "while", "begin", "let", "try", "struct", "module", "do", "quote", "macro"}
    files = [os.path.join(ROOT, "julia", "Krotov", sub, f) for sub in ("src", "test")
             for f in sorted(os.listdir(os.path.join(ROOT, "julia", "Krotov", sub)))]
    files.append(os.path.join(ROOT, "julia", "reference_vectors.jl"))
    assert len(files) >= 7
    for path in files:
        name = os.path.relpath(path, ROOT)
        s = _jl_strip(open(path, encoding="utf-8").read())
        stack, par, sq, line = [], 0, 0, 1
        for m in re.finditer(r"\n|[\[\]\(\)]|:?[^\W\d]\w*!?", s):
            t = m.group(0)
            if t == "\n":
                line += 1
            elif t in "()":
                par += 1 if t == "(" else -1
            elif t in "[]":
                sq += 1 if t == "[" else -1
            elif t.startswith(":") or sq > 0:
                continue
            elif t in openers:
                if not (t in ("for", "if") and par > 0):  # (generators inside parentheses need no `end`)
                    stack.append((t, line))
            elif t == "end":
                assert stack, f"{name}:{line}: `end` without an opener"
                stack.pop()
            assert par >= 0 and sq >= 0, f"{name}:{line}: closing bracket without an opener"
        assert not stack, f"{name}: unclosed {stack[-3:]}"
        assert par == 0 and sq == 0, f"{name}: unbalanced brackets"


# ---- the host driver on an oracle-backed engine (tests/oracle_engine.py) ---------------------------------------------
@pytest.fixture
def oracle_engine(monkeypatch):
    """`KrotovCuda` replaced by the oracle-backed stand-in: the product's host driver runs on CPU (test-only)."""
    import importlib

    import oracle_engine as E

    monkeypatch.setattr(importlib.import_module("krotov_jl_b200.workspace"), "KrotovCuda", E.OracleEngine)
    before = E.OracleEngine.created
    yield E
    assert E.OracleEngine.created > before


def test_host_driver_reproduces_the_oracle_loop_bit_for_bit(oracle_engine):
    """optimize() -> KrotovWrk -> krotov_initial_fw_prop / krotov_iteration -> engine calls -> update_result, with the
    engine's arithmetic done by the oracle: the pulse buffers, their swap, tau / J_T and the records must come out
    exactly as the oracle's own loop of src/optimize.jl:161-235 produces them (built-in chi, user chi, continue_from)."""
    from oracle import krotov_oracle as O
    from util import run_product

    for w in (W.c1_tls(), W.dummy_dense(d=10, n_traj=3, n_controls=2, n_grid=51, functional="ss")):
        ref = O.optimize_krotov(W.to_oracle(w), 4)
        got = run_product(w, 4)
        assert np.array_equal(got["pulses"], ref["pulses"])
        assert np.abs(np.array(got["J_T"]) - np.array(ref["J_T"])).max() < 5e-16  # (J_T is evaluated by the product's functional)
        assert np.array_equal(np.array(got["g_a_int"]), np.array(ref["g_a_int"]))
        # a user-supplied chi (KROTOV_CHI_HOST: chi(T) formed on the host and pushed with set_chi)
        user = run_product(w, 4, chi=lambda Psi, trajs, tau=None: K.chi_ss(Psi, trajs, tau=tau) if w.functional == "ss"
                           else K.chi_sm(Psi, trajs, tau=tau))
        assert np.abs(user["pulses"] - ref["pulses"]).max() < 1e-14
        # two iterations, then two more from the result (the pulses make the round trip midpoints -> grid -> midpoints)
        a = run_product(w, 2)
        b = run_product(w, 4, continue_from=a["result"])
        assert b["result"].iter == 4 and np.abs(b["pulses"] - ref["pulses"]).max() < 1e-11


def test_second_order_host_path_matches_general_formula(oracle_engine):
    """`sigma` through the product's host path (chi(T) - sigma/2 Psi(T) pushed with set_chi, sigma.refresh after
    update_result) against the oracle's general second-order update with a stored previous trajectory."""
    from oracle import krotov_oracle as O
    from util import run_product

    for w, a0 in ((W.c1_tls(), 1.0), (W.dummy_dense(d=10, n_traj=3, n_controls=2, n_grid=51, functional="sm"), 0.2)):
        for make in (lambda: -1.3 * a0, lambda: (lambda t: -0.8 * a0), lambda: K.NumericalSigma(a0, 0.1 * a0)):
            ref = O.optimize_krotov(W.to_oracle(w), 4, sigma=make())
            got = run_product(w, 4, sigma=make())
            assert np.abs(np.array(got["J_T"]) - np.array(ref["J_T"])).max() < 1e-12
            assert np.abs(got["pulses"] - ref["pulses"]).max() < 1e-12
        first = O.optimize_krotov(W.to_oracle(w), 4)
        assert np.abs(first["pulses"] - ref["pulses"]).max() > 1e-3
    # refresh receives what it needs to re-estimate A
    seen = []

    class S(K.Sigma):
        def __call__(self, t):
            return -0.5

        def refresh(self, **info):
            seen.append(info)

    w = W.c1_tls()
    got = run_product(w, 2, sigma=S())
    assert len(seen) == 2
    i = seen[-1]
    assert set(i) >= {"forward_states", "forward_states0", "chi_states", "J_T", "J_T_prev", "optimized_pulses", "guess_pulses",
                      "trajectories", "result"}
    assert i["J_T"] == got["J_T"][2] and i["J_T_prev"] == got["J_T"][1]
    assert np.array_equal(i["forward_states"][0], got["result"].states[0])
    tau_prev = got["tau"][1]
    assert np.allclose(i["chi_states"][0], tau_prev[0] * w.target[0], atol=1e-15)  # chi_sm, N = 1, BEFORE the fold
    A = K.numerical_estimate_A(i["forward_states"], i["forward_states0"], i["chi_states"], i["J_T"] - i["J_T_prev"])
    assert np.isfinite(A)


def test_sigma_argument_errors(oracle_engine):
    w = W.c1_tls()
    with pytest.raises(K.ArgumentError, match="varies over the time grid"):
        K.optimize(to_problem(w, sigma=lambda t: -1.0 - t, iter_stop=1), method=K.Krotov)
    with pytest.raises(K.ArgumentError, match="skip_initial_forward_propagation"):
        K.optimize(to_problem(w, sigma=-1.0, skip_initial_forward_propagation=True, iter_stop=1), method=K.Krotov)
    wn = W.dummy_dense(d=6, n_traj=2, n_controls=1, n_grid=11)
    wn.H0 = [wn.H0[0] - 0.1j * np.eye(6)]
    with pytest.raises(K.ArgumentError, match="Hermitian"):
        K.optimize(to_problem(wn, sigma=-1.0, iter_stop=1), method=K.Krotov)


def test_product_never_touches_the_oracle_or_a_cpu_fallback():
    """The oracle (and the oracle-backed engine the CPU tests inject) is test infrastructure: nothing under
    krotov.jl_b200/, include/ or julia/ may import, link or name it, and the product's engine has exactly one way to
    compute -- the handle of libkrotov_cuda (`krotov_create` fails without a GPU, see test_create_without_gpu_fails_loudly)."""
    bad = []
    for top in ("krotov.jl_b200", "include", "julia"):
        for folder, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".h", ".jl")):
                    continue
                with open(os.path.join(folder, f), encoding="utf-8") as fh:
                    for n, line in enumerate(fh, 1):
                        if re.search(r"\b(import|from|include|dlopen|CDLL)\b.*\boracle", line) or "oracle_engine" in line or "libkrotov_oracle" in line:
                            bad.append(f"{os.path.relpath(os.path.join(folder, f), ROOT)}:{n}: {line.strip()}")
    assert not bad, bad
    import importlib

    eng = importlib.import_module("krotov_jl_b200.engine")
    ws = importlib.import_module("krotov_jl_b200.workspace")
    assert ws.KrotovCuda is eng.KrotovCuda  # (outside the tests that patch it, the workspace builds the CUDA engine)


# ---- two ranks over gloo: the product's multi-rank HOST path on the oracle-backed engine -----------------------------------
def _gloo_driver_worker(rank, world, port, out, functional, mode, use_sigma):
    import importlib

    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import oracle_engine as E
        from krotov_jl_b200.distributed import Comm

        importlib.import_module("krotov_jl_b200.workspace").KrotovCuda = E.OracleEngine
        comm = Comm(device=rank)
        w = _two_rank_workload(functional)
        hist = {"J_T": []}

        def cb(wrk, it, eps_new, eps_old):
            hist["J_T"].append(wrk.result.J_T)
            hist["pulses"] = np.array([np.array(e) for e in eps_new])
            hist["shard"] = wrk._shard
            hist["tau"] = np.array(wrk.result.tau_vals)

        kw = dict(sigma=K.NumericalSigma(0.3, 0.05)) if use_sigma else {}
        res = K.optimize(to_problem(w, iter_stop=3, callback=cb, multi_gpu=mode, **kw), method=K.Krotov, comm=comm)
        out.put((rank, hist["J_T"], hist["pulses"], hist["shard"], res.message, np.array(res.states), hist["tau"],
                 E.OracleEngine.created))
    finally:
        dist.destroy_process_group()


def _two_rank_workload(functional):
    w = W.dummy_dense(d=8, n_traj=6, n_controls=2, n_grid=31, functional=functional, seed=21)
    w.H0 = [w.H0[0], w.H0[0] * 1.2]  # two generators, three trajectories each: the shards are cut between them
    w.Hc = [w.Hc[0], [w.Hc[0][0] * 0.8, w.Hc[0][1]]]
    w.gen_of_traj = np.array([0, 0, 0, 1, 1, 1])
    return w


@pytest.mark.parametrize("functional,mode,use_sigma", [("sm", "shard", False), ("ss", "shard", True), ("re", "shard", False),
                                                       ("sm", "replicate", True)])
def test_gloo_world2_host_driver_matches_one_rank(functional, mode, use_sigma):
    """optimize(problem, comm=Comm) on two CPU processes (gloo): sharding of the trajectories (`shard_bounds`, generator
    runs stay together), the per-iteration gathers of tau and states, the global J_T_sm coefficient through
    `set_chi_coeffs`, the second-order boundary condition per shard, replicas with identical pulses -- everything the
    host does for several ranks, with the engines' arithmetic (and the per-step cross-rank sum of the overlaps, which the
    CUDA kernels exchange over NVLink) done by the oracle-backed engine.  Against the one-process oracle run."""
    import torch.multiprocessing as mp
    from oracle import krotov_oracle as O

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() + 37 * ["sm", "ss", "re"].index(functional) + 211 * use_sigma + 503 * (mode == "replicate")) % 2000
    procs = [ctx.Process(target=_gloo_driver_worker, args=(r, 2, port, q, functional, mode, use_sigma)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, J0, P0, s0, m0, st0, tau0, made0), (r1, J1, P1, s1, m1, st1, tau1, made1) = res
    assert m0 == m1 == "Reached maximum number of iterations" and made0 == made1 == 1
    assert (s0, s1) == (((0, 3), (3, 6)) if mode == "shard" else ((0, 6), (0, 6)))
    assert J0 == J1 and np.array_equal(P0, P1) and np.array_equal(st0, st1) and np.array_equal(tau0, tau1)
    ref = O.optimize_krotov(W.to_oracle(_two_rank_workload(functional)), 3,
                            sigma=K.NumericalSigma(0.3, 0.05) if use_sigma else None)
    assert np.abs(np.array(J0) - np.array(ref["J_T"])).max() < 1e-12
    assert np.abs(P0 - ref["pulses"]).max() < 1e-12
    assert np.abs(st0 - ref["states"]).max() < 1e-12 and np.abs(tau0 - ref["tau"][-1]).max() < 1e-12


def test_committed_bench_lines_follow_the_contract():
    """The JSON lines bench.py printed on the B200 boxes (committed under profiles/) carry every key of the bench
    contract, and their derived numbers are consistent with one another."""
    import json

    for name, n in (("r2_bench_c4_1gpu_final.json", 1), ("r2_bench_c4_2gpu_replicate.json", 2),
                    ("r2_bench_c4_8gpu_replicate.json", 8)):
        with open(os.path.join(ROOT, "profiles", name)) as fh:
            d = json.load(fh)
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                    "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
            assert key in d, (name, key)
        assert d["n_gpus"] == n and d["warmup"] >= 3 and d["dtype"] == "f64" and d["data"] == "synthetic"
        assert d["vs_baseline"] is None  # BASELINE.md holds no published number for this metric
        assert "workload" in d["config"] and "model" not in d["config"]
        for key in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
            assert key in d["e2e"]
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
        assert 0 < d["e2e"]["value"] < d["value"]  # end to end includes what the device-timed value does not
        assert d["gpu_launches"] >= d["steps"]
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        r = d["roofline"]
        for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert key in r
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0 < r["frac"] < 1
        # value = whole-job state-timesteps over the device time of the timed iterations
        st = 2 * 1024 * 2000
        assert abs(d["value"] - st / (d["ms_per_step"] * 1e-3)) / d["value"] < 1e-9
        if n == 1:
            c = d["cpu_baseline"]
            for key in ("value", "unit", "cores", "kind", "sample"):
                assert key in c
            assert c["kind"] == "port" and c["cores"] > 1
            assert abs(r["achieved"] - r["algorithmic_bytes_per_launch"] / (d["ms_per_step"] * 1e-3) / 1e9) / r["achieved"] < 1e-9
            t5 = d["extra_configs"]["C5 dense d=4096 N=64, N_T=20 of 10000 (every step costs the same)"]["roofline_fp64_tensor"]
            assert abs(t5["frac"] - t5["achieved"] / t5["peak"]) < 1e-12 and t5["frac"] < 1
