"""Controls that enter the generators through several (operator, amplitude) terms, tied to one control
(``krotov_set_control_terms``): a drive in a rotating frame, a drive with its ac-Stark shift, ensemble members that see
one control through different distortions."""
import importlib
import os

import numpy as np
import pytest

import krotov_jl_b200 as K
import terms_reference as R
import workloads as W
from krotov_jl_b200.controls import get_control_terms

RTOL_JT, ATOL_JT, ATOL_PULSE = 1e-10, 5e-13, 1e-9
ERR_ARG = 1  # KROTOV_ERR_ARG


def run(case, comm=None, **kwargs):
    """Optimise ``case`` through the public API; per-iteration J_T, per-control g_a, final per-control pulses."""
    hist = dict(J_T=[], g_a_int=[])

    def record(wrk, it, eps_new, eps_old):
        hist["J_T"].append(wrk.result.J_T)
        if it > 0:
            hist["g_a_int"].append(np.array(wrk.g_a_int))
        hist["pulses"] = np.array([np.array(e) for e in eps_new])
        hist["info"] = wrk.engine.info()
        hist["engine"] = wrk.engine

    kwargs.setdefault("rethrow_exceptions", True)
    hist["result"] = K.optimize(case.problem(callback=record, **kwargs), method=K.Krotov, comm=comm)
    return hist


def assert_close(got, ref, tol_JT=1e-12, tol_pulse=1e-12, tol_ga=1e-12):
    assert np.abs(np.asarray(got["J_T"]) - np.asarray(ref["J_T"])).max() <= tol_JT, (got["J_T"], ref["J_T"])
    assert np.abs(np.asarray(got["pulses"]) - np.asarray(ref["pulses"])).max() <= tol_pulse
    assert np.abs(np.asarray(got["g_a_int"]) - np.asarray(ref["g_a_int"])).max() <= tol_ga


def assert_parity(got, ref):
    """BASELINE tolerances (the oracle computes in another order)."""
    ref_JT = np.asarray(ref["J_T"])
    assert np.all(np.abs(np.asarray(got["J_T"]) - ref_JT) <= RTOL_JT * np.abs(ref_JT) + ATOL_JT)
    assert np.abs(got["pulses"] - np.asarray(ref["pulses"])).max() <= ATOL_PULSE
    assert np.abs(np.asarray(got["g_a_int"]) - np.asarray(ref["g_a_int"])).max() <= 1e-11


@pytest.fixture
def oracle_engine(monkeypatch):
    monkeypatch.setattr(importlib.import_module("krotov_jl_b200.workspace"), "KrotovCuda", R.TermsOracleEngine)
    R.TermsOracleEngine.calls.clear()
    made = []
    init = R.TermsOracleEngine.__init__

    def spy(self, **kw):
        made.append(kw)
        init(self, **kw)

    monkeypatch.setattr(R.TermsOracleEngine, "__init__", spy)
    return made


# ---- CPU: term building ----------------------------------------------------------------------------------------------
def test_term_building_sums_splits_masks_and_orders():
    X = np.array([[0, 1], [1, 0]], complex)
    Y = np.array([[0, -1j], [1j, 0]], complex)
    Z = np.diag([1.0, -1.0]).astype(complex)
    e, f = (lambda t: 0.1), (lambda t: 0.2)
    cos = lambda t: np.cos(t)  # noqa: E731
    a_cos, a_sin = K.ShapedAmplitude(e, cos), K.ShapedAmplitude(e, np.sin)
    a_cos2 = K.ShapedAmplitude(e, cos)  # same key and the same shape object as a_cos: the same term
    g1 = K.hamiltonian(Z, (X, a_cos), (Y, f), (Y, a_cos2), (Z, a_sin))
    g2 = K.hamiltonian(Z, (X, e), (Z, f))
    controls = K.get_controls([g1, g2])
    terms, ops = get_control_terms([g1, g2], controls)
    assert [c for c, _ in terms] == [0, 1, 0, 0]  # term l = control l for l < L, the further terms after them
    assert terms[0][1] is a_cos and terms[2][1] is a_sin and terms[3][1] is None and terms[1][1] is None
    assert np.array_equal(ops[0][0], X + Y) and np.array_equal(ops[0][1], Y) and np.array_equal(ops[0][2], Z)
    assert ops[0][3] is None  # g1 has no direct eps term
    assert ops[1][0] is None and ops[1][2] is None and np.array_equal(ops[1][1], Z) and np.array_equal(ops[1][3], X)


def test_untied_problem_builds_todays_arrays_without_a_setter_call(oracle_engine):
    """`(H1, eps), (H2, eps)` is one term with the operator H1 + H2, as before: no term map reaches the engine."""
    w = W.c1_tls(n_grid=41)
    sy = np.array([[0, -1j], [1j, 0]], complex)
    H = K.hamiltonian(w.H0[0], (w.Hc[0][0], w.controls[0]), (sy, w.controls[0]))
    problem = K.ControlProblem([K.Trajectory(w.psi0[0], H, target_state=w.target[0])], w.tlist, prop_method=K.Cheby,
                               J_T=K.J_T_sm, lambda_a=1.0, iter_stop=1, print_iters=False)
    K.optimize(problem, method=K.Krotov)
    assert R.TermsOracleEngine.calls == []
    kw = oracle_engine[0]
    assert len(kw["Hc"]) == 1 and len(kw["Hc"][0]) == 1
    assert np.array_equal(kw["Hc"][0][0], w.Hc[0][0] + sy)
    assert kw["update_shape"].shape == (1, 40) and np.array_equal(kw["lambda_a"], [1.0])


@pytest.mark.parametrize("name", sorted(R.CASES))
def test_oracle_against_exact_vectors(name):
    case = R.CASES[name]()
    gold = R.load_golden(name)
    p, tc = case.oracle_arrays()
    assert list(tc) == gold["term_ctrl"]
    for method, tol in (("expm", 1e-14), ("cheby", 1e-12)):
        h = R.optimize_terms(p, tc, iter_stop=case.iters, prop_method=method)
        assert_close(h, gold, tol, tol, tol)


@pytest.mark.parametrize("name", sorted(R.CASES))
def test_host_driver_per_control_results_against_exact_vectors(name, oracle_engine):
    case = R.CASES[name]()
    gold = R.load_golden(name)
    got = run(case)
    assert len(R.TermsOracleEngine.calls) == 1 and list(R.TermsOracleEngine.calls[0]) == gold["term_ctrl"]
    res = got["result"]
    assert len(res.optimized_controls) == case.C and got["pulses"].shape[0] == case.C
    assert all(len(g) == case.C for g in got["g_a_int"])  # per control, not double-counted
    assert_close(got, gold)


def test_terms_of_one_control_differ_between_generators_in_their_shapes_only():
    """Per-generator shapes of one amplitude function make separate terms; a generator that maps the control through
    another function (polynomial, parametrization) than the other generators do is refused before any device work."""
    w = W.c1_tls(n_grid=21)
    eps = w.controls[0]
    trajs = lambda *gens: [K.Trajectory(w.psi0[0], g, target_state=w.target[0]) for g in gens]  # noqa: E731
    gens = [K.hamiltonian(w.H0[0], (w.Hc[0][0], K.ShapedAmplitude(eps, s))) for s in (np.cos, np.sin)]
    wrk = K.KrotovWrk.__new__(K.KrotovWrk)
    wrk.controls = (eps,)
    wrk._terms, wrk._term_ops = get_control_terms(gens, wrk.controls)
    wrk._check_term_functions()
    assert [c for c, _ in wrk._terms] == [0, 0]
    stark = K.hamiltonian(w.H0[0], (w.Hc[0][0], eps), (w.Hc[0][0], K.PolynomialAmplitude(eps, [0, 0, 1])))
    plain = K.hamiltonian(w.H0[0], (w.Hc[0][0], eps))
    with pytest.raises(K.ArgumentError):
        K.optimize(K.ControlProblem(trajs(stark, plain), w.tlist, prop_method=K.Cheby, J_T=K.J_T_sm, lambda_a=1.0,
                                    iter_stop=1, print_iters=False, rethrow_exceptions=True), method=K.Krotov)


def _gloo_terms_worker(rank, world, port, out):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        importlib.import_module("krotov_jl_b200.workspace").KrotovCuda = R.TermsOracleEngine
        from krotov_jl_b200.distributed import Comm

        got = run(R.CASES["two_generators_shapes"](), comm=Comm(device=0), multi_gpu="shard")
        h = {k: np.asarray(got[k]).tolist() for k in ("J_T", "g_a_int", "pulses")}
        out.put((rank, h))
    finally:
        dist.destroy_process_group()


def test_gloo_two_ranks_match_one_rank(oracle_engine):
    """The tie after the cross-rank sum: two gloo ranks (one shard of the ensemble each, oracle engine) agree with one."""
    import torch.multiprocessing as mp

    one = run(R.CASES["two_generators_shapes"]())
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_terms_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, h in res:
        assert_close(h, one, 1e-13, 1e-13, 1e-13)


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(R.CASES))
def test_exact_vectors_on_the_warp_kernel(name):
    case = R.CASES[name]()
    got = run(case)
    assert got["info"]["path"] == 1 and got["info"]["kernel"] != 1  # the warp kernel, the one-thread kernel bypassed
    assert_close(got, R.load_golden(name))


def _engine_pair(w):
    """Two handles of one problem: control 0 as the tied pair (H1, eps), (H2, eps) and as one term eps (H1 + H2)."""
    from krotov_jl_b200 import _lib as B
    from krotov_jl_b200.cheby import ChebyDirection
    from krotov_jl_b200.engine import KrotovCuda

    H1 = w.Hc[0][0]
    H2 = 0.5 * H1.conj() + 0.1 * np.diag(np.arange(w.d)).astype(complex)
    eps = K.discretize_on_midpoints(w.controls[0], w.tlist)
    kw = dict(tlist=w.tlist, H0=w.H0, gen_of_traj=w.gen_of_traj, psi0=w.psi0, target=w.target,
              functional=B.CHI_SM, n_traj_global=w.N)
    S = K.discretize_on_midpoints(w.update_shape, w.tlist)
    tied = KrotovCuda(Hc=[[H1, H2]], update_shape=np.stack([S, S]), lambda_a=[w.lambda_a] * 2, **kw)
    one = KrotovCuda(Hc=[[H1 + H2]], update_shape=S[None], lambda_a=[w.lambda_a], **kw)
    for backward in (False, True):
        adj = (lambda m: m.conj().T) if backward else (lambda m: m)
        cd = ChebyDirection([adj(h) for h in w.H0], [[adj(H1 + H2)]], w.tlist, backward, [eps])
        cd.push(tied, B.BACKWARD if backward else B.FORWARD)
        cd.push(one, B.BACKWARD if backward else B.FORWARD)
    return tied, one, eps


@pytest.mark.gpu
def test_tied_linear_terms_reproduce_the_summed_operator():
    tied, one, eps = _engine_pair(W.c2_transmon_x(n_grid=201))
    tied.set_control_terms([0, 0])
    g1, g2 = eps[None].copy(), np.stack([eps, eps])
    tied.forward(g2)
    one.forward(g1)
    for _ in range(3):
        n2, ga2 = tied.iterate(g2)
        n1, ga1 = one.iterate(g1)
        assert np.array_equal(n2[0], n2[1]) and ga2[1] == 0.0
        assert np.abs(n2[0] - n1[0]).max() <= 1e-12 and abs(ga2[0] - ga1[0]) <= 1e-12
        assert np.abs(tied.tau() - one.tau()).max() <= 1e-12
        g1, g2 = n1, n2
    tied.close()
    one.close()


def _ensemble_case():
    return R.rotating_frame_ensemble(n_samples=8, n_grid=201)


@pytest.mark.gpu
def test_ensemble_multi_cta_and_emulated_ranks():
    case = _ensemble_case()
    got = run(case)
    assert got["info"]["grid_blocks"] > 1
    p, tc = case.oracle_arrays()
    assert_parity(got, R.optimize_terms(p, tc, 2))
    for mode in ("shard", "replicate"):
        two = run(case, emulate_ranks=2, multi_gpu=mode)
        assert len(two["J_T"]) == case.iters + 1
        allp = two["engine"].pulses_all  # every rank's copy, term rows: the tie runs on identical bits everywhere
        assert all(np.array_equal(allp[r], allp[0]) for r in range(len(allp)))
        assert np.array_equal(allp[0][0], allp[0][1])
        assert_same_run(two, got, mode)


def assert_same_run(two, one, mode):
    """replicate: the forward sweep of every rank IS the one-rank sweep -- bit for bit; shard: the CTA partials are cut
    differently, the fixed-point sums then differ in the last bits (the tolerance of the untied multi-rank tests)."""
    if mode == "replicate":
        assert np.array_equal(two["pulses"], one["pulses"]) and list(two["J_T"]) == list(one["J_T"])
        assert np.array_equal(np.array(two["g_a_int"]), np.array(one["g_a_int"]))
    else:
        assert np.abs(np.asarray(two["pulses"]) - one["pulses"]).max() < 1e-12
        assert np.abs(np.array(two["J_T"]) - np.array(one["J_T"])).max() < 1e-12
        assert np.abs(np.array(two["g_a_int"]) - np.array(one["g_a_int"])).max() < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dense", "dense_cluster_sweep", "sparse_sweep", "sparse_stream", "reloaded_rows"])
def test_block_paths(kind, monkeypatch):
    kw = {}
    if kind == "dense":
        monkeypatch.setenv("KROTOV_NO_DSWEEP", "1")
        w = W.dummy_dense(d=40, n_traj=6, n_controls=2, n_grid=31, seed=3)
    elif kind == "dense_cluster_sweep":
        w = W.dummy_dense(d=100, n_traj=20, n_controls=1, n_grid=21, seed=101)
    elif kind == "reloaded_rows":
        monkeypatch.setenv("KROTOV_NO_PREG", "1")
        w = W.dummy_dense(d=12, n_traj=5, n_controls=2, n_grid=31, seed=4)
    else:
        if kind == "sparse_stream":
            monkeypatch.setenv("KROTOV_NO_SWEEP", "1")
        w = W.spin_chain(n_spins=6, n_traj=8, n_grid=31)
        kw = {"force_path": 3}
    case = R.tie_workload(w)
    got = run(case, **kw)
    assert got["info"]["path"] == {"reloaded_rows": 1, "dense": 2, "dense_cluster_sweep": 2}.get(kind, 3)
    p, tc = case.oracle_arrays()
    assert_parity(got, R.optimize_terms(p, tc, 2))


@pytest.mark.gpu
def test_block_path_graph_replay_equals_direct_launches(monkeypatch):
    monkeypatch.setenv("KROTOV_NO_DSWEEP", "1")
    case = R.tie_workload(W.dummy_dense(d=40, n_traj=6, n_controls=2, n_grid=31, seed=3))
    case.iters = 6
    a = run(case)
    assert a["info"]["path"] == 2 and a["info"]["graph_replays"] >= 2
    monkeypatch.setenv("KROTOV_NO_GRAPH", "1")
    b = run(case)
    assert b["info"]["graph_replays"] == 0
    assert np.array_equal(a["pulses"], b["pulses"]) and a["J_T"] == b["J_T"]


@pytest.mark.gpu
def test_c_abi_arguments_identity_map_and_resources():
    from krotov_jl_b200 import _lib as B

    live0 = B.lib().krotov_live_device_objects()
    w = W.c2_transmon_x(n_grid=101)
    tied, one, eps = _engine_pair(w)
    g2 = np.stack([eps, eps])

    def code(f, *a):
        with pytest.raises(B.KrotovCudaError) as e:
            f(*a)
        return e.value.code

    assert code(tied.set_control_terms, [1, 0]) == ERR_ARG  # not in order of first appearance
    assert code(tied.set_control_terms, [0, 2]) == ERR_ARG  # out of range
    assert code(tied.set_control_terms, [0, -1]) == ERR_ARG
    tied.set_control_terms([0, 0])
    bad = g2.copy()
    bad[1, 3] = np.nextafter(bad[1, 3], 1.0)  # tied guess rows must be bitwise equal
    assert code(tied.forward, bad) == ERR_ARG
    tied.forward(g2)
    assert code(tied.iterate, bad) == ERR_ARG
    # NULL and the identity map both restore the untied state: bit for bit what a handle never tied computes
    ref = None
    for m in ("never", None, [0, 1]):
        t2, _, _ = _engine_pair(w)
        if m != "never":
            t2.set_control_terms([0, 0])
            t2.set_control_terms(m)
        t2.forward(g2)
        out = [t2.iterate(g2)]
        out.append(t2.iterate(out[0][0]))
        out = (np.array([o[0] for o in out]), np.array([o[1] for o in out]), t2.tau())
        if ref is None:
            ref = out
        assert all(np.array_equal(a, b) for a, b in zip(out, ref))
        t2.close()
    tied.close()
    one.close()
    # tied update_shape / lambda_a rows must agree
    from krotov_jl_b200.engine import KrotovCuda

    S = K.discretize_on_midpoints(w.update_shape, w.tlist)
    base = dict(tlist=w.tlist, H0=w.H0, Hc=[[w.Hc[0][0], w.Hc[0][0]]], gen_of_traj=w.gen_of_traj, psi0=w.psi0,
                target=w.target, functional=B.CHI_SM)
    for shp, lam in ((np.stack([S, 0.5 * S]), [w.lambda_a] * 2), (np.stack([S, S]), [w.lambda_a, 2 * w.lambda_a])):
        e = KrotovCuda(update_shape=shp, lambda_a=lam, **base)
        assert code(e.set_control_terms, [0, 0]) == ERR_ARG
        e.close()
    assert B.lib().krotov_live_device_objects() == live0


def _mg_worker(rank, world, port, mode, q):
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "tests")]
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from krotov_jl_b200.distributed import Comm

        got = run(_ensemble_case(), comm=Comm(device=rank), multi_gpu=mode)
        q.put((rank, np.asarray(got["pulses"]).tolist(), list(got["J_T"]), np.asarray(got["g_a_int"]).tolist()))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["shard", "replicate"])
def test_two_gpus(mode):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    import torch.multiprocessing as mp

    one = run(_ensemble_case())
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_mg_worker, args=(r, 2, port, mode, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, pulses, J, ga in res:
        assert_same_run(dict(pulses=pulses, J_T=J, g_a_int=ga), one, mode)
