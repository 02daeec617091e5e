"""Two ranks on two GPUs: trajectories sharded, per-step overlap sums exchanged in-kernel over NVLink -- by the
hierarchical fixed-point sum (default: local accumulator, the completing add forwards one add per rank), by the one-hop
sum (`KROTOV_XCHG=onehop`: every CTA adds into every rank's accumulator) and by the mailbox protocol
(`KROTOV_XCHG=mbox`: rank sums pushed into the peers' mailboxes; also the dense path's protocol).
Needs >= 2 CUDA devices (skipped on the single-GPU box); run with `gpurun --gpus 2`.  The same protocols run on ONE
device in tests/test_parity_gpu.py (`emulate_ranks`, all ranks' CTAs in one cooperative launch)."""
import os

import numpy as np
import pytest

import workloads as W

pytestmark = pytest.mark.gpu


def _make(kind, n_samples, n_grid):
    if kind == "c4":
        return W.c4_ensemble(n_samples=n_samples, n_grid=n_grid)
    if kind == "chain":  # sparse generator: the persistent ELL sweep (or its launch-per-term stream)
        return W.spin_chain(n_spins=7, n_traj=n_samples, n_grid=n_grid, functional="sm")
    return W.dummy_dense(d=64, n_traj=n_samples, n_controls=2, n_grid=n_grid, functional=kind, seed=5)


_BIG = 1e13


def _big_chi(states, trajectories, tau=None):
    """chi of J_T_sm scaled by 1e13 (with lambda_a scaled alike the optimisation is unchanged, but the overlap sums
    leave the fixed-point range of the one-hop sums)."""
    n = len(trajectories)
    s = sum(t.weight * x for t, x in zip(trajectories, tau))
    return [_BIG * (t.weight / n**2) * s * t.target_state for t in trajectories]


def _worker(rank, world, port, kind, n_samples, n_grid, iters, q, env=None):
    import sys

    os.environ.update(env or {})

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import krotov_jl_b200 as K
        from krotov_jl_b200.distributed import Comm
        from util import to_problem

        comm = Comm(device=rank)
        w = _make(kind, n_samples, n_grid)
        hist = {"J_T": [], "shard": None}
        live = K._lib.lib().krotov_live_device_objects
        hist["live"] = [live()]

        def cb(wrk, it, eps_new, eps_old):
            if it == 0 and (env or {}).get("TEST_RECONNECT"):
                # connecting again drops the peer mappings of the first connect before it maps the peers anew
                hist["live"].append(live())
                comm.connect(wrk.engine)
                hist["live"].append(live())
            hist["fallback"] = hist.get("fallback", 0) + wrk.engine.info()["fallback_steps"]
            hist["J_T"].append(wrk.result.J_T)
            hist["pulses"] = np.array([np.array(e) for e in eps_new])
            hist["shard"] = wrk._shard
            hist["ga"] = np.array(wrk.g_a_int)

        extra = {}
        if (env or {}).get("TEST_BIG_CHI"):
            extra = dict(chi=_big_chi, lambda_a=_BIG * w.lambda_a)
        if kind == "chain":
            extra["force_path"] = 3
        extra["multi_gpu"] = (env or {}).get("TEST_MULTI_GPU", "shard")
        res = K.optimize(to_problem(w, iter_stop=iters, callback=cb, device=rank, **extra), method=K.Krotov, comm=comm)
        hist["live"].append(live())
        q.put((rank, hist["J_T"], hist["pulses"], hist["shard"], res.message, np.array(res.states), hist["ga"],
               hist["fallback"], hist["live"]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("kind,n_samples,n_grid,env", [
    ("c4", 8, 201, {}), ("c4", 64, 101, {}), ("c4", 2, 101, {}), ("c4", 64, 101, {"KROTOV_XCHG": "onehop"}),
    ("c4", 64, 101, {"KROTOV_XCHG": "onehop", "KROTOV_XACC_STRIDE": "16"}),
    ("c4", 8, 201, {"KROTOV_XCHG": "mbox"}), ("c4", 64, 101, {"KROTOV_NO_XACC": "1"}),
    ("c4", 8, 41, {"TEST_BIG_CHI": "1"}), ("c4", 8, 41, {"TEST_BIG_CHI": "1", "KROTOV_XCHG": "onehop"}),
    ("sm", 20, 21, {}), ("ss", 9, 21, {}), ("sm", 20, 21, {"KROTOV_NO_SWEEP_RANKS": "1"}),
    ("chain", 40, 21, {}), ("chain", 40, 21, {"KROTOV_NO_SWEEP_RANKS": "1"}),
    ("c4", 8, 201, {"TEST_MULTI_GPU": "replicate"}), ("c4", 64, 101, {"TEST_MULTI_GPU": "replicate"}),
    ("c4", 3, 101, {"TEST_MULTI_GPU": "auto"}), ("c4", 8, 201, {"TEST_MULTI_GPU": "replicate", "TEST_RECONNECT": "1"})])
def test_two_ranks_match_single_gpu(kind, n_samples, n_grid, env):
    """kind c4: warp path (in-kernel exchange of the comm warps); kinds sm/ss: dense generators (d = 64: the cluster
    sweep, rank sums through the mailboxes from inside the sweep; with KROTOV_NO_SWEEP_RANKS the DMMA stream with the
    exchange in update_kernel); kind chain: sparse generator (the ELL sweep, or its stream)."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from util import run_product

    iters = 2
    single = run_product(_make(kind, n_samples, n_grid), iters, **({"force_path": 3} if kind == "chain" else {}))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + os.getpid() % 1000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, n_samples, n_grid, iters, q, env)) for r in range(2)]
    for p in procs:
        p.start()
    out = sorted([q.get(timeout=300) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, J0, P0, s0, m0, st0, ga0, fb0, live0), (r1, J1, P1, s1, m1, st1, ga1, fb1, live1) = out
    for live in (live0, live1):  # every rank gives back all it allocated and mapped
        assert live[-1] == live[0]
        if env.get("TEST_RECONNECT"):
            assert live[1] == live[2] > live[0]
    assert m0 == m1 == "Reached maximum number of iterations"
    n_traj = 4 * n_samples if kind == "c4" else n_samples
    replicated = env.get("TEST_MULTI_GPU") in ("replicate", "auto")
    if replicated:
        # replicated forward sweep: every rank holds everything and must reproduce the one-GPU run bit for bit
        assert s0 == s1 == (0, n_traj)
        assert np.array_equal(P0, single["pulses"]) and J0 == list(single["J_T"]) and np.array_equal(st0, st1)
        assert np.array_equal(st0, np.array(single["result"].states))
    else:
        assert s0 == (0, n_traj // 2) and s1 == (n_traj // 2, n_traj)
    # replicas must hold bit-identical pulses (every rank applies the same rank-ordered sum)
    assert np.array_equal(P0, P1) and J0 == J1 and np.array_equal(ga0, ga1)
    # and agree with the single-GPU run up to the summation order of the overlap sums
    assert np.abs(np.array(J0) - np.array(single["J_T"])).max() < 1e-12
    assert np.abs(P0 - single["pulses"]).max() < 1e-12
    assert np.abs(st0 - np.array(single["result"].states)).max() < 1e-11
    if env.get("TEST_BIG_CHI"):
        # partials beyond 2^28: every CTA of both ranks redid those steps with the mailbox protocol
        assert fb0 > n_grid // 2 and fb1 > n_grid // 2
    elif kind == "c4":
        assert fb0 == 0 and fb1 == 0
