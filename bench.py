#!/usr/bin/env python
"""bench.py -- Krotov iterations/s and state-timesteps/s of the B200 hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--samples S] [--n-grid G] [--dump-outputs DIR]

A "step" is ONE Krotov iteration (backward sweep + sequential update + forward sweep,
src/optimize.jl:279-371 of the reference) over the whole workload.  The workload is BASELINE.json's
config C4 -- the robust two-transmon CNOT ensemble: 256 Hamiltonian samples x 4 basis states = 1024
trajectories, d = 25, L = 2 controls, N_T = 2000 -- which fits one GPU; with --gpus N the SAME 1024
trajectories are sharded over N ranks (strong scaling, as BASELINE.json words it: "sharded 1/2/4/8 GPUs").

value  = state-timesteps/s (2 N N_T per iteration) from the device time of the timed iterations (CUDA
         events on the launch stream inside libkrotov_cuda, inputs resident in HBM), max over ranks.
e2e    = the same metric through the public API `optimize(problem, method=Krotov)`: every iteration copies
         the guess pulses host->device and the new pulses, g_a integrals and tau device->host, and runs the
         reference's host bookkeeping (range checks, J_T, callbacks).
--impl reference times the CPU restatement of the reference (oracle/krotov_oracle.c, OpenMP over
trajectories like the reference's @threadsif) on a bounded sample of the same workload: Julia is not
installed in this image, so the reference itself cannot run (see DESIGN.md).
--dump-outputs DIR writes what the last timed iteration returned (see dump_outputs) as float64 .npy files; the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import workloads as W  # noqa: E402

METRIC = "state_timesteps_per_s"
UNIT = "state-timesteps/s"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, sampled through NVML in a thread
    (an `nvidia-smi -lms` child process was measured to perturb the launches it is supposed to watch)."""

    def __init__(self, index=0, period=0.05):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.thread = None

    def prepare(self):
        """NVML initialisation (tens of ms, and not the same on every rank): done before the run, never between the
        barrier that opens the timed region and the first timed launch -- with several ranks the ranks that are ready
        first launch and wait IN the kernel for the last one, which counts as device time."""
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def start(self):
        if getattr(self, "nv", None) is None:
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def smem_roofline(n_traj, n_steps, terms_per_step, width, sm_count, sm_mhz, ms_launch):
    """The resource that actually binds the warp kernel: the shared-memory crossbar (128 B/clk/SM).  One Chebyshev
    term moves (W+1) warp-wide 512-byte accesses per trajectory (W LDS.128 gathers + 1 STS.128)."""
    moved = float(n_traj) * n_steps * terms_per_step * (width + 1) * 512.0
    peak = 128.0 * sm_count * sm_mhz * 1e6
    return {"achieved": moved / (ms_launch * 1e-3) / 1e9, "unit": "GB/s", "peak": peak / 1e9,
            "frac": moved / (ms_launch * 1e-3) / peak, "bytes_per_launch": moved,
            "peak_source": "128 B/clk/SM (B300_MICROARCH.md) x SMs x max SM clock; tools/chain_bench.cu reaches 92 % of "
                           "it with this kernel's inner loop (profiles/r1_chain_bench.txt)",
            "note": "algorithmic: N x N_T x (m_fw + m_bw - 2) terms x (W+1) x 512 B; the backward sweep alone runs at "
                    "~80 % of this roof, the forward sweep waits ~40 % of every time step for the grid-wide sum "
                    "(DESIGN.md 4.1)"}


def host_cores():
    """Host threads the CPU arm may use: the cores this process is allowed to run on.  `torch.distributed.run`
    exports OMP_NUM_THREADS=1 to its workers, so the OpenMP default must never be relied on -- the count is passed
    explicitly to the C restatement (oracle/c_oracle.py `n_threads`)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_baseline_sample(workload_full, samples, iters, n_threads=0):
    """Time the C restatement on a bounded sample: the first `samples` ensemble members of the workload."""
    from oracle import c_oracle

    n_threads = n_threads or host_cores()
    w = W.c4_ensemble(n_samples=samples, n_grid=len(workload_full.tlist))
    p = W.to_oracle(w)
    out = c_oracle.optimize_krotov_c(p, iters, n_threads=n_threads)
    st = 2.0 * w.N * w.N_T * iters
    return {"value": st / out["secs"], "unit": UNIT, "cores": out["threads"], "kind": "port",
            "iterations_per_s_at_sample": iters / out["secs"],
            "sample": f"{samples} of 256 ensemble samples ({w.N} trajectories), N_T={w.N_T}, {iters} iteration(s), "
                      f"{out['secs']:.2f} s; C restatement of Krotov.jl (Julia not installed), OpenMP over trajectories"}


DMMA_PEAK_TFLOPS = 37.1  # self-measured FP64 mma.sync peak on this pool's B200 (tools/microbench.cu, profiles/r1_microbench_fp64.txt)
DFMA_PEAK_TFLOPS = 34.2


def extra_configs(K, to_problem, peaks):
    """The other BASELINE configs, timed by the same run (device time from the handle, CUDA events on the launch
    stream): C1, C2, C3 at full size on the persistent one-launch kernels, and C5 at full WIDTH (d = 4096, 64
    trajectories) over 20 time steps, both sweeps, on the FP64 DMMA path -- every time step of C5 costs the same, so
    the per-step figures carry to N_T = 10000.  Each entry names the roof that binds it."""
    out = {}

    def run(w, iters, warm):
        ms, info = [], {}

        def cb(wrk, it, *a):
            if it >= 1:
                i = wrk.engine.info()
                ms.append(i["ms_last"])
                info.update(i)

        res = K.optimize(to_problem(w, iter_stop=warm + iters, callback=cb), method=K.Krotov)
        if res.message.startswith("Exception"):
            raise RuntimeError(res.message)
        return float(np.mean(ms[warm:])), info, res

    kernels = {1: "krotov_warp_kernel / krotov_tiny_kernel (one persistent launch per iteration)",
               2: "dense_gemm_kernel<8> (FP64 DMMA, stream-K) + build_G_kernel + update_kernel",
               3: "sparse_sweep_kernel / spmm_kernel"}
    for name, make, iters in (("C1 TLS d=2 N=1 N_T=500", W.c1_tls, 10), ("C2 transmon X d=3 N=2 N_T=500", W.c2_transmon_x, 10),
                              ("C3 two-transmon d=25 N=4 N_T=2000", W.c3_two_transmon, 5)):
        try:
            w = make()
            ms, info, res = run(w, iters, 2)
            out[name] = {"ms_per_iteration": ms, "iterations_per_s": 1e3 / ms,
                         "state_timesteps_per_s": 2.0 * w.N * w.N_T / (ms * 1e-3),
                         "us_per_time_step_both_sweeps": 1e3 * ms / w.N_T, "launches_per_iteration": info["launches_last"],
                         "grid": [info["grid_blocks"], info["block_threads"]], "m": info["m_fw"], "J_T_last": res.J_T,
                         "kernel": kernels[info["path"]] if info["grid_blocks"] > 1 or info["block_threads"] > 32 else
                         "krotov_tiny_kernel (one warp, one thread per trajectory)",
                         "bound": "latency of the serial chain (one trajectory per warp / thread; neither HBM nor FP64 "
                                  "is loaded: %.2g GB/s, %.2g GFLOP/s)" % (
                                      16.0 * w.d * w.N * (2 * w.N_T + 1) / (ms * 1e-3) / 1e9,
                                      2.0 * w.N * w.N_T * (info["m_fw"] - 1) * 8 * info["nnz_union"] / (ms * 1e-3) / 1e9)}
        except Exception as exc:  # an extra config never costs the headline
            out[name] = {"error": str(exc)}
    try:
        n_grid = 21
        w = W.c5_dense(d=4096, n_traj=64, n_grid=n_grid)
        ms, info, res = run(w, 1, 1)
        N_T, m, dp = w.N_T, info["m_fw"], 4096
        gemms = N_T * (2 * (m - 1) + w.L)  # (m-1) per direction and step + the overlap GEMM of every control
        flops = gemms * 8.0 * dp * dp * w.N
        gen_bytes = gemms * 16.0 * dp * dp
        out["C5 dense d=4096 N=64, N_T=%d of 10000 (every step costs the same)" % N_T] = {
            "ms_per_iteration": ms, "ms_per_time_step_both_sweeps": ms / N_T,
            "s_per_iteration_at_N_T_10000": ms / N_T * 10000 * 1e-3,
            "state_timesteps_per_s": 2.0 * w.N * N_T / (ms * 1e-3), "launches_per_iteration": info["launches_last"],
            "m": m, "kernel": kernels[info["path"]], "J_T_last": res.J_T,
            "roofline_fp64_tensor": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": DMMA_PEAK_TFLOPS,
                                     "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / DMMA_PEAK_TFLOPS,
                                     "flops_per_iteration": flops,
                                     "formula": "8 dp^2 N x [(m-1) x 2 + L] GEMMs per time step x N_T, over the WHOLE "
                                                "iteration (generator builds, updates, storage and launch gaps included)",
                                     "peak_source": "self-measured mma.sync.m8n8k4.f64 peak (tools/microbench.cu); "
                                                    "MEASURED_PEAKS.json has no FP64 figure"},
            "roofline_hbm_generator": {"achieved": gen_bytes / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                       "frac": gen_bytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                       "note": "16 dp^2 bytes of generator per GEMM if nothing stayed in L2"}}
    except Exception as exc:
        out["C5 dense d=4096 N=64"] = {"error": str(exc)}
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(folder, pulses, g_a_int, res):
    """The arrays a caller of the timed path receives from its last iteration, as float64 .npy files (complex arrays
    with a trailing [re, im] axis): the new pulses (L, N_T), the g_a integrals (L,), tau (N, 2), the forward-propagated
    final states (N, d, 2) and J_T (1,).  Beyond DUMP_BYTES in all, tau and the states are cut to a fixed, seeded
    sample of trajectories whose indices go to trajectory_index.npy."""
    def re_im(a):
        a = np.asarray(a, np.complex128)
        return np.stack([a.real, a.imag], axis=-1)

    out = {"pulses": np.asarray(pulses, np.float64), "g_a_int": np.asarray(g_a_int, np.float64),
           "tau": re_im(res.tau_vals), "states": re_im(np.array(res.states)), "J_T": np.array([res.J_T], np.float64)}
    n = out["states"].shape[0]
    per_traj = out["states"][0].nbytes + out["tau"][0].nbytes + 8
    keep = (DUMP_BYTES - out["pulses"].nbytes - 4096) // per_traj
    if keep < n:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        out["tau"], out["states"] = out["tau"][rows], out["states"][rows]
        out["trajectory_index"] = rows.astype(np.float64)
    os.makedirs(folder, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(folder, name + ".npy"), np.ascontiguousarray(a))


def run_reference(args):
    """`--impl reference`: CPU restatement on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = min(args.samples, args.ref_samples)
    from oracle import c_oracle

    c_oracle.build()
    # each "step" is one iteration on the bounded sample; warm-up iterations are run and discarded
    w = W.c4_ensemble(n_samples=sample, n_grid=args.n_grid)
    p = W.to_oracle(w)
    t0 = time.time()
    n_threads = args.ref_threads or host_cores()
    if n_threads == 1 and (os.cpu_count() or 1) > 1 and not args.ref_threads:
        # a single-threaded CPU arm on a multi-core box is not the baseline BASELINE.json asks for
        raise SystemExit(f"reference arm would run on 1 of {os.cpu_count()} cores (affinity "
                         f"{sorted(os.sched_getaffinity(0))}); pass --ref-threads to force")
    out = c_oracle.optimize_krotov_c(p, args.warmup + args.steps, n_threads=n_threads)
    # the C oracle reports the loop time of all iterations; per-iteration time is uniform
    secs_per_iter = out["secs"] / (args.warmup + args.steps)
    st = 2.0 * w.N * w.N_T
    value = st / secs_per_iter
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs_per_iter, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "iterations_per_s": 1.0 / secs_per_iter,
        "config": {"workload": f"C4 robust two-transmon CNOT ensemble, bounded sample: {sample} of {args.samples} "
                               f"samples x 4 basis states = {w.N} trajectories, d=25, L=2, N_T={w.N_T}",
                   "note": "iterations/s is per iteration of the SAMPLE; state-timesteps/s is size-independent"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": out["threads"], "kind": "port",
                         "sample": f"{sample} samples ({w.N} trajectories), {args.warmup + args.steps} iterations, "
                                   f"{out['secs']:.2f} s loop time"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--samples", type=int, default=256, help="ensemble samples (256 = BASELINE C4)")
    ap.add_argument("--n-grid", type=int, default=2001, help="time-grid points (2001 = BASELINE C4)")
    ap.add_argument("--ref-samples", type=int, default=32, help="bounded sample for the CPU arm")
    ap.add_argument("--ref-threads", type=int, default=0, help="host threads of the CPU arm (0 = all cores this "
                    "process may run on; never the OpenMP default, which torchrun pins to 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the C1/C2/C3/C5 block of the JSON line")
    ap.add_argument("--multi-gpu", choices=["auto", "shard", "replicate"], default="auto",
                    help="several ranks: shard the trajectories (per-step exchange) or replicate the forward sweep")
    ap.add_argument("--scaling", choices=["strong", "weak"], default="strong",
                    help="strong: the BASELINE ensemble sharded over the ranks; weak: --samples per rank")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed iteration to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    if args.impl == "reference":
        run_reference(args)
        return

    # stdout carries exactly ONE JSON line: anything a library prints there (NCCL's version banner, ...) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch

    import krotov_jl_b200 as K
    from util import to_problem

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        from krotov_jl_b200.distributed import Comm

        comm = Comm(device=local_rank)

    n_samples = args.samples * (world if args.scaling == "weak" else 1)
    w = W.c4_ensemble(n_samples=n_samples, n_grid=args.n_grid)
    N, N_T, d, L = w.N, w.N_T, w.d, w.L
    steps, warmup = args.steps, max(args.warmup, 3)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            comm.barrier()
            torch.cuda.synchronize()

    # ---- timed run through the public API; device time is read from the handle after every iteration
    dev_ms, launches, marks = [], [], {}
    sampler = ClockSampler(local_rank)
    sampler.prepare()

    def cb(wrk, it, eps_new, eps_old):
        marks.setdefault("wall", []).append(time.perf_counter())
        if it >= 1:
            info = wrk.engine.info()
            dev_ms.append(info["ms_last"])
            marks.setdefault("rank_wait", []).append(round(info.get("ms_rank_wait", 0.0), 3))
            launches.append(info["launches_last"])
            marks["info"] = info
        if it == warmup:
            sampler.start()
            barrier()
            marks["t0"] = time.perf_counter()
            marks["wall"][-1] = marks["t0"]  # per-iteration list starts where the timed region starts
        if it == warmup + steps:
            barrier()
            marks["t1"] = time.perf_counter()
            marks["clocks"] = sampler.stop()
            if args.dump_outputs:
                marks["pulses"] = np.array([np.array(e) for e in eps_new])
                marks["g_a_int"] = np.array(wrk.g_a_int)
        marks["J_T"] = wrk.result.J_T
        marks["m_fw"] = int(wrk.fw_settings.coeff_count.max())
        marks["m_bw"] = int(wrk.bw_settings.coeff_count.max())
        marks["shard"] = wrk._shard

    problem = to_problem(w, iter_stop=warmup + steps, callback=cb, device=local_rank, multi_gpu=args.multi_gpu)
    res = K.optimize(problem, method=K.Krotov, comm=comm)
    if res.message.startswith("Exception"):
        raise SystemExit(f"optimisation failed: {res.message}")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, marks["pulses"], marks["g_a_int"], res)

    timed_ms = np.array(dev_ms[warmup:warmup + steps])
    dev_total_ms = float(timed_ms.sum())
    wall_s = marks["t1"] - marks["t0"]
    per_rank = None
    if world > 1:
        # per-rank record (device ms and host wall ms of every timed iteration, time spent at the rank barrier): the line
        # reports the MAX over ranks, this shows where it comes from
        mine = {"rank": rank, "dev_ms": [round(float(x), 2) for x in timed_ms],
                "wall_ms": [round(1e3 * (b - a), 2) for a, b in zip(marks["wall"][warmup:warmup + steps], marks["wall"][warmup + 1:warmup + steps + 1])],
                "timed_region_ms": round(1e3 * wall_s, 2), "J_T_last": marks["J_T"], "rank_wait_ms": marks.get("rank_wait", [])[warmup:warmup + steps]}
        per_rank = comm.all_gather_object(mine)
        t = torch.tensor([dev_total_ms, wall_s], dtype=torch.float64, device="cuda")
        import torch.distributed as dist

        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_total_ms, wall_s = float(t[0]), float(t[1])
    st_per_iter = 2.0 * N * N_T
    value = st_per_iter * steps / (dev_total_ms * 1e-3)
    e2e = st_per_iter * steps / wall_s

    if rank == 0:
        peaks, peak_src = load_peaks()
        info = marks["info"]
        m = max(marks["m_fw"], marks["m_bw"])
        # algorithmic bytes per launch (SURVEY.md 8d): the chi trajectory written once and read once
        lo, hi = marks["shard"]
        n_loc = hi - lo
        alg_bytes = 16.0 * d * n_loc * (2 * N_T + 1)
        ms_launch = dev_total_ms / steps
        ach_gbs = alg_bytes / (ms_launch * 1e-3) / 1e9
        nnz = info["nnz_union"]
        flops = 2.0 * n_loc * N_T * (m - 1) * 8 * nnz + n_loc * N_T * L * 8 * (nnz + d)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if world == 1 and args.samples == 256 and args.n_grid == 2001 and os.path.exists(tpath):
            with open(tpath) as fh:  # measured once under ncu for exactly this launch shape
                traffic = json.load(fh).get("krotov_warp_kernel<6,2,256,32> on C4 (1024 trajectories, N_T=2000)")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": dev_total_ms / steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "iterations_per_s": steps / (dev_total_ms * 1e-3),
            "config": {"workload": f"C4 robust two-transmon CNOT ensemble: {n_samples} samples x 4 basis states = "
                                   f"{N} trajectories, d={d}, L={L}, N_T={N_T}, Chebyshev m={m}",
                       "parallelism": (f"backward sweep sharded over {world} GPUs, forward sweep replicated on each"
                                       if info.get("exchange") == 5 else f"trajectories sharded over {world} GPU(s)"),
                       "l2": "chi trajectory (%.0f MB per GPU) is larger than L2; no flush needed" % (info["hbm_bytes_state"] / 1e6),
                       "grid": [info["grid_blocks"], info["block_threads"]], "J_T_last": marks["J_T"],
                       **({"rank_barrier_wait_ms_last": round(info.get("ms_rank_wait", 0.0), 3)} if info.get("exchange") == 5 else {}),
                       **({"exchange": {1: "per time step, in-kernel: every CTA adds its fixed-point partial into its rank's "
                                           "accumulator; the add that completes a word forwards the rank sum with one add per "
                                           "rank over NVLink (hierarchical sum)",
                                        2: "per time step, in-kernel over NVLink: every CTA adds its fixed-point partial into "
                                           "every rank's accumulator (one hop)",
                                        3: "per time step, in-kernel over NVLink: rank sums pushed into the peers' mailboxes",
                                        4: "per time step, in-kernel: hierarchical sum, rank sums forwarded with plain stores "
                                           "into per-rank slots over NVLink",
                                        5: "none per time step: every rank holds all trajectories; the backward sweep is "
                                           "sharded and writes chi to every rank over NVLink (one rank barrier per iteration), "
                                           "the time-serial forward sweep runs on every rank (replicated forward sweep)"}.get(info.get("exchange"), "?")} if world > 1 else {})},
            "e2e": {"value": e2e, "unit": UNIT, "iterations_per_s": steps / wall_s,
                    "h2d_bytes_per_step": L * N_T * 8, "d2h_bytes_per_step": L * N_T * 8 + L * 8 + n_loc * 16,
                    "ms_per_step_each": [round(1e3 * (b - a), 2) for a, b in zip(marks["wall"][warmup:warmup + steps], marks["wall"][warmup + 1:warmup + steps + 1])]},
            "gpu_launches": int(sum(launches[warmup:warmup + steps])),
            "clocks": marks["clocks"],
            "roofline": {"bound": "hbm", "achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": ach_gbs / peaks["hbm_gbs"], "traffic": traffic,
                         "traffic_source": "profiles/r2_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of ONE "
                                           "ncu --set full capture of this launch shape (profiles/r2_warp_kernel_ncu_full.txt), "
                                           "NOT measured in this run; "
                                           "1.25x the algorithmic bytes because d = 25 states sit in 32-entry records",
                         "peak_source": peak_src,
                         "kernel": "krotov_warp_kernel", "algorithmic_bytes_per_launch": alg_bytes,
                         "note": "the fused kernel keeps all Chebyshev vectors on chip, so HBM traffic is only the chi "
                                 "trajectory; the binding resource is the shared-memory crossbar (see roofline_smem "
                                 "and DESIGN.md 4.1)"},
            "roofline_smem": smem_roofline(n_loc, N_T, marks["m_fw"] + marks["m_bw"] - 2, info["ell_width"],
                                           info["sm_count"], marks["clocks"]["sm_max_mhz"] or 1965.0, ms_launch),
            "roofline_fp64": {"achieved_tflops": flops / (ms_launch * 1e-3) / 1e12, "flops_per_launch": flops,
                              "peak_tflops": 34.2, "peak_source": "self-measured DFMA peak on this pool's B200 "
                              "(tools/microbench.cu, profiles/r1_microbench_fp64.txt; DMMA: 37.1)",
                              "frac": flops / (ms_launch * 1e-3) / 1e12 / 34.2,
                              "bound": "not the FP64 pipe: shared-memory crossbar (roofline_smem) in the sweeps, exchange "
                                       "latency between the time steps of the forward sweep"},
        }
        if per_rank is not None:
            line["per_rank"] = per_rank
        if world == 1 and not args.no_extra_configs and args.samples == 256:
            line["extra_configs"] = extra_configs(K, to_problem, peaks)
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline_sample(w, min(args.samples, 128), 2)
            except Exception as exc:  # the baseline is a report, never a reason to lose the GPU number
                line["cpu_baseline"] = {"error": str(exc)}
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
