"""Device time per Krotov iteration of C4 at full size (256 samples, 2001 grid points) with the control entering
linearly, through a polynomial (eps + 2 eps^2 on control 0) and through TanhParametrization on both controls.  The
non-linear forms add the comm warp's amplitude evaluation (amp_eval_cold, with a tanh for the parametrization) between
the exchange and barrier B of every time step.

    python tools/gpu_amplitude_cost.py [--iters 8] [--reps 3] [--out profiles/r3_amplitude_cost.txt]

Records krotov_info.ms_last (CUDA events around the launches of one krotov_iterate) for every iteration after the first
two, and the GPU name and power limit read in the same run.  Needs a GPU."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import krotov_jl_b200 as K  # noqa: E402
import sat_reference as S  # noqa: E402
import workloads as W  # noqa: E402


def run(kind, iters):
    w = W.c4_ensemble()
    params = [None] * len(w.controls)
    if kind == "polynomial":
        w.amp_poly = [[0.0, 1.0, 2.0]] + [None] * (len(w.controls) - 1)
    elif kind == "tanh":
        a = [max(float(np.abs(K.discretize(c, w.tlist)).max()), 0.1) for c in w.controls]
        params = [K.TanhParametrization(-2 * x, 2 * x) for x in a]
    ms = []

    def cb(wrk, it, *_):
        if it >= 3:  # iterations 1 and 2 include first launches and the first spectral-range updates
            ms.append(wrk.engine.info()["ms_last"])

    K.optimize(S.param_problem(w, params, iter_stop=iters, callback=cb), method=K.Krotov)
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [f"GPU: {gpu}", "C4 full size (256 samples, 2001 grid points, 2 controls), one GPU; ms = krotov_info.ms_last "
             f"per iteration (iterations 3..{a.iters}), {a.reps} runs per kind, kinds alternated"]
    res = {k: [] for k in ("linear", "polynomial", "tanh")}
    for _ in range(a.reps):
        for k in res:
            res[k] += run(k, a.iters)
    for k, v in res.items():
        v = np.array(v)
        lines.append(f"{k:10s} median {np.median(v):8.3f} ms  min {v.min():8.3f}  max {v.max():8.3f}  (n={v.size})")
    base = np.median(res["linear"])
    for k in ("polynomial", "tanh"):
        d = np.median(res[k]) - base
        lines.append(f"{k} - linear: {d:+.3f} ms per iteration = {1e3 * d / 2000:+.4f} us per forward time step")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
