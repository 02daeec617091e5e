"""Device time per Krotov iteration of C4 at full size (256 samples, 2001 grid points) with control 0 entering
  - linear:  (H_re, eps_0)                                               -- two controls, two terms
  - shaped:  (H_re, ShapedAmplitude(eps_0, cos(D t)))                     -- two controls, two terms, non-linear path
  - cos/sin: the shaped term and (conj(H_re)/2, ShapedAmplitude(eps_0, sin(D t))) tied to it -- three terms
and a rotating-frame problem with two controls, each a cos/sin pair (four terms: the runtime-L row-reloading instance,
the register-resident rows stop at three terms).  The tied forms add the comm warp's tie (tie_sum_cold) between the
exchange and barrier B of every time step.

    python tools/gpu_control_terms_cost.py [--iters 8] [--reps 3] [--out profiles/r3_control_terms_cost.txt]

Records krotov_info.ms_last (CUDA events around the launches of one krotov_iterate) for every iteration after the first
two, the kernel that ran (krotov_info.kernel) and the GPU name and power limit read in the same run.  Needs a GPU."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import krotov_jl_b200 as K  # noqa: E402
import terms_reference as R  # noqa: E402
import workloads as W  # noqa: E402

KERNELS = {1: "tiny", 2: "preg", 3: "seq_preg", 4: "pair", 5: "reload", 6: "dmma_stream", 7: "dense_sweep",
           8: "sparse_sweep", 9: "sparse_stream"}


def case(kind):
    w = W.c4_ensemble()
    c = R.tie_workload(w)  # terms: control 0 (cos), control 1, control 0 (sin)
    if kind == "linear":
        c.ops, c.term_ctrl, c.poly, c.shape = [r[:2] for r in c.ops], [0, 1], [None, None], [None, None]
    elif kind == "shaped":
        c.ops, c.term_ctrl, c.poly, c.shape = [r[:2] for r in c.ops], [0, 1], [None, None], c.shape[:2]
    elif kind == "four_terms":  # control 1 as a cos/sin pair as well
        D = 2 * np.pi * 1.5 / float(w.tlist[-1])
        c.ops = [r + [0.5 * r[1].conj()] for r in c.ops]
        c.term_ctrl, c.poly = [0, 1, 0, 1], [None] * 4
        c.shape = [c.shape[0], lambda t: np.cos(D * t), c.shape[2], lambda t: np.sin(D * t)]
        c.guess = [c.guess[0], lambda t, g=c.guess[0]: 0.5 * g(t)]
    return c


def run(kind, iters):
    ms, info = [], {}

    def cb(wrk, it, *_):
        if it >= 3:  # iterations 1 and 2 include first launches and the first spectral-range updates
            ms.append(wrk.engine.info()["ms_last"])
            info.update(wrk.engine.info())

    c = case(kind)
    c.iters = iters
    K.optimize(c.problem(callback=cb), method=K.Krotov)
    return ms, KERNELS.get(info.get("kernel"), info.get("kernel")), info.get("grid_blocks")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [f"GPU: {gpu}", "C4 full size (256 samples, 2001 grid points), one GPU; ms = krotov_info.ms_last per iteration "
             f"(iterations 3..{a.iters}), {a.reps} runs per kind, kinds alternated"]
    kinds = ("linear", "shaped", "cos_sin", "four_terms")
    res = {k: [] for k in kinds}
    meta = {}
    for _ in range(a.reps):
        for k in kinds:
            ms, kern, blocks = run(k, a.iters)
            res[k] += ms
            meta[k] = (kern, blocks)
    for k, v in res.items():
        v = np.array(v)
        lines.append(f"{k:10s} median {np.median(v):8.3f} ms  min {v.min():8.3f}  max {v.max():8.3f}  (n={v.size})  "
                     f"kernel {meta[k][0]}, {meta[k][1]} CTAs")
    for k, b in (("shaped", "linear"), ("cos_sin", "shaped"), ("four_terms", "cos_sin")):
        d = np.median(res[k]) - np.median(res[b])
        lines.append(f"{k} - {b}: {d:+.3f} ms per iteration = {1e3 * d / 2000:+.4f} us per forward time step")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
