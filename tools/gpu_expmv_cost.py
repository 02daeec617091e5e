"""Device time per Krotov iteration under prop_method=Cheby and prop_method=Expmv (krotov_info.ms_last, medians) for
C1-C4 and a damped-qubit ensemble; card name and power limit from the same run.

    python tools/gpu_expmv_cost.py [out_path]     (default profiles/r3_expmv_cost.txt)"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402

import expmv_reference as X  # noqa: E402
import krotov_jl_b200 as K  # noqa: E402
import workloads as W  # noqa: E402
from util import run_product  # noqa: E402

ITERS = 6  # the first iteration (range events, first launch) is dropped from the median

CASES = [("C1 tls (d=2, N_T=500)", W.c1_tls), ("C2 transmon (d=3, N_T=500)", W.c2_transmon_x),
         ("C3 two transmons (d=25, N_T=2000)", W.c3_two_transmon),
         ("C4 ensemble 1024 traj (d=25, N_T=2000)", lambda: W.c4_ensemble(n_samples=256)),
         ("damped qubit ensemble 300 traj (d=4, N_T=2000)", lambda: X.damped_ensemble(n_samples=300, n_grid=2001, T=40.0))]


def measure(make, method):
    ms = []

    def cb(wrk, it, *_):
        if it > 1:
            ms.append(wrk.engine.info()["ms_last"])

    h = run_product(make(), ITERS, prop_method=method, callback=cb)
    info = h["info"]
    return float(np.median(ms)), info["m_fw"], info["kernel"]


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_expmv_cost.txt")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    lines = [f"card: {card}", f"device ms per Krotov iteration (krotov_info.ms_last), median of iterations 2..{ITERS}",
             f"{'case':48s} {'Cheby ms':>9s} {'terms':>6s} {'Expmv ms':>9s} {'m*s':>6s}  Expmv/Cheby"]
    for name, make in CASES:
        cm, cterms, _ = measure(make, K.Cheby) if not name.startswith("damped") else (float("nan"), 0, 0)
        em, eterms, kern = measure(make, K.Expmv)
        assert kern == K._lib.KERNEL_TAYLOR
        lines.append(f"{name:48s} {cm:9.3f} {cterms:6d} {em:9.3f} {eterms:6d}  {em / cm:10.2f}")
        print(lines[-1], flush=True)
    lines.append("damped ensemble: Chebyshev not run (its window misses strong decay, see tests/test_expmv.py)")
    with open(out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
