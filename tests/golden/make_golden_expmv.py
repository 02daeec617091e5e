"""Exact-propagator vector of a dissipative problem (the propagator `prop_method=Expmv` exists for): the driven qubit
with amplitude damping in Liouville space, gamma = 1 and 2, two density-matrix trajectories, J_T_re
(tests/expmv_reference.py damped_qubit), optimised by the 40-digit loop of tests/mp_reference.py with mpmath.expm per
interval.

    python tests/golden/make_golden_expmv.py"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import expmv_reference as X  # noqa: E402
import mp_reference as M  # noqa: E402
import workloads as W  # noqa: E402

ITERS = 3
h = M.krotov_exact_general(W.to_oracle(X.damped_qubit()), ITERS)
out = {"source": f"tests/mp_reference.py krotov_exact_general(expmv_reference.damped_qubit()), mpmath dps=40, "
                 "mpmath.expm per interval", "iters": ITERS, "J_T": h["J_T"], "g_a_int": h["g_a_int"], "pulses": h["pulses"],
       "tau_re": [t.real for t in h["tau"]], "tau_im": [t.imag for t in h["tau"]]}
with open(os.path.join(HERE, "damped_qubit_exact40.json"), "w") as fh:
    json.dump(out, fh)
print("damped_qubit", out["J_T"])
