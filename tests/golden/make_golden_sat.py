"""Golden vector for bounded (saturating) amplitudes that does NOT come from the oracle: the two-level system of
test/test_tls_optimization.jl:12-63 with the control entering through TanhParametrization(-0.5, 0.5), i.e.
H = -sz/2 + 0.5 tanh(u) sx, optimised in 50-digit arithmetic with the closed-form propagator of every interval
(tests/sat_reference.py tls_tanh_exact).

    python tests/golden/make_golden_sat.py"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import mpmath as mp  # noqa: E402

import sat_reference as S  # noqa: E402

CASES = {"c1_tls_tanh_exact50": dict(iters=5, amp_poly=(0.0, 0.5), amp_sat=1.0)}

for name, kw in CASES.items():
    h = S.tls_tanh_exact(**kw)
    out = {"source": "tests/sat_reference.py tls_tanh_exact(%s), mpmath dps=50" % ", ".join(f"{k}={v}" for k, v in kw.items()),
           "J_T": [float(x) for x in h["J_T"]], "J_T_30_digits": [mp.nstr(x, 30) for x in h["J_T_mp"]],
           "g_a_int": h["g_a_int"], "pulses": h["pulses"], "amp_poly": list(kw["amp_poly"]), "amp_sat": kw["amp_sat"]}
    with open(os.path.join(HERE, name + ".json"), "w") as fh:
        json.dump(out, fh)
    print(name, out["J_T_30_digits"])
