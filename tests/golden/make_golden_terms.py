"""Golden vectors for controls that enter through several (operator, amplitude) terms, NOT from the oracle: the problems
of tests/terms_reference.py CASES optimised in 40-digit arithmetic with mpmath.expm for every interval
(terms_reference.krotov_exact_terms).

    python tests/golden/make_golden_terms.py"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import terms_reference as R  # noqa: E402

for name, make in R.CASES.items():
    case = make()
    p, term_ctrl = case.oracle_arrays()
    h = R.krotov_exact_terms(p, term_ctrl, iters=case.iters, dps=40)
    out = {"source": f"tests/terms_reference.py krotov_exact_terms(CASES[{name!r}]()), mpmath dps=40",
           "iters": case.iters, "term_ctrl": [int(c) for c in term_ctrl], **h}
    with open(R.golden_path(name), "w") as fh:
        json.dump(out, fh)
    print(name, out["J_T"])
