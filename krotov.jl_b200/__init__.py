"""krotov_jl_b200 -- B200-native Krotov iteration behind the API of JuliaQuantumControl/Krotov.jl.

    from krotov_jl_b200 import *
    problem = ControlProblem([Trajectory(psi0, hamiltonian(H0, (H1, eps)), target_state=tgt)], tlist,
                             iter_stop=5, prop_method=Cheby, J_T=J_T_sm, lambda_a=1.0)
    result = optimize(problem, method=Krotov)

The package directory is ``krotov.jl_b200/`` (not importable by that name); ``krotov_jl_b200.py`` at the
repo root registers it under the import name ``krotov_jl_b200``.  Host code here mirrors the reference's
interface; all propagation runs in ``libkrotov_cuda.so`` (``csrc/``), with no CPU fallback.
"""
from .controls import discretize, discretize_on_midpoints, get_control_derivs, get_controls
from .errors import ArgumentError, ErrorException
from .functionals import J_T_re, J_T_sm, J_T_ss, chi_re, chi_sm, chi_ss, make_chi, taus
from .generators import (Generator, LogisticParametrization, LogisticSqParametrization, ParametrizedAmplitude,
                         PolynomialAmplitude, ShapedAmplitude, SquareParametrization, TanhParametrization,
                         TanhSqParametrization, hamiltonian)
from .optimize import (Cheby, Expmv, Krotov, finalize_result, krotov_initial_fw_prop, krotov_iteration,
                       make_krotov_print_iters, make_print_iters, optimize, optimize_krotov, update_result,
                       update_sigma)
from .problem import ControlProblem, Trajectory
from .result import KrotovResult
from .second_order import NumericalSigma, Sigma, numerical_estimate_A
from .shapes import blackman, box, flattop
from .cheby import cheby_coeffs, specrange, transform_control_ranges
from .workspace import IdDict, KrotovWrk
from .engine import KrotovCuda
from ._lib import KrotovCudaError

__version__ = "0.1.0"
