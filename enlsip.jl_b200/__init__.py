"""enlsip.jl_b200 -- B200-native batched ENLSIP Gauss-Newton engine behind the Enlsip.jl API.

Host-side mirror of the reference interface for the hot path (``CnlsModel`` / ``solve!`` /
``status`` / ``solution`` / ``sum_sq_residuals``; reference src/cnls_model.jl:145-221,
src/solver.jl:62-91) over the C ABI of ``include/enlsip_b200.h``.  The product path is the CUDA
library only: importing works without a GPU, but every solve raises if the extension or a CUDA
device is missing -- there is no CPU fallback.
"""
from . import capi, synth
from .model import (CnlsModel, UserFamily, solve, solve_b, status, solution, sum_sq_residuals, constraints_values,
                    total_nb_constraints, dict_status_codes, evaluate, gn_step)
from .model_large import LargeCnlsModel, LargeUserFamily, shard_rows, solve_large

__all__ = ["capi", "synth", "CnlsModel", "UserFamily", "solve", "solve_b", "status", "solution", "sum_sq_residuals",
           "constraints_values", "total_nb_constraints", "dict_status_codes", "evaluate", "gn_step", "LargeCnlsModel", "LargeUserFamily", "shard_rows",
           "solve_large"]
