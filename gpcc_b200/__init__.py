"""gpcc_b200 -- host-side mirror of the GPCC.jl public API over the sm_100a CUDA library.

The exported names, keyword arguments and return shapes follow the reference
(/root/reference/src/GPCC.jl:30-31, src/gpccfixdelay_marginaliseb.jl:46-53,351,
src/getprobabilities.jl:1-20, src/uniformpriordelay.jl:10-16) so that the parity tests read like the
reference's README.  All arithmetic on the hot path happens in libgpcc_b200.so (CUDA); this package only
marshals arrays.  Julia callers bind the same C ABI through julia/GPCC_B200.jl (see INTEGRATION.md).
"""
from .api import (Context, Problem, gpcc, gpccgrid, getprobabilities, uniformpriordelay, Uniform, MvNormal,  # noqa: F401
                  OU, rbf, matern32, matern52, initial_solutions, default_context, GpccError, performcv, cv_folds,
                  FitState, StateSpaceFitState, comm_unique_id, simulatedata_device)
from .synthetic import simulatetwolightcurves, simulatethreelightcurves, simulatedata, synthetic_bands  # noqa: F401,E402
