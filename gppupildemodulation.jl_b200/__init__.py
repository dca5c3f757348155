"""gppd-b200: B200-native (sm_100a) implementation of GPPupilDemodulation.jl's
``demodulateall`` hot path behind the reference's own interface.

    import gppd_b200 as gp
    output, param, likelihood = gp.demodulateall(times, cmplxV)

The numerics live in ``libgppd.so`` (hand-written CUDA, C ABI in
``include/gppd.h``); this package is the host-side mirror of the reference's
Julia API.  There is no CPU fallback: without the built library and a B200 the
calls raise ``GppdError``.
"""
from . import sharding, synthetic  # noqa: F401
from ._lib import GppdError, Handle, build, default_handle  # noqa: F401
from .api import (D1, D2, D3, D4, FC, FT, HIGH, LOW, M_2PI, NORMAL, OFF, SC,  # noqa: F401
                  TRANSIENT, Diode, FaintStates, MetState, ModulationNoOffsets,
                  ModulationWithOffsets, Side, buildfaintparameters, buildstates, covariances,
                  demodulateall, ellipse_keys, ellipses, idx, process_table, processmetrology, read_stefan_file,
                  table_windows, uncertainty_keys, window_uncertainty_columns)
