"""unconfined_b200 -- B200-native evaluator of klkuhlm/unconfined's double-precision
Laplace-Hankel drawdown solutions (the loop nest driver.f90:100-231 of the reference).

The product is the C-ABI shared library ``libunconfined_b200.so`` (include/unconfined_b200.h,
hand-written sm_100a kernels).  This package is the thin host-side mirror used from Python:
``api`` binds the C ABI with ctypes (host arrays) and with torch device pointers (resident
arrays); ``build`` compiles the library in-tree with nvcc.  There is no CPU fallback: every
evaluation call raises if the library or a CUDA device is missing.
"""
from .api import (UncParams, Params, UncError, lib, eval_grid, eval_points, eval_points_device,  # noqa: F401
                  eval_grid_device, eval_screens, eval_screens_device, eval_points_dz,
                  eval_points_dz_device, j0_zeros, split_index, zlay, device_count, set_device,
                  measure_fp64_peak, device_info, kernel_launch_count, shutdown, last_error,
                  set_carry, force_kernel, debug_cbesk01)
from .build import build  # noqa: F401
