"""timberborn_support_solver_b200 — B200 (sm_100a) upper-bound engine for Timberborn ceiling-support placement.

The product is libtss.so (include/tss.h, sources under csrc/); this package is the host-side mirror of the reference
library's interface for the feasibility-and-bound path, bound to it through ctypes.  Importing the package needs
the built library; creating an Engine needs a CUDA device.  There is no CPU fallback.
"""
from ._lib import LIB_PATH, SIGNATURES, load  # noqa: F401
from .api import (INTERRUPTED, KERNEL_AUTO, KERNEL_HALF_WARP, KERNEL_PAIR, KERNEL_THREAD, KERNEL_WARP, KERNEL_WINDOW_PLACEMENTS, PLATFORMS_DEFAULT, SAT, UNSAT, Cnf, DeviceCnf, Encoding, EncodingVars, Engine,  # noqa: F401
                  GpuBoundSolver, Platform, PlatformDef, PlatformLayout, PlatformLimits, Project, Search, TssError, card_limit_classes,
                  ValidationResult, World, WorldGrid, render_world, solver_loop, weight_loop)

load()  # fail loudly at import time if libtss.so is missing or does not export every declared symbol
