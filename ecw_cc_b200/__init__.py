"""ecw_cc_b200 — B200-native (sm_100a) coupled-cluster residual path of ECW_CC.

Host-side mirror of the reference's `CCSD.GCC` / `CCS.Gccs` method surface
(same names, argument order and return conventions) over a C-ABI CUDA library
(`libecw_b200.so`, declared in include/ecw_b200.h).  There is no CPU fallback:
every compute call needs a CUDA device and the built library.
"""
from ._lib import lib, build, LIB_PATH, EcwError  # noqa: F401
from .eris import DeviceEris  # noqa: F401
from .CCSD import GCC, gamma_CCSD  # noqa: F401
from .CCS import Gccs  # noqa: F401
from .devops import DevOps  # noqa: F401
from .utilities import subdiff  # noqa: F401
from .Solver_GS import Solver_CCSD  # noqa: F401
from .harness import Solver_CCS, Solver_ES  # noqa: F401  (test harness: callers of the path, see harness/__init__.py)
from . import exp_pot  # noqa: F401
from . import molint  # noqa: F401
from . import maps  # noqa: F401

__all__ = ["GCC", "Gccs", "Solver_CCSD", "Solver_CCS", "Solver_ES", "DevOps", "DeviceEris", "subdiff", "gamma_CCSD", "build", "lib", "EcwError"]
