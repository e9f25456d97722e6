"""rlfluidcontrol_b200 -- B200-native batched Lilypad AFCCylinder environments.

The product is the C-ABI shared library `librlfc.so` (include/rlfc.h) built from csrc/ for sm_100a;
this package is the thin Python mirror of the reference's environment interface
(clientLilypad/AFCCylinder.pde + clientCFD.pde) on top of it.  There is no CPU fallback: creating an
environment without the CUDA library / a CUDA device raises.
"""
from .env import AFCCylinderBatch, RlfcError, Config, EnvParams, load_library, library_path, default_init_state  # noqa: F401
from .env import STAT_NAMES, flow_stats_from_sums  # noqa: F401
from .records import parse_record  # noqa: F401

__version__ = "0.1.0"
