"""versatilefilmgrain_b200 -- B200-native (sm_100a) back end for the VFGS hardware-layer hot path.

The product is the C-ABI shared library ``libvfgs_b200.so`` (sources in ``csrc/``, interface in
``include/vfgs_hw.h`` + ``include/vfgs_b200.h``). This package only builds it and mirrors its
interface for Python callers (tests, bench); there is no Python or CPU compute path.
"""
from .api import Job, Session, VfgsHw, VfgsError, load_library, LIB_PATH  # noqa: F401
from .build import build  # noqa: F401
