"""
yet_another_wizz_b200 -- B200-native pair-counting engine behind the public API
of yet_another_wizz (`crosscorrelate` / `autocorrelate`).

Only the hot path lives here (SURVEY.md section 8): CUDA kernels + C ABI under
`csrc/`, and the thin Python host that mirrors the reference's interface for
that path.  There is no CPU fallback.
"""

from ._lib import YawbError
from .binning import Binning
from .catalog import Catalog, InconsistentPatchesError
from .config import Configuration
from .coordinates import AngularCoordinates, AngularDistances
from .corrfunc import CorrFunc, ScalarCorrFunc
from .engine import DeviceCatalog, Engine, EngineGroup
from .measurements import (PatchLinkage, autocorrelate, autocorrelate_scalar, autocorrelate_tomographic,
                           crosscorrelate, crosscorrelate_scalar, crosscorrelate_tomographic)
from .randoms import BoxRandoms

__all__ = [
    "AngularCoordinates", "AngularDistances", "Binning", "BoxRandoms", "Catalog", "Configuration", "CorrFunc",
    "DeviceCatalog", "Engine", "EngineGroup", "InconsistentPatchesError", "PatchLinkage", "ScalarCorrFunc", "YawbError",
    "autocorrelate", "autocorrelate_scalar", "autocorrelate_tomographic", "crosscorrelate", "crosscorrelate_scalar",
    "crosscorrelate_tomographic",
]
__version__ = "0.1.0"
