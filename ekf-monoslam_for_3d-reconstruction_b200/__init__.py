"""B200-native MonoSLAM EKF hot path (predict / active-search match / update) behind the reference's
VSlamFilter interface.  The compute path is libekf_b200.so (hand-written sm_100a CUDA, C ABI in
include/ekf_b200.h); this package is the thin Python host mirror used by tests and bench.py.

The directory name is not a valid Python identifier; import it with `load_package()` from the
repository root's `ekfb200.py` shim, which registers it as module `ekf_b200`.
"""
from . import _abi, dist, keyframes, synth  # noqa: F401
from ._abi import EkfBatchDesc, EkfConfig, EkfFeatureInfo, EkfStepStats, default_config  # noqa: F401
from .build import build  # noqa: F401


def __getattr__(name):  # lazy: importing the package must not require the built library
    if name in ("VSlamFilter", "EkfError", "match_batch", "FilterBatch", "systematic_ancestors", "nccl_unique_id", "load_nccl"):
        from . import filter as _f
        return getattr(_f, name)
    if name == "lib":
        from ._lib import lib as _l
        return _l
    raise AttributeError(name)
