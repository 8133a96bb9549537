"""fastselect_b200 -- B200-native (sm_100a) Relief-family feature scoring.

Drop-in for the GPU backend of ``fast_select.{ReliefF, SURF, MultiSURF, TuRF}``
(reference: src/fast_select/__init__.py:1-10) and, on the same one-hot tensor-core kernels, of the
joint-count selectors ``fast_select.{mRMR, CFS}`` / ``fast_select.mutual_information``, plus this
project's own ``MDR`` (two-locus interaction search on a bit-sliced count kernel).  The
estimators call hand-written CUDA through the C ABI in ``include/fastselect_b200.h``; nothing here
falls back to a CPU.
"""
from . import _mi as mutual_information
from ._mdr import MDR
from ._mi import CFS, mRMR
from ._relief import MultiSURF, ReliefF, SURF
from ._shard import enable_distributed, set_gpus
from ._turf import TuRF

__all__ = ["ReliefF", "SURF", "MultiSURF", "TuRF", "mRMR", "CFS", "MDR", "mutual_information", "enable_distributed", "set_gpus"]
__version__ = "0.1.0"
