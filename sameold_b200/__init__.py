"""sameold_b200 — B200-native batched SAME/EAS receiver engine (hot path of cbs228/sameold, rebuilt for sm_100a).

The package is a thin host layer over the CUDA engine (sameold_b200/csrc -> sameold_b200/_build/libsame_b200.so, C ABI
in include/same_engine.h).  Importing the receiver classes does not need a GPU; building an engine does — there is no
CPU fallback anywhere in this package.
"""
from .receiver import (  # noqa: F401
    EqualizerBuilder,
    Message,
    SameBatchReceiver,
    SameEngineError,
    SameMultiReceiver,
    SameReceiver,
    SameReceiverBuilder,
    SameReceiverEvent,
    state_info,
)
from .build import build_native  # noqa: F401

__version__ = "0.1.0"
