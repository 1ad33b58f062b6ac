"""tron_b200 -- B200-native batched 2-player TRON environment + GPU replay ring.

Hot path of ckawoalt/Deep-Q-Learning_TRON (Game.step / state_for_player / pop_up / replay), rebuilt
as hand-written sm_100a CUDA kernels behind a C ABI (include/tron_b200.h).  Python here is only the
host-side mirror of the reference's object surface plus a vectorised batch API; torch is used for
device memory and streams.  There is no CPU fallback: compute calls raise if the CUDA library or a
GPU is missing.
"""
from . import _abi as abi  # noqa: F401

__all__ = ["abi", "lib", "BatchedTron", "ReplayRing", "StateRing"]


def __getattr__(name):  # lazy: importing the package must not require torch / a built library
    if name == "lib":
        from . import _lib
        return _lib
    if name == "BatchedTron":
        from .batch_env import BatchedTron
        return BatchedTron
    if name == "ReplayRing":
        from .replay import ReplayRing
        return ReplayRing
    if name == "StateRing":
        from .replay import StateRing
        return StateRing
    raise AttributeError(name)
