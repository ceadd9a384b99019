"""v2ce_toolbox_b200 -- B200 (sm_100a) implementation of the V2CE video->continuous-events
hot path behind the reference's own Python API (v2ce.py / scripts/*).

Host code is Python/PyTorch plumbing (device memory, streams, torch.distributed); every
device computation is hand-written CUDA in libv2ce_b200.so, reached through the C ABI of
include/v2ce_b200.h.  No CPU fallback: CPU tensors and a missing library raise.
"""
from ._lib import V2ceError, load  # noqa: F401
from .clip_stream import ClipStream  # noqa: F401
from .voxelize import events_to_voxels  # noqa: F401

__version__ = '0.1.0'
