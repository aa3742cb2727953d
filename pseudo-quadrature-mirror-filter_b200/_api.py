from .design import (center_pad_next_pow_2, get_prototype, get_qmf_bank, kaiser_filter, loss_wc, make_odd)
from .pqmf import (PQMF, CachedPQMF, classic_forward, classic_inverse, polyphase_forward, polyphase_inverse, reverse_half)
from . import _lib
from ._lib import launch_count, library_paths
from .sharding import shard_rows
from .streaming import StreamGraph, StreamPool

__all__ = [
    "PQMF", "CachedPQMF", "reverse_half", "polyphase_forward", "polyphase_inverse", "classic_forward", "classic_inverse",
    "get_prototype", "get_qmf_bank", "kaiser_filter", "loss_wc", "center_pad_next_pow_2", "make_odd", "launch_count",
    "library_paths", "shard_rows", "StreamGraph", "StreamPool",
]
