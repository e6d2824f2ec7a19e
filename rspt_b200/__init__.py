"""rspt_b200 -- B200-native (sm_100a) implementation of rspt's signal-packer hot path.

Only what the path needs: `csrc/` (CUDA kernels + the C ABI of include/rspt_gpu.h), the C++
drop-in for lib_rspt/signal_packer.h, and this thin Python host mirror.  There is no CPU path.
"""
from ._lib import KINDS, RsptError  # noqa: F401


def __getattr__(name):
    # torch is imported lazily so that `import rspt_b200` (and the symbol-export test) works
    # in processes that never touch the GPU
    if name in ("SignalPacker", "CompressedBatch", "CompressedStore", "crc32c", "synth_ecg", "prdn"):
        from . import packer
        return getattr(packer, name)
    if name in ("shard_range", "allgather_totals", "place_offsets"):
        from . import dist
        return getattr(dist, name)
    raise AttributeError(name)
