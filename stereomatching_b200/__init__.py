"""stereomatching_b200 -- B200-native (sm_100a) replacement for the CUDA side of
chrg127/stereomatching's block-matching hot path, behind a C ABI.

The product is ``libstereo_b200.so`` (include/stereo_b200.h, csrc/); this package is
the thin ctypes binding used by tests and bench.py.  There is no CPU fallback.
"""
from .api import (  # noqa: F401
    BEST, EDGES1, EDGES2, GHOST, KERNEL_AUTO, KERNEL_BITSLICE, KERNEL_DIRECT, MATCH, OUTPUT, SCORE,
    SCORE_ALL, SM_ERR_DEGENERATE, SYMBOLS, WEB, WEB_FILLED, WRAP, MultiGpuBands, MultiGpuBatch, PinnedBuffer, StereoContext,
    StereoError, band_rows, device_count, lib, OPT_EDGES_FP64, OPT_PIPE_GROUP, OPT_ROW_RUNS,
    INFO_WARPS_PER_SM, INFO_PAIRS_PER_LAUNCH, INFO_TMEM_COLUMNS, INFO_EDGE_THRESHOLDS, INFO_KERNEL_SHAPE, INFO_ROW_RUNS,
    SHAPE_HALF, SHAPE_TWO_WORDS, SHAPE_SEG8, SHAPE_C2, SHAPE_HP, SHAPE_MULTI, SHAPE_BITSLICE, SHAPE_DIRECT,
)
