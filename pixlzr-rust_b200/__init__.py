"""pixlzr_b200 — B200-native (sm_100a) implementation of the pixlzr hot path.

Layout
  csrc/        hand-written CUDA kernels + the C ABI (include/pixlzr_b200.h) + the host container stage
  _native.py   ctypes binding of libpixlzr_b200.so (fails loudly if the library is missing)
  api.py       host-side mirror of the reference's public API (Pixlzr, PixlzrBlock, FilterType,
               process, get_block_variance, ...) on top of the C ABI
  build.py     in-tree nvcc build
"""
from .api import (  # noqa: F401
    ErrorReport,
    FilterType,
    OptimalCurve,
    Pixlzr,
    PixlzrBlock,
    RateDistortion,
    Strategy,
    StrategyReport,
    get_block_variance,
    get_block_variance_directionally,
    image_error,
    parse_shrinking_factor,
    payload_error,
    process,
    process_by_strategy,
    process_custom,
    psnr_of,
    rd_curve,
    rdo_curve,
    reduce_image_section,
    sse_budget,
    tree_process,
    tree_process_custom,
)
from . import _native as native  # noqa: F401
from . import sharding  # noqa: F401
from . import cli  # noqa: F401
