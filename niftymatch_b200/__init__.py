"""niftymatch_b200 -- B200-native (sm_100a) SIFT detect/describe + brute-force k=2 matching
behind the public API of gift-surg/NiftyMatch.

The product is the C-ABI shared library (include/nm_b200.h, niftymatch_b200/csrc/) and
the C++ drop-in headers (include/nm/).  This Python package is plumbing for tests and
benchmarks: it binds the C-ABI with ctypes and uses torch only for device memory,
streams and torch.distributed.
"""
from ._lib import load, NmError, LIB_PATH, SiftParamsC  # noqa: F401
from .sift import SiftParams, SiftBatch, gaussian_taps, grayscale, cast_u8, undistort_map  # noqa: F401
from .match import match, match_top2, merge_top2, match_pairs, match_pairs_span, set_engine, get_engine, tc_probe  # noqa: F401
from .ransac import (align_points, align_pairs_span, ransac, ransac_batch, ransac_hypotheses, refine, refine_batch,  # noqa: F401
                     adjust_chain, TRANSLATION, SIMILARITY, HOMOGRAPHY, MOSAIC, TRANSFER)
from .dist import shard_bounds, match_sharded, frame_range, register_stream  # noqa: F401
from .mosaic import Mosaic, Placement, place, render_stream  # noqa: F401
