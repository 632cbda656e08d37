"""fade_b200 -- B200 (sm_100a) implementation of `fade annotate`'s soft-clip realignment path.

The product is `libfadegpu.so` (C ABI in include/fadegpu.h + include/fadehost.h, CUDA kernels in
fade_b200/csrc).  This package is the thin Python host layer used by the tests and bench.py; it
mirrors the reference's `annotate` loop (source/anno.d:16-110) on top of the C ABI.  There is no
CPU fallback: importing works anywhere, computing needs the built library and a CUDA device.
"""
from ._lib import FadeGpuError, build, lib, lib_path  # noqa: F401
from .api import (Batch, Context, Job, Params, Record, annotate_records, default_params,  # noqa: F401
                  MAX_OPS, PairResults, PAIR_RESULT_DTYPE, ScoreResults)
