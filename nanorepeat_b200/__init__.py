"""nanorepeat_b200 -- B200 (sm_100a) drop-in for NanoRepeat's repeat-size estimation hot path.

Host-side mirror of the reference's operator interface for that path:

    round1_and_round2_estimation(data_type, repeat_region, num_cpu)   # nanoRepeat_bam.py:334
    round3_estimation(data_type, fast_mode, repeat_region, num_cpu)   # nanoRepeat_bam.py:446

and of the callers either side of it (anchoring: Step 1; joint: nanoRepeat-joint's grid rounds; phasing: the 1-D allele
phasing; pipeline: Steps 1-4 for many regions in memory), backed by libnanorepeat_b200.so (CUDA kernels + C ABI,
include/nanorepeat_b200.h).  There is no CPU compute
fallback: importing works anywhere, calling an estimation function without the built library or without a
B200 raises.
"""
from .presets import get_preset_for_minimap2, get_scoring, DATA_TYPES          # noqa: F401
from .repeat_region import Read, RepeatRegion                                  # noqa: F401
from .estimation import (round1_and_round2_estimation, round3_estimation,     # noqa: F401
                         round3_estimation_for1read, estimate_regions, install)
from . import engine, sharding, pymm2_shim, joint, anchoring, phasing          # noqa: F401
from .sharding import estimate_regions_sharded, quantify_regions_sharded       # noqa: F401
from .pipeline import quantify_regions                                         # noqa: F401

__version__ = "0.1.0"
