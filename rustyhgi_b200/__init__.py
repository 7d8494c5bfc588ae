"""rustyhgi_b200 -- B200-native implementation of RustyHGI's hierarchical-grid encode/decode loop.

The product is rustyhgi_b200/libhgi_b200.so (CUDA, sm_100a) behind the C ABI in include/hgi.h;
this package is the thin host-side mirror of the crate's API used by tests and bench.py.
"""
from ._lib import HgiError, HgiLibraryError, LIB_PATH, lib  # noqa: F401
from .api import (Archive, Context, Crossed, Decoder, Encoder, Grid, InterpolationType, LeftTop, Linear,  # noqa: F401
                  Metadata, NoOp, Pool, QuantizationLevel, PATH_PER_LEVEL, PATH_TILE, PATH_TILE_GENERIC, PATH_TILE_TMA, error_metrics, histogram, plan_region, rgb_to_luma)
from . import sharding  # noqa: F401

lib()  # fail at import time if the CUDA library is missing
