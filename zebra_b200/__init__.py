"""zebra_b200 -- B200-native replacement for the query hot path of emmyoh/zebra.

LSH hyperplane hashing and batched candidate scoring run in hand-written sm_100a CUDA kernels behind the
C ABI of include/zebra_b200.h (libzebra_b200.so); this package is the thin host mirror of the reference's
LSHIndex / Database / metric API.  There is no CPU fallback.
"""
from . import _ffi
from ._ffi import ZebraError
from .database import Database, DatabaseEmbeddingModel
from .distance import (BrayCurtisDistance, CanberraDistance, ChebyshevDistance, CosineDistance, HammingDistance,
                       L2Distance, L2SquaredDistance, L3Distance, L4Distance, ManhattanDistance, MinkowskiDistance,
                       PNormDistance, bits_to_f64, f64_to_bits, point_is_above)
from .index import Forest, LSHIndex, LSHIndexOptions, comm_unique_id, recall_at_k, synth_fill_device

__all__ = [
    "Database", "DatabaseEmbeddingModel", "LSHIndex", "LSHIndexOptions", "Forest", "CosineDistance", "L2Distance",
    "L2SquaredDistance", "ChebyshevDistance", "CanberraDistance", "BrayCurtisDistance", "ManhattanDistance", "L3Distance",
    "L4Distance", "HammingDistance", "MinkowskiDistance", "PNormDistance", "ZebraError", "bits_to_f64", "f64_to_bits", "point_is_above", "comm_unique_id",
    "synth_fill_device", "recall_at_k",
]
