"""mahout_b200 -- B200-native (sm_100a) sketch-similarity hot path of jalhajj/mahout.

The product is libmahout_b200.so (C ABI in include/mahout_b200.h); this package is the thin
host-side mirror of the reference's operator API over that ABI.  No CPU fallback exists.
"""
from ._native import (CMException, InexactError, NativeError, LIB_PATH)  # noqa: F401
from .sketch import (Context, DoubleCountMinSketch, HashFunction, HashFunctionBuilder,  # noqa: F401
                     SizedBank, SketchBank, cm_dims, default_context)

__all__ = ["Context", "DoubleCountMinSketch", "HashFunction", "HashFunctionBuilder", "SizedBank", "SketchBank",
           "cm_dims", "default_context", "CMException", "InexactError", "NativeError", "LIB_PATH"]
