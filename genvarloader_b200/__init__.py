"""genvarloader_b200 -- B200-native haplotype reconstruction + track realignment behind GenVarLoader's
`Dataset` API.  CUDA only: importing the kernels without the built library raises (no CPU fallback)."""
from ._insertion_fill import Constant, FlankSample, InsertionFill, Interpolate, Repeat5p, Repeat5pNormalized

__all__ = ["Dataset", "Engine", "AnnotatedHaps", "Ragged", "RaggedAnnotatedHaps", "InsertionFill", "Repeat5p",
           "Repeat5pNormalized", "Constant", "FlankSample", "Interpolate", "Reference", "DummyVariant", "RaggedAlleles",
           "RaggedVariants", "RaggedIntervals", "VarWindowOpt"]


def __getattr__(name):  # torch + the CUDA library are loaded on first use
    if name in ("Dataset",):
        from ._dataset import Dataset

        return Dataset
    if name == "Reference":
        from ._open import Reference

        return Reference
    if name == "Engine":
        from ._engine import Engine

        return Engine
    if name in ("AnnotatedHaps", "Ragged", "RaggedAnnotatedHaps", "DummyVariant", "RaggedAlleles", "RaggedVariants", "RaggedIntervals",
                "VarWindowOpt"):
        from . import _types

        return getattr(_types, name)
    raise AttributeError(name)
