"""mhaq_b200 — B200 (sm_100a) native fake-quantization hot path for MHAQ-style QAT.

Importing the package loads the in-tree CUDA shared library through its C ABI
(``include/mhaq_fq.h``).  There is no CPU fallback: a missing library is an
ImportError, a CPU tensor is a RuntimeError.
"""
from . import _lib  # noqa: F401  (fails loudly if the CUDA library is not built)
from .ops import (  # noqa: F401
    PackedCodes,
    fake_quant,
    pack_codes,
    quantize_codes,
    unpack_codes,
    quantize_eval,
    philox_noise,
    row_stats,
    set_device_philox_state,
)

__all__ = ["fake_quant", "quantize_codes", "quantize_eval", "philox_noise", "row_stats",
           "set_device_philox_state", "PackedCodes", "pack_codes", "unpack_codes"]
