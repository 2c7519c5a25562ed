"""B200-native in-loop filter chain of VTM 2.1 (deblocking -> SAO -> ALF).

The product is the C-ABI CUDA library ``libilf_b200.so`` (include/ilf_b200.h, csrc/) plus the C++ shim that
keeps the reference's LoopFilter / SampleAdaptiveOffset / AdaptiveLoopFilter class interfaces (shim/).
This Python package is a thin ctypes binding of the C ABI used by the tests and bench.py.
"""
from .ilf import BAND_ABOVE, BAND_BELOW, IlfError, IlfHashPart, InLoopFilter, hash_combine, lib_path, load_library, pinned_planes  # noqa: F401
from . import bands  # noqa: F401
