"""bzip2_b200 -- B200 (sm_100a) bzip2 compressor behind libbz2's C API.

The product is the shared library ``bzip2_b200/libbz2_b200.so`` (CUDA kernels + C ABI + the
libbz2-compatible C front end).  This package is only a thin ctypes loader used by the tests,
``bench.py`` and ``__graft_entry__``; it adds no compute of its own and has no CPU fallback:
every call fails loudly if the library is missing or no CUDA device is usable.
"""
from .binding import (  # noqa: F401
    LIB_PATH, Bz2B200Error, Engine, Multi, Stats, bzlib, compress, compress_bound, build_library, load,
)
