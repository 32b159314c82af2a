"""CPU: the batch entry points' bound and argument checks (bz2b200_compress_bound, bz2b200_compress_batch_*)."""
import ctypes as C

import numpy as np
import pytest

import support as S
from bzip2_b200 import binding

EPARAM = -1


def _inputs():
    rng = np.random.default_rng(11)
    for n in list(range(0, 64)) + [100, 255, 256, 1000, 2047, 3000]:
        yield f"random{n}", S.gen_random(n, seed=n + 1)
        yield f"text{n}", S.gen_text(n, seed=n + 7)
        yield f"runs{n}", S.gen_runs(n, seed=n + 3) if n else np.zeros(0, np.uint8)
    for n in (17, 300, 2999):
        yield f"byte_runs{n}", np.full(n, rng.integers(0, 256), np.uint8)


@pytest.mark.parametrize("level", [1, 9])
def test_compress_bound_covers_small_inputs(lib, level):
    for name, x in _inputs():
        bound = lib.bz2b200_compress_bound(level, x.size)
        got = len(S.orc_compress(x, level))
        assert bound >= got, f"{name}: bound {bound} < {got} bytes"


@pytest.mark.parametrize("level", [1, 9])
def test_compress_bound_covers_sizes_around_a_block(lib, level):
    nmax = 100000 * level - 19
    for n in (nmax - 1, nmax, nmax + 1, nmax + 2):
        for x in (S.gen_random(n, seed=n), S.gen_text(n, seed=n)):
            assert lib.bz2b200_compress_bound(level, n) >= len(S.orc_compress(x, level))


def test_compress_bound_rejects_bad_levels(lib):
    assert lib.bz2b200_compress_bound(0, 100) == 0
    assert lib.bz2b200_compress_bound(10, 100) == 0


def test_batch_param_errors_need_no_gpu(lib):
    src = np.zeros(16, np.uint8)
    dst = np.zeros(4096, np.uint8)
    offs = np.array([0, 8, 16], np.uint64)
    out_offs = np.zeros(3, np.uint64)
    crcs = np.zeros(2, np.uint32)
    u64p = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
    u32p = crcs.ctypes.data_as(C.POINTER(C.c_uint32))
    st = binding.Stats()
    for f in (lib.bz2b200_compress_batch_host, lib.bz2b200_compress_batch_device):
        # NULL engine
        assert f(None, src.ctypes.data, u64p(offs), 2, dst.ctypes.data, dst.size, u64p(out_offs), u32p, 0, C.byref(st)) == EPARAM
        assert f(None, src.ctypes.data, u64p(offs), 0, dst.ctypes.data, dst.size, u64p(out_offs), u32p, 0, C.byref(st)) == EPARAM
        # NULL offsets (checked before the engine is used: a bogus handle is never dereferenced)
        bogus = C.c_void_p(0x10)
        assert f(bogus, src.ctypes.data, None, 2, dst.ctypes.data, dst.size, u64p(out_offs), u32p, 0, C.byref(st)) == EPARAM
    h = C.c_void_p()
    assert lib.bz2b200_engine_create_batch(None, 0, 9, 0, 64) == EPARAM
    if lib.bz2b200_device_count() == 0:
        assert lib.bz2b200_engine_create_batch(C.byref(h), 0, 9, 0, 64) == -2        # BZ2B200_ENODEV
