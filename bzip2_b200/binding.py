"""ctypes loader for libbz2_b200.so (include/bz2_b200.h and include/bzlib.h)."""
import ctypes as C
import os
import subprocess
import functools
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbz2_b200.so")

BZ_RUN, BZ_FLUSH, BZ_FINISH = 0, 1, 2
BZ_OK, BZ_RUN_OK, BZ_FLUSH_OK, BZ_FINISH_OK, BZ_STREAM_END = 0, 1, 2, 3, 4
BZ_SEQUENCE_ERROR, BZ_PARAM_ERROR, BZ_MEM_ERROR, BZ_OUTBUFF_FULL, BZ_CONFIG_ERROR = -1, -2, -3, -8, -9


class Bz2B200Error(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [("in_bytes", C.c_uint64), ("out_bytes", C.c_uint64), ("n_blocks", C.c_uint32),
                ("n_windows", C.c_uint32), ("sum_nblock", C.c_uint64), ("sum_nmtf", C.c_uint64),
                ("n_power_blocks", C.c_uint32), ("combined_crc", C.c_uint32),
                ("ms_total", C.c_float), ("ms_s1", C.c_float), ("ms_s2", C.c_float), ("ms_s3", C.c_float),
                ("ms_s4", C.c_float), ("bwt_rounds", C.c_uint32), ("kernel_launches", C.c_uint32), ("out_bits", C.c_uint64),
                ("ms_span", C.c_float)]


class BzStream(C.Structure):
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_uint), ("total_in_lo32", C.c_uint),
                ("total_in_hi32", C.c_uint), ("next_out", C.c_void_p), ("avail_out", C.c_uint),
                ("total_out_lo32", C.c_uint), ("total_out_hi32", C.c_uint), ("state", C.c_void_p),
                ("bzalloc", C.c_void_p), ("bzfree", C.c_void_p), ("opaque", C.c_void_p)]


def build_library(verbose=False):
    """Compile every CUDA source for sm_100a (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.check_call(["make", "-C", os.path.join(HERE, "csrc"), "-j8"], stdout=out)
    return LIB_PATH


EXPORTS = [
    # include/bz2_b200.h
    "bz2b200_device_count", "bz2b200_last_error", "bz2b200_version", "bz2b200_engine_create",
    "bz2b200_engine_create_bounded", "bz2b200_engine_destroy", "bz2b200_engine_set_stream", "bz2b200_engine_set_verbosity", "bz2b200_compress_host", "bz2b200_compress_device", "bz2b200_stream_begin",
    "bz2b200_stream_feed", "bz2b200_debug_keep", "bz2b200_debug_fetch",
    "bz2b200_scan_create", "bz2b200_scan_rescan", "bz2b200_scan_boundary", "bz2b200_scan_destroy", "bz2b200_concat_bits",
    "bz2b200_multi_create", "bz2b200_multi_destroy", "bz2b200_multi_engines", "bz2b200_multi_compress",
    "bz2b200_compress_bound", "bz2b200_engine_create_batch", "bz2b200_compress_batch_host", "bz2b200_compress_batch_device",
    # include/bzlib.h
    "BZ2_bzCompressInit", "BZ2_bzCompress", "BZ2_bzCompressEnd", "BZ2_bzBuffToBuffCompress",
    "BZ2_bzWriteOpen", "BZ2_bzWrite", "BZ2_bzWriteClose", "BZ2_bzWriteClose64", "BZ2_bzlibVersion",
    "BZ2_bzDecompressInit", "BZ2_bzDecompress", "BZ2_bzDecompressEnd", "BZ2_bzBuffToBuffDecompress",
    "BZ2_bzReadOpen", "BZ2_bzReadClose", "BZ2_bzReadGetUnused", "BZ2_bzRead",
    "BZ2_bzopen", "BZ2_bzdopen", "BZ2_bzread", "BZ2_bzwrite", "BZ2_bzflush", "BZ2_bzclose", "BZ2_bzerror",
]


@functools.lru_cache(None)
def load():
    if not os.path.exists(LIB_PATH):
        raise Bz2B200Error(f"{LIB_PATH} is missing: run __graft_entry__.build() (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, sz = C.c_void_p, C.c_size_t
    lib.bz2b200_device_count.restype = C.c_int
    lib.bz2b200_last_error.restype = C.c_char_p
    lib.bz2b200_version.restype = C.c_char_p
    lib.bz2b200_engine_create.restype = C.c_int
    lib.bz2b200_engine_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, sz]
    lib.bz2b200_engine_create_bounded.restype = C.c_int
    lib.bz2b200_engine_create_bounded.argtypes = [C.POINTER(vp), C.c_int, C.c_int, sz]
    lib.bz2b200_engine_destroy.restype = None
    lib.bz2b200_engine_destroy.argtypes = [vp]
    lib.bz2b200_engine_set_stream.restype = C.c_int
    lib.bz2b200_engine_set_stream.argtypes = [vp, vp]
    lib.bz2b200_compress_host.restype = C.c_int
    lib.bz2b200_compress_host.argtypes = [vp, vp, sz, vp, C.POINTER(sz), C.c_uint, C.POINTER(Stats)]
    lib.bz2b200_compress_device.restype = C.c_int
    lib.bz2b200_compress_device.argtypes = [vp, vp, sz, vp, sz, C.POINTER(sz), C.c_uint, C.POINTER(Stats)]
    lib.bz2b200_stream_begin.restype = C.c_int
    lib.bz2b200_stream_begin.argtypes = [vp]
    lib.bz2b200_debug_keep.restype = C.c_int
    lib.bz2b200_debug_keep.argtypes = [vp, C.c_int]
    lib.bz2b200_debug_fetch.restype = C.c_int
    lib.bz2b200_debug_fetch.argtypes = [vp, C.c_char_p, vp, sz, C.POINTER(sz)]
    lib.bz2b200_scan_create.restype = C.c_int
    lib.bz2b200_scan_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, vp, sz, C.c_int, C.c_uint64, C.c_int]
    lib.bz2b200_scan_rescan.restype = C.c_int
    lib.bz2b200_scan_rescan.argtypes = [vp, vp, sz, C.c_int, C.c_uint64, C.c_int]
    lib.bz2b200_scan_boundary.restype = C.c_int
    lib.bz2b200_scan_boundary.argtypes = [vp, sz, sz, C.c_uint, C.POINTER(sz), C.POINTER(C.c_uint32)]
    lib.bz2b200_scan_destroy.restype = None
    lib.bz2b200_scan_destroy.argtypes = [vp]
    lib.bz2b200_concat_bits.restype = C.c_int
    lib.bz2b200_concat_bits.argtypes = [C.c_int, vp, C.c_uint64, vp, C.c_uint64]
    lib.BZ2_bzCompressInit.restype = C.c_int
    lib.BZ2_bzCompressInit.argtypes = [C.POINTER(BzStream), C.c_int, C.c_int, C.c_int]
    lib.BZ2_bzCompress.restype = C.c_int
    lib.BZ2_bzCompress.argtypes = [C.POINTER(BzStream), C.c_int]
    lib.BZ2_bzCompressEnd.restype = C.c_int
    lib.BZ2_bzCompressEnd.argtypes = [C.POINTER(BzStream)]
    lib.BZ2_bzBuffToBuffCompress.restype = C.c_int
    lib.BZ2_bzBuffToBuffCompress.argtypes = [vp, C.POINTER(C.c_uint), vp, C.c_uint, C.c_int, C.c_int, C.c_int]
    lib.BZ2_bzlibVersion.restype = C.c_char_p
    lib.BZ2_bzDecompressInit.restype = C.c_int
    lib.BZ2_bzDecompressInit.argtypes = [C.POINTER(BzStream), C.c_int, C.c_int]
    lib.BZ2_bzDecompress.restype = C.c_int
    lib.BZ2_bzDecompress.argtypes = [C.POINTER(BzStream)]
    lib.BZ2_bzDecompressEnd.restype = C.c_int
    lib.BZ2_bzDecompressEnd.argtypes = [C.POINTER(BzStream)]
    lib.BZ2_bzBuffToBuffDecompress.restype = C.c_int
    lib.BZ2_bzBuffToBuffDecompress.argtypes = [vp, C.POINTER(C.c_uint), vp, C.c_uint, C.c_int, C.c_int]
    lib.BZ2_bzopen.restype = vp
    lib.BZ2_bzopen.argtypes = [C.c_char_p, C.c_char_p]
    lib.BZ2_bzdopen.restype = vp
    lib.BZ2_bzdopen.argtypes = [C.c_int, C.c_char_p]
    lib.BZ2_bzread.restype = C.c_int
    lib.BZ2_bzread.argtypes = [vp, vp, C.c_int]
    lib.BZ2_bzwrite.restype = C.c_int
    lib.BZ2_bzwrite.argtypes = [vp, vp, C.c_int]
    lib.BZ2_bzflush.restype = C.c_int
    lib.BZ2_bzflush.argtypes = [vp]
    lib.BZ2_bzclose.restype = None
    lib.BZ2_bzclose.argtypes = [vp]
    lib.BZ2_bzerror.restype = C.c_char_p
    lib.BZ2_bzerror.argtypes = [vp, C.POINTER(C.c_int)]
    lib.bz2b200_multi_create.restype = C.c_int
    lib.bz2b200_multi_create.argtypes = [C.POINTER(vp), C.POINTER(C.c_int), C.c_int, C.c_int, sz]
    lib.bz2b200_multi_destroy.restype = None
    lib.bz2b200_multi_destroy.argtypes = [vp]
    lib.bz2b200_multi_engines.restype = C.c_int
    lib.bz2b200_multi_engines.argtypes = [vp]
    lib.bz2b200_multi_compress.restype = C.c_int
    lib.bz2b200_multi_compress.argtypes = [vp, vp, C.POINTER(vp), sz, vp, C.POINTER(sz), C.c_uint, C.POINTER(Stats)]
    lib.bz2b200_pool_clear.restype = None
    lib.bz2b200_compress_bound.restype = sz
    lib.bz2b200_compress_bound.argtypes = [C.c_int, sz]
    lib.bz2b200_engine_create_batch.restype = C.c_int
    lib.bz2b200_engine_create_batch.argtypes = [C.POINTER(vp), C.c_int, C.c_int, sz, sz]
    u64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    for name in ("bz2b200_compress_batch_host", "bz2b200_compress_batch_device"):
        getattr(lib, name).restype = C.c_int
        getattr(lib, name).argtypes = [vp, vp, u64p, sz, vp, sz, u64p, u32p, C.c_uint, C.POINTER(Stats)]
    return lib


def _check(rc, what):
    if rc != 0:
        raise Bz2B200Error(f"{what} failed: rc={rc}: {load().bz2b200_last_error().decode()}")


def _ptr(a):
    return a.ctypes.data if a.size else None


def _u64p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint64)) if a is not None else None


def compress_bound(level, n):
    """Worst-case size of one stream of n input bytes (the reference's BuffToBuff bound, 1% + 600 bytes)."""
    return load().bz2b200_compress_bound(level, n)


class Engine:
    """One GPU compression engine (bz2b200_engine_*)."""

    def __init__(self, level=9, device=0, window_bytes=0, max_items=0):
        """max_items != 0: an engine whose windows hold up to max_items inputs of a batch call (engine_create_batch)."""
        self.lib = load()
        self.h = C.c_void_p()
        self.level = level
        if max_items:
            _check(self.lib.bz2b200_engine_create_batch(C.byref(self.h), device, level, window_bytes, max_items),
                   "engine_create_batch")
        else:
            _check(self.lib.bz2b200_engine_create(C.byref(self.h), device, level, window_bytes), "engine_create")

    def close(self):
        if self.h:
            self.lib.bz2b200_engine_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        _check(self.lib.bz2b200_engine_set_stream(self.h, cuda_stream_ptr), "set_stream")

    def compress(self, data, flags=0):
        a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data, np.uint8)
        cap = int(a.size * 1.02) + 24576 * (a.size // (100000 * self.level - 19) + 2) + 1024
        out = np.empty(cap, np.uint8)
        n = C.c_size_t(cap)
        st = Stats()
        _check(self.lib.bz2b200_compress_host(self.h, _ptr(a), a.size, out.ctypes.data, C.byref(n), flags, C.byref(st)),
               "compress_host")
        self.stats = st
        return out[: n.value].tobytes()

    def compress_device(self, d_src_ptr, n, d_dst_ptr, dst_cap, flags=0):
        """Input and output are device pointers (e.g. torch tensor .data_ptr())."""
        out_len = C.c_size_t(0)
        st = Stats()
        _check(self.lib.bz2b200_compress_device(self.h, d_src_ptr, n, d_dst_ptr, dst_cap, C.byref(out_len), flags, C.byref(st)),
               "compress_device")
        self.stats = st
        return out_len.value

    def compress_batch_raw(self, src, offsets, dst_cap=None, flags=0):
        """One bz2b200_compress_batch_host call on a flat uint8 array and its item offsets (n+1, offsets[0] = 0).
        Returns (rc, dst array, out_offsets, stream_crcs); raises only when the library is missing."""
        src = np.ascontiguousarray(src, np.uint8)
        offs = np.ascontiguousarray(offsets, np.uint64)
        n = offs.size - 1
        if dst_cap is None:
            dst_cap = sum(compress_bound(self.level, int(x)) for x in np.diff(offs))
        dst = np.empty(max(dst_cap, 1), np.uint8)
        out_offs = np.zeros(n + 1, np.uint64)
        crcs = np.zeros(max(n, 1), np.uint32)
        st = Stats()
        rc = self.lib.bz2b200_compress_batch_host(self.h, _ptr(src), _u64p(offs), n, dst.ctypes.data, dst_cap,
                                                  _u64p(out_offs), crcs.ctypes.data_as(C.POINTER(C.c_uint32)), flags,
                                                  C.byref(st))
        self.stats = st
        return rc, dst, out_offs, crcs[:n]

    def compress_batch(self, items, flags=0):
        """Compress every item to its own complete .bz2 stream in one call (bz2b200_compress_batch_host)."""
        arrs = [np.frombuffer(x, dtype=np.uint8) if isinstance(x, (bytes, bytearray)) else np.ascontiguousarray(x, np.uint8)
                for x in items]
        offs = np.zeros(len(arrs) + 1, np.uint64)
        offs[1:] = np.cumsum([a.size for a in arrs], dtype=np.uint64)
        src = np.concatenate(arrs) if arrs else np.zeros(0, np.uint8)
        rc, dst, out_offs, crcs = self.compress_batch_raw(src, offs, flags=flags)
        _check(rc, "compress_batch_host")
        self.stream_crcs = crcs
        return [dst[int(out_offs[k]):int(out_offs[k + 1])].tobytes() for k in range(len(arrs))]

    def compress_batch_device(self, d_src_ptr, offsets, d_dst_ptr, dst_cap, flags=0, stream_crcs=None):
        """Device input and output (e.g. torch tensor .data_ptr()); offsets: host array of n+1 item offsets.
        Returns the numpy array of n+1 stream offsets in the destination."""
        offs = np.ascontiguousarray(offsets, np.uint64)
        n = offs.size - 1
        out_offs = np.zeros(n + 1, np.uint64)
        crcp = None
        if stream_crcs is not None:
            assert stream_crcs.dtype == np.uint32 and stream_crcs.size >= n
            crcp = stream_crcs.ctypes.data_as(C.POINTER(C.c_uint32))
        st = Stats()
        _check(self.lib.bz2b200_compress_batch_device(self.h, d_src_ptr, _u64p(offs), n, d_dst_ptr, dst_cap, _u64p(out_offs),
                                                      crcp, flags, C.byref(st)), "compress_batch_device")
        self.stats = st
        return out_offs

    def fetch(self, name, dtype, count=None):
        cap = (1 << 28)
        dt = np.dtype(dtype)
        # ask for the natural size first
        buf = np.empty(cap // dt.itemsize if count is None else count, dtype=dt)
        got = C.c_size_t(0)
        _check(self.lib.bz2b200_debug_fetch(self.h, name.encode(), buf.ctypes.data, buf.nbytes, C.byref(got)), f"debug_fetch({name})")
        return buf[: got.value // dt.itemsize].copy()


class Multi:
    """Several engines on one stream (bz2b200_multi_*): devices=[0, 1, 2, 3] shards by block over four GPUs,
    devices=[0, 0] keeps two windows in flight on one."""

    def __init__(self, devices, level=9, window_bytes=0):
        self.lib = load()
        self.h = C.c_void_p()
        self.level = level
        self.devices = list(devices)
        arr = (C.c_int * len(self.devices))(*self.devices)
        _check(self.lib.bz2b200_multi_create(C.byref(self.h), arr, len(self.devices), level, window_bytes), "multi_create")

    def close(self):
        if self.h:
            self.lib.bz2b200_multi_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def out_cap(self, n):
        return int(n * 1.02) + 24576 * (n // (100000 * self.level - 19) + 2) + 1024

    def compress_ptr(self, src_ptr, n, dst_ptr, cap, flags=0, d_srcs=None):
        """src_ptr: host pointer (or None with d_srcs = one device pointer per engine); dst_ptr: host pointer."""
        out_len = C.c_size_t(cap)
        st = Stats()
        ds = None
        if d_srcs is not None:
            ds = (C.c_void_p * len(d_srcs))(*d_srcs)
        _check(self.lib.bz2b200_multi_compress(self.h, src_ptr, ds, n, dst_ptr, C.byref(out_len), flags, C.byref(st)), "multi_compress")
        self.stats = st
        return out_len.value

    def compress(self, data, flags=0):
        a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data, np.uint8)
        cap = self.out_cap(a.size)
        out = np.empty(cap, np.uint8)
        n = self.compress_ptr(_ptr(a), a.size, out.ctypes.data, cap, flags)
        return out[:n].tobytes()


def compress(data, level=9):
    """BZ2_bzBuffToBuffCompress through the libbz2-compatible entry point."""
    lib = load()
    a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else np.ascontiguousarray(data, np.uint8)
    cap = int(a.size * 1.02) + 24576 * (a.size // (100000 * level - 19) + 2) + 1024
    out = np.empty(cap, np.uint8)
    n = C.c_uint(cap)
    src = a.ctypes.data if a.size else out.ctypes.data
    rc = lib.BZ2_bzBuffToBuffCompress(out.ctypes.data, C.byref(n), src, a.size, level, 0, 0)
    if rc != BZ_OK:
        raise Bz2B200Error(f"BZ2_bzBuffToBuffCompress rc={rc}: {lib.bz2b200_last_error().decode()}")
    return out[: n.value].tobytes()


class bzlib:
    """Streaming API mirror (BZ2_bzCompressInit / BZ2_bzCompress / BZ2_bzCompressEnd) for tests."""

    def __init__(self, level=9):
        self.lib = load()
        self.strm = BzStream()
        rc = self.lib.BZ2_bzCompressInit(C.byref(self.strm), level, 0, 0)
        if rc != BZ_OK:
            raise Bz2B200Error(f"BZ2_bzCompressInit rc={rc}: {self.lib.bz2b200_last_error().decode()}")
        self.out = bytearray()

    def call(self, data, action, out_chunk=1 << 16):
        """One BZ2_bzCompress call; returns (rc, consumed)."""
        a = np.frombuffer(bytes(data), dtype=np.uint8).copy() if len(data) else np.zeros(1, np.uint8)
        ob = np.empty(out_chunk, np.uint8)
        self.strm.next_in = a.ctypes.data
        self.strm.avail_in = len(data)
        self.strm.next_out = ob.ctypes.data
        self.strm.avail_out = out_chunk
        rc = self.lib.BZ2_bzCompress(C.byref(self.strm), action)
        produced = out_chunk - self.strm.avail_out
        self.out += ob[:produced].tobytes()
        return rc, len(data) - self.strm.avail_in

    def end(self):
        return self.lib.BZ2_bzCompressEnd(C.byref(self.strm))


def decompress_stream(data, in_chunk=1 << 16, out_chunk=1 << 16):
    """Host decoder through BZ2_bzDecompressInit / BZ2_bzDecompress / BZ2_bzDecompressEnd.
    Returns (rc, output bytes, input bytes left unread)."""
    lib = load()
    strm = BzStream()
    rc = lib.BZ2_bzDecompressInit(C.byref(strm), 0, 0)
    if rc != BZ_OK:
        raise Bz2B200Error(f"BZ2_bzDecompressInit rc={rc}")
    src = np.frombuffer(bytes(data), dtype=np.uint8).copy() if len(data) else np.zeros(1, np.uint8)
    ob = np.empty(out_chunk, np.uint8)
    out = bytearray()
    pos = 0
    rc = BZ_OK
    while True:
        take = min(in_chunk, len(data) - pos)
        strm.next_in = src.ctypes.data + pos
        strm.avail_in = take
        while True:
            strm.next_out = ob.ctypes.data
            strm.avail_out = out_chunk
            rc = lib.BZ2_bzDecompress(C.byref(strm))
            out += ob[:out_chunk - strm.avail_out].tobytes()
            if rc != BZ_OK or strm.avail_out > 0:
                break
        pos += take - strm.avail_in
        if rc != BZ_OK or (strm.avail_in == 0 and pos >= len(data)):
            break
    lib.BZ2_bzDecompressEnd(C.byref(strm))
    return rc, bytes(out), len(data) - pos


def decompress(data, cap):
    """BZ2_bzBuffToBuffDecompress. Returns (rc, bytes)."""
    lib = load()
    src = np.frombuffer(bytes(data), dtype=np.uint8).copy() if len(data) else np.zeros(1, np.uint8)
    dst = np.empty(max(cap, 1), np.uint8)
    n = C.c_uint(cap)
    rc = lib.BZ2_bzBuffToBuffDecompress(dst.ctypes.data, C.byref(n), src.ctypes.data, len(data), 0, 0)
    return rc, dst[:n.value].tobytes()
