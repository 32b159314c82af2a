"""Regenerates tests/golden/ref_checks.json: the known answers of the differential tests that used to need the
reference library built from its source tree (test_oracle_vs_ref.py, test_decoder.py, test_gpu_scale.py).

They are minted from the stock libbzip2 installed on the system (1.0.8; the run stops if it cannot be found).
The compressor of stock libbzip2 and the reference differ in one known place: the origPtr they choose among
equal rotations, i.e. for a block that is an exact power u^q (q >= 2).  So

  * before minting, every committed reference golden (sample*.bz2, streams.json, powers_random.json) whose
    blocks are all power-free must be reproduced byte for byte, or nothing is written;
  * a compressed-stream answer is stored only for an input whose blocks are all power-free, and null otherwise
    (the tests check those cases against the committed reference goldens or not at all).

  python tests/golden/make_ref_checks.py
"""
import ctypes as C
import ctypes.util
import functools
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import support as S  # noqa: E402
from golden.make_golden import stream_cases  # noqa: E402

OUT = os.path.join(HERE, "ref_checks.json")
BZ_FINISH, BZ_FINISH_OK, BZ_STREAM_END = 2, 3, 4


class BzStream(C.Structure):
    _fields_ = [("next_in", C.c_void_p), ("avail_in", C.c_uint), ("total_in_lo32", C.c_uint),
                ("total_in_hi32", C.c_uint), ("next_out", C.c_void_p), ("avail_out", C.c_uint),
                ("total_out_lo32", C.c_uint), ("total_out_hi32", C.c_uint), ("state", C.c_void_p),
                ("bzalloc", C.c_void_p), ("bzfree", C.c_void_p), ("opaque", C.c_void_p)]


class EState(C.Structure):
    """The leading fields of libbzip2's compressor state (bzlib_private.h), up to nMTF."""
    _fields_ = [("strm", C.c_void_p), ("mode", C.c_int32), ("state", C.c_int32), ("avail_in_expect", C.c_uint32),
                ("arr1", C.c_void_p), ("arr2", C.c_void_p), ("ftab", C.c_void_p), ("origPtr", C.c_int32),
                ("ptr", C.c_void_p), ("block", C.c_void_p), ("mtfv", C.c_void_p), ("zbits", C.c_void_p),
                ("workFactor", C.c_int32), ("state_in_ch", C.c_uint32), ("state_in_len", C.c_int32),
                ("rNToGo", C.c_int32), ("rTPos", C.c_int32),
                ("nblock", C.c_int32), ("nblockMAX", C.c_int32), ("numZ", C.c_int32), ("state_out_pos", C.c_int32),
                ("nInUse", C.c_int32), ("inUse", C.c_uint8 * 256), ("unseqToSeq", C.c_uint8 * 256),
                ("bsBuff", C.c_uint32), ("bsLive", C.c_int32), ("blockCRC", C.c_uint32), ("combinedCRC", C.c_uint32),
                ("verbosity", C.c_int32), ("blockNo", C.c_int32), ("blockSize100k", C.c_int32), ("nMTF", C.c_int32)]


@functools.lru_cache(None)
def _lib():
    name = ctypes.util.find_library("bz2")
    if name is None:
        raise SystemExit("make_ref_checks: no libbz2 on this system")
    lib = C.CDLL(name)
    vp = C.c_void_p
    lib.BZ2_bzlibVersion.restype = C.c_char_p
    lib.BZ2_bzBuffToBuffCompress.argtypes = [vp, C.POINTER(C.c_uint), vp, C.c_uint, C.c_int, C.c_int, C.c_int]
    lib.BZ2_bzBuffToBuffDecompress.argtypes = [vp, C.POINTER(C.c_uint), vp, C.c_uint, C.c_int, C.c_int]
    lib.BZ2_bzCompressInit.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    lib.BZ2_bzCompress.argtypes = [vp, C.c_int]
    lib.BZ2_bzCompressEnd.argtypes = [vp]
    lib.BZ2_blockSort.argtypes = [vp]
    return lib


def _init(level):
    strm = BzStream()
    assert _lib().BZ2_bzCompressInit(C.byref(strm), level, 0, 0) == 0
    s = EState.from_address(strm.state)
    # the layout above is the library's: these hold right after BZ2_bzCompressInit (bzlib.c)
    assert s.strm == C.addressof(strm) and s.blockSize100k == level and s.nblockMAX == 100000 * level - 19
    assert s.workFactor == 30 and s.ptr == s.arr1 and s.mtfv == s.arr1 and s.block == s.arr2 and not s.zbits
    return strm, s


def compress(data, level):
    """BZ2_bzBuffToBuffCompress, workFactor 0"""
    a = S.as_u8(data)
    out = np.zeros(int(a.size * 1.02) + 1000, np.uint8)
    n = C.c_uint(out.size)
    src = a.ctypes.data if a.size else out.ctypes.data
    assert _lib().BZ2_bzBuffToBuffCompress(out.ctypes.data, C.byref(n), src, a.size, level, 0, 0) == 0
    return out[: n.value].tobytes()


def trace(data, level):
    """The blocks BZ2_bzCompress(BZ_FINISH) cuts: per block (post-RLE1 bytes, CRC, origPtr, nMTF, nInUse).
    The output window is sized so that each call that returns BZ_FINISH_OK has compressed exactly one block and left
    its output pending (the first call takes one byte: a call that moves no byte at all is a sequence error); the
    call that returns BZ_STREAM_END only drains the last one."""
    a = S.as_u8(data)
    strm, s = _init(level)
    sink = np.empty(1 << 21, np.uint8)
    strm.next_in, strm.avail_in = (a.ctypes.data if a.size else sink.ctypes.data), a.size
    strm.next_out, strm.avail_out = sink.ctypes.data, 1
    blocks = []
    try:
        while True:
            rc = _lib().BZ2_bzCompress(C.byref(strm), BZ_FINISH)
            assert rc in (BZ_FINISH_OK, BZ_STREAM_END), rc
            if rc == BZ_FINISH_OK and s.nblock > 0:
                blk = np.ctypeslib.as_array(C.cast(s.block, C.POINTER(C.c_uint8)), (s.nblock,)).copy()
                blocks.append({"block": blk, "crc": s.blockCRC, "orig_ptr": s.origPtr, "n_mtf": s.nMTF, "n_in_use": s.nInUse})
            if rc == BZ_STREAM_END:
                return blocks
            strm.next_out, strm.avail_out = sink.ctypes.data, s.numZ - s.state_out_pos
    finally:
        _lib().BZ2_bzCompressEnd(C.byref(strm))


def block_sort(blk):
    """BZ2_blockSort on one post-RLE1 block: (BWT bytes, origPtr)"""
    a = S.as_u8(blk)
    strm, s = _init(9)
    try:
        C.memmove(s.block, a.ctypes.data, a.size)
        s.nblock = a.size
        _lib().BZ2_blockSort(strm.state)
        sa = np.ctypeslib.as_array(C.cast(s.ptr, C.POINTER(C.c_uint32)), (a.size,)).astype(np.int64)
        return a[(sa - 1) % a.size], int(s.origPtr)
    finally:
        _lib().BZ2_bzCompressEnd(C.byref(strm))


def is_power(blk):
    """blk == u^q for some q >= 2: then some rotations are equal"""
    n = blk.size
    return any(np.array_equal(blk[p:], blk[:-p]) for p in range(1, n // 2 + 1) if n % p == 0)


def power_free(data, level):
    return all(not is_power(b["block"]) for b in trace(data, level))


def stream_answer(data, level):
    """sha256 and length of the stream, or None when a block is an exact power"""
    if not power_free(data, level):
        return None
    out = compress(data, level)
    return {"sha256": hashlib.sha256(out).hexdigest(), "out_len": len(out)}


def check_against_reference_goldens():
    for i in (1, 2, 3):
        with open(os.path.join(HERE, f"sample{i}.ref"), "rb") as f, open(os.path.join(HERE, f"sample{i}.bz2"), "rb") as g:
            assert compress(f.read(), i) == g.read(), f"sample{i}"
    gold = json.load(open(os.path.join(HERE, "streams.json")))
    checked = 0
    for name, data, level in stream_cases():
        got = stream_answer(data, level)
        if got is not None:
            assert got["sha256"] == gold[name]["sha256"], name
            checked += 1
    for g in json.load(open(os.path.join(HERE, "powers_random.json")))[::3]:
        d = S.random_power_case(g["seed"], g["p"], g["alpha"], g["q"])
        for level in (1, 9):
            got = stream_answer(d, level)
            if got is not None:
                assert got["sha256"] == g[f"sha_L{level}"], (g, level)
                checked += 1
    print(f"{_lib().BZ2_bzlibVersion().decode()}: {checked} committed reference streams reproduced")


# ----------------------------------------------------------------------------- the cases (shared with the tests)
def fuzz_small_cases():
    rng = np.random.default_rng(2024)
    for it in range(250):
        n = int(rng.integers(0, 4000))
        alpha = int(rng.integers(1, 257))
        mode = it % 4
        if mode == 0:
            d = rng.integers(0, alpha, n, dtype=np.uint8)
        elif mode == 1:
            d = np.repeat(rng.integers(0, alpha, n // 7 + 1, dtype=np.uint8), rng.integers(1, 300, n // 7 + 1))[:n].astype(np.uint8)
        elif mode == 2:
            d = np.resize(rng.integers(0, alpha, int(rng.integers(1, 40)), dtype=np.uint8), n)
        else:
            d = S.gen_text(n, seed=it + 1)
        level = int(rng.integers(1, 10))
        yield it, mode, d, level


MULTIBLOCK = [("text", 1_200_000, 1), ("random", 700_000, 2), ("runs", 3_000_000, 1), ("p1000", 450_000, 1), ("mixed", 900_000, 2)]


def multiblock_input(gen, n):
    return {"text": S.gen_text, "random": S.gen_random, "runs": S.gen_runs, "p1000": S.gen_period1000,
            "mixed": lambda k: S.gen_mixed(k, seg=100_000)}[gen](n)


def tail_merge_input():
    return (np.arange(99981 + 1, dtype=np.uint32) % 251).astype(np.uint8)


def stage_input():
    return S.gen_text(150_000)


def decoder_cases():
    import bz2
    d = S.gen_text(60_000, 2).tobytes()
    z = bz2.compress(d, 1)
    cases = [z, z[:-1], z[:100], z[:4], z[:3], b"", b"BZh", b"BZh9", b"BZx9" + z[4:], z + b"tail",
             b"j", b"Bj", b"BZh9j", b"BZh91j", b"BZh9\x17\x72\x45\x38\x50", b"BZh9\x17\x72\x45\x38\x51",
             b"BZh9\x17\x72\x45\x38\x50\x90\0\0\0\0", b"BZh9\x17\x72\x45\x38\x50\x90\0\0\0\1"]
    bad = bytearray(z); bad[12] ^= 0x40; cases.append(bytes(bad))
    bad = bytearray(z); bad[-1] ^= 0x01; cases.append(bytes(bad))
    return d, cases


def level_sweep_input():
    return S.gen_text(30_000_000, seed=5)


def main():
    check_against_reference_goldens()
    res = {"library": _lib().BZ2_bzlibVersion().decode()}
    res["fuzz_small"] = [stream_answer(d, level) for _, _, d, level in fuzz_small_cases()]
    print("fuzz_small:", sum(x is not None for x in res["fuzz_small"]), "of", len(res["fuzz_small"]), "power-free")
    res["multiblock"] = {f"{g}-{n}-{lv}": stream_answer(multiblock_input(g, n), lv) for g, n, lv in MULTIBLOCK}
    assert all(res["multiblock"].values())
    d = tail_merge_input()
    res["tail_merge"] = dict(stream_answer(d, 1), n_blocks=len(trace(d, 1)))
    blocks = trace(stage_input(), 1)
    assert not any(is_power(b["block"]) for b in blocks)
    bwt, op = block_sort(blocks[0]["block"])
    assert op == blocks[0]["orig_ptr"]
    res["stage_functions"] = {"nblock": [int(b["block"].size) for b in blocks], "crc": [int(b["crc"]) for b in blocks],
                              "block0_sha256": hashlib.sha256(blocks[0]["block"]).hexdigest(),
                              "bwt0_sha256": hashlib.sha256(bwt).hexdigest(), "orig_ptr0": op,
                              "n_mtf0": int(blocks[0]["n_mtf"]), "n_in_use0": int(blocks[0]["n_in_use"])}
    d, cases = decoder_cases()
    codes = []
    for c in cases:
        row = []
        for cap in (len(d), len(d) - 1, 10):
            dst = np.zeros(max(cap, 1), np.uint8)
            src = S.as_u8(c)
            n = C.c_uint(cap)
            rc = _lib().BZ2_bzBuffToBuffDecompress(dst.ctypes.data, C.byref(n), src.ctypes.data if src.size else dst.ctypes.data, src.size, 0, 0)
            row.append([rc, hashlib.sha256(dst[: n.value]).hexdigest() if rc == 0 else None])
        codes.append(row)
    res["decoder_codes"] = codes
    d = level_sweep_input()
    res["level_sweep"] = {str(lv): stream_answer(d, lv) for lv in range(1, 10)}
    assert all(res["level_sweep"].values())
    with open(OUT, "w") as f:
        json.dump(res, f, indent=0, sort_keys=True)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
