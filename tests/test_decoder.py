"""Host decoder behind BZ2_bzDecompress* / BZ2_bzBuffToBuffDecompress / BZ2_bzopen-bzread
(bzip2_b200/csrc/bzlib_decode.c): outside the accelerated path, present so the library covers the
reference's whole libbz2 surface (bzlib.h:100-271).  Checked against the golden vectors, Python's
bz2 module and the return codes of libbzip2's own decoder (tests/golden/ref_checks.json)."""
import bz2
import ctypes as C
import hashlib
import json
import os
import random

import numpy as np
import pytest

import support
from bzip2_b200 import binding

GOLD = os.path.join(os.path.dirname(__file__), "golden")
BZ_OK, BZ_STREAM_END = 0, 4
BZ_DATA_ERROR, BZ_DATA_ERROR_MAGIC, BZ_UNEXPECTED_EOF, BZ_OUTBUFF_FULL = -4, -5, -7, -8


def _samples():
    for i in (1, 2, 3):
        with open(os.path.join(GOLD, f"sample{i}.bz2"), "rb") as f:
            z = f.read()
        with open(os.path.join(GOLD, f"sample{i}.ref"), "rb") as f:
            r = f.read()
        yield i, z, r


def test_golden_vectors_one_shot():
    for i, z, r in _samples():
        rc, out = binding.decompress(z, len(r))
        assert rc == BZ_OK and out == r, i
        rc, _ = binding.decompress(z, len(r) - 1)
        assert rc == BZ_OUTBUFF_FULL
        rc, _ = binding.decompress(z[:-1], len(r) + 16)
        assert rc == BZ_UNEXPECTED_EOF
        rc, _ = binding.decompress(z[: len(z) // 2], len(r) + 16)
        assert rc == BZ_UNEXPECTED_EOF


@pytest.mark.parametrize("in_chunk,out_chunk", [(1, 1 << 16), (5000, 5000), (1 << 20, 7), (3, 11)])
def test_golden_vectors_streaming(in_chunk, out_chunk):
    for i, z, r in _samples():
        if in_chunk * out_chunk < 100 and i != 1:
            continue
        rc, out, left = binding.decompress_stream(z, in_chunk, out_chunk)
        assert rc == BZ_STREAM_END and out == r and left == 0, i


def test_fuzz_against_python_bz2():
    rng = random.Random(7)
    for t in range(120):
        n = rng.choice([0, 1, 2, 5, 49, 50, 51, 100, 1000, 50000, 250000])
        kind = rng.randrange(5)
        if kind == 0:
            d = rng.randbytes(n)
        elif kind == 1:
            d = bytes(rng.choice(b"ab") for _ in range(n))
        elif kind == 2:
            d = bytes([7]) * n
        elif kind == 3:
            d = (b"hello world " * (n // 12 + 1))[:n]
        else:
            d = bytes(support.gen_runs(max(n, 1), t))[:n]
        z = bz2.compress(d, rng.randint(1, 9))
        rc, out = binding.decompress(z, n + 1)
        assert rc == BZ_OK and out == d, (t, n, kind)
        rc, out, left = binding.decompress_stream(z, rng.choice([1, 17, 4096]), rng.choice([1 << 16, 100]))
        assert rc == BZ_STREAM_END and out == d and left == 0, (t, n, kind)


def test_oracle_streams_round_trip():
    # multi-block streams at -1, including the RLE1 corner cases the compressor tests use
    for name, data in [("text", support.gen_text(450_000, support.TEXT_SEED)),
                       ("runs", support.gen_runs(700_000, 3)),
                       ("same", np.full(1_000_000, 65, np.uint8)),
                       ("rand", support.gen_random(250_000, 5))]:
        raw = bytes(data)
        z = support.orc_compress(raw, 1)
        rc, out = binding.decompress(z, len(raw))
        assert rc == BZ_OK and out == raw, name
        rc, out, left = binding.decompress_stream(z, 777, 33333)
        assert rc == BZ_STREAM_END and out == raw and left == 0, name


def test_trailing_bytes_and_concatenated_streams():
    a, b = b"first stream " * 1000, b"second" * 10
    za, zb = bz2.compress(a), bz2.compress(b)
    for in_chunk in (1, 100, 1 << 20):
        rc, out, left = binding.decompress_stream(za + zb, in_chunk)
        assert rc == BZ_STREAM_END and out == a and left == len(zb), in_chunk
        rc, out, left = binding.decompress_stream(za + b"\x00garbage", in_chunk)
        assert rc == BZ_STREAM_END and out == a and left == 8


def test_corruption_is_reported():
    d = support.gen_text(120_000, 11).tobytes()
    z = bytearray(bz2.compress(d, 1))
    rc, _ = binding.decompress(bytes(z[:2]) + b"x" + bytes(z[3:]), len(d))
    assert rc == BZ_DATA_ERROR_MAGIC
    rc, _ = binding.decompress(b"BZh0" + bytes(z[4:]), len(d))
    assert rc == BZ_DATA_ERROR_MAGIC
    bad = bytearray(z)
    bad[10] ^= 0x01                      # block CRC field
    rc, _ = binding.decompress(bytes(bad), len(d))
    assert rc == BZ_DATA_ERROR
    bad = bytearray(z)
    bad[-2] ^= 0x10                      # combined CRC
    rc, _ = binding.decompress(bytes(bad), len(d))
    assert rc == BZ_DATA_ERROR
    rng = random.Random(3)
    for _ in range(60):                  # any flipped payload bit must be an error, never a crash
        bad = bytearray(z)
        p = rng.randrange(4, len(z))
        bad[p] ^= 1 << rng.randrange(8)
        rc, out = binding.decompress(bytes(bad), len(d) + 1000)
        assert rc in (BZ_DATA_ERROR, BZ_UNEXPECTED_EOF, BZ_OUTBUFF_FULL, BZ_DATA_ERROR_MAGIC), (p, rc)


def test_same_codes_as_reference_decoder():
    """Return code and output of BZ2_bzBuffToBuffDecompress on good, truncated and damaged streams, as libbzip2's
    decoder gives them (tests/golden/ref_checks.json, make_ref_checks.py)."""
    from golden.make_ref_checks import decoder_cases
    gold = json.load(open(os.path.join(GOLD, "ref_checks.json")))["decoder_codes"]
    d, cases = decoder_cases()
    assert len(cases) == len(gold)
    for i, (c, row) in enumerate(zip(cases, gold)):
        for cap, (want, want_sha) in zip((len(d), len(d) - 1, 10), row):
            got, out = binding.decompress(c, cap)
            assert got == want, (i, cap, got, want)
            if want == BZ_OK:
                assert hashlib.sha256(out).hexdigest() == want_sha, (i, cap)


def test_zlib_style_file_read(tmp_path):
    lib = binding.load()
    d = support.gen_text(300_000, 9).tobytes()
    p = tmp_path / "x.bz2"
    p.write_bytes(bz2.compress(d, 3) + b"EXTRA")
    h = lib.BZ2_bzopen(str(p).encode(), b"r")
    assert h
    out = bytearray()
    buf = C.create_string_buffer(10_000)
    while True:
        n = lib.BZ2_bzread(h, buf, 10_000)
        assert n >= 0
        if n == 0:
            break
        out += buf.raw[:n]
    err = C.c_int(99)
    assert lib.BZ2_bzerror(h, C.byref(err)) == b"OK" and err.value == 0
    lib.BZ2_bzclose(h)
    assert bytes(out) == d
    assert lib.BZ2_bzopen(str(tmp_path / "missing.bz2").encode(), b"r") is None
    # a truncated file is an error, not a short read
    p.write_bytes(bz2.compress(d, 3)[:-5])
    h = lib.BZ2_bzopen(str(p).encode(), b"rs")
    got = 0
    while True:
        n = lib.BZ2_bzread(h, buf, 10_000)
        if n <= 0:
            break
        got += n
    assert n == -1
    assert lib.BZ2_bzerror(h, C.byref(err)) == b"UNEXPECTED_EOF" and err.value == BZ_UNEXPECTED_EOF
    lib.BZ2_bzclose(h)


def test_decompress_param_and_sequence_errors():
    lib = binding.load()
    assert lib.BZ2_bzDecompressInit(None, 0, 0) == -2
    s = binding.BzStream()
    assert lib.BZ2_bzDecompressInit(C.byref(s), 5, 0) == -2
    assert lib.BZ2_bzDecompressInit(C.byref(s), 0, 2) == -2
    assert lib.BZ2_bzDecompress(None) == -2
    assert lib.BZ2_bzDecompressEnd(None) == -2
    s2 = binding.BzStream()
    assert lib.BZ2_bzDecompress(C.byref(s2)) == -2          # never initialised
    assert lib.BZ2_bzDecompressInit(C.byref(s), 0, 1) == 0
    assert lib.BZ2_bzDecompressEnd(C.byref(s)) == 0
    assert lib.BZ2_bzDecompressEnd(C.byref(s)) == -2        # state already released
    n = C.c_uint(10)
    assert lib.BZ2_bzBuffToBuffDecompress(None, C.byref(n), b"x", 1, 0, 0) == -2


def test_cli_decompress_and_test_modes(tmp_path):
    import subprocess
    cli = os.path.join(os.path.dirname(binding.LIB_PATH), "bzip2-b200")
    d = support.gen_text(200_000, 4).tobytes()
    (tmp_path / "a.bz2").write_bytes(bz2.compress(d, 2) + bz2.compress(b"more"))
    (tmp_path / "b.tbz2").write_bytes(bz2.compress(d) + b"garbage!")
    (tmp_path / "c.bz2").write_bytes(bz2.compress(d)[:-9])
    (tmp_path / "d.bz2").write_bytes(b"plain text, not bzip2")
    run = lambda *a: subprocess.run([cli, *a], cwd=tmp_path, capture_output=True)
    assert run("-t", "a.bz2", "b.tbz2").returncode == 0
    assert run("-t", "c.bz2").returncode == 2
    assert run("-t", "d.bz2").returncode == 2
    r = run("-dc", "a.bz2")
    assert r.returncode == 0 and r.stdout == d + b"more"
    assert run("-dk", "a.bz2", "b.tbz2").returncode == 0
    assert (tmp_path / "a").read_bytes() == d + b"more" and (tmp_path / "a.bz2").exists()
    assert (tmp_path / "b.tar").read_bytes() == d
    assert run("-d", "a.bz2").returncode == 1                 # output exists
    assert run("-df", "a.bz2").returncode == 0 and not (tmp_path / "a.bz2").exists()
    assert run("-d", "c.bz2").returncode == 2 and not (tmp_path / "c").exists() and (tmp_path / "c.bz2").exists()
    r = subprocess.run([cli, "-d"], input=bz2.compress(d), capture_output=True)
    assert r.returncode == 0 and r.stdout == d
