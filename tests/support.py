"""Shared test/bench support: ctypes bindings for the checkers and workload generators.

Nothing here is product code.  `oracle()` is our CPU restatement (oracle/liboracle.so),
`ref()` is the unmodified reference compiled from /root/reference (oracle/_ref/libbz2_ref.so,
present only when it was built in the authoring container and shipped with the snapshot).
"""
import ctypes as C
import os
import subprocess
import functools
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
GOLDEN = os.path.join(ROOT, "tests", "golden")

u8p = C.POINTER(C.c_uint8)


def _p(a, t=C.c_uint8):
    return a.ctypes.data_as(C.POINTER(t))


class OrcBlock(C.Structure):
    _fields_ = [("in_begin", C.c_uint64), ("in_end", C.c_uint64), ("nblock", C.c_int32), ("crc", C.c_uint32)]


class RefRec(C.Structure):
    _fields_ = [("in_end", C.c_uint64), ("nblock", C.c_int32), ("block_crc", C.c_uint32),
                ("comb_crc", C.c_uint32), ("orig_ptr", C.c_int32), ("n_mtf", C.c_int32),
                ("n_in_use", C.c_int32), ("num_z", C.c_int32)]


@functools.lru_cache(None)
def oracle():
    path = os.path.join(ORACLE_DIR, "liboracle.so")
    if not os.path.exists(path):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)
    lib = C.CDLL(path)
    lib.orc_crc.restype = C.c_uint32
    lib.orc_crc.argtypes = [u8p, C.c_uint64]
    lib.orc_rle1_split.restype = C.c_int64
    lib.orc_rle1_split.argtypes = [u8p, C.c_uint64, C.c_int, C.c_int, C.POINTER(OrcBlock), C.c_int64]
    lib.orc_rle1_emit.restype = C.c_int32
    lib.orc_rle1_emit.argtypes = [u8p, C.c_uint64, C.c_uint64, u8p, u8p]
    lib.orc_bwt.restype = C.c_int32
    lib.orc_bwt.argtypes = [u8p, C.c_int32, u8p, C.POINTER(C.c_int32)]
    lib.orc_tie_offset.restype = C.c_int32
    lib.orc_tie_offset.argtypes = [u8p, C.c_int32, C.c_int32]
    lib.orc_mtf.restype = C.c_int32
    lib.orc_mtf.argtypes = [u8p, C.c_int32, u8p, C.POINTER(C.c_uint16), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.orc_make_code_lengths.restype = None
    lib.orc_make_code_lengths.argtypes = [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32, C.c_int32]
    lib.orc_send_mtf.restype = None
    lib.orc_send_mtf.argtypes = [C.POINTER(C.c_uint16), C.c_int32, u8p, C.POINTER(C.c_int32), u8p, C.POINTER(C.c_uint64)]
    lib.orc_send_mtf_tables.restype = C.c_int32
    lib.orc_send_mtf_tables.argtypes = [C.POINTER(C.c_uint16), C.c_int32, u8p, C.POINTER(C.c_int32), u8p,
                                        C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_uint64)]
    lib.orc_compress.restype = C.c_int64
    lib.orc_compress.argtypes = [u8p, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_int32), u8p, C.c_uint64]
    lib.gen_text.restype = C.c_uint64
    lib.gen_text.argtypes = [u8p, C.c_uint64, u8p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32,
                             C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]
    lib.gen_random.restype = None
    lib.gen_random.argtypes = [u8p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.gen_tile.restype = None
    lib.gen_tile.argtypes = [u8p, C.c_uint64, u8p, C.c_uint64, C.c_uint64]
    lib.gen_runs.restype = None
    lib.gen_runs.argtypes = [u8p, C.c_uint64, C.POINTER(C.c_uint64)]
    return lib


def have_ref():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libbz2_ref.so"))


@functools.lru_cache(None)
def ref():
    path = os.path.join(ORACLE_DIR, "_ref", "libbz2_ref.so")
    # RTLD_DEEPBIND: the product library exports the same BZ2_* names.
    lib = C.CDLL(path, mode=os.RTLD_LOCAL | os.RTLD_DEEPBIND)
    lib.BZ2_bzBuffToBuffCompress.restype = C.c_int
    lib.BZ2_bzBuffToBuffCompress.argtypes = [u8p, C.POINTER(C.c_uint), u8p, C.c_uint, C.c_int, C.c_int, C.c_int]
    lib.BZ2_bzBuffToBuffDecompress.restype = C.c_int
    lib.BZ2_bzBuffToBuffDecompress.argtypes = [u8p, C.POINTER(C.c_uint), u8p, C.c_uint, C.c_int, C.c_int]
    lib.ref_trace.restype = C.c_int
    lib.ref_trace.argtypes = [u8p, C.c_uint64, C.c_int, C.POINTER(RefRec), C.c_int, C.c_int, u8p, u8p, C.c_uint64,
                              C.POINTER(C.c_uint64)]
    lib.ref_bwt.restype = C.c_int
    lib.ref_bwt.argtypes = [u8p, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
    lib.ref_mtf.restype = C.c_int
    lib.ref_mtf.argtypes = [u8p, C.c_int, u8p, C.POINTER(C.c_uint16), C.POINTER(C.c_int), C.POINTER(C.c_int32),
                            C.POINTER(C.c_int)]
    lib.ref_send_mtf.restype = C.c_int
    lib.ref_send_mtf.argtypes = [C.POINTER(C.c_uint16), C.c_int, u8p, u8p, C.c_int, C.POINTER(C.c_int64)]
    lib.ref_make_code_lengths.restype = None
    lib.ref_make_code_lengths.argtypes = [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int, C.c_int]
    lib.ref_crc.restype = C.c_uint32
    lib.ref_crc.argtypes = [u8p, C.c_uint64]
    return lib


# ----------------------------------------------------------------------------- wrappers
def as_u8(data):
    if isinstance(data, (bytes, bytearray)):
        return np.frombuffer(bytes(data), dtype=np.uint8).copy() if len(data) else np.zeros(0, np.uint8)
    return np.ascontiguousarray(data, dtype=np.uint8)


def _buf(a):
    return _p(a) if a.size else C.cast(C.create_string_buffer(1), u8p)


def ref_compress(data, level=9):
    a = as_u8(data)
    cap = int(a.size * 1.02) + 1000
    out = np.zeros(cap, np.uint8)
    n = C.c_uint(cap)
    rc = ref().BZ2_bzBuffToBuffCompress(_p(out), C.byref(n), _buf(a), a.size, level, 0, 0)
    assert rc == 0, rc
    return out[: n.value].tobytes()


def ref_decompress(comp, out_size):
    a = as_u8(comp)
    out = np.zeros(max(out_size, 1), np.uint8)
    n = C.c_uint(out.size)
    rc = ref().BZ2_bzBuffToBuffDecompress(_p(out), C.byref(n), _p(a), a.size, 0, 0)
    assert rc == 0, rc
    return out[: n.value].tobytes()


def ref_trace(data, level=9, want_block=-1):
    a = as_u8(data)
    maxb = a.size // (100000 * level - 30) + 3
    recs = (RefRec * maxb)()
    blk = np.zeros(900016, np.uint8)
    cap = int(a.size * 1.02) + 1000
    out = np.zeros(cap, np.uint8)
    olen = C.c_uint64(0)
    nb = ref().ref_trace(_buf(a), a.size, level, recs, maxb, want_block, _p(blk), _p(out), cap, C.byref(olen))
    assert nb >= 0, nb
    return [recs[i] for i in range(nb)], blk, out[: olen.value].tobytes()


def ref_bwt(block):
    a = as_u8(block)
    out = np.zeros(a.size + 1, np.uint32)
    op = C.c_int(0)
    rc = ref().ref_bwt(_p(a), a.size, _p(out, C.c_uint32), C.byref(op))
    assert rc == 0
    return out[: a.size].astype(np.uint8), op.value


def orc_split(data, level=9, tail_merge=1):
    a = as_u8(data)
    maxb = (a.size + a.size // 4) // (100000 * level - 30) + 3       # RLE1 turns a run of four into five bytes
    blocks = (OrcBlock * maxb)()
    nb = oracle().orc_rle1_split(_buf(a), a.size, level, tail_merge, blocks, maxb)
    assert 0 <= nb <= maxb
    return [blocks[i] for i in range(nb)]


def orc_rle1_emit(data, begin, end):
    a = as_u8(data)
    out = np.zeros((end - begin) * 5 // 4 + 16, np.uint8)
    inuse = np.zeros(256, np.uint8)
    n = oracle().orc_rle1_emit(_buf(a), begin, end, _p(out), _p(inuse))
    return out[:n].copy(), inuse


def orc_bwt(block):
    a = as_u8(block)
    out = np.zeros(a.size, np.uint8)
    op = C.c_int32(0)
    q = oracle().orc_bwt(_p(a), a.size, _p(out), C.byref(op))
    return out, op.value, q


def orc_tie_offset(block, q):
    """g with origPtr_ref = lo + g for an exact power block u^q (oracle/tie_order.c)."""
    a = as_u8(block)
    return int(oracle().orc_tie_offset(_buf(a), a.size, q))


def orc_mtf(bwt, inuse):
    a = as_u8(bwt)
    iu = as_u8(inuse)
    mtfv = np.zeros(a.size + 2, np.uint16)
    freq = np.zeros(258, np.int32)
    nu = C.c_int32(0)
    n = oracle().orc_mtf(_p(a), a.size, _p(iu), _p(mtfv, C.c_uint16), _p(freq, C.c_int32), C.byref(nu))
    return mtfv[:n].copy(), freq, nu.value


def orc_send_mtf_tables(mtfv, freq, inuse):
    """Stage 4's decisions for one block: (nGroups, selectors, code lengths [6][258], halvings [4 passes][6 tables],
    bits of the coded section from the symbol map on)."""
    m = np.ascontiguousarray(mtfv, dtype=np.uint16)
    f = np.ascontiguousarray(freq, dtype=np.int32)
    iu = as_u8(inuse)
    sel = np.zeros((m.size + 49) // 50 + 1, np.uint8)
    lens = np.zeros((6, 258), np.int32)
    halv = np.zeros((4, 6), np.int32)
    bits = C.c_uint64(0)
    ng = oracle().orc_send_mtf_tables(_p(m, C.c_uint16), m.size, _p(iu), _p(f, C.c_int32), _p(sel), _p(lens, C.c_int32),
                                      _p(halv, C.c_int32), C.byref(bits))
    return ng, sel[: (m.size + 49) // 50].copy(), lens, halv, bits.value


def orc_compress(data, level=9, tail_merge=1, force_orig_ptr=None):
    a = as_u8(data)
    cap = int(a.size * 1.3) + 100000
    out = np.zeros(cap, np.uint8)
    fp = None
    if force_orig_ptr is not None:
        fo = np.ascontiguousarray(force_orig_ptr, dtype=np.int32)
        fp = _p(fo, C.c_int32)
    n = oracle().orc_compress(_buf(a), a.size, level, tail_merge, fp, _p(out), cap)
    assert n > 0, n
    return out[:n].tobytes()


# ----------------------------------------------------------------------------- stage 2 parameters
def hist_stride(level, hist_log2=18):
    """k-gram bins reserved per block (engine_new, csrc/engine.cu; BZ2_B200_HIST_LOG2 = hist_log2)"""
    nmax = 100000 * level - 19
    s = 1 << 16
    while s < (1 << hist_log2) and s < nmax // 4:
        s <<= 1
    if hist_log2 > 18 and s < nmax * 2:
        s = 1 << hist_log2
    return s


def codemap(ninuse, stride, maxk=24):
    """k_codemap (csrc/stage2_bwt.cu): (k, nbins, bits per symbol, m) of a block with `ninuse` symbols.  The k-gram
    sort starts at depth k with ninuse^k buckets; a text key holds the next m symbols in m * bits <= 51 bits."""
    k, bins = 1, max(ninuse, 1)
    while ninuse > 1 and k < maxk and bins * ninuse <= stride:
        bins *= ninuse
        k += 1
    bits = 1
    while (1 << bits) < ninuse:
        bits += 1
    return k, bins, bits, min(51 // bits, 48)


# ----------------------------------------------------------------------------- generators
@functools.lru_cache(None)
def _vocab():
    toks = open(os.path.join(GOLDEN, "vocab.txt"), "rb").read().split()
    blob = np.frombuffer(b"".join(toks), dtype=np.uint8).copy()
    lens = np.array([len(t) for t in toks], dtype=np.int32)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32)
    return blob, offs, lens


TEXT_SEED = 0x0123456789ABCDEF


def gen_text(n, seed=TEXT_SEED, out=None):
    """SURVEY.md 8(d) C2: Zipf text over the words0-3 vocabulary."""
    blob, offs, lens = _vocab()
    if out is None:
        out = np.empty(n, np.uint8)
    st = C.c_uint64(seed)
    til = C.c_int32(0)
    oracle().gen_text(_p(out), n, _p(blob), _p(offs, C.c_int32), _p(lens, C.c_int32), len(lens), C.byref(st), C.byref(til))
    return out


def gen_random(n, seed=2, out=None):
    if out is None:
        out = np.empty(n, np.uint8)
    st = C.c_uint64(seed)
    oracle().gen_random(_p(out), n, C.byref(st))
    return out


def gen_tile(n, unit, out=None):
    u = as_u8(unit)
    if out is None:
        out = np.empty(n, np.uint8)
    oracle().gen_tile(_p(out), n, _p(u), u.size, 0)
    return out


def gen_period1000(n):
    return gen_tile(n, gen_random(1000, seed=1))


def gen_runs(n, seed=3):
    out = np.empty(n, np.uint8)
    st = C.c_uint64(seed)
    oracle().gen_runs(_p(out), n, C.byref(st))
    return out


def gen_mixed(n, seg=1 << 20):
    """C4-style mix: text / binary-ish / random segments (segment size scaled down for tests)."""
    out = np.empty(n, np.uint8)
    kinds = 0
    pos = 0
    while pos < n:
        m = min(seg, n - pos)
        k = kinds % 3
        if k == 0:
            out[pos:pos + m] = gen_text(m, seed=TEXT_SEED + kinds)
        elif k == 1:
            base = gen_random(4096, seed=77 + kinds)
            out[pos:pos + m] = np.resize(np.concatenate([base, base[::-1] // 3, np.repeat(base[:512], 7)]), m)
        else:
            out[pos:pos + m] = gen_random(m, seed=1000 + kinds)
        pos += m
        kinds += 1
    return out


def gen_c4(n, seg=64 << 20):
    """SURVEY 8(d) config C4: segments cycling T, B, R.  T = the C2 text generator (one continuing stream),
    B = sample1.ref || sample2.ref (311,036 bytes of real binary, tests/golden/) tiled, R = raw xorshift64*
    bytes (seed 2, one continuing stream)."""
    nseg = (n + seg - 1) // seg
    n_t = sum(min(seg, n - k * seg) for k in range(nseg) if k % 3 == 0)
    n_r = sum(min(seg, n - k * seg) for k in range(nseg) if k % 3 == 2)
    text = gen_text(max(n_t, 1), TEXT_SEED)
    rnd = gen_random(max(n_r, 1), 2)
    with open(os.path.join(GOLDEN, "sample1.ref"), "rb") as f1, open(os.path.join(GOLDEN, "sample2.ref"), "rb") as f2:
        binary = np.frombuffer(f1.read() + f2.read(), np.uint8)
    out = np.empty(n, np.uint8)
    tp = rp = 0
    for k in range(nseg):
        pos = k * seg
        m = min(seg, n - pos)
        if k % 3 == 0:
            out[pos:pos + m] = text[tp:tp + m]; tp += m
        elif k % 3 == 1:
            out[pos:pos + m] = np.resize(binary, m)
        else:
            out[pos:pos + m] = rnd[rp:rp + m]; rp += m
    return out


def power_stream_cases():
    """Inputs whose blocks are exact powers u^q (golden streams minted from the reference).  The first six have
    units with a single B* suffix (closed form on the GPU), the rest several (tie-order replay)."""
    yield "zeros_2M_L9", np.zeros(2_000_000, np.uint8), 9
    yield "zeros_700k_L1", np.zeros(700_000, np.uint8), 1
    yield "ff_1M_L5", np.full(1_000_000, 255, np.uint8), 5
    yield "aab_2M_L9", gen_tile(2_000_000, b"aab"), 9
    yield "aab_500k_L1", gen_tile(500_000, b"aab"), 1
    yield "period7_400k_L1", gen_tile(400_000, b"1234567"), 1
    rec7 = gen_tile(420_000, b"ab\ncd\n.")                  # 7-byte records: every full block at -1 is (rec)^14283
    yield "rec7_420k_L1", rec7, 1
    yield "rec7_420k_L5", rec7, 5
    yield "rec7_420k_L9", rec7, 9
    yield "abcabd_600k_L2", gen_tile(600_000, b"abcabd"), 2
    yield "aabb_900k_L3", gen_tile(900_000, b"aabb"), 3
    yield "abcdcb_1M_L1", gen_tile(1_000_000, b"abcdcb"), 1
    yield "rec21_350k_L1", gen_tile(350_000, b"id,name,value\n1,ab,2\n"), 1


def random_power_case(seed, p, alpha, q):
    """u = p seeded bytes over an alphabet of `alpha`, tiled q times (tests/golden/powers_random.json)."""
    u = gen_random(p, seed=seed).astype(np.uint32) % alpha + (48 if alpha < 200 else 0)
    return np.tile(u.astype(np.uint8), q)


def long_repeat_cases():
    """Inputs with long NON-tandem repeats (a copy of the same data hundreds of kB further on): the shapes the
    repeat passes of stage 2 (2e) exist for.  (name, uint8 array); seeded, so they double as golden stream cases."""
    rng = np.random.default_rng(5)
    r300 = rng.integers(0, 256, 300_000, dtype=np.uint8)
    txt = gen_text(260_000, seed=9)
    edited = txt.copy()
    edited[100_000] ^= 1                                     # second copy differs in one byte
    binary = np.frombuffer(open(os.path.join(GOLDEN, "sample1.ref"), "rb").read() + open(os.path.join(GOLDEN, "sample2.ref"), "rb").read(), np.uint8)
    few = rng.integers(0, 4, 5_000, dtype=np.uint8) + 65
    return [
        ("random300k_x3", np.resize(r300, 2_000_000)),                      # every rotation has a twin 300 kB further on
        ("random130k_x7", np.resize(r300[:130_000], 1_700_000)),            # up to seven copies per block: several keys per visit
        ("text_twice_edited", np.concatenate([txt, edited, txt[:150_000]])),
        ("binary_tiled", np.resize(binary, 1_900_000)),                     # the C4 binary third
        ("period5000_4sym", np.resize(few, 1_500_000)),
        ("random_then_copy_shifted", np.concatenate([r300[:200_000], few, r300[:200_000], r300[50_000:250_000]])),
    ]
