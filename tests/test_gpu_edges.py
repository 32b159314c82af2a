"""GPU: the BWT and Huffman kernels at the edges of their parameters, block by block against the oracle.

The rest of the GPU suite feeds whole streams of a few generators through the default build.  Stage 2 changes its
behaviour with the block's alphabet (k-gram depth k, bits per symbol, text-key width m, aggregated or direct count
pass), the level's bin budget, the size class of every segment and the switches read at engine creation; stage 4 has a
halve-and-retry loop that ordinary data never reaches.  Every case here goes through check_window(), which compares each
stage of every block with the oracle, and asserts that it reached the path it is aimed at."""
import bz2
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import support as S
import bzip2_b200 as B

pytestmark = pytest.mark.gpu

HDR_BITS = 48 + 32 + 1 + 24             # block magic, CRC, randomised bit, origPtr: stage 4's bit count includes them
ALPHAS = [2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 61, 63, 64, 65, 127, 128, 129, 200, 255, 256]
CLASS_EDGES = [2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 256, 257, 512, 513, 1024, 1025, 2048, 2049, 4096, 4097, 8192, 8193,
               20_000, 70_000]


def nmax(level):
    return 100000 * level - 19


@pytest.fixture(scope="module")
def engines():
    """One default engine per level, shared by the cases of this file; closed when the module ends."""
    live = {}

    def get(level):
        if level not in live:
            while live:
                live.pop(next(iter(live))).close()
            live[level] = B.Engine(level=level)
        return live[level]
    try:
        yield get
    finally:
        for e in live.values():
            e.close()


def check_window(eng, data, level, blocks=None, whole=True):
    """Compress `data` (one window) and compare every stage of the chosen blocks (default: all) with the oracle:
    block split, input offsets, CRC, RLE1 output, inUse and its size, BWT and origPtr, the MTF values and their
    counts, stage 4's table count, selectors, code lengths and coded size.  With `whole`, the stream must also equal
    orc_compress.  Returns (stream, per-block facts) for the coverage assertions of the callers."""
    data = S.as_u8(data)
    out = eng.compress(data)
    assert eng.stats.n_windows == 1
    split = S.orc_split(data, level)
    X = eng.fetch("X", np.uint32).astype(np.int64)
    P = eng.fetch("P", np.uint32)
    assert len(X) - 1 == len(split)
    assert [int(x) for x in np.diff(X)] == [b.nblock for b in split]
    assert [int(p) for p in P[:-1]] == [b.in_begin for b in split] and int(P[-1]) == data.size
    assert [int(c) for c in eng.fetch("crc", np.uint32)] == [b.crc for b in split]
    enc = eng.fetch("enc", np.uint8)
    bwt = eng.fetch("bwt", np.uint8)
    mtfv = eng.fetch("mtfv", np.uint16)
    nmtf = eng.fetch("nmtf", np.uint32)
    op = eng.fetch("origptr", np.uint32)
    inuse = eng.fetch("inuse", np.uint8).reshape(-1, 256)
    ninuse = eng.fetch("ninuse", np.uint32)
    freq = eng.fetch("mtffreq", np.int32).reshape(-1, 258)
    ngroups = eng.fetch("ngroups", np.uint32)
    sel = eng.fetch("sel", np.uint8)
    hlen = eng.fetch("hlen", np.uint8).reshape(-1, 6, 258)
    bits = eng.fetch("bits", np.uint64)
    facts = []
    for b in (range(len(split)) if blocks is None else blocks):
        blk = split[b]
        x0, x1 = int(X[b]), int(X[b + 1])
        where = f"block {b} of {len(split)}"
        e_exp, iu_exp = S.orc_rle1_emit(data, blk.in_begin, blk.in_end)
        assert np.array_equal(enc[x0:x1], e_exp), f"S1 enc {where}"
        assert np.array_equal(inuse[b], iu_exp), f"inUse {where}"
        assert int(ninuse[b]) == int(iu_exp.sum()), f"nInUse {where}"
        bw_exp, op_exp, q = S.orc_bwt(e_exp)
        assert np.array_equal(bwt[x0:x1], bw_exp), f"S2 BWT {where}"
        assert int(op[b]) == op_exp, f"S2 origPtr {where}"
        m_exp, f_exp, _ = S.orc_mtf(bw_exp, iu_exp)
        assert int(nmtf[b]) == len(m_exp), f"S3 nMTF {where}"
        assert np.array_equal(mtfv[x0 + b: x0 + b + len(m_exp)], m_exp), f"S3 mtfv {where}"
        assert np.array_equal(freq[b], f_exp), f"S3 mtfFreq {where}"
        ng, sel_exp, len_exp, halv, cbits = S.orc_send_mtf_tables(m_exp, f_exp, iu_exp)
        assert int(ngroups[b]) == ng, f"S4 nGroups {where}"
        s0 = (x0 + b) // 50 + b
        assert np.array_equal(sel[s0: s0 + len(sel_exp)], sel_exp), f"S4 selectors {where}"
        assert np.array_equal(hlen[b].astype(np.int32), len_exp), f"S4 code lengths {where}"
        assert int(bits[b]) == HDR_BITS + cbits, f"S4 coded bits {where}"
        facts.append({"n": x1 - x0, "ninuse": int(ninuse[b]), "nmtf": len(m_exp), "halvings": int(halv.sum()), "q": q})
    if whole:
        assert out == S.orc_compress(data, level)
    return out, facts


# ------------------------------------------------------------------ generators
def cap_runs(a, cap=3):
    """drop every byte that would extend a run beyond `cap`: RLE1 then leaves the data alone"""
    if a.size == 0:
        return a
    starts = np.r_[True, a[1:] != a[:-1]]
    first = np.flatnonzero(starts)
    pos = np.arange(a.size) - first[np.cumsum(starts) - 1]
    return a[pos < cap]


def run_free(rng, n, syms):
    """i.i.d. symbols from `syms` with runs cut to 3: inUse is exactly the symbols drawn"""
    syms = np.asarray(syms, np.uint8)
    out = cap_runs(syms[rng.integers(0, syms.size, 2 * n + 16)])
    assert out.size >= n
    return out[:n]


def edited_twice(rng, n, syms):
    """run-free data that contains a long copy of itself with a few substitutions: the copy keeps doubling rounds and
    the repeat passes busy at the block's key width"""
    half = run_free(rng, n // 2 + 64, syms)
    copy = half.copy()
    at = rng.integers(0, copy.size, 6)
    copy[at] = np.asarray(syms, np.uint8)[rng.integers(0, len(syms), at.size)]
    out = cap_runs(np.concatenate([half, copy]))
    while out.size < n:
        out = cap_runs(np.concatenate([out, run_free(rng, n - out.size + 8, syms)]))
    return out[:n]


def runs251(rng, n_enc, others, long_every=40):
    """Bytes whose RLE1 output uses only `others` + [251]: runs of the other symbols are 1-3 long, runs of 251 are 1-3
    long or whole multiples of 255 (each 255-chunk encodes to five 251s).  The long 251-stretches give the largest
    k-gram key of the block (all symbols = the top code).  Returns input bytes whose RLE1 output is about n_enc long."""
    others = np.asarray(others, np.uint8)
    vals, lens = [], []
    enc = 0
    turn = 0
    while enc < n_enc:
        if turn % 2 == 0:
            v = int(others[rng.integers(0, others.size)])
            ln = int(rng.integers(1, 4))
            vals.append(v); lens.append(ln); enc += ln
        else:
            if rng.integers(0, long_every) == 0:
                q = int(rng.integers(1, 5))
                vals.append(251); lens.append(255 * q); enc += 5 * q
            else:
                ln = int(rng.integers(1, 4))
                vals.append(251); lens.append(ln); enc += ln
        turn += 1
    return np.repeat(np.asarray(vals, np.uint8), lens)


def geometric(seed, n, ratio, nsym):
    rng = np.random.default_rng(seed)
    p = ratio ** np.arange(nsym)
    return rng.choice(nsym, n, p=p / p.sum()).astype(np.uint8)


# ------------------------------------------------------------------ alphabet sweep
def alphabet_window(level, shape, seed):
    """one block per alphabet size: every segment is exactly nmax run-free bytes and ends where the next one starts
    with a different byte, so the split puts each alphabet in a block of its own"""
    rng = np.random.default_rng(seed)
    segs, alphas = [], []
    for a in ALPHAS:
        syms = np.sort(rng.choice(256, a, replace=False))
        while True:
            seg = run_free(rng, nmax(level), syms) if shape == "iid" else edited_twice(rng, nmax(level), syms)
            if not segs or seg[0] != segs[-1][-1]:
                break
        segs.append(seg)
        alphas.append(a)
    return np.concatenate(segs), alphas


@pytest.mark.parametrize("level", [1, 3, 9])
def test_alphabet_sweep(engines, level):
    seen = set()
    for shape, seed in (("iid", 10 + level), ("copy", 20 + level)):
        data, alphas = alphabet_window(level, shape, seed)
        _, facts = check_window(engines(level), data, level)
        assert [f["ninuse"] for f in facts] == alphas, shape
        stride = S.hist_stride(level)
        for f in facts:
            k, nbins, bits, m = S.codemap(f["ninuse"], stride)
            seen.add((stride, bits, f["ninuse"] <= 128 and nbins < (1 << 19)))
    # one block of a single symbol: 255-runs of 251 encode to 251 only
    d = np.full(255 * (nmax(level) // 5 + 7), 251, np.uint8)
    _, facts = check_window(engines(level), d, level)
    assert all(f["ninuse"] == 1 for f in facts) and facts[0]["q"] > 1
    assert {b for _, b, _ in seen} == set(range(1, 9))                  # bits per symbol 1..8
    assert {agg for _, _, agg in seen} == {True, False}                  # both count passes
    assert {s for s, _, _ in seen} == {{1: 1 << 16, 3: 1 << 17, 9: 1 << 18}[level]}


# ------------------------------------------------------------------ size classes of the refinement sorts
def class_edge_windows():
    """Single-block windows at -9 (byte alphabet: k = 2, m = 6, so a segment is resolved in round 0 unless its
    rotations agree on 8 bytes).  S copies of a marker start with 0xFF and a marker id, and no other byte is 0xFF, so
    the k-gram bucket of that pair holds exactly S rotations.  Three kinds per S:
      short  marker of 2 bytes, distinct tails: a round-0 segment of S that the text keys resolve;
      long   marker of 12 bytes, distinct tails: the S rotations reach the doubling rounds together;
      ties   marker of 2 bytes, tails that start with one of three 12-byte strings: equal keys in runs of about S/3
             inside the segment in round 0 and again in the first doubling round.
    The copies of all kinds are shuffled and packed into blocks of up to 850 kB (a kind never straddles two)."""
    rng = np.random.default_rng(99)
    shared = [rng.integers(0, 255, 12, dtype=np.uint8) for _ in range(3)]
    groups = []
    mid = 0
    for s in CLASS_EDGES:
        for kind in ("short", "long", "ties"):
            if s == 70_000 and kind != "short":
                continue                     # 70 000 copies of a longer record do not fit one block
            mid += 1
            marker = np.r_[np.uint8(255), np.uint8(mid), rng.integers(0, 255, 10 if kind == "long" else 0, dtype=np.uint8)]
            tails = rng.integers(0, 255, (s, 8), dtype=np.uint8)
            if kind == "ties":
                pick = rng.integers(0, 3, s)
                tails = np.concatenate([np.stack([shared[i] for i in pick]), tails], axis=1)
            recs = np.concatenate([np.broadcast_to(marker, (s, marker.size)), tails], axis=1)
            groups.append(recs)
    windows, cur, size = [], [], 0
    for recs in sorted(groups, key=lambda r: -r.size):
        if size + recs.size > 850_000 and cur:
            windows.append(cur); cur, size = [], 0
        cur.append(recs); size += recs.size
    windows.append(cur)
    out = []
    for w in windows:
        rows = [r for recs in w for r in recs]
        order = rng.permutation(len(rows))
        out.append(np.concatenate([rows[i] for i in order]))
    return out


_TRACE = re.compile(r"\[bz2b200\] round (\d+):((?: c\d+=\d+/\d+)+)")


def class_trace():
    """BZ2_B200_TRACE=1 lines of the class-edge windows: {round: {class: segments}} summed over windows.  trace_on()
    reads the variable once per process, so the windows run in a child process."""
    here = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import bzip2_b200 as B, test_gpu_edges as T\n"
            "e = B.Engine(level=9)\n"
            "try:\n"
            "    [e.compress(w) for w in T.class_edge_windows()]\n"
            "finally:\n"
            "    e.close()\n") % (S.ROOT, here)
    env = dict(os.environ, BZ2_B200_TRACE="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    rounds = {}
    for m in _TRACE.finditer(r.stderr):
        per = rounds.setdefault(int(m.group(1)), {})
        for c, cnt in re.findall(r"c(\d+)=(\d+)/", m.group(2)):
            per[int(c)] = per.get(int(c), 0) + int(cnt)
    return rounds


def test_size_class_edges(engines):
    for w in class_edge_windows():
        check_window(engines(9), w, 9)
    rounds = class_trace()
    assert 0 in rounds and len(rounds) >= 2
    first = {c for c, n in rounds[0].items() if n}
    later = {c for r, per in rounds.items() if r >= 1 for c, n in per.items() if n}
    # Every class in round 0 (64-bit text keys) and in some doubling round (rank keys).  Not aimed at: k_refine_large
    # with 2 radix passes (doubling rounds in blocks of <= 65536 encoded bytes).  A segment of more than 8192 rotations
    # that agree on 8 bytes needs 8193 non-overlapping copies (more than 65536 bytes) unless the copies overlap, and
    # overlapping copies are a tandem repeat that k_resolve_periodic settles before the sort.
    assert first == set(range(12)), sorted(first)
    assert later == set(range(12)), sorted(later)


# ------------------------------------------------------------------ block sizes
BLOCK_SIZES = list(range(1, 41)) + [1023, 1024, 1025, 4095, 4096, 4097, 8191, 8192, 8193, 65535, 65536, 65537]


def test_block_size_edges(engines):
    """k >= n (the `deep` path of k_seg_init), the halo wrap of k_kgram, and the tile edges of the k-gram and MTF
    passes.  n counts encoded bytes.  A one-symbol block is all 251 (255-runs encode to five 251s, 1-3 more stay as
    they are), which cannot make n = 4 mod 5."""
    rng = np.random.default_rng(5)
    eng = engines(9)
    checked = 0
    for n in BLOCK_SIZES:
        for a in (1, 2, 3, 256):
            if a == 1:
                if n % 5 == 4:
                    continue
                d = np.full(255 * (n // 5) + n % 5, 251, np.uint8)
            else:
                d = run_free(rng, n, np.sort(rng.choice(256, a, replace=False)))
            _, facts = check_window(eng, d, 9)
            assert [f["n"] for f in facts] == [n], (n, a)
            checked += 1
    assert checked == len(BLOCK_SIZES) * 4 - sum(1 for n in BLOCK_SIZES if n % 5 == 4)


# ------------------------------------------------------------------ Huffman
@pytest.mark.parametrize("level,seed,n,ratio,nsym", [
    (1, 40, 800_000, 0.6, 40),
    (9, 1, 850_000, 0.5, 20),
    (9, 2, 850_000, 0.6, 30),
    (9, 4, 850_000, 0.55, 25),
])
def test_huffman_length_limit(engines, level, seed, n, ratio, nsym):
    """Geometric i.i.d. sources: some table builds exceed 17 bits and take k_huff_lengths' halve-and-retry loop."""
    d = geometric(seed, n, ratio, nsym)
    _, facts = check_window(engines(level), d, level)
    assert sum(f["halvings"] for f in facts) > 0


NMTF_TARGETS = [49, 50, 51, 199, 200, 201, 599, 600, 601, 1199, 1200, 1201, 2399, 2400, 2401, 2449, 2450, 2451]


def find_nmtf(target):
    """A small seeded input whose block has exactly `target` MTF symbols (bounded search)."""
    for seed in range(64):
        rng = np.random.default_rng(1000 * target + seed)
        alpha = int(rng.choice([40, 128, 256]))
        for n in range(target - 12, target + 12):
            d = rng.integers(0, alpha, max(n, 1), dtype=np.uint8)
            enc, iu = S.orc_rle1_emit(d, 0, d.size)
            bw, _, _ = S.orc_bwt(enc)
            m, _, _ = S.orc_mtf(bw, iu)
            if len(m) == target:
                return d
    return None


def test_ngroups_thresholds(engines):
    """nGroups changes at nMTF = 200, 600, 1200 and 2400; selectors at multiples of 50."""
    eng = engines(9)
    for t in NMTF_TARGETS:
        d = find_nmtf(t)
        assert d is not None, t
        _, facts = check_window(eng, d, 9)
        assert facts[0]["nmtf"] == t


# ------------------------------------------------------------------ top of the position field
def test_highest_flat_positions():
    """A 100 MiB window of runs of exactly four (random, differing bytes) encodes to 1.25x its size, about 131.1 M
    bytes, near the 2^27 limit of the small-class worklist's position field.  The window's last blocks hold the highest
    flat positions; the whole stream must equal a small-window engine's and decode."""
    n = 100 << 20
    rng = np.random.default_rng(7)
    vals = (np.cumsum(rng.integers(1, 256, n // 4)) % 256).astype(np.uint8)
    data = np.repeat(vals, 4)
    eng = B.Engine(level=1, window_bytes=n)
    try:
        nb = len(S.orc_split(data, 1))
        out, _ = check_window(eng, data, 1, blocks=range(nb - 3, nb), whole=False)
        assert int(eng.fetch("X", np.uint32)[-1]) == n // 4 * 5
        assert int(eng.fetch("X", np.uint32)[-1]) > 0.97 * (1 << 27)
    finally:
        eng.close()
    small = B.Engine(level=1, window_bytes=8 << 20)
    try:
        assert small.compress(data) == out
        assert small.stats.n_windows > 10
    finally:
        small.close()
    assert bz2.decompress(out) == data.tobytes()


# ------------------------------------------------------------------ switches read at engine creation
def switch_window(level):
    """Text, the 2- and 3-symbol 251-run constructions, a long repeat and exact powers, in one window of several
    blocks.  Block 0 is exactly nmax run-free bytes, so block 1 is all 251: an exact power that is not the first block
    of a sub-batch of 2 or 5."""
    rng = np.random.default_rng(40 + level)
    nm = nmax(level)
    while True:
        first = run_free(rng, nm, np.arange(256))
        if first[-1] != 251:
            break
    parts = [first, np.full(255 * (nm // 5 + 30), 251, np.uint8), S.gen_text(2 * nm, seed=level)]
    parts.append(runs251(rng, 2 * nm + nm // 4, [int(rng.integers(0, 250))]))
    parts.append(runs251(rng, 2 * nm + nm // 4, [int(v) for v in rng.choice(250, 2, replace=False)]))
    r = rng.integers(0, 256, nm // 3, dtype=np.uint8)
    parts.append(np.resize(r, 3 * nm))                                   # every rotation has twins nm/3 further on
    if nm % 3 == 0:
        parts.append(S.gen_tile(3 * nm + 7, b"abc"))                     # blocks inside it are rotations of abc^q
    return np.concatenate(parts)


SWITCHES = ([("BZ2_B200_S2_GROUP", str(g)) for g in (1, 2, 5)] + [("BZ2_B200_HIST_LOG2", str(h)) for h in range(16, 23)]
            + [("BZ2_B200_CHAIN", "0")])


@pytest.mark.parametrize("level", [1, 9])
def test_switch_invariance(monkeypatch, level):
    data = switch_window(level)
    win = int(data.size * 1.1) + (1 << 20)
    eng = B.Engine(level=level, window_bytes=win)
    try:
        exp, facts = check_window(eng, data, level)
    finally:
        eng.close()
    small = [i for i, f in enumerate(facts) if f["ninuse"] in (2, 3)]
    powers = [i for i, f in enumerate(facts) if f["q"] > 1]
    assert {facts[i]["ninuse"] for i in small} == {2, 3}
    assert 1 in powers, powers
    for name, value in SWITCHES:
        monkeypatch.setenv(name, value)
        eng = B.Engine(level=level, window_bytes=win)
        try:
            assert eng.compress(data) == exp, (name, value)
        finally:
            eng.close()
        monkeypatch.delenv(name)
