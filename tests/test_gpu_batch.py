"""GPU: many independent inputs in one call (bz2b200_compress_batch_*).  Every item's stream must equal the single-input
GPU call on that item and the CPU oracle; the index, the CRCs, the packing rule, the device path, the item mode of
stage 1 and the trace text are checked against what the single-stream path produces."""
import bz2
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import support as S
import bzip2_b200 as B
from bzip2_b200 import binding

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPARAM, EOUTFULL = -1, -5
TAIL_STREAMED, NO_HEADER = 1, 2


def nmax(level):
    return 100000 * level - 19


def no_runs(n, seed):
    """n bytes without two equal neighbours: the RLE1 output is the input, so n is also the encoded size."""
    d = np.random.default_rng(seed).integers(1, 256, n)
    return (np.cumsum(d) % 256).astype(np.uint8)


def window_caps(level, window_bytes, max_items):
    """engine_new's window capacity and block slots (engine.cu)."""
    w = window_bytes or (96 << 20)
    w = max(w, (nmax(level) + 16) * 52)
    w = min(w, 100 << 20)
    enc_cap = w + w // 4 + 4096
    return w, min(enc_cap // nmax(level) + 2 + max_items, 4096)


def predict_windows(level, window_bytes, max_items, sizes):
    """The packing rule: close a window before the item that would exceed its input bytes or block slots; an item
    larger than a window runs through the single-stream window loop (its own windows, counted by the caller)."""
    win, slots_cap = window_caps(level, window_bytes, max_items)
    slots = lambda n: (n + n // 4 + 64) // nmax(level) + 1  # noqa: E731
    windows, big, W, s, open_ = 0, [], 0, 0, False
    for n in sizes:
        if n > win or slots(n) > slots_cap:
            if open_:
                windows += 1
            open_, W, s = False, 0, 0
            big.append(n)
            continue
        if open_ and (W + n > win or s + slots(n) > slots_cap):
            windows += 1
            W, s = 0, 0
        open_ = True
        W += n
        s += slots(n)
    return windows + (1 if open_ else 0), big


def item_mix(level):
    n = nmax(level)
    items = [b"", b"a", b"", bytes(range(2, 42))]
    items += [S.gen_random(k, seed=k).tobytes() for k in (2, 3, 5, 17, 40)]
    items += [S.gen_text(30_000, seed=4).tobytes(), S.gen_random(20_000, seed=5).tobytes(), S.gen_runs(50_000, seed=6).tobytes()]
    items += [S.gen_tile(7 * 3000, b"ab\ncd\n.").tobytes(), S.gen_tile(5000, b"aab").tobytes(), b"\x00" * 4000]
    for k in (n - 1, n, n + 1, n + 2):
        items.append(no_runs(k, k).tobytes())
    items.append(b"")
    return items


@pytest.fixture(scope="module")
def batch_engines():
    engines = {}

    def get(level, window_bytes=0, max_items=64):
        key = (level, window_bytes, max_items)
        if key not in engines:
            while len(engines) >= 2:
                engines.pop(next(iter(engines))).close()
            engines[key] = B.Engine(level=level, window_bytes=window_bytes, max_items=max_items)
        return engines[key]

    yield get
    for e in engines.values():
        e.close()


def check_items(e, items, flags, single=None):
    got = e.compress_batch(items, flags)
    tail_merge = 0 if flags & TAIL_STREAMED else 1
    for k, (x, g) in enumerate(zip(items, got)):
        exp = S.orc_compress(np.frombuffer(x, np.uint8), e.level, tail_merge=tail_merge)
        assert g == exp, f"item {k} ({len(x)} bytes): batch stream differs from the oracle"
        if single is not None:
            assert single.compress(x, flags) == g, f"item {k}: batch stream differs from the single-input call"
    return got


@pytest.mark.parametrize("flags", [0, TAIL_STREAMED])
@pytest.mark.parametrize("level", [1, 5, 9])
def test_item_mix(batch_engines, engine_for, level, flags):
    e = batch_engines(level)
    got = check_items(e, item_mix(level), flags, single=engine_for(level))
    assert got[0] == got[2] and len(got[0]) == 14                     # an empty item: header and trailer only


def test_power_stream_cases(batch_engines):
    by_level = {}
    for name, x, level in S.power_stream_cases():
        if x.size <= 1_000_000:
            by_level.setdefault(level, []).append(x.tobytes())
    for level, items in by_level.items():
        check_items(batch_engines(level), [b"xy"] + items + [b"z"], 0)


def test_item_larger_than_the_window(batch_engines, engine_for):
    level = 1
    e = batch_engines(level, window_bytes=1, max_items=64)            # the smallest window the level allows
    win, _ = window_caps(level, 1, 64)
    big = S.gen_text(win + 300_000, seed=12).tobytes()
    items = [b"abc", S.gen_random(5000, seed=1).tobytes(), big, b"", S.gen_text(7000, seed=3).tobytes(), big[:win]]
    for flags in (0, TAIL_STREAMED):
        check_items(e, items, flags, single=engine_for(level))
        assert e.stats.n_windows >= predict_windows(level, 1, 64, [len(x) for x in items])[0] + 2   # + the big item's own


def test_item_boundaries_do_not_merge(batch_engines, engine_for):
    """Each pair below would encode differently as one stream: runs and chunks must be cut at every item start."""
    items = [b"xyzaaa", b"aabcd",                                   # a run of five across the seam
             b"q" + b"z" * 255, b"z" * 10,                          # a 255-byte run ends exactly at an item end
             b"ab" + b"c" * 2, b"c" * 2 + b"de",                    # runs of four span the seam
             b"m" * 4, b"m" * 4, b"m" * 3, b"m",                    # whole items that are runs
             b"k" * 300, b"k" * 251, b"", b"k" * 4]
    for level in (1, 9):
        for flags in (0, TAIL_STREAMED):
            got = check_items(batch_engines(level), items, flags, single=engine_for(level))
            assert b"".join(got) != engine_for(level).compress(b"".join(items), flags)


def test_packing_edges(batch_engines):
    level, max_items = 1, 64
    e = batch_engines(level, window_bytes=1, max_items=max_items)
    win, slots_cap = window_caps(level, 1, max_items)
    cases = {
        "fill_slots": [S.gen_text(900, seed=k).tobytes() for k in range(slots_cap)],
        "one_more": [S.gen_text(900, seed=k).tobytes() for k in range(slots_cap + 1)],
        "fill_win": [S.gen_text(win // 4, seed=1).tobytes()] * 3 + [S.gen_text(win - 3 * (win // 4), seed=2).tobytes()],
    }
    for name, items in cases.items():
        w, big = predict_windows(level, 1, max_items, [len(x) for x in items])
        assert not big
        check_items(e, items, 0)
        assert e.stats.n_windows == w, name
    assert predict_windows(level, 1, max_items, [len(x) for x in cases["fill_slots"]])[0] == 1
    assert predict_windows(level, 1, max_items, [len(x) for x in cases["one_more"]])[0] == 2
    assert sum(map(len, cases["fill_win"])) == win


def test_many_items_many_windows(batch_engines, engine_for):
    rng = np.random.default_rng(7)
    sizes = rng.integers(0, 400, 5000)
    sizes[::97] = 0
    gens = (S.gen_text, S.gen_random, S.gen_runs)
    items = [gens[k % 3](int(n), seed=k + 1).tobytes() if n else b"" for k, n in enumerate(sizes)]
    level = 1
    e = batch_engines(level, window_bytes=1, max_items=64)
    got = check_items(e, items, 0)
    w, _ = predict_windows(level, 1, 64, list(sizes))
    assert e.stats.n_windows == w and w > 10
    assert e.stats.in_bytes == sum(sizes) and e.stats.out_bits == 8 * sum(map(len, got)) and e.stats.combined_crc == 0
    # a default engine (no extra slots) gives the same bytes
    assert engine_for(level).compress_batch(items) == got


def _trailer_crc(stream):
    bits = np.unpackbits(np.frombuffer(stream, np.uint8))
    magic = np.unpackbits(np.frombuffer((0x177245385090).to_bytes(6, "big"), np.uint8))
    for pad in range(8):
        p = bits.size - pad - 80
        if p >= 32 and np.array_equal(bits[p:p + 48], magic):
            return int("".join(map(str, bits[p + 48:p + 80])), 2)
    raise AssertionError("no trailer")


def test_index_decode_and_crcs(batch_engines, engine_for):
    level = 9
    e = batch_engines(level)
    items = item_mix(level)[:14]
    offs = np.zeros(len(items) + 1, np.uint64)
    offs[1:] = np.cumsum([len(x) for x in items])
    rc, dst, out_offs, crcs = e.compress_batch_raw(np.frombuffer(b"".join(items), np.uint8), offs)
    assert rc == 0
    whole = dst[:int(out_offs[-1])].tobytes()
    assert bz2.decompress(whole) == b"".join(items)                    # stdlib: a multi-stream decoder
    rest, out = whole, b""
    while rest:
        r, part, left = binding.decompress_stream(rest)
        assert r == binding.BZ_STREAM_END
        out += part
        rest = rest[len(rest) - left:]
    assert out == b"".join(items)
    single = engine_for(level)
    for k, x in enumerate(items):
        s = whole[int(out_offs[k]):int(out_offs[k + 1])]
        r, part = binding.decompress(s, len(x) + 16)
        assert r == binding.BZ_OK and part == x
        assert int(crcs[k]) == _trailer_crc(s)
        single.compress(x)
        assert int(crcs[k]) == single.stats.combined_crc


def test_device_path(batch_engines, lib):
    torch = pytest.importorskip("torch")
    level = 5
    e = batch_engines(level)
    items = item_mix(level)
    src = np.frombuffer(b"".join(items), np.uint8)
    offs = np.zeros(len(items) + 1, np.uint64)
    offs[1:] = np.cumsum([len(x) for x in items])
    rc, hdst, houts, hcrcs = e.compress_batch_raw(src, offs)
    assert rc == 0
    total = int(houts[-1])
    d_src = torch.from_numpy(src.copy()).cuda()
    d_dst = torch.full((total + 4096,), 0xA5, dtype=torch.uint8, device="cuda")
    crcs = np.zeros(len(items), np.uint32)
    outs = e.compress_batch_device(d_src.data_ptr(), offs, d_dst.data_ptr() + 1, total + 100, stream_crcs=crcs)
    assert np.array_equal(outs, houts) and np.array_equal(crcs, hcrcs)
    got = d_dst.cpu().numpy()
    assert got[1:1 + total].tobytes() == hdst[:total].tobytes()
    assert (got[0] == 0xA5) and (got[1 + total:] == 0xA5).all()
    # one byte short: EOUTFULL, and nothing past dst_cap is written
    d_dst.fill_(0xA5)
    out_offs = np.zeros(len(items) + 1, np.uint64)
    u64p = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
    st = binding.Stats()
    f = lib.bz2b200_compress_batch_device
    rc = f(e.h, d_src.data_ptr(), u64p(offs), len(items), d_dst.data_ptr(), total - 1, u64p(out_offs), None, 0, C.byref(st))
    assert rc == EOUTFULL
    torch.cuda.synchronize()
    assert (d_dst.cpu().numpy()[total - 1:] == 0xA5).all()
    bad = offs.copy()
    bad[3] = bad[4] + 1                                                 # offsets that decrease
    assert f(e.h, d_src.data_ptr(), u64p(bad), len(items), d_dst.data_ptr(), total, u64p(out_offs), None, 0, C.byref(st)) == EPARAM
    nz = offs.copy()
    nz[0] = 1
    assert f(e.h, d_src.data_ptr(), u64p(nz), len(items), d_dst.data_ptr(), total, u64p(out_offs), None, 0, C.byref(st)) == EPARAM
    assert f(e.h, d_src.data_ptr(), u64p(offs), len(items), d_dst.data_ptr(), total, u64p(out_offs), None, NO_HEADER,
             C.byref(st)) == EPARAM
    # n_items = 0 writes nothing
    assert f(e.h, d_src.data_ptr(), u64p(offs), 0, d_dst.data_ptr(), 0, u64p(out_offs), None, 0, C.byref(st)) == 0
    assert int(out_offs[0]) == 0


def test_item_aware_stage1_directly(batch_engines):
    """One batch window: X, P, crc and bitoff are the per-item single-call tables, shifted by the item's place."""
    level = 1
    e = batch_engines(level)
    e.lib.bz2b200_debug_keep(e.h, 1)
    items = [S.gen_text(250_000, seed=1).tobytes(), b"", b"aaaa" + b"b" * 300, S.gen_random(130_000, seed=2).tobytes(),
             b"x", S.gen_runs(220_000, seed=3).tobytes()]
    got = e.compress_batch(items)
    assert e.stats.n_windows == 1
    nb = e.stats.n_blocks
    X = e.fetch("X", np.uint32, nb + 1)
    P = e.fetch("P", np.uint32, nb + 1)
    crc = e.fetch("crc", np.uint32, nb)
    bitoff = e.fetch("bitoff", np.uint64, nb + 1)
    single = B.Engine(level=level, window_bytes=1 << 20)
    single.lib.bz2b200_debug_keep(single.h, 1)
    b0, ebase, pbase, obase = 0, 0, 0, 0
    for x, s in zip(items, got):
        if x:
            assert single.compress(x) == s
            k = single.stats.n_blocks
            sX = single.fetch("X", np.uint32, k + 1)
            sP = single.fetch("P", np.uint32, k + 1)
            assert np.array_equal(X[b0:b0 + k + 1], sX + ebase)
            assert np.array_equal(P[b0:b0 + k + 1], sP + pbase)
            assert np.array_equal(crc[b0:b0 + k], single.fetch("crc", np.uint32, k))
            assert np.array_equal(bitoff[b0:b0 + k], single.fetch("bitoff", np.uint64, k + 1)[:k] + 8 * obase)
            b0 += k
            ebase += int(sX[-1])
        pbase += len(x)
        obase += len(s)
    assert b0 == nb
    single.close()


TRACE_SCRIPT = r"""
import sys, ctypes as C
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import numpy as np, support as S, bzip2_b200 as B
items = [S.gen_text(150_000, seed=1).tobytes(), b"", b"a" * 1000, S.gen_random(120_000, seed=2).tobytes(), b"q"]
e = B.Engine(level=1, max_items=64)
e.lib.bz2b200_engine_set_verbosity(e.h, 3)
if sys.argv[2] == "batch":
    out = e.compress_batch(items)
else:
    out = [e.compress(x) for x in items]
sys.stdout.write(str(sum(map(len, out))))
"""


def test_trace_text_equals_single_calls():
    def run(mode):
        r = subprocess.run([sys.executable, "-c", TRACE_SCRIPT, ROOT, mode], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        return r.stdout, r.stderr
    b, s = run("batch"), run("single")
    assert b == s
    assert s[1].count("final combined CRC") == 5 and "block 1:" in s[1]


def _cli_tree(d, n_small=300):
    rng = np.random.default_rng(21)
    d.mkdir()
    names = []
    gens = (S.gen_text, S.gen_random, S.gen_runs)
    for k in range(n_small):
        n = int(rng.integers(0, 20_000))
        (d / f"f{k:03d}.txt").write_bytes(gens[k % 3](n, seed=k + 1).tobytes() if n else b"")
        names.append(f"f{k:03d}.txt")
    (d / "large.txt").write_bytes(S.gen_text(9 << 20, seed=5).tobytes())          # above the CLI's small-file limit
    (d / "empty.txt").write_bytes(b"")
    (d / "old.bz2").write_bytes(bz2.compress(b"already compressed"))
    return names[:150] + ["large.txt", "empty.txt", "missing.txt", "old.bz2"] + names[150:]


def test_cli_batches_small_files(tmp_path):
    cli = os.path.join(ROOT, "bzip2_b200", "bzip2-b200")
    runs = {}
    for mode in ("batch", "stream"):
        d = tmp_path / mode
        args = _cli_tree(d)
        env = dict(os.environ)
        if mode == "stream":
            env["BZ2_B200_CLI_STREAM"] = "1"
        c = subprocess.run([cli, "-1", "-c", "-v"] + args, cwd=d, env=env, capture_output=True, timeout=900)
        r = subprocess.run([cli, "-1", "-v"] + args, cwd=d, env=env, capture_output=True, timeout=900)
        outs = {p.name: p.read_bytes() for p in sorted(d.iterdir())}
        runs[mode] = (c, r, outs, args)
    (cb, rb, ob, args), (cs, rs, os_, _) = runs["batch"], runs["stream"]
    assert rb.returncode == rs.returncode == 1 and cb.returncode == cs.returncode == 1
    assert ob == os_                                                # same outputs, same inputs removed
    assert rb.stderr == rs.stderr and cb.stderr == cs.stderr        # same lines in argument order
    assert cb.stdout == cs.stdout
    done = [a for a in args if a not in ("missing.txt", "old.bz2")]
    assert cb.stdout == b"".join(ob[a + ".bz2"] for a in done)       # -c: the per-file streams back to back
    assert all(a not in ob for a in done) and "old.bz2" in ob
    lines = rb.stderr.decode().splitlines()
    order = [next(i for i, ln in enumerate(lines) if f" {a}" in ln or f"file {a}" in ln) for a in args]
    assert order == sorted(order)
