"""GPU: byte parity at the scale the bench runs, the literal drop-in CLI, and the reference decoder round trip.

* window scale (VERDICT r1 weak #6): 120-200 MB inputs -- two full windows of ~111 blocks at -9, ~1200 blocks at -1 --
  compared byte for byte with the unmodified reference (oracle/_ref, shipped with the snapshot) and, where that is
  absent, through sha256 goldens minted from it (tests/golden/large_streams.json, make_golden.py --large);
* drop-in CLI (SURVEY 8b, INTEGRATION.md 1): the reference's UNMODIFIED bzip2.c, compiled against include/bzlib.h and
  linked with libbz2_b200.so (oracle/_ref/bzip2_ref_on_b200, built by oracle/Makefile in the authoring container),
  against the reference's own binary on the same files -- its 5000-byte BZ2_bzWrite trickle, bzip2.c:350-358;
* C5 (SURVEY 8d): every level -1..-9, output equal to the reference's stream and decoded back to the input.
"""
import bz2
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import support as S
import bzip2_b200 as B

pytestmark = pytest.mark.gpu
G = S.GOLDEN
REF_DIR = os.path.join(S.ORACLE_DIR, "_ref")
REF_CLI = os.path.join(REF_DIR, "bzip2_ref")
RELINKED = os.path.join(REF_DIR, "bzip2_ref_on_b200")


def _large(name):
    return {"text_200M_L9": lambda: S.gen_text(200_000_000),
            "c4_200M_L9": lambda: S.gen_c4(200_000_000, seg=64 << 20),
            "text_120M_L1": lambda: S.gen_text(120_000_000, seed=7)}[name]()


@pytest.mark.parametrize("name", ["text_200M_L9", "c4_200M_L9", "text_120M_L1"])
def test_window_scale_byte_parity(engine_for, name):
    gold = json.load(open(os.path.join(G, "large_streams.json")))[name]
    d = _large(name)
    eng = engine_for(gold["level"])
    out = eng.compress(d)
    assert eng.stats.n_windows >= 2
    assert len(out) == gold["out_len"]
    assert hashlib.sha256(out).hexdigest() == gold["sha256"]
    if S.have_ref() and name != "text_120M_L1":          # the reference itself, byte for byte, on the same box
        assert out == S.ref_compress(d, gold["level"])


def test_window_scale_sharded_four_ranks(engine_for):
    """Four ranks, one stream: the sharded result equals the golden of the reference's single stream."""
    from bzip2_b200 import sharding as sh
    gold = json.load(open(os.path.join(G, "large_streams.json")))["c4_200M_L9"]
    data = _large("c4_200M_L9")
    world = 4
    shards = [np.ascontiguousarray(data[r * data.size // world:(r + 1) * data.size // world]) for r in range(world)]
    halos = sh.make_halos(shards, 64 << 20)
    backends = {}

    def make(r):
        backends[r] = sh.GpuBackend(9, 0)
        return backends[r]
    out, infos = sh.run_threads(world, make, shards, halos, 9)
    for b in backends.values():
        b.eng.close()
    assert hashlib.sha256(bytes(out)).hexdigest() == gold["sha256"]


@pytest.mark.skipif(not (os.path.exists(REF_CLI) and os.path.exists(RELINKED)), reason="oracle/_ref binaries not shipped")
@pytest.mark.parametrize("level", [1, 9])
def test_reference_cli_relinked(tmp_path, level):
    data = np.concatenate([S.gen_mixed(4_300_000, seg=1 << 19), S.gen_tile(700_000, b"ab\ncd\n."), np.zeros(300_000, np.uint8)]).tobytes()
    src = tmp_path / "input.dat"
    src.write_bytes(data)
    ref = subprocess.run([REF_CLI, f"-{level}", "-c", str(src)], capture_output=True)
    assert ref.returncode == 0, ref.stderr
    ours = subprocess.run([RELINKED, f"-{level}", "-c", str(src)], capture_output=True)
    assert ours.returncode == 0, ours.stderr
    assert ours.stdout == ref.stdout
    # file mode: same name handling, same bytes, input kept with -k
    r = subprocess.run([RELINKED, f"-{level}", "-k", str(src)], capture_output=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "input.dat.bz2").read_bytes() == ref.stdout and src.exists()
    # and the reference decodes it
    dec = subprocess.run([REF_CLI, "-dc", str(tmp_path / "input.dat.bz2")], capture_output=True)
    assert dec.returncode == 0 and dec.stdout == data
    # -vv: the library's per-block trace (compress.c:831-834, :877-878) is the reference's, line for line
    tr_ref = subprocess.run([REF_CLI, f"-{level}", "-vv", "-c", str(src)], capture_output=True)
    tr_ours = subprocess.run([RELINKED, f"-{level}", "-vv", "-c", str(src)], capture_output=True)
    pick = lambda err: [ln for ln in err.decode().splitlines() if ln.startswith("    block ") or "final combined CRC" in ln]
    assert tr_ours.stdout == ref.stdout
    assert len(pick(tr_ref.stderr)) >= 3 and pick(tr_ours.stderr) == pick(tr_ref.stderr)


def test_level_sweep_reference_decoder(engine_for):
    """C5 at test size: -1..-9 on 30 MB of text, each output the reference's own stream (tests/golden/ref_checks.json,
    make_ref_checks.py) and decoded back to the input."""
    from golden.make_ref_checks import level_sweep_input
    gold = json.load(open(os.path.join(G, "ref_checks.json")))["level_sweep"]
    d = level_sweep_input()
    want = hashlib.sha256(d.tobytes()).hexdigest()
    for level in range(1, 10):
        out = engine_for(level).compress(d)
        assert len(out) == gold[str(level)]["out_len"] and hashlib.sha256(out).hexdigest() == gold[str(level)]["sha256"], level
        assert hashlib.sha256(bz2.decompress(out)).hexdigest() == want, level


def test_own_cli_whole_file_paths(tmp_path):
    """bzip2-b200 reads regular files whole: small files share one input-sized engine, a large file is spread over the
    engines of BZ2_B200_DEVICES; the bytes are those of the streaming loop (every input byte in BZ_RUN mode)."""
    cli = os.path.join(os.path.dirname(B.LIB_PATH), "bzip2-b200")
    ndev = max(1, B.load().bz2b200_device_count())
    files = {"a.txt": S.gen_text(70_000, seed=1), "b.bin": S.gen_random(2_500_000, seed=9), "c.rec": S.gen_tile(420_000, b"ab\ncd\n."),
             "empty": np.zeros(0, np.uint8), "big.dat": S.gen_mixed(130_000_000, seg=1 << 22),
             "edge.dat": (np.arange(99_981 + 1, dtype=np.uint32) % 251).astype(np.uint8)}
    for name, d in files.items():
        (tmp_path / name).write_bytes(d.tobytes())
    env = dict(os.environ, BZ2_B200_DEVICES=",".join(str(i % ndev) for i in range(3)), BZ2_B200_WINDOW_MB="32")
    r = subprocess.run([cli, "-1", "-k"] + [str(tmp_path / n) for n in files], capture_output=True, env=env)
    assert r.returncode == 0, r.stderr
    for name, d in files.items():
        got = (tmp_path / (name + ".bz2")).read_bytes()
        if d.size <= 3_000_000:
            assert got == S.orc_compress(d, 1, tail_merge=0), name
        else:
            streamed = subprocess.run([cli, "-1", "-c", str(tmp_path / name)], capture_output=True,
                                      env=dict(os.environ, BZ2_B200_CLI_STREAM="1"))
            assert streamed.returncode == 0 and streamed.stdout == got, name
            dec = subprocess.run([REF_CLI, "-dc", str(tmp_path / (name + ".bz2"))], capture_output=True) if os.path.exists(REF_CLI) else None
            if dec is not None:
                assert dec.returncode == 0 and hashlib.sha256(dec.stdout).digest() == hashlib.sha256(d.tobytes()).digest()
