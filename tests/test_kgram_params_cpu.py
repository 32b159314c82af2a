"""CPU: the parameters stage 2 derives from a block's alphabet (k_codemap) and the bin budget (engine_new), checked
for every level, every accepted BZ2_B200_HIST_LOG2 and every alphabet size against the widths of the words they are
packed into.

The count pass of the k-gram sort (k_kgram<KG_HISTOFF, true>) aggregates a tile's k-grams in a shared-memory table
whose slot word is key + 1 above a 13-bit count, so the aggregated path is only sound while key + 1 < 2^19.  Which
blocks take it is read from the kernel's own condition in csrc/stage2_bwt.cu, so this test fails if that guard loses
its bin limit."""
import os
import re

import support as S

CSRC = os.path.join(S.ROOT, "bzip2_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _const(src, name):
    m = re.search(r"constexpr\s+\w+\s+" + name + r"\s*=\s*([^;]+);", src)
    assert m, name
    return int(eval(m.group(1).replace("u", "")))          # "1u << 19" -> 1 << 19


def _agg_rule():
    """The condition under which k_kgram's count pass aggregates per tile, as a function of (ninuse, nbins)."""
    src = _src("stage2_bwt.cu")
    m = re.search(r"if \(AGG && ([^{]*)\)\s*\{", src)
    assert m, "aggregated count path not found in k_kgram"
    cond = m.group(1)
    for name in re.findall(r"\bKG_[A-Z_]+\b", cond):
        cond = cond.replace(name, str(_const(src, name)))
    cond = cond.replace("p.kg_agg_alpha", str(_const(src, "KG_AGG_MAX_ALPHA")))
    cond = re.sub(r"(\d+)u\b", r"\1", cond).replace("&&", " and ").replace("p.nbins[b]", "nbins").replace("base", "ninuse")
    return eval("lambda ninuse, nbins: " + cond)


def _tag_bits():
    src = _src("stage2_bwt.cu")
    m = re.search(r"tagw = \(key \+ 1u\) << (\d+);", src)
    assert m
    return 32 - int(m.group(1))


def _accepted_hist_log2():
    m = re.search(r"if \(v >= (\d+) && v <= (\d+)\) hist_log2", _src("engine.cu"))
    assert m
    return range(int(m.group(1)), int(m.group(2)) + 1)


def _cases():
    maxk = _const(_src("stage2_bwt.cu"), "KG_MAXK")
    for level in range(1, 10):
        for hl in _accepted_hist_log2():
            stride = S.hist_stride(level, hl)
            for a in range(1, 257):
                yield level, hl, stride, a, S.codemap(a, stride, maxk)


def test_hist_stride_model():
    assert [S.hist_stride(lv) for lv in (1, 3, 9)] == [1 << 16, 1 << 17, 1 << 18]      # default budget per level
    assert list(_accepted_hist_log2()) == list(range(16, 23))
    for level in range(1, 10):
        for hl in _accepted_hist_log2():
            s = S.hist_stride(level, hl)
            assert s & (s - 1) == 0 and (1 << 16) <= s <= (1 << 22)      # the tie replay keeps 65536 ints there


def test_codemap_fits_its_words():
    src = _src("stage2_bwt.cu")
    ms_lbits = _const(src, "MS_LBITS")
    lg_lbits = 13                                          # k_refine_radix<1024>: CAP 8192 > 4096 -> 13 local-index bits
    agg = _agg_rule()
    tag_bits = _tag_bits()
    n_agg = n_direct = 0
    for level, hl, stride, a, (k, nbins, bits, m) in _cases():
        where = (level, hl, a, k, nbins)
        assert nbins <= stride, where
        assert nbins == max(a, 1) ** k, where
        assert (1 << bits) >= a, where
        assert m * bits <= 51, where
        assert m * bits + lg_lbits <= 64 and m * bits + ms_lbits <= 64, where   # text key over the local index
        if agg(a, nbins):
            n_agg += 1
            assert (nbins - 1) + 1 < (1 << tag_bits), where                     # the largest key's tag fits
        else:
            n_direct += 1
    assert n_agg and n_direct


def test_rank_and_position_fields():
    """Rank keys of the doubling rounds sit over a 12-bit local index in u32 words (medium sort, radix CTAs up to
    4096); the small-class worklist packs the flat position into 27 bits."""
    src = _src("stage2_bwt.cu")
    ms_lbits = _const(src, "MS_LBITS")
    nmax = 100000 * 9 - 19
    assert nmax - 1 < 1 << (32 - ms_lbits)
    win = 100 << 20                                        # engine_new clamps the window to 100 MiB
    enc_cap = win + win // 4 + 4096
    assert enc_cap < 1 << 27


def test_old_guard_would_overflow():
    """Without the bin limit, alphabets of 2-7 symbols at HIST_LOG2 >= 19 get keys whose tag does not fit."""
    over = set()
    for level, hl, stride, a, (k, nbins, bits, m) in _cases():
        if a <= 128 and nbins > (1 << 19) - 1:
            over.add((hl, a))
    assert (19, 2) in over and (20, 3) in over and (22, 7) in over
    assert not any(hl <= 18 for hl, _ in over)
