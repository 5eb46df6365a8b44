"""T1: CUDA MTF+RLE2 (bz2b200_mtf_rle2) vs the oracle's rle2_mtf_encode restatement (rle2_mtf.rs:23-177)."""
import numpy as np
import pytest

import bwtcraft
from bzip2_rust_b200 import corpus
from inputs import small_cases

pytestmark = pytest.mark.gpu


def _check(engine, ref, bwt, name=""):
    sym, freq, smap = engine.rle2_mtf_encode(bwt)
    rs, rf, rm = ref.rle2_mtf_encode(bwt)
    assert len(sym) == len(rs), "%s: m differs %d vs %d" % (name, len(sym), len(rs))
    assert np.array_equal(sym, rs), "%s: symbols differ at %s" % (name, np.nonzero(sym != rs)[0][:5])
    assert np.array_equal(freq, rf), name
    assert list(smap) == list(rm), name


def test_small_cases(engine, ref):
    for name, data in small_cases():
        _, bwt, _ = ref.bwt_encode(data, ref.SPEC_FAST)
        _check(engine, ref, bwt, name)
        _check(engine, ref, data, name + "/raw")      # any byte string is a valid input of this stage


def test_chunk_boundaries(engine, ref):
    # zero runs and first occurrences straddling the 1024-byte chunk edges
    rng = np.random.default_rng(3)
    for n in (1023, 1024, 1025, 2047, 2048, 2049, 4096, 5000):
        _check(engine, ref, bytes(n), "zeros%d" % n)
        _check(engine, ref, b"\x07" * n, "sevens%d" % n)
        a = np.zeros(n, dtype=np.uint8)
        a[rng.integers(0, n, 5)] = rng.integers(1, 255, 5)
        _check(engine, ref, a.tobytes(), "sparse%d" % n)
        a = np.repeat(rng.integers(0, 256, n // 100 + 1, dtype=np.uint8), 100)[:n]
        _check(engine, ref, a.tobytes(), "runs100_%d" % n)


def test_all_256_symbols(engine, ref):
    rng = np.random.default_rng(4)
    a = rng.integers(0, 256, 100_000, dtype=np.uint8)
    _check(engine, ref, a.tobytes(), "rand256")       # eob = 257: freq[256] truncation case of SURVEY B.3
    a = np.concatenate([np.arange(256, dtype=np.uint8)[::-1], np.zeros(5000, dtype=np.uint8), np.arange(256, dtype=np.uint8)])
    _check(engine, ref, a.tobytes(), "desc_then_zero")


def _used_value_blocks():
    """[(name, block)] for the four register layouts of k_mtf_emit3, chosen by the count of used byte values (at most
    32, 64 or 128, or more): 1, 2, 32, 33, 64, 65, 128, 129, 255 and 256 values, placed lowest, spread out (0 and 255
    included) and highest.  A block spans four CH-byte chunks, has a run across the first chunk edge and one value
    that is used in the last chunk only; blocks of exactly CH and CH + 1 bytes end the list."""
    ch = bwtcraft.GEO["CH"]
    rng = np.random.default_rng(6)
    out = []

    def fill(vals, n):
        a = np.repeat(rng.choice(vals, n), rng.integers(1, 4, n))[:n]      # short runs of random values
        a[:len(vals)] = rng.permutation(vals)                              # every value is used
        return a

    for count in (1, 2, 32, 33, 64, 65, 128, 129, 255, 256):
        spread = [127] if count == 1 else [i * 255 // (count - 1) for i in range(count)]
        for place, vals in (("low", list(range(count))), ("spread", spread), ("high", list(range(256 - count, 256)))):
            vals = np.array(vals, dtype=np.uint8)
            late = vals[len(vals) // 2] if count > 1 else None
            early = vals[vals != late] if count > 1 else vals
            n = 3 * ch + ch // 2
            a = fill(early, n)
            a[ch - 5:ch + 7] = early[-1]                                       # a run across the first chunk edge
            if late is not None:
                a[n - ch // 4::7] = late                                       # first used in the last chunk
            out.append(("used%d_%s" % (count, place), a.tobytes()))
        for n in (ch, ch + 1):
            vals = np.array(spread, dtype=np.uint8)
            out.append(("used%d_n%d" % (count, n), fill(vals, n).tobytes()))
    return out


def test_used_value_counts_at_the_emit_layout_edges(engine, ref):
    blocks = _used_value_blocks()
    for name, blk in blocks:
        assert len(set(blk)) == int(name[4:].split("_")[0]), name
        _check(engine, ref, blk, name)
    crcs = [ref.crc(b) for _, b in blocks]
    got = engine.compress_blocks([b for _, b in blocks], crcs)      # all four layouts in one launch
    for (name, blk), c, (gb, gpad) in zip(blocks, crcs, got):
        rb, rpad, _ = ref.compress_block(blk, c, ref.SPEC_FAST)
        assert (gb, gpad) == (rb, rpad), name


def test_full_size_block(engine, ref):
    blk = corpus.text(899_981, 41).tobytes()
    _, bwt, _ = ref.bwt_encode(blk, ref.SPEC_FAST)
    _check(engine, ref, bwt, "text900k")
    blk = corpus.repetitive(899_000, 42).tobytes()
    _, bwt, _ = ref.bwt_encode(blk, ref.SPEC_FAST)
    _check(engine, ref, bwt, "rep900k")
