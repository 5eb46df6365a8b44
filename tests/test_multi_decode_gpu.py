"""bz2b200_decompress_stream_multi: `decompress` (decompress.rs:38) over several ranks of ONE process.  The input is cut
into byte windows; each rank finds the magics of its windows, receives the block chain from the window before, and copies
its bytes straight to their place in the output.  On a single-GPU box the ranks share the GPU (device ids repeat).
BZ2B200_MULTI_DEC_WINDOW makes windows small, so that streams of a few MB give many windows per rank and stream
boundaries can be put on window edges.  The output and the return codes must be those of the single-GPU call."""
import bz2
import ctypes as C

import numpy as np
import pytest
import torch

import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus

pytestmark = pytest.mark.gpu


def _devices(world):
    n = torch.cuda.device_count()
    return [r % n for r in range(world)]


def _rc(fn, *a):
    try:
        fn(*a)
    except bz.Bz2B200Error as e:
        return e.rc
    return bz.OK


def _raw(m, s, cap):
    """(rc, *out_len) of one call with an output buffer of `cap` bytes."""
    a = np.frombuffer(s, dtype=np.uint8)
    out = np.empty(max(cap, 1), dtype=np.uint8)
    ln = C.c_size_t()
    rc = m._L.bz2b200_decompress_stream_multi(m._h, a.ctypes.data, a.size, out.ctypes.data, cap, C.byref(ln))
    return rc, ln.value, out


@pytest.fixture(scope="module")
def data():
    return np.concatenate([corpus.text(2_000_000, 51), corpus.repetitive(1_000_000, 52),
                           corpus.random_bytes(1_000_000, 53)]).tobytes()


@pytest.fixture(scope="module")
def streams(engine, data):
    return [engine.compress(data, 1), engine.compress(data, 9), bz2.compress(data, 9)]


@pytest.mark.parametrize("world", [2, 3, 8])
def test_worlds_decode_the_input(engine, data, streams, world, monkeypatch):
    monkeypatch.setenv("BZ2B200_MULTI_DEC_WINDOW", "100000")             # 8 to 40 windows: several per rank
    big = corpus.text(world * (8 << 20) + 4096, 54)                      # large enough for the multi-rank compressor
    m = bz.MultiEngine(_devices(world))
    try:
        for s in streams:
            assert m.decompress(s) == data
            assert engine.decompress(s) == data
            st = m.stats()
            assert st["h2d_bytes"] >= len(s) and st["d2h_bytes"] == len(data)
        assert m.compress(big, 9) == engine.compress(big, 9)             # the compressor on the same context in between
        for s in streams:
            assert m.decompress(s, max_out=len(data)) == data
    finally:
        m.close()


def test_stream_boundaries_on_window_edges(engine):
    """Concatenated streams (own and libbz2's, mixed levels, an empty one, a later one with a larger level); the window
    size puts one window edge 0, 1, 2, 7 and 10 bytes before and after each boundary, so that footers, "BZh" headers and
    first block magics straddle edges.  A large last stream keeps every boundary in the first half of the input."""
    parts = [engine.compress(corpus.text(300_000, 61), 1), bz2.compress(corpus.repetitive(300_000, 62).tobytes(), 3),
             bz2.compress(b""), engine.compress(corpus.text(500_000, 63), 9), bz2.compress(corpus.text(300_000, 64).tobytes(), 9),
             engine.compress(corpus.random_bytes(1_500_000, 65), 9)]
    cat = b"".join(parts)
    want = bz2.decompress(cat)
    assert engine.decompress(cat) == want
    bounds = np.cumsum([len(p) for p in parts])[:-1]
    m = bz.MultiEngine(_devices(3))
    try:
        for b in bounds:
            for d in (0, 1, -1, 2, -2, 7, -7, 10, -10):
                w = int(b) + d
                assert 2 * w <= len(cat)
                with pytest.MonkeyPatch.context() as mp:
                    mp.setenv("BZ2B200_MULTI_DEC_WINDOW", str(w))
                    assert m.decompress(cat) == want, (int(b), d)
    finally:
        m.close()


def test_chance_magics(engine, data, streams, monkeypatch):
    """BZ2B200_MULTI_DEC_CHANCE adds a spurious block candidate at the first bit of every window and between any two
    candidates (inside block data: the range of the block before is cut, its walk finishes code by code); such
    candidates stay off the chain.  Also with BZ2B200_DEC_RANGE_LIMIT cutting every range."""
    monkeypatch.setenv("BZ2B200_MULTI_DEC_WINDOW", "150000")
    monkeypatch.setenv("BZ2B200_MULTI_DEC_CHANCE", "1")
    m = bz.MultiEngine(_devices(3))
    try:
        for s in streams:
            assert m.decompress(s) == data
        for limit in ("700", "100000"):
            monkeypatch.setenv("BZ2B200_DEC_RANGE_LIMIT", limit)
            assert m.decompress(streams[1]) == data, limit
    finally:
        m.close()


def test_randomised_block(engine, ref, monkeypatch):
    """A legacy randomised block (built as in test_decode_gpu.test_randomised_block), decoded on the multi path."""
    from test_decode_gpu import _rand_flips
    data = corpus.text(300_000, 33).tobytes() + b"q" * 1000 + corpus.random_bytes(5000, 34).tobytes()
    (crc, rle1, last, consumed), = list(ref.rle1_blocks(data, 9))
    r = bytearray(rle1)
    for p in _rand_flips(len(r)):
        r[p] ^= 1
    packed, pad, _ = ref.compress_block(bytes(r), crc, ref.SPEC_FAST)
    pb = bytearray(packed)
    pb[10] |= 0x80
    stream = bz.merge_streams(9, [(bytes(pb), len(pb) * 8 - pad, [crc])])
    stream = stream + engine.compress(data, 1)                           # and a second stream after it
    monkeypatch.setenv("BZ2B200_MULTI_DEC_WINDOW", "40000")
    m = bz.MultiEngine(_devices(2))
    try:
        assert m.decompress(stream) == data + data
    finally:
        m.close()


def test_single_defects_give_the_single_gpu_code(engine, monkeypatch):
    data = corpus.text(1_500_000, 71).tobytes()
    s = engine.compress(data, 9)
    mid = bytearray(s)
    mid[len(s) // 2] ^= 0x10                                             # inside a block
    foot = bytearray(s)
    foot[-2] ^= 0x01                                                     # inside the footer's combined CRC
    cases = {"block bit": bytes(mid), "footer crc": bytes(foot), "trailing garbage": s + b"garbage after the stream",
             "truncated": s[:len(s) * 2 // 3], "not bzip2": b"not a bzip2 stream at all " * 40_000, "short": b"BZh91AY&SY"}
    monkeypatch.setenv("BZ2B200_MULTI_DEC_WINDOW", "65536")
    m = bz.MultiEngine(_devices(3))
    try:
        for name, bad in cases.items():
            want = _rc(engine.decompress, bad, 1 << 24)
            assert want != bz.OK, name
            assert _rc(m.decompress, bad, 1 << 24) == want, name
            assert m.decompress(s) == data, name                         # the context still works
        assert _rc(engine.decompress, cases["footer crc"], 1 << 24) == bz.E_CRC
        assert _rc(engine.decompress, cases["trailing garbage"], 1 << 24) == bz.E_FORMAT
    finally:
        m.close()


def test_output_capacity(engine, monkeypatch):
    rep = corpus.repetitive(2_000_000, 81).tobytes()                     # compresses far more than 8:1
    s = engine.compress(rep, 9) + bz2.compress(corpus.text(600_000, 82).tobytes(), 9)
    want = engine.decompress(s)
    monkeypatch.setenv("BZ2B200_MULTI_DEC_WINDOW", "20000")
    m = bz.MultiEngine(_devices(2))
    try:
        rc, ln, _ = _raw(m, s, len(want) - 1)
        assert rc == bz.E_CAP and ln == len(want)
        rc, ln, out = _raw(m, s, ln)
        assert rc == bz.OK and out[:ln].tobytes() == want
        assert m.decompress(s) == want                                   # first guess too small: one retry
    finally:
        m.close()


def test_small_inputs_take_the_single_gpu_path(engine):
    m = bz.MultiEngine(_devices(4))
    try:
        for d in (b"", b"x", corpus.text(1_000_000, 91).tobytes()):
            for s in (engine.compress(d, 9), bz2.compress(d, 1)):
                assert m.decompress(s) == engine.decompress(s) == d
                if d:
                    rc, ln, _ = _raw(m, s, len(d) - 1)
                    assert rc == bz.E_CAP and ln == len(d)
    finally:
        m.close()


def test_large_stream_world4(engine):
    """More than 1 GiB of output, default windows (24 MiB of input each)."""
    data = np.tile(corpus.text(64 << 20, 101), 17)
    s = engine.compress(data, 9)
    m = bz.MultiEngine(_devices(4))
    try:
        out = np.empty(data.size, dtype=np.uint8)
        a = np.frombuffer(s, dtype=np.uint8)
        assert m.decompress_into(a.ctypes.data, a.size, out.ctypes.data, out.size) == data.size
        assert np.array_equal(out, data)
    finally:
        m.close()


def test_all_visible_gpus(engine):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    data = corpus.text(n * 30_000_000, 2)
    s = engine.compress(data, 9)
    m = bz.MultiEngine(list(range(n)))
    try:
        assert m.decompress(s, max_out=data.size) == data.tobytes()
    finally:
        m.close()
