"""Decoder conformance: the hand-built streams of tests/bz2craft.py (code lengths up to 20, any selector count, any BWT
string, RLE1 run tails, per-stream block sizes, ...) through every decode path, against libbz2.

Each case goes through the one-call decoder (bz2b200_decompress_stream), the streaming decoder with a sink and in test
mode with small windows (bz2b200_dstream_*), and the multi-context decoder on two ranks with small windows
(bz2b200_decompress_stream_multi).  The dstream and multi paths get the case behind a filler stream of a few MB, so that
it is decoded in a later window.  Where libbz2 accepts a case every path returns its bytes; where libbz2 rejects it every
path returns the same code, and the contexts then still decode a good stream."""
import io

import numpy as np
import pytest
import torch

import bz2craft as bc
import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus

pytestmark = pytest.mark.gpu
CODES = {"E_FORMAT": bz.E_FORMAT, "E_CRC": bz.E_CRC}


def _result(fn):
    try:
        return bz.OK, fn()
    except bz.Bz2B200Error as e:
        return e.rc, None


def _dstream(engine, s, sink):
    out = io.BytesIO() if sink else None
    d = bz.DStream(engine, out)
    try:
        d.write(s)
    finally:
        d.close()
    return out.getvalue() if sink else d.total_out


@pytest.fixture(scope="module")
def engine():
    """This module's own context, closed at its end.  The dstream paths give a context about 225 MB of page-locked
    staging and output buffers, which it keeps while it lives.  The session's context must not carry them into later
    modules, where they would add to the process's peak resident set."""
    eng = bz.Engine()
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def filler(engine):
    """A stream of 5 MB that hardly compresses: more than the dstream's 4 MiB look-ahead, several multi windows."""
    data = corpus.random_bytes(5_000_000, 41).tobytes()
    return engine.compress(data, 9), data


@pytest.fixture(scope="module")
def multi():
    n = torch.cuda.device_count()
    m = bz.MultiEngine([0, 1 % n])
    yield m
    m.close()


def _paths(engine, multi, filler, s, monkeypatch):
    """{path: (rc, bytes decoded -- for test mode their count)}; the windowed paths decode filler + s."""
    fs = filler[0] + s
    res = {"decompress": _result(lambda: engine.decompress(s))}
    monkeypatch.delenv("BZ2B200_DSTREAM_WINDOW", raising=False)
    res["dstream"] = _result(lambda: _dstream(engine, fs, True))
    monkeypatch.setenv("BZ2B200_DSTREAM_WINDOW", str(1 << 20))
    res["dstream test mode"] = _result(lambda: _dstream(engine, fs, False))
    monkeypatch.setenv("BZ2B200_MULTI_DEC_WINDOW", str(1 << 20))
    res["multi"] = _result(lambda: multi.decompress(fs))
    return res


@pytest.mark.parametrize("name", list(bc.CASES))
def test_case_on_every_decode_path(engine, multi, filler, name, monkeypatch):
    data, want, code = bc.CASES[name]()
    lib = bc.libbz2(data)
    res = _paths(engine, multi, filler, data, monkeypatch)
    if code == "ok":
        assert lib == want is not None
        pre = filler[1]
        expect = {"decompress": want, "dstream": pre + want, "dstream test mode": len(pre) + len(want), "multi": pre + want}
        for path, (rc, got) in res.items():
            assert rc == bz.OK, (path, rc)
            assert got == expect[path], path
        return
    assert lib is None
    assert {path: rc for path, (rc, _) in res.items()} == dict.fromkeys(res, CODES[code])
    good, out = filler                                                   # the contexts are fine after the error
    assert engine.decompress(good) == out
    assert multi.decompress(good) == out
    assert _dstream(engine, good, False) == len(out)


def _keys(n, rng):
    return sorted({k for k in (0, 31, 32, 2048, n - 1, int(rng.integers(0, n))) if k < n})


def test_bwt_decode_every_key_of_small_blocks(engine):
    """bz2b200_bwt_decode against libbz2's rule (n steps from the origin pointer, P = stable argsort of L), n = 1..70,
    every key: the true BWT of a text (one LF cycle, every key a rotation) and a random string (several cycles)."""
    rng = np.random.default_rng(17)
    for n in range(1, 71):
        text = bytes(rng.integers(97, 100, n, dtype=np.uint8))
        for L in (bc.bwt(text)[0], bytes(rng.integers(97, 100, n, dtype=np.uint8))):
            for key in range(n):
                assert engine.bwt_decode(key, L) == bc.ibwt(L, key), (n, L, key)


@pytest.mark.parametrize("n", [2047, 2048, 2049, 65535, 65537, 900000])
def test_bwt_decode_large_blocks(engine, n):
    """Around the 2048-row coarse splitters and at the largest block: keys on regular and coarse splitter rows, the last
    row and a random one, for a true BWT (one cycle: every key gives a rotation) and for random strings (a few cycles;
    sorted: n cycles of length 1)."""
    rng = np.random.default_rng(n)
    _, single = engine.bwt_encode(corpus.text(n, n % 1000).tobytes())
    rand = rng.integers(0, 256, n, dtype=np.uint8)
    for L in (bytes(single), rand.tobytes(), np.sort(rand).tobytes()):
        for key in _keys(n, rng):
            assert engine.bwt_decode(key, L) == bc.ibwt(L, key), (n, key)
