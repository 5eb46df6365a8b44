"""bz2b200_dstream_*: `decompress` (decompress.rs:38) as a pipeline -- .bz2 input in pieces, checked output through a sink
on a library thread.  Whatever the piece sizes and the window size (BZ2B200_DSTREAM_WINDOW), the sink receives the bytes
of the whole-buffer call, and an input with a single defect gives that call's return code; test mode (no sink) runs
every check without downloading.  Windows decode up to 4 MiB before their end (LOOK), so small windows put the decode
edge where a test wants it."""
import bz2
import ctypes as C
import io
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOOK = 4 << 20


def _pieces(rng, n_small=20, n=30, hi=3_000_000):
    return [1] * n_small + [int(x) for x in rng.integers(1, hi, n)]


def _run(engine, s, pieces=(), test=False):
    """(rc, total_in, total_out, bytes the sink received or None) of one dstream over `s`."""
    out = None if test else io.BytesIO()
    rc = bz.OK
    d = None
    try:
        with bz.DStream(engine, out) as d:
            pos = 0
            for p in pieces:
                if pos >= len(s):
                    break
                d.write(s[pos:pos + p])
                pos += p
            if pos < len(s):
                d.write(s[pos:])
    except bz.Bz2B200Error as e:
        rc = e.rc
    return rc, d.total_in, d.total_out, (None if test else out.getvalue())


def _rc(fn, *a):
    try:
        fn(*a)
    except bz.Bz2B200Error as e:
        return e.rc
    return bz.OK


@pytest.fixture(scope="module")
def data():
    return np.concatenate([corpus.text(9_000_000, 61), corpus.repetitive(9_000_000, 62), corpus.random_bytes(3_000_000, 63),
                           corpus.text(2_500_000, 64)]).tobytes()


@pytest.fixture(scope="module")
def streams(engine, data):
    s9 = engine.compress(data, 9)
    small = corpus.text(700_000, 65).tobytes()
    cat = engine.compress(small, 1) + bz2.compress(b"") + s9 + engine.compress(b"", 5)
    return {"engine -1": engine.compress(data, 1), "engine -9": s9, "bz2 -9": bz2.compress(data, 9), "concatenation": cat}


def test_pieces_and_windows_give_the_whole_buffer_output(engine, data, streams, monkeypatch):
    rng = np.random.default_rng(11)
    for name, s in streams.items():
        want = bz2.decompress(s)
        assert engine.decompress(s) == want, name
        for win in (None, 100_000, 1 << 20):
            if win is None:
                monkeypatch.delenv("BZ2B200_DSTREAM_WINDOW", raising=False)
            else:
                monkeypatch.setenv("BZ2B200_DSTREAM_WINDOW", str(win))
            rc, ti, to, got = _run(engine, s, _pieces(rng))
            assert rc == bz.OK and got == want and ti == len(s) and to == len(want), (name, win)
            rc, ti, to, _ = _run(engine, s, _pieces(rng), test=True)
            assert rc == bz.OK and ti == len(s) and to == len(want), (name, win, "test mode")


def test_chance_magics_do_not_change_the_output(engine, streams, monkeypatch):
    """BZ2B200_MULTI_DEC_CHANCE adds a spurious candidate at every window's first bit and between any two candidates,
    also in the carried tail and the look-ahead."""
    monkeypatch.setenv("BZ2B200_MULTI_DEC_CHANCE", "1")
    rng = np.random.default_rng(12)
    for win in (None, 100_000, 1 << 20):
        if win is None:
            monkeypatch.delenv("BZ2B200_DSTREAM_WINDOW", raising=False)
        else:
            monkeypatch.setenv("BZ2B200_DSTREAM_WINDOW", str(win))
        for name, s in streams.items():
            rc, ti, to, got = _run(engine, s, _pieces(rng))
            assert rc == bz.OK and got == bz2.decompress(s), (name, win)


def test_stream_boundaries_on_window_edges(engine):
    """The window size puts the first window's decode edge (W - LOOK) 0, 1, 2, 7 and 10 bytes before and after every
    stream boundary, so that footers, "BZh" headers and first block magics straddle it.  The large last stream keeps the
    first window from being the last one."""
    parts = [engine.compress(corpus.text(300_000, 61), 1), bz2.compress(corpus.repetitive(300_000, 62).tobytes(), 3),
             bz2.compress(b""), engine.compress(corpus.text(500_000, 63), 9), bz2.compress(corpus.text(300_000, 64).tobytes(), 9),
             engine.compress(corpus.random_bytes(6_000_000, 65), 9)]
    cat = b"".join(parts)
    want = bz2.decompress(cat)
    assert engine.decompress(cat) == want
    bounds = np.cumsum([len(p) for p in parts])[:-1]
    rng = np.random.default_rng(13)
    for b in bounds:
        for d in (0, 1, -1, 2, -2, 7, -7, 10, -10):
            w = LOOK + int(b) + d
            assert w < len(cat)
            with pytest.MonkeyPatch.context() as mp:
                mp.setenv("BZ2B200_DSTREAM_WINDOW", str(w))
                rc, ti, to, got = _run(engine, cat, [int(x) for x in rng.integers(1, 2_000_000, 8)])
                assert rc == bz.OK and got == want, (int(b), d)
                rc, _, to, _ = _run(engine, cat, [len(cat)], test=True)
                assert rc == bz.OK and to == len(want), (int(b), d)


def test_single_defects_give_the_whole_buffer_code(engine, monkeypatch):
    data = np.concatenate([corpus.text(1_500_000, 71), corpus.random_bytes(5_000_000, 70)]).tobytes()
    s = engine.compress(data, 9)                                         # with 64 KiB windows: several decode windows
    mid = bytearray(s)
    mid[len(s) // 2] ^= 0x10                                             # inside a block
    bcrc = bytearray(s)
    bcrc[11] ^= 0x01                                                     # the first block's stored CRC (bytes 10..13)
    cases = {"block bit": (bytes(mid), data), "block crc": (bytes(bcrc), data),
             "missing footer": (s[:-10], data), "truncated": (s[:len(s) * 2 // 3], data),
             "trailing garbage": (s + b"garbage after the stream", data), "bad magic": (b"BZx" + s[3:], b""),
             "not bzip2": (b"not a bzip2 stream at all " * 40_000, b"")}
    for win in (None, 65536):
        if win is None:
            monkeypatch.delenv("BZ2B200_DSTREAM_WINDOW", raising=False)
        else:
            monkeypatch.setenv("BZ2B200_DSTREAM_WINDOW", str(win))
        for name, (bad, truth) in cases.items():
            want = _rc(engine.decompress, bad, 1 << 24)
            assert want in (bz.E_FORMAT, bz.E_CRC), name
            rc, ti, _, got = _run(engine, bad, [1, 1, 5, 100_000, 300_000])
            assert rc == want and truth.startswith(got), (name, win)
            assert _run(engine, bad, [len(bad)], test=True)[0] == want, (name, win)
        assert _rc(engine.decompress, cases["block crc"][0], 1 << 24) == bz.E_CRC
    for short in (b"", b"B", b"BZh91AY&SY"):                             # the one-call path: E_ARG; a stream: E_FORMAT at close
        assert _rc(engine.decompress, short, 1 << 24) == bz.E_ARG
        assert _run(engine, short)[0] == bz.E_FORMAT
        assert _run(engine, short, test=True)[0] == bz.E_FORMAT
    assert engine.decompress(s) == data                                  # the context still works


def test_combined_crc_across_windows(engine, monkeypatch):
    """A stream that spans at least five windows: its combined CRC is folded across them; a wrong one is E_CRC."""
    data = np.concatenate([corpus.random_bytes(7_000_000, 72), corpus.text(3_000_000, 73)]).tobytes()
    s = engine.compress(data, 9)
    win = 1 << 20
    assert len(s) > LOOK + 3 * win
    monkeypatch.setenv("BZ2B200_DSTREAM_WINDOW", str(win))
    rc, _, _, got = _run(engine, s, [3_000_000] * 5)
    assert rc == bz.OK and got == data
    foot = bytearray(s)
    foot[-2] ^= 0x01                                                     # inside the footer's combined CRC
    assert _rc(engine.decompress, bytes(foot), 1 << 25) == bz.E_CRC
    rc, _, _, got = _run(engine, bytes(foot), [3_000_000] * 5)
    assert rc == bz.E_CRC and got == data                                # every block passed its own CRC
    assert _run(engine, bytes(foot), test=True)[0] == bz.E_CRC


def test_larger_than_memory_test_mode(engine):
    """More than 16 GiB of output through one dstream in test mode: the same 256 MiB stream written again and again."""
    rep = corpus.repetitive(256 << 20, 91)
    s = engine.compress(rep, 9)
    reps = (16 << 30) // rep.size + 1
    with bz.DStream(engine) as d:
        for _ in range(reps):
            d.write(s)
    assert d.total_in == reps * len(s) and d.total_out == reps * rep.size > (16 << 30)


_CHILD = r"""
import json, sys, zlib
sys.path.insert(0, sys.argv[1])
import bzip2_rust_b200 as bz
assert "torch" not in sys.modules
s = open(sys.argv[2], "rb").read()
reps = int(sys.argv[3])
class Crc:
    n, crc = 0, 0
    def write(self, b):
        self.n += len(b)
        self.crc = zlib.crc32(b, self.crc)
eng = bz.Engine(0)
sink = Crc()
with bz.DStream(eng, sink) as d:
    for _ in range(reps):
        for off in range(0, len(s), 16 << 20):
            d.write(s[off:off + (16 << 20)])
eng.close()
# this process's own peak: ru_maxrss would also hold the parent's, which subprocess (vfork, then exec) passes on
hwm = [int(l.split()[1]) for l in open("/proc/self/status") if l.startswith("VmHWM:")][0]
print(json.dumps({"n": sink.n, "crc": sink.crc, "total_out": d.total_out, "torch": "torch" in sys.modules,
                  "peak_rss_kib": hwm}))
"""


def test_larger_than_memory_bounded_rss(engine, tmp_path):
    """About 4.25 GiB through a counting, CRC-ing sink in a process that does not import torch: the output is exact and
    the peak resident set stays under 2 GiB (the whole-buffer path would need more than 4 GiB for the output alone)."""
    rep = corpus.repetitive(256 << 20, 92)
    s = engine.compress(rep, 9)
    reps = 17
    crc = 0
    for _ in range(reps):
        crc = zlib.crc32(rep, crc)
    path = tmp_path / "rep.bz2"
    path.write_bytes(s)
    del rep
    r = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(path), str(reps)], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["n"] == res["total_out"] == reps * (256 << 20) > (4 << 30)
    assert res["crc"] == crc and not res["torch"]
    assert res["peak_rss_kib"] < (2 << 20), res


def test_sink_errors_and_bad_arguments(engine):
    class Full(io.RawIOBase):
        def write(self, b):
            raise OSError("disk full")
    s = engine.compress(corpus.text(3_000_000, 74), 9)
    with pytest.raises(OSError):
        with bz.DStream(engine, Full()) as d:
            d.write(s)
    assert "dstream: the sink reported an error" in bz.load_library().bz2b200_last_error(engine._h).decode()
    L = bz.load_library()
    h = C.c_void_p()
    assert L.bz2b200_dstream_open(engine._h, bz.SINK(), None, C.byref(h)) == bz.OK
    assert L.bz2b200_dstream_write(h, None, 5) == bz.E_ARG              # no data but a length
    assert L.bz2b200_dstream_close(h, None, None) == bz.E_FORMAT        # nothing was written
    # the context still compresses and decompresses
    d = corpus.text(1_000_000, 75).tobytes()
    z = engine.compress(d, 9)
    assert bz2.decompress(z) == d and engine.decompress(z) == d
    assert _run(engine, z)[3] == d


def _cli(args, cwd, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bz2b200_cli.py")] + args, cwd=cwd, env=env,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)


def test_cli_streams_and_removes_a_partial_output(engine, tmp_path):
    d = str(tmp_path)
    a = np.concatenate([corpus.text(4_000_000, 76), corpus.random_bytes(2_000_000, 77)]).tobytes()
    z = engine.compress(a, 9) + bz2.compress(corpus.text(500_000, 78).tobytes(), 3)
    open(os.path.join(d, "a.bz2"), "wb").write(z)
    env = dict(os.environ, BZ2B200_DSTREAM_WINDOW="200000")             # many windows
    r = _cli(["-d", "a.bz2"], d, env)
    assert r.returncode == 0, r.stderr
    assert open(os.path.join(d, "a"), "rb").read() == bz2.decompress(z)
    r = _cli(["-t", "a.bz2"], d, env)
    assert r.returncode == 0, r.stderr
    r = _cli(["-d", "-c", "a.bz2"], d, env)
    assert r.returncode == 0 and r.stdout == bz2.decompress(z)
    bad = bytearray(z)
    bad[len(z) // 2] ^= 0x04
    open(os.path.join(d, "bad.bz2"), "wb").write(bytes(bad))
    r = _cli(["-d", "bad.bz2"], d, env)
    assert r.returncode == 2 and not os.path.exists(os.path.join(d, "bad"))
    assert _cli(["-t", "bad.bz2"], d, env).returncode == 2
