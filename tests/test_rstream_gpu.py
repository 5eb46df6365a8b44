"""bz2b200_rstream: bz2b200_recover on an input that arrives in pieces, window by window, in bounded memory.

Most cases compare with Engine.recover (the whole-input path) on the same bytes: the entries field for field, the sink's
bytes and the totals, for several window sizes (BZ2B200_RSTREAM_WINDOW) and piece sizes.  The crafted-edge cases place
the first window's edge, at input byte WF - DEC_LOOK, exactly where a rule of the windowed driver matters."""
import ctypes as C
import io
import json
import os
import random
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import bz2craft as bc
import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus
from test_recover_gpu import big, flip, magics, still_decodes, without  # noqa: F401  (big: the 200-block fixture)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
MiB = 1 << 20
DEC_MAX_INPUT = 0xFFFFFF00 * 4


def _look():
    """DEC_LOOK, read from the source the way bwtcraft.py reads the sort's geometry."""
    text = open(os.path.join(ROOT, "bzip2_rust_b200", "csrc", "pump.cuh")).read()
    m = re.search(r"constexpr size_t DEC_LOOK = (\d+)u << (\d+);", text)
    return int(m.group(1)) << int(m.group(2))


LOOK = _look()


def fields(es):
    return [(e.bit, e.end_bit, e.out_off, e.out_len, e.crc, e.status, e.flags) for e in es]


def pieces_of(s, how, seed=0):
    if how == "whole":
        return [s]
    if isinstance(how, int):
        return [s[i:i + how] for i in range(0, len(s), how)]
    rnd = random.Random(seed)                       # "random": 1 .. 3 MiB
    out, i = [], 0
    while i < len(s):
        k = rnd.randint(1, 3 * MiB)
        out.append(s[i:i + k])
        i += k
    return out


def rstream(engine, s, monkeypatch, window=None, how="whole", sink=True):
    if window is None:
        monkeypatch.delenv("BZ2B200_RSTREAM_WINDOW", raising=False)
    else:
        monkeypatch.setenv("BZ2B200_RSTREAM_WINDOW", str(window))
    out = io.BytesIO() if sink else None
    with bz.RStream(engine, out) as r:
        for p in pieces_of(s, how):
            r.write(p)
    assert r.total_in == len(s) and r.nent == len(r.entries)
    return r.total_out, r.entries, out.getvalue() if sink else None


def same_as_recover(engine, s, monkeypatch, windows, hows, want=None):
    out = io.BytesIO()
    total, ents = engine.recover(s, out)
    if want is not None:
        assert out.getvalue() == want
    for w in windows:
        for how in hows:
            t2, e2, o2 = rstream(engine, s, monkeypatch, w, how)
            assert (t2, fields(e2)) == (total, fields(ents)), (w, how)
            assert o2 == out.getvalue(), (w, how)
    return ents


# ---- the existing inputs ------------------------------------------------------------------------------------------
W_SMALL = [None, MiB]


def test_golden_streams(engine, monkeypatch):
    g = json.load(open(os.path.join(HERE, "golden", "streams.json")))
    ins = [bytes.fromhex(h) for h in g["app_e"].values()] + [bytes.fromhex(e["stream_hex"]) for e in g["small"]]
    for e in g["generated"]:
        data = corpus.mix1m(e["seed"], e["n"]).tobytes() if e["gen"] == "mix1m" else \
            getattr(corpus, e["gen"])(e["n"], e["seed"]).tobytes()
        ins.append(engine.compress(data, e["level"]))
    for s in ins:
        same_as_recover(engine, s, monkeypatch, W_SMALL, ["whole", 65536])
    same_as_recover(engine, ins[0], monkeypatch, [1024], [1])        # one byte at a time, on a small input


@pytest.mark.parametrize("name", sorted(bc.CASES))
def test_crafted_cases(engine, monkeypatch, name):
    s, _, _ = bc.CASES[name]()
    same_as_recover(engine, s, monkeypatch, W_SMALL, ["whole"])
    still_decodes(engine)


def test_multi_stream_and_mixed_levels(engine, monkeypatch):
    import bz2
    a, b, c = corpus.text(1_500_000, 3).tobytes(), corpus.mix1m(4, 700_000).tobytes(), corpus.random_bytes(300_000, 5).tobytes()
    s = engine.compress(a, 1) + bz2.compress(b, 9) + engine.compress(c, 5) + bz2.compress(b"", 3)
    ents = same_as_recover(engine, s, monkeypatch, W_SMALL + [1024], ["whole", 4096], want=a + b + c)
    assert sum(1 for e in ents if e.flags & bz.REC_FOOTER) == 4


# ---- the damage matrix --------------------------------------------------------------------------------------------
WINDOWS = [MiB, 5 * MiB, 3 * MiB + 13]
HOWS = [4096, "random", "whole"]


def _damage(case, big):
    data, s, starts, blocks, foot = big
    if case == "data":
        return flip(s, blocks[5] + 2000)
    if case == "crc":
        return flip(s, blocks[64] + 48 + 7)
    if case == "magic":
        return flip(s, blocks[129] + 20)
    if case == "deleted_byte":
        cut = (blocks[60] + 4000) // 8
        return s[:cut] + s[cut + 1:]
    if case == "truncated":
        return s[:(blocks[130] + 5000) // 8]
    if case == "header":
        return b"XXXX" + s[4:]
    if case == "footer":
        return flip(s, foot[-1] + 48 + 3)
    if case == "every_tenth":
        d = s
        for k in range(0, len(blocks), 10):
            d = flip(d, blocks[k] + 3000)
        return d
    raise AssertionError(case)


@pytest.mark.parametrize("case", ["intact", "data", "crc", "magic", "deleted_byte", "truncated", "header", "footer",
                                  "every_tenth"])
def test_damage_matrix(engine, big, monkeypatch, case):
    d = big[1] if case == "intact" else _damage(case, big)
    same_as_recover(engine, d, monkeypatch, WINDOWS, HOWS)


def test_garbage_between_and_after_streams(engine, monkeypatch):
    a, b = corpus.text(2_000_000, 31).tobytes(), corpus.mix1m(32, 900_000).tobytes()
    sa, sb = engine.compress(a, 2), engine.compress(b, 9)
    junk = corpus.random_bytes(100_003, 33).tobytes()
    for d in (sa + junk + sb, sa + sb + junk, junk + sa + junk + sb + junk):
        same_as_recover(engine, d, monkeypatch, WINDOWS, HOWS, want=a + b)


# ---- crafted window edges: the first edge at input byte e, with WF = e + DEC_LOOK -----------------------------------
def at_edge(engine, s, monkeypatch, edge_byte, how="whole"):
    assert len(s) > edge_byte + LOOK                                # the first window is not the last one
    return same_as_recover(engine, s, monkeypatch, [edge_byte + LOOK], [how])


@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_edge_at_a_block_magic(engine, big, monkeypatch, delta):
    data, s, starts, blocks, _ = big
    for k in (30, 31):
        at_edge(engine, s, monkeypatch, blocks[k] // 8 + delta)
        at_edge(engine, flip(s, blocks[k] + 2000), monkeypatch, blocks[k] // 8 + delta, 4096)


def test_edge_inside_a_damaged_block(engine, big, monkeypatch):
    data, s, starts, blocks, _ = big
    d = flip(s, blocks[40] + 2000)
    ents = at_edge(engine, d, monkeypatch, (blocks[40] + 6000) // 8)
    assert [e.bit for e in ents if e.status and not e.flags & bz.REC_FOOTER] == [blocks[40]]


def test_edge_inside_an_intact_block_with_chance_magics(engine, big, monkeypatch):
    """The edge lies inside an intact block, so `cover` crosses it; with the knob, a chance candidate lies past it."""
    data, s, starts, blocks, _ = big
    d = flip(s, blocks[90] + 30)
    monkeypatch.setenv("BZ2B200_MULTI_DEC_CHANCE", "1")
    out = io.BytesIO()
    total, ents = engine.recover(d, out)

    def intact(es):
        return [(e.bit, e.end_bit, e.out_off, e.out_len, e.flags) for e in es if e.status == bz.OK and not e.flags & bz.REC_FOOTER]
    for k in (20, 21):
        edge = (blocks[k] + blocks[k + 1]) // 16                   # the middle of block k: chance candidates lie past it
        for how in ("whole", 4096):
            t2, e2, o2 = rstream(engine, d, monkeypatch, edge + LOOK, how)
            assert (t2, o2) == (total, out.getvalue())
            assert intact(e2) == intact(ents)


@pytest.mark.parametrize("before", [1, 8, 64])
def test_edge_before_a_rescued_block(engine, big, monkeypatch, before):
    """Block k is intact and the magic of k + 1 is flipped: the rescue bit (k's end) lies at or past the edge."""
    data, s, starts, blocks, _ = big
    k = 50
    d = flip(s, blocks[k + 1] + 20)
    ents = at_edge(engine, d, monkeypatch, (blocks[k + 1] - before) // 8)
    assert [e.bit for e in ents if e.flags & bz.REC_NO_MAGIC] == [blocks[k + 1]]
    assert not [e for e in ents if e.status]


def test_edge_at_a_footer(engine, monkeypatch):
    a, b = corpus.text(3_000_000, 41).tobytes(), corpus.random_bytes(6_000_000, 42).tobytes()
    s = engine.compress(a, 1) + engine.compress(b, 3)
    f = [bit for bit, foot in magics(s) if foot][0]
    for edge in (f // 8 - 1, f // 8, f // 8 + 1, (f + 80) // 8, (f + 80) // 8 + 4):
        ents = at_edge(engine, s, monkeypatch, edge)
        assert [e.status for e in ents if e.flags & bz.REC_FOOTER] == [bz.OK, bz.OK]
    d = flip(s, f + 48 + 3)                                         # a damaged footer at the edge
    at_edge(engine, d, monkeypatch, f // 8)


def test_edge_in_garbage_between_streams(engine, monkeypatch):
    a, b = corpus.text(2_000_000, 51).tobytes(), corpus.random_bytes(5_000_000, 52).tobytes()
    sa, sb = engine.compress(a, 2), engine.compress(b, 9)
    junk = corpus.random_bytes(100_003, 53).tobytes()
    d = sa + junk + sb
    for edge in (len(sa) + 10, len(sa) + 50_000, len(sa) + len(junk) - 1):
        at_edge(engine, d, monkeypatch, edge)
    assert engine.recover(d)[0] == len(a) + len(b)


# ---- past the one-call bound ----------------------------------------------------------------------------------------
def test_past_the_one_call_bound(engine, monkeypatch):
    """268 copies of a 64 MB -9 stream of random bytes (> DEC_MAX_INPUT), one damaged in a block that spans an edge.
    Only one copy is held in host memory.  About 17.2 GB pass through the default 64 MiB windows."""
    monkeypatch.delenv("BZ2B200_RSTREAM_WINDOW", raising=False)
    n = 64_000_000
    s = engine.compress(corpus.random_bytes(n, 61).tobytes(), 9)
    c = len(s)
    copies = DEC_MAX_INPUT // c + 1
    blocks = [e.bit for e in engine.recover(s)[1] if not e.flags & bz.REC_FOOTER]
    # the first own-range edge (k + 1) * 64 MiB - DEC_LOOK past the middle that lies inside a copy, 2 MB from its ends
    wf = 64 * MiB
    for k in range(copies * c // (2 * wf), copies * c // wf):
        j, rel = divmod((k + 1) * wf - LOOK, c)
        if 2_000_000 < rel < c - 2_000_000:
            break
    rel *= 8
    i = max(x for x in range(len(blocks)) if blocks[x] < rel)
    assert blocks[i] < rel < blocks[i + 1]
    d = flip(s, blocks[i] + 2000)
    want_total, want = engine.recover(d)
    bad = [e for e in want if e.status and not e.flags & bz.REC_FOOTER]
    assert len(bad) == 1
    seen = {"n": 0, "bad": [], "footers_bad": [], "last": None}

    def on_entries(es):
        seen["n"] += len(es)
        for e in es:
            if e.status:
                (seen["footers_bad"] if e.flags & bz.REC_FOOTER else seen["bad"]).append(e)
        seen["last"] = es[-1]
    with bz.RStream(engine, None, on_entries) as r:
        for x in range(copies):
            r.write(d if x == j else s)
    assert r.total_in == copies * c > DEC_MAX_INPUT
    assert r.total_out == want_total + (copies - 1) * n
    assert r.nent == seen["n"] and not r.entries
    assert [(e.status, e.bit - 8 * j * c) for e in seen["bad"]] == [(bad[0].status, bad[0].bit)]
    assert [e.status for e in seen["footers_bad"]] == [bz.E_FORMAT]
    assert seen["last"].flags & bz.REC_FOOTER


# ---- API behaviour --------------------------------------------------------------------------------------------------
def _open_raw(engine, sink, report):
    h = C.c_void_p()
    return engine._L.bz2b200_rstream_open(engine._h, sink, report, None, C.byref(h)), h


def _close_raw(engine, h):
    t = C.c_uint64()
    return engine._L.bz2b200_rstream_close(h, C.byref(t), C.byref(t), C.byref(t))


def test_callback_errors_are_sticky(engine, big, monkeypatch):
    monkeypatch.setenv("BZ2B200_RSTREAM_WINDOW", str(MiB))
    s = big[1]
    a = np.frombuffer(s, dtype=np.uint8)
    for sink, report in ((bz.SINK(lambda u, p, n: 1), bz.REC_REPORT()),
                         (bz.SINK(), bz.REC_REPORT(lambda u, p, n: 1)),
                         (bz.SINK(lambda u, p, n: 0), bz.REC_REPORT(lambda u, p, n: 1))):
        rc, h = _open_raw(engine, sink, report)
        assert rc == bz.OK
        rcs = [engine._L.bz2b200_rstream_write(h, a.ctypes.data + off, min(MiB, a.size - off))
               for off in range(0, a.size, MiB)]
        assert set(rcs) <= {bz.OK, bz.E_ARG}
        if bz.E_ARG in rcs:                                     # sticky: every later write returns it
            assert rcs[rcs.index(bz.E_ARG):] == [bz.E_ARG] * (len(rcs) - rcs.index(bz.E_ARG))
        assert _close_raw(engine, h) == bz.E_ARG
        assert "rstream: " in engine._L.bz2b200_last_error(engine._h).decode()
    still_decodes(engine)


def test_python_exceptions_are_raised(engine, big):
    s = big[1]
    with pytest.raises(ZeroDivisionError):
        with bz.RStream(engine, type("W", (), {"write": lambda self, b: 1 / 0})()) as r:
            r.write(s)
    with pytest.raises(KeyError):
        with bz.RStream(engine, None, lambda es: {}["x"]) as r:
            r.write(s)
    still_decodes(engine)


def test_close_without_input(engine):
    rc, h = _open_raw(engine, bz.SINK(), bz.REC_REPORT())
    assert rc == bz.OK
    assert _close_raw(engine, h) == bz.E_ARG
    with pytest.raises(bz.Bz2B200Error):
        bz.RStream(engine).close()


def test_one_stream_per_context(engine):
    r = bz.RStream(engine)
    with pytest.raises(bz.Bz2B200Error):
        bz.DStream(engine)
    with pytest.raises(bz.Bz2B200Error):
        bz.RStream(engine)
    r.write(engine.compress(b"abc" * 1000, 9))
    r.close()
    d = bz.DStream(engine)
    with pytest.raises(bz.Bz2B200Error):
        bz.RStream(engine)
    d.write(engine.compress(b"abc" * 1000, 9))
    d.close()
    still_decodes(engine)


def test_entries_come_after_their_bytes(engine, big, monkeypatch):
    monkeypatch.setenv("BZ2B200_RSTREAM_WINDOW", str(3 * MiB + 13))
    s = _damage("every_tenth", big)
    got = [0]
    checked = [0]

    class Out:
        def write(self, b):
            got[0] += len(b)

    def on_entries(es):
        for e in es:
            assert got[0] >= e.out_off + e.out_len
            checked[0] += 1
    with bz.RStream(engine, Out(), on_entries) as r:
        for p in pieces_of(s, "random", 7):
            r.write(p)
    assert checked[0] == r.nent > 200 and got[0] == r.total_out
    still_decodes(engine)


# ---- the command line ---------------------------------------------------------------------------------------------
def test_cli_recover_from_stdin(engine, big):
    data, s, starts, blocks, _ = big
    d = flip(flip(s, blocks[40] + 2000), blocks[100] + 20)
    cli = [sys.executable, os.path.join(ROOT, "tools", "bz2b200_cli.py"), "--recover"]
    env = dict(os.environ, BZ2B200_RSTREAM_WINDOW=str(MiB))
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "bad.bz2")
        open(f, "wb").write(d)
        r1 = subprocess.run(cli + [f], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        r2 = subprocess.run(cli + ["-"], input=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
        assert r1.returncode == r2.returncode == 2
        assert r2.stdout == open(os.path.join(td, "bad.recovered"), "rb").read() == without(data, starts, {40})
        assert r2.stderr.decode().replace("bz2b200: -: ", "bz2b200: %s: " % f) == r1.stderr.decode()
