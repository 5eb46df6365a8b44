"""bz2b200_recover: every intact block of a damaged .bz2 input, and a report of what was lost.

The oracle is libbz2 itself: an entry's bits [bit, end_bit) are wrapped as a one-block stream ("BZh9", a block magic, the
bits after the entry's 48 magic bits, a footer whose combined CRC is the block's stored CRC) and decoded with Python's bz2.
Every intact entry must decode to exactly the bytes recover gave for it.  The damage tests take the expected output
from the input: an engine-compressed file minus the input slices (Engine.stream_plan) of the blocks they damage."""
import bz2
import ctypes as C
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import bz2craft as bc
import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
BLOCK_MAGIC, END_MAGIC = 0x314159265359, 0x177245385090


# ---- the oracle ---------------------------------------------------------------------------------------------------
def magics(data):
    """Sorted (bit, is_footer) of every block and footer magic: bytes.find in the 8 bit-shifted copies of `data`."""
    data = bytes(data)
    n = len(data)
    x = int.from_bytes(data, "big")
    found = []
    for sh in range(8):
        y = ((x << sh) & ((1 << (8 * n)) - 1)).to_bytes(n, "big") if sh else data
        for magic, foot in ((BLOCK_MAGIC, False), (END_MAGIC, True)):
            pat = magic.to_bytes(6, "big")
            i = y.find(pat)
            while i >= 0:
                found.append((8 * i + sh, foot))
                i = y.find(pat, i + 1)
    return sorted(found)


def bits(data, a, b):
    """The bits [a, b) of `data` as an int."""
    lo, hi = a // 8, (b + 7) // 8
    v = int.from_bytes(bytes(data[lo:hi]), "big")
    return (v >> (hi * 8 - b)) & ((1 << (b - a)) - 1)


def wrap(data, a, b):
    """'BZh9' + a block magic + bits [a + 48, b) + a footer whose combined CRC is the block's stored CRC."""
    crc = bits(data, a + 48, a + 80)
    v, nb = int.from_bytes(b"BZh9", "big"), 32
    for val, ln in ((BLOCK_MAGIC, 48), (bits(data, a + 48, b), b - a - 48), (END_MAGIC, 48), (crc, 32)):
        v, nb = (v << ln) | val, nb + ln
    pad = (-nb) % 8
    return (v << pad).to_bytes((nb + pad) // 8, "big")


def libbz2_block(data, a, b):
    """libbz2's decode of the bits [a, b) as one block, None where it rejects them."""
    try:
        return bz2.decompress(wrap(data, a, b))
    except (OSError, ValueError, EOFError):
        return None


# ---- helpers ------------------------------------------------------------------------------------------------------
def recover(engine, s):
    out = io.BytesIO()
    total, ents = engine.recover(s, out)
    return total, ents, out.getvalue()


def check_universal(s, total, ents, out):
    """Every intact block entry is libbz2's decode of its bits; the sink got their concatenation."""
    assert total == len(out) == sum(e.out_len for e in ents)
    pos = 0
    for e in ents:
        assert e.out_off == pos
        if e.flags & bz.REC_FOOTER:
            assert e.out_len == 0 and e.end_bit == e.bit + 80
            continue
        if e.status == bz.OK:
            assert libbz2_block(s, e.bit, e.end_bit) == out[pos:pos + e.out_len], e
        else:
            assert e.out_len == 0 and e.status in (bz.E_FORMAT, bz.E_CRC)
        pos += e.out_len
    bits_seen = [e.bit for e in ents]
    assert bits_seen == sorted(bits_seen)


def check_intact(engine, s):
    total, ents, out = recover(engine, s)
    check_universal(s, total, ents, out)
    assert out == engine.decompress(s)
    assert all(e.status == bz.OK for e in ents), [e for e in ents if e.status]
    assert not any(e.flags & bz.REC_NO_MAGIC for e in ents)
    return ents


def flip(s, bit):
    b = bytearray(s)
    b[bit // 8] ^= 0x80 >> (bit % 8)
    return bytes(b)


def still_decodes(engine):
    data = corpus.text(300_000, 9).tobytes()
    assert engine.decompress(engine.compress(data, 9)) == data


# ---- intact inputs: the one-call result ---------------------------------------------------------------------------
def test_golden_streams_give_the_one_call_result(engine):
    g = json.load(open(os.path.join(HERE, "golden", "streams.json")))
    for hexs in g["app_e"].values():
        check_intact(engine, bytes.fromhex(hexs))
    for e in g["small"]:
        check_intact(engine, bytes.fromhex(e["stream_hex"]))
    for e in g["generated"]:
        data = corpus.mix1m(e["seed"], e["n"]).tobytes() if e["gen"] == "mix1m" else \
            getattr(corpus, e["gen"])(e["n"], e["seed"]).tobytes()
        check_intact(engine, engine.compress(data, e["level"]))


@pytest.mark.parametrize("name", sorted(bc.CASES))
def test_crafted_cases(engine, name):
    s, _, code = bc.CASES[name]()
    if code == "ok":
        check_intact(engine, s)
        return
    total, ents, out = recover(engine, s)           # a rejected case: no fault, only libbz2-checked bytes
    check_universal(s, total, ents, out)
    still_decodes(engine)


def test_multi_stream_and_mixed_levels(engine):
    a, b, c = corpus.text(1_500_000, 3).tobytes(), corpus.mix1m(4, 700_000).tobytes(), corpus.random_bytes(300_000, 5).tobytes()
    s = engine.compress(a, 1) + bz2.compress(b, 9) + engine.compress(c, 5) + bz2.compress(b"", 3)
    ents = check_intact(engine, s)
    assert sum(1 for e in ents if e.flags & bz.REC_FOOTER) == 4


# ---- the damage matrix --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big(engine):
    """20 MB of alternating text and random megabytes at -1: about 200 blocks, several batches of 128."""
    parts = [corpus.text(1_000_000, 20 + i) if i % 2 == 0 else corpus.random_bytes(1_000_000, 20 + i) for i in range(20)]
    data = np.concatenate(parts).tobytes()
    s = engine.compress(data, 1)
    starts = [int(x) for x in engine.stream_plan(data, 1)]
    mags = magics(s)
    blocks = [b for b, foot in mags if not foot]
    assert len(blocks) == len(starts) - 1 > 128
    return data, s, starts, blocks, [b for b, foot in mags if foot]


def without(data, starts, lost):
    return b"".join(data[starts[k]:starts[k + 1]] for k in range(len(starts) - 1) if k not in lost)


def damaged_blocks(ents):
    return [e for e in ents if e.status != bz.OK and not e.flags & bz.REC_FOOTER]


def run_damaged(engine, s, want):
    total, ents, out = recover(engine, s)
    check_universal(s, total, ents, out)
    assert out == want
    return ents


def footers(ents):
    return [e for e in ents if e.flags & bz.REC_FOOTER]


def test_intact_big_file(engine, big):
    data, s, starts, blocks, foot = big
    ents = check_intact(engine, s)
    assert [e.bit for e in ents if not e.flags & bz.REC_FOOTER] == blocks
    assert [e.status for e in footers(ents)] == [bz.OK]


@pytest.mark.parametrize("k", [0, 5, 127, 128, 150])
def test_bit_in_block_data(engine, big, k):
    data, s, starts, blocks, _ = big
    ents = run_damaged(engine, flip(s, blocks[k] + 2000), without(data, starts, {k}))
    assert [e.bit for e in damaged_blocks(ents)] == [blocks[k]]
    assert [e.status for e in footers(ents)] == [bz.E_FORMAT]


@pytest.mark.parametrize("k", [0, 64, 140])
def test_bit_in_stored_crc(engine, big, k):
    data, s, starts, blocks, _ = big
    ents = run_damaged(engine, flip(s, blocks[k] + 48 + 7), without(data, starts, {k}))
    assert [(e.bit, e.status) for e in damaged_blocks(ents)] == [(blocks[k], bz.E_CRC)]


@pytest.mark.parametrize("k", [1, 100, 128, 129, 200])
def test_bit_in_block_magic(engine, big, k):
    """The block before k is intact and ends where k starts: k is decoded there, and nothing is lost."""
    data, s, starts, blocks, _ = big
    k = min(k, len(blocks) - 1)
    d = flip(s, blocks[k] + 20)
    ents = run_damaged(engine, d, data)
    assert not damaged_blocks(ents)
    nm = [e for e in ents if e.flags & bz.REC_NO_MAGIC]
    assert [e.bit for e in nm] == [blocks[k]]
    assert [e.status for e in footers(ents)] == [bz.OK]
    if shutil.which("bzip2recover") and shutil.which("bzip2"):
        data_k = without(data, starts, {k - 1, k})               # it loses blocks k - 1 and k
        assert b"".join(bzip2recover_pieces(d)) == data_k


def test_deleted_byte(engine, big):
    data, s, starts, blocks, _ = big
    k = 60
    cut = (blocks[k] + 4000) // 8
    d = s[:cut] + s[cut + 1:]
    ents = run_damaged(engine, d, without(data, starts, {k}))
    later = [e.bit for e in ents if not e.flags & bz.REC_FOOTER and e.status == bz.OK and e.bit > blocks[k]]
    assert later == [b - 8 for b in blocks[k + 1:]]                # the later blocks at their shifted bit phases


def test_truncated(engine, big):
    data, s, starts, blocks, _ = big
    k = 130
    d = s[:(blocks[k] + 5000) // 8]
    ents = run_damaged(engine, d, data[:starts[k]])
    assert not footers(ents)


def test_header_overwritten(engine, big):
    data, s, starts, blocks, _ = big
    ents = run_damaged(engine, b"XXXX" + s[4:], data)
    assert not damaged_blocks(ents) and [e.status for e in footers(ents)] == [bz.OK]


def test_garbage_between_and_after_streams(engine):
    a, b = corpus.text(2_000_000, 31).tobytes(), corpus.mix1m(32, 900_000).tobytes()
    sa, sb = engine.compress(a, 2), engine.compress(b, 9)
    junk = corpus.random_bytes(100_003, 33).tobytes()
    for d in (sa + junk + sb, sa + sb + junk, junk + sa + junk + sb + junk):
        ents = run_damaged(engine, d, a + b)
        assert [e.status for e in footers(ents)] == [bz.OK, bz.OK]


def test_damaged_footer(engine, big):
    data, s, starts, blocks, foot = big
    ents = run_damaged(engine, flip(s, foot[-1] + 48 + 3), data)
    assert not damaged_blocks(ents)
    assert [e.status for e in footers(ents)] == [bz.E_CRC]


def test_every_tenth_block(engine, big):
    data, s, starts, blocks, _ = big
    d = s
    lost = set(range(0, len(blocks), 10))
    for k in lost:
        d = flip(d, blocks[k] + 3000)
    ents = run_damaged(engine, d, without(data, starts, lost))
    assert {e.bit for e in damaged_blocks(ents)} >= {blocks[k] for k in lost}


# ---- knobs, capacity, sinks ---------------------------------------------------------------------------------------
def test_chance_magics_change_nothing(engine, big, monkeypatch):
    data, s, starts, blocks, _ = big
    d = flip(flip(s, blocks[7] + 2000), blocks[90] + 30)
    total, ents, out = recover(engine, d)
    monkeypatch.setenv("BZ2B200_MULTI_DEC_CHANCE", "1")
    total2, ents2, out2 = recover(engine, d)
    check_universal(d, total2, ents2, out2)
    assert out2 == out and total2 == total

    def intact(es):
        return [(e.bit, e.end_bit, e.out_off, e.out_len, e.flags) for e in es if e.status == bz.OK and not e.flags & bz.REC_FOOTER]
    assert intact(ents2) == intact(ents)


def _raw(engine, s, sink, cap):
    a = np.frombuffer(s, dtype=np.uint8)
    ents = (bz.RecEntry * max(cap, 1))()
    nent, total = C.c_uint32(), C.c_uint64()
    rc = engine._L.bz2b200_recover(engine._h, a.ctypes.data, a.size, sink, None, ents, cap, C.byref(nent), C.byref(total))
    return rc, nent.value, total.value, list(ents[:min(cap, nent.value)])


def test_capacity_and_sinks(engine, big):
    data, s, starts, blocks, _ = big
    d = flip(s, blocks[3] + 2000)
    total, ents, out = recover(engine, d)
    got = []
    sink = bz.SINK(lambda u, p, n: got.append(C.string_at(p, n)) or 0)
    rc, nent, tot, few = _raw(engine, d, sink, 5)
    assert (rc, nent, tot) == (bz.E_CAP, len(ents), total)
    assert b"".join(got) == out                                      # the scan ran to the end
    assert [(e.bit, e.status) for e in few] == [(e.bit, e.status) for e in ents[:5]]
    rc, nent, tot, none = _raw(engine, d, bz.SINK(), len(ents))      # report only
    assert (rc, nent, tot) == (bz.OK, len(ents), total)
    assert [(e.bit, e.end_bit, e.out_off, e.out_len, e.crc, e.status, e.flags) for e in none] == \
        [(e.bit, e.end_bit, e.out_off, e.out_len, e.crc, e.status, e.flags) for e in ents]
    rc, *_ = _raw(engine, d, bz.SINK(lambda u, p, n: 1), len(ents))
    assert rc == bz.E_ARG
    with pytest.raises(ZeroDivisionError):
        engine.recover(d, type("W", (), {"write": lambda self, b: 1 / 0})())
    still_decodes(engine)


# ---- the command line ---------------------------------------------------------------------------------------------
def _cli(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bz2b200_cli.py")] + list(args),
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE)


def test_cli_recover(engine, big):
    data, s, starts, blocks, _ = big
    with tempfile.TemporaryDirectory() as td:
        good = os.path.join(td, "good.bz2")
        open(good, "wb").write(s)
        r = _cli("--recover", good)
        assert r.returncode == 0, r.stderr
        assert open(os.path.join(td, "good.recovered"), "rb").read() == data
        assert b"damaged" not in r.stderr and b"lost" not in r.stderr
        assert _cli("--recover", good).returncode == 1                   # exists: -f needed
        bad = os.path.join(td, "bad.bz2")
        k = 40
        d = flip(s, blocks[k + 20] + 2000)
        junk = corpus.random_bytes(5000, 3).tobytes()
        open(bad, "wb").write(d[:(blocks[k] + 900) // 8] + d[(blocks[k] + 9000) // 8:] + junk)
        r = _cli("--recover", "-f", bad)
        assert r.returncode == 2
        lines = r.stderr.decode().splitlines()
        assert sum("damaged block at input bits [%d," % blocks[k] in ln for ln in lines) == 1, lines
        assert sum("damaged block at input bits" in ln for ln in lines) == 2, lines
        end = 8 * (len(d) - (blocks[k] + 9000) // 8 + (blocks[k] + 900) // 8 + len(junk))
        assert sum(("lost input bits" in ln and ", %d), output offset" % end in ln) for ln in lines) == 1, lines
        assert open(os.path.join(td, "bad.recovered"), "rb").read() == without(data, starts, {k, k + 20})
        cut = os.path.join(td, "cut.bz2")                             # ends right after its last block: no footer
        open(cut, "wb").write(s[:(big[4][-1] + 7) // 8])
        r = _cli("--recover", cut)
        assert r.returncode == 2 and open(os.path.join(td, "cut.recovered"), "rb").read() == data
        r = _cli("--recover", "-c", "-q", bad)
        assert r.returncode == 2 and r.stderr == b"" and r.stdout == without(data, starts, {k, k + 20})


def bzip2recover_pieces(d):
    """The pieces bzip2recover writes for `d` that pass bzip2 -t, in order, decoded."""
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "x.bz2")
        open(f, "wb").write(d)
        subprocess.run(["bzip2recover", f], cwd=td, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        out = []
        for p in sorted(x for x in os.listdir(td) if x.startswith("rec")):
            r = subprocess.run(["bzip2", "-dc", os.path.join(td, p)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            if r.returncode == 0:
                out.append(r.stdout)
        return out
