"""Crafted BWT blocks at the edges of the GPU suffix sort, and a numpy model of its list state.

The GPU sort (csrc/bwt.cu) picks its path at fixed sizes: k_init_ranks scans rows in tiles of RT and sends every group
of the 8-byte sort to the LOC list (at most LCAP rows) or the BIG list; k_refine_local reads the LOC list in windows of
LW entries and owns the groups that start in the first LTILE = LW - LCAP of them, ranking groups of at most SCAP by
all-pairs counting and larger ones by LSD passes; k_list_refine splits the BIG list in tiles of RT.  Whether a natural
block reaches any of these edges is chance, and two kinds of mistake never show in the output bytes: a LOC-sized group
sent down the BIG path, and a resolved rotation kept in the next list.  The blocks built here place groups at exact
SA rows and list offsets, and list_model() predicts the list lengths that bz2b200_get_bwt_stats reports.

The geometry is read from the CUDA sources, so the crafted edges move with it.
"""
import functools
import os
import re

import numpy as np

_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bzip2_rust_b200", "csrc")


def _read_int(fname, pattern):
    with open(os.path.join(_CSRC, fname)) as f:
        m = re.search(pattern, f.read(), re.M)
    assert m, "%s: no match for %r: the geometry moved, update tests/bwtcraft.py" % (fname, pattern)
    return int(m.group(1))


def geometry():
    """The sort's and MTF's fixed sizes, as the sources define them by default."""
    g = dict(
        LW=_read_int("bwt.cu", r"^#define BZ_LW (\d+)\s*$"),
        LCAP=_read_int("bwt.cu", r"^#define BZ_LCAP (\d+)\s*$"),
        SCAP=_read_int("bwt.cu", r"^#define BZ_SCAP (\d+)\s*$"),
        RT=_read_int("common.cuh", r"^constexpr int BZ_THREADS = (\d+);") * _read_int("bwt.cu", r"^constexpr int RT_IPT = (\d+);"),
        CH=_read_int("mtf.cu", r"^#define BZ_MTF_CH (\d+)\s*$"),
    )
    g["LTILE"] = g["LW"] - g["LCAP"]
    return g


GEO = geometry()


# ------------------------------------------------------------------------------------------------------------------
# model
# ------------------------------------------------------------------------------------------------------------------
def _groups(heads_by_row, rows):
    """Offsets and sizes, in the list `rows` (SA rows in order), of the groups whose head rows are heads_by_row[rows]."""
    if len(rows) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    h = heads_by_row[rows]
    st = np.flatnonzero(np.r_[True, h[1:] != h[:-1]])
    return st, np.diff(np.r_[st, len(rows)])


def list_model(block, lcap=None):
    """Model of bz_bwt_batch on one block.

    Rotations are sorted by their cyclic 8-byte prefix.  A rotation is LOC when its depth-8 group has at most `lcap`
    members and BIG otherwise, for good.  Round h (8, 16, ...) lists the rotations that are still tied, in SA-row order,
    or nothing once h >= n.  A round refines the LOC list with key2 = rank[(s+h) mod n] (rank = the group's first row)
    and then the BIG list, whose key2 already sees the ranks the LOC step just wrote, as the GPU orders its kernels.
    Those ranks are finer than depth h, so a BIG group can split sooner than a pure depth-h rule says: on natural text
    the two rules give different list lengths (the bytes are the same).

    Returns dict(key, bwt, sa, spans8, rounds) where spans8 = (start row, size, big) of every depth-8 group of more
    than one row and rounds[i] = dict(h, loc, big, loc_groups, big_groups, left): list lengths, (offset, size,
    subgroups after the refinement) of each group in its list, and the rows still tied after the refinement.
    """
    lcap = GEO["LCAP"] if lcap is None else lcap
    a = np.frombuffer(bytes(block), dtype=np.uint8)
    n = len(a)
    assert n >= 1
    k = np.zeros(n, dtype=np.uint64)
    for q in range(8):                                      # big-endian cyclic prefix: a block with n < 8 wraps
        k = (k << np.uint64(8)) | np.roll(a, -q).astype(np.uint64)
    sa = np.argsort(k, kind="stable")
    ks = k[sa]
    rows = np.arange(n)
    head = np.r_[True, ks[1:] != ks[:-1]]
    hrow = np.maximum.accumulate(np.where(head, rows, 0))
    rank = np.empty(n, np.int64)
    rank[sa] = hrow
    size = np.bincount(hrow, minlength=n)[hrow]
    big_rot = np.zeros(n, bool)
    big_rot[sa] = size > lcap
    st = np.flatnonzero(head)
    sz = np.diff(np.r_[st, n])
    m = sz > 1
    spans8 = list(zip(st[m].tolist(), sz[m].tolist(), (sz[m] > lcap).tolist()))
    rounds = []
    h = 8
    while h < n:
        hrow = rank[sa]
        size = np.bincount(hrow, minlength=n)[hrow]
        tied = size > 1
        if not tied.any():
            break
        is_big = big_rot[sa]
        rnd = dict(h=h)
        for name, lrows in (("loc", np.flatnonzero(tied & ~is_big)), ("big", np.flatnonzero(tied & is_big))):
            off, gsz = _groups(hrow, lrows)
            sub = np.zeros(len(off), np.int64)
            if len(lrows):
                s = sa[lrows]
                g = hrow[lrows]
                k2 = rank[(s + h) % n]
                o = np.lexsort((k2, g))
                s, g, k2 = s[o], g[o], k2[o]
                new = np.r_[True, (g[1:] != g[:-1]) | (k2[1:] != k2[:-1])]
                sa[lrows] = s
                rank[s] = lrows[np.maximum.accumulate(np.where(new, np.arange(len(lrows)), 0))]
                sub = np.add.reduceat(new.astype(np.int64), off)
            rnd[name] = len(lrows)
            rnd[name + "_groups"] = list(zip(off.tolist(), gsz.tolist(), sub.tolist()))
        hrow = rank[sa]
        rnd["left"] = int((np.bincount(hrow, minlength=n)[hrow] > 1).sum())
        rounds.append(rnd)
        h *= 2
    return dict(key=int(rank[0]), bwt=a[(sa - 1) % n].tobytes(), sa=sa, spans8=spans8, rounds=rounds)


_MODELS = {}


def model_of(block):
    """list_model(block), computed once per process."""
    key = bytes(block)
    if key not in _MODELS:
        _MODELS[key] = list_model(key)
    return _MODELS[key]


def batch_stats(models):
    """What bwt_stats() reports after one batch of these blocks: rounds, list_sum, big_sum."""
    return dict(rounds=max((len(m["rounds"]) for m in models), default=0),
                list_sum=sum(r["loc"] + r["big"] for m in models for r in m["rounds"]),
                big_sum=sum(r["big"] for m in models for r in m["rounds"]))


# ------------------------------------------------------------------------------------------------------------------
# builders
# ------------------------------------------------------------------------------------------------------------------
# A block is a sequence of records: a word followed by a tag that no other record has.  Byte ranges keep the parts
# apart: word leads are 0x01..0x3f, so the rotations that start at a lead sort first and in lead order; everything
# else in a word is 0x40..0xff and every tag byte 0x80..0xfe, so all other rotations sort after them.  The rows and
# list offsets of the lead rotations therefore follow from the words alone.
class Block:
    def __init__(self):
        self.records = []          # (lead, word body) in sort order of the lead rotations
        self._g = 0

    def _body(self, w):
        """w - 1 bytes after the lead: the group number (two bytes) and a position byte, repeated, so that no 8 bytes
        of one word recur in another word or at another offset of the same word."""
        g = self._g
        self._g += 1
        assert g < 127 * 127
        out = bytearray()
        j = 0
        while len(out) < w - 1:
            out += bytes([0x80 + g // 127, 0x80 + g % 127, 0x40 + j % 64])
            j += 1
        return bytes(out[:w - 1])

    def singles(self, lead, count):
        """`count` rotations that sort alone, one SA row each."""
        self.records += [(lead, b"")] * count

    def groups(self, lead, size, count=1, w=8, tail=None):
        """`count` groups of `size` rotations tied to depth w (w - 1 shared bytes after the lead).  tail = list of
        (copies, extra bytes): the members go on with different words, so that the group splits at depth w."""
        for _ in range(count):
            body = self._body(w)
            if tail is None:
                self.records += [(lead, body)] * size
            else:
                assert sum(c for c, _ in tail) == size
                for c, t in tail:
                    self.records += [(lead, body + self._body(t + 1))] * c

    def bytes(self):
        """Tags are (k mod 127, k / 127, k mod 127) for record k: neighbouring records differ in the first and the last
        tag byte, so that no rotation ties two records of a small group to each other or to the next group."""
        n = len(self.records)
        out = bytearray()
        for k, (lead, body) in enumerate(self.records):
            assert 0 < lead < 0x40
            f = 0x80 + k % 127
            slow = [0x80 + (k // 127) % 127] + ([0x80 + k // (127 * 127)] if n > 127 * 127 else [])
            out += bytes([lead]) + body + bytes([f] + slow + [f])
        return bytes(out)


def _fill_pairs(b, lead, count, w):
    """LOC groups of 2 (and one of 3 when count is odd) that add exactly `count` entries to the lists up to round w."""
    assert count >= 0 and count != 1, count
    if count % 2:
        b.groups(lead, 3, 1, w)
        count -= 3
    b.groups(lead, 2, count // 2, w)


def rows_block(placements):
    """Groups at exact SA rows: placements = [(row, size)], filled in between with rotations that sort alone."""
    b = Block()
    lead, row = 1, 0
    for start, size in sorted(placements):
        assert start >= row
        b.singles(lead, start - row)
        b.groups(lead + 1, size)
        lead += 2
        row = start + size
    return b.bytes()


def loc_block(placements, w, d, lt):
    """Groups at exact LOC offsets in every round up to h = w: placements = [(offset, size, word length)], the gaps
    filled with groups of 2 and 3 of word length w (they resolve in round w).  More such groups at the end bring the
    LOC list of round w to a length of lt k + d: the rotations inside the words add groups of their own there."""
    def build(pad):
        b = Block()
        lead, off = 1, 0
        for start, size, wl in sorted(placements):
            _fill_pairs(b, lead, start - off, w)
            b.groups(lead + 1, size, 1, wl)
            lead += 2
            off = start + size
        _fill_pairs(b, lead, pad, w)
        return b.bytes()

    def loc_len(blk):
        return next((r["loc"] for r in list_model(blk)["rounds"] if r["h"] == w), 0) if blk else 0

    base = loc_len(build(0))
    total = base + 2 + (d - base - 2) % lt
    blk = build(total - base)
    assert loc_len(blk) == total
    return blk


@functools.lru_cache(maxsize=None)
def crafted():
    """crafted_blocks() of the default geometry, built once per process."""
    return tuple(crafted_blocks())


def crafted_blocks(geo=GEO):
    """[(name, block)]: the blocks that reach the edges of coverage_table()."""
    RT, LT, LCAP, SCAP = geo["RT"], geo["LTILE"], geo["LCAP"], geo["SCAP"]
    out = []
    # k_init_ranks: groups of LCAP and LCAP + 1 rows inside a tile, on its last row, ending on it, and across its edge
    # after member 1, LCAP / 2 and LCAP - 1; every placement has a tile of its own
    for size in (LCAP, LCAP + 1):
        offs = [7, RT - 1, RT - size, RT - LCAP // 2, RT - (LCAP - 1)]
        out.append(("init_rows_%d" % size, rows_block([(2 * i * RT + o, size) for i, o in enumerate(offs)])))
    # a group of 2 RT rows aligned to the tiles, and one that leaves a tile without a head
    out.append(("init_tile_without_head", rows_block([(RT, 2 * RT), (4 * RT - 1, RT + 500)])))
    # k_refine_local, once for round 8 (w = 8) and once for round 16 (w = 16), with LOC lengths next to a multiple of
    # LTILE.  Groups with 2 w shared bytes (factor 2) stay whole through the refinement of round w.
    lay1 = [(LT - 1, LCAP, 1), (2 * LT, 2, 1), (2 * LT + 2, SCAP, 2), (2 * LT + 2 + SCAP, SCAP + 1, 1),
            (2 * LT + 8 + 2 * SCAP, 2 * SCAP, 2)]
    lay2 = [(LT, SCAP, 1)] + [(2 * LT + i * (SCAP + 1), SCAP + 1, 1) for i in range(LT // (SCAP + 1) + 1)] + \
           [(4 * LT, LCAP, 1), (4 * LT + LCAP, 3 * SCAP // 2, 2)]
    for lay, name, ds in ((lay1, "loc_window", (-1, 0)), (lay2, "loc_medium", (1, -1))):
        for w, d in zip((8, 16), ds):
            out.append(("%s_w%d" % (name, w), loc_block([(o, s, f * w) for o, s, f in lay], w, d, LT)))
    out.append(("loc_len_w8", loc_block([], 8, 0, LT)))
    out.append(("loc_len_w16", loc_block([], 16, 1, LT)))
    # BIG path: list lengths around LCAP and the tiles of k_list_refine
    for sizes in ((LCAP + 1,), (RT,), (RT + 1,), (RT, RT), (LCAP + 1, 2 * RT - LCAP)):
        b = Block()
        for i, s in enumerate(sizes):
            b.groups(1 + i, s)
        out.append(("big_" + "_".join(map(str, sizes)), b.bytes()))
    # a BIG group that splits into LOC-sized groups that stay on the BIG path for another round
    b = Block()
    q = LCAP // 2
    b.groups(1, 4 * q, tail=[(q, 16)] * 4)
    out.append(("big_splits_to_loc_size", b.bytes()))
    # termination: periodic blocks, and ties that last until 2h first reaches n
    for n, unit in ((9, b"abc"), (16, b"ab"), (17, b"a"), (1024, b"abcd"), (1025, b"abcde"), (900_000, b"abc")):
        out.append(("periodic_%d" % n, unit * (n // len(unit))))
    # two rotations of a^(n-1) b share n - 2 bytes: the last tie resolves in round h with h < n <= 2h
    for n in (16, 2048):
        out.append(("last_tie_at_2h_%d" % n, b"a" * (n - 1) + b"b"))
    for n in range(1, 9):
        out.append(("tiny_%d" % n, b"aaaaaaab"[:n]))
    return out


# ------------------------------------------------------------------------------------------------------------------
# coverage
# ------------------------------------------------------------------------------------------------------------------
def _any_span(m, pred):
    return any(pred(s, z) for s, z, _ in m["spans8"])


def _loc(m, pred, min_h=8):
    return any(pred(o, z, sub) for r in m["rounds"] if r["h"] >= min_h for o, z, sub in r["loc_groups"])


def _big(m, pred):
    return any(pred(o, z, sub) for r in m["rounds"] for o, z, sub in r["big_groups"])


def coverage_table(geo=GEO):
    """[(edge name, predicate(model, n))]: every edge must hold for at least one crafted block."""
    RT, LT, LCAP, SCAP = geo["RT"], geo["LTILE"], geo["LCAP"], geo["SCAP"]
    t = []
    for size in (LCAP, LCAP + 1):
        t += [
            ("init: %d rows inside one tile" % size, lambda m, n, z=size: _any_span(m, lambda s, y: y == z and s // RT == (s + y - 1) // RT)),
            ("init: %d rows from a tile's last row" % size, lambda m, n, z=size: _any_span(m, lambda s, y: y == z and s % RT == RT - 1)),
            ("init: %d rows ending on a tile's last row" % size, lambda m, n, z=size: _any_span(m, lambda s, y: y == z and (s + y) % RT == 0)),
        ]
        for k in (1, LCAP // 2, LCAP - 1):
            t.append(("init: %d rows across a tile edge after member %d" % (size, k),
                      lambda m, n, z=size, k=k: _any_span(m, lambda s, y: y == z and (s + k) % RT == 0)))
    t += [
        ("init: a tile without a head", lambda m, n: _any_span(m, lambda s, y: (s // RT + 2) * RT <= s + y)),
        ("init: %d rows aligned to the tiles" % (2 * RT), lambda m, n: _any_span(m, lambda s, y: y == 2 * RT and s % RT == 0)),
    ]
    for h, when in ((8, "round 8"), (16, "round >= 16")):
        for size in (2, SCAP, SCAP + 1, LCAP):
            t.append(("local %s: group of %d" % (when, size), lambda m, n, z=size, h=h: _loc(m, lambda o, y, s: y == z, h)))
        t += [
            ("local %s: group at offset %d k, k >= 2" % (when, LT), lambda m, n, h=h: _loc(m, lambda o, y, s: o >= 2 * LT and o % LT == 0, h)),
            ("local %s: group at offset %d (next tile)" % (when, LT), lambda m, n, h=h: _loc(m, lambda o, y, s: o == LT, h)),
            ("local %s: %d members at offset %d mod %d (window full)" % (when, LCAP, LT - 1, LT),
             lambda m, n, h=h: _loc(m, lambda o, y, s: y == LCAP and o % LT == LT - 1, h)),
            ("local %s: one tile owns %d groups of %d" % (when, LT // (SCAP + 1) + 1, SCAP + 1),
             lambda m, n, h=h: any(sum(1 for o, y, _ in r["loc_groups"] if y == SCAP + 1 and o // LT == tt) == LT // (SCAP + 1) + 1
                                   for r in m["rounds"] if r["h"] >= h for tt in range(r["loc"] // LT + 1))),
            ("local %s: medium group stays tied" % when, lambda m, n, h=h: _loc(m, lambda o, y, s: y > SCAP and s == 1, h)),
            ("local %s: small group stays tied" % when, lambda m, n, h=h: _loc(m, lambda o, y, s: 1 < y <= SCAP and s == 1, h)),
        ]
        for d in (-1, 0, 1):
            t.append(("local %s: LOC length %d k %+d" % (when, LT, d),
                      lambda m, n, d=d, h=h: any(r["loc"] >= LT - 1 and (r["loc"] - d) % LT == 0 for r in m["rounds"] if r["h"] >= h)))
    for length in (LCAP + 1, RT, RT + 1, 2 * RT, 2 * RT + 1):
        t.append(("big: list length %d" % length, lambda m, n, z=length: any(r["big"] == z for r in m["rounds"])))
    t += [
        ("big: group across a %d-entry tile edge" % RT, lambda m, n: _big(m, lambda o, y, s: o // RT != (o + y - 1) // RT)),
        ("big: LOC-sized groups stay on the BIG path",
         lambda m, n: any(1 < y <= LCAP for r in m["rounds"][1:] for o, y, s in r["big_groups"])),
    ]
    for size in (9, 16, 17, 1024, 1025, 900_000):
        t.append(("end: periodic, n = %d" % size, lambda m, n, z=size: n == z and m["rounds"] and m["rounds"][-1]["left"] > 0))
    t.append(("end: the last tie resolves in the round where 2h first reaches n",
              lambda m, n: m["rounds"] and m["rounds"][-1]["left"] == 0 and m["rounds"][-1]["h"] * 2 >= n))
    for size in range(1, 9):
        t.append(("end: n = %d has no rounds" % size, lambda m, n, z=size: n == z and not m["rounds"]))
    return t
