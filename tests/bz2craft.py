"""bz2craft: a bit-exact .bz2 writer with every field under the caller's control, and the plain model of what libbz2
decodes from it.

The encoders the suite otherwise uses (ours, libbz2's) only write what a real compressor writes: code lengths of at most
17, as many selectors as groups, true BWTs.  The format allows more, and libbz2 1.0.8 -- the decode authority -- accepts
it.  A `Block` here fixes each field of one block: the symbol map (also 16-ranges flagged with an empty second-level
word), the randomised bit, `origPtr`, the table count, the selector list and its declared length, every table's code
lengths and the start value / delta walk that encodes them, the block CRC, and the symbol sequence (MTF/RLE2 symbols
with EOB, or derived from a BWT string).  `craft` lays blocks out in streams (level digit, combined CRC, several
streams, trailing bytes) and returns the bytes with the model output:
    inverse BWT by libbz2's rule (text position i = L[P^(i+1)(origPtr)], P = rows stably sorted by byte, n steps)
    -> de-randomisation -> inverse RLE1 (a count byte follows every 4 equal bytes; a block may end without one).
Pure Python and numpy; bits are packed with numpy, so a 900 000-symbol block takes about a second."""
import bz2
import ctypes
import zlib
from dataclasses import dataclass, field

import numpy as np

BLOCK_MAGIC = 0x314159265359
END_MAGIC = 0x177245385090
_REV8 = bytes(int(f"{i:08b}"[::-1], 2) for i in range(256))


def crc32(data):
    """CRC-32/BZIP2 (MSB first): the reflected zlib CRC of the bit-reversed bytes, bit-reversed."""
    return int(f"{zlib.crc32(bytes(data).translate(_REV8)):032b}"[::-1], 2)


def combine(crcs):
    c = 0
    for b in crcs:
        c = (((c << 1) | (c >> 31)) & 0xFFFFFFFF) ^ b
    return c


def rnums():
    """BZ2_rNums, the format's 512 randomisation distances, from libbz2 itself."""
    return list((ctypes.c_int32 * 512).in_dll(ctypes.CDLL("libbz2.so.1.0"), "BZ2_rNums"))


# ---- the model ----------------------------------------------------------------------------------------------------
def unmtf(syms, used):
    """MTF/RLE2 symbols (EOB last, or absent) -> the BWT string L.  RUNA/RUNB add (s + 1) << k copies of the list front."""
    lst = list(used)
    eob = len(used) + 1
    out, run, k = [], 0, 0
    for s in syms:
        s = int(s)
        if s <= 1:
            run += (s + 1) << k
            k += 1
            continue
        if run:
            out.append(bytes([lst[0]]) * run)
            run, k = 0, 0
        if s == eob:
            break
        v = lst.pop(s - 1)
        lst.insert(0, v)
        out.append(bytes([v]))
    if run:
        out.append(bytes([lst[0]]) * run)
    return b"".join(out)


def mtf_rle2(L, used):
    """The BWT string L -> MTF/RLE2 symbols with EOB (run lengths in bijective base 2, RUNA = 0, RUNB = 1)."""
    lst = list(used)
    syms, z = [], 0

    def flush(z):
        while z > 0:
            z -= 1
            syms.append(z & 1)
            z >>= 1
    for c in L:
        p = lst.index(c)
        if p == 0:
            z += 1
            continue
        flush(z)
        z = 0
        syms.append(p + 1)
        lst.insert(0, lst.pop(p))
    flush(z)
    syms.append(len(used) + 1)
    return syms


def lf(L):
    """P: row j of the stably sorted rows is row P[j] of L."""
    return np.argsort(np.frombuffer(bytes(L), dtype=np.uint8), kind="stable")


def ibwt(L, key):
    """libbz2's rule: text position i (0-based) = L[P^(i+1)(key)], exactly n steps whatever the cycles of P."""
    P = lf(L).tolist()
    Lb = bytes(L)
    out = bytearray(len(Lb))
    t = key
    for i in range(len(Lb)):
        t = P[t]
        out[i] = Lb[t]
    return bytes(out)


def derandomize(x):
    x = bytearray(x)
    t, pos, k = rnums(), 0, 0
    while pos < len(x):
        p = pos + t[k % 512] - 2
        if p < len(x):
            x[p] ^= 1
        pos += t[k % 512]
        k += 1
    return bytes(x)


def rle1_decode(b):
    """Inverse RLE1, or None for a block that ends with four equal bytes and no count byte: libbz2 then reads a count
    from past the block's end and reports the block corrupt (unRLE_obuf_to_output_FAST)."""
    out, i, n = bytearray(), 0, len(b)
    run, prev = 0, -1
    while i < n:
        c = b[i]
        i += 1
        if run == 4:
            out += bytes([prev]) * c
            run, prev = 0, -1
            continue
        run = run + 1 if c == prev else 1
        prev = c
        out.append(c)
    return None if run == 4 else bytes(out)


def pick_key(L, rng):
    """A random origin pointer for which both readings of the walk's last step agree (L[P^n(key)] == L[key]), or any
    key if there is none: keeps a case with a made-up L about what it tests rather than the multi-cycle rule."""
    P = lf(L)
    n = len(L)
    Lb = np.frombuffer(bytes(L), dtype=np.uint8)
    seen = np.zeros(n, dtype=bool)
    good = []
    for s in range(n):
        if seen[s]:
            continue
        cyc = [s]
        seen[s] = True
        t = int(P[s])
        while t != s:
            cyc.append(t)
            seen[t] = True
            t = int(P[t])
        c = np.array(cyc)
        good.extend(c[Lb[np.roll(c, -(n % len(c)))] == Lb[c]].tolist())
    return int(rng.choice(good)) if good else int(rng.integers(0, n))


# ---- Huffman tables -----------------------------------------------------------------------------------------------
def codes(lengths):
    """Canonical codes as libbz2 assigns them (BZ2_hbAssignCodes): by length, then by symbol.  None where the code does not
    fit its length (an oversubscribed table)."""
    out = [None] * len(lengths)
    ok = [1 <= l <= 20 for l in lengths]
    if not any(ok):
        return out
    vec = 0
    for n in range(min(l for l, o in zip(lengths, ok) if o), max(l for l, o in zip(lengths, ok) if o) + 1):
        for i, l in enumerate(lengths):
            if l == n:
                out[i] = vec if vec < (1 << n) else None
                vec += 1
        vec <<= 1
    return out


def complete_lengths(alpha, maxlen):
    """Lengths of a complete prefix code over `alpha` symbols whose longest code is `maxlen`: 1, 2, ..., maxlen, maxlen,
    then the longest leaf shorter than maxlen split in two until there are `alpha` leaves.  Ascending."""
    ls = list(range(1, maxlen)) + [maxlen, maxlen]
    assert alpha >= len(ls) and alpha <= 1 << maxlen
    while len(ls) < alpha:
        i = max(j for j, l in enumerate(ls) if l < maxlen)
        ls[i:i + 1] = [ls[i] + 1, ls[i] + 1]
    return sorted(ls)


def fixed_lengths(alpha):
    return [max(1, (alpha - 1).bit_length())] * alpha


# ---- the writer ---------------------------------------------------------------------------------------------------
class Bits:
    """MSB-first bit writer: (value, width <= 32) items, packed with numpy at the end."""

    def __init__(self):
        self.v, self.w = [], []
        self.n = 0

    def put(self, v, w):
        if w > 32:
            self.put(v >> 32, w - 32)
            v, w = v & 0xFFFFFFFF, 32
        if w:
            self.v.append(np.array([v], dtype=np.uint64))
            self.w.append(np.array([w], dtype=np.uint8))
            self.n += w

    def put_array(self, v, w):
        v = np.asarray(v, dtype=np.uint64)
        w = np.asarray(w, dtype=np.uint8)
        self.v.append(v)
        self.w.append(w)
        self.n += int(w.sum(dtype=np.int64))

    def tobytes(self):
        if not self.v:
            return b""
        v = np.concatenate(self.v)
        w = np.concatenate(self.w).astype(np.int64)
        bits = []
        for i in range(0, v.size, 1 << 16):              # in slices: the 64-bit temporaries stay small
            cv, cw = v[i:i + (1 << 16)], w[i:i + (1 << 16)]
            rv = np.repeat(cv, cw)
            sh = np.repeat(np.cumsum(cw), cw) - 1 - np.arange(int(cw.sum()))   # bits below this one in its item
            bits.append(((rv >> sh.astype(np.uint64)) & np.uint64(1)).astype(np.uint8))
        return np.packbits(np.concatenate(bits)).tobytes()


@dataclass
class Block:
    """One block.  `syms` are the MTF/RLE2 symbols including EOB; `used` the byte values of the symbol map (ascending).
    Unset fields take what a plain encoder would write: two tables of fixed-length codes, table 0 for every group, the
    CRC of the model output.  `selectors` holds table numbers, written move-to-front coded; an entry >= ngroups is
    written as that raw MTF index (an invalid stream).  Groups past the end of the list use its last entry's table.
    `paths[(t, s)]` lists the lengths the delta walk of table t passes through before it settles on symbol s's length.
    `phase`: extra selectors (MTF index 0, one bit each) are added so that the symbol data starts at this bit offset
    mod 32 of the file."""
    syms: list
    used: list
    key: int
    rand: int = 0
    crc: int = None
    ngroups: int = 2
    selectors: list = None
    nselectors: int = None
    lengths: list = None
    starts: list = None
    paths: dict = field(default_factory=dict)
    extra_l1: tuple = ()
    phase: int = None
    L: bytes = None

    @staticmethod
    def from_bwt(L, key, used=None, **kw):
        used = sorted(set(L)) if used is None else list(used)
        return Block(syms=mtf_rle2(L, used), used=used, key=key, L=bytes(L), **kw)

    @property
    def alpha(self):
        return len(self.used) + 2

    def bwt(self):
        if self.L is None:
            self.L = unmtf(self.syms, self.used)
        return self.L

    def output(self):
        """What libbz2 decodes from this block, or None where it rejects the block (origPtr outside it, an open run at
        its end)."""
        if "_out" not in self.__dict__:
            L = self.bwt()
            x = None
            if 0 <= self.key < len(L):
                x = ibwt(L, self.key)
                x = rle1_decode(derandomize(x) if self.rand else x)
            self._out = x
        return self._out

    def block_crc(self):
        if self.crc is not None:
            return self.crc
        out = self.output()
        return crc32(out) if out is not None else 0

    def write(self, w):
        alpha, T = self.alpha, self.ngroups
        nsym = len(self.syms)
        ngrp = (nsym + 49) // 50
        sels = list(self.selectors) if self.selectors is not None else [0] * ngrp
        lengths = [list(l) for l in self.lengths] if self.lengths is not None else [fixed_lengths(alpha)] * T
        crc = self.block_crc()
        w.put(BLOCK_MAGIC, 48)
        w.put(crc, 32)
        w.put(self.rand, 1)
        w.put(self.key, 24)
        his = {u >> 4 for u in self.used} | set(self.extra_l1)
        l1 = sum(0x8000 >> h for h in his)
        w.put(l1, 16)
        for h in sorted(his):
            w.put(sum(0x8000 >> (u & 15) for u in self.used if u >> 4 == h), 16)
        w.put(T, 3)
        # selectors, move-to-front coded
        mtf, sel_bits = list(range(max(T, 1))), []
        for s in sels:
            if s >= T:
                sel_bits.append(s)
                continue
            j = mtf.index(s)
            mtf.insert(0, mtf.pop(j))
            sel_bits.append(j)
        # code lengths: 5-bit start, then per symbol a walk (10 = +1, 11 = -1) ended by 0
        tab = Bits()
        for t in range(len(lengths)):
            cur = self.starts[t] if self.starts is not None else lengths[t][0]
            tab.put(cur, 5)
            for s in range(alpha):
                for target in list(self.paths.get((t, s), ())) + [lengths[t][s]]:
                    while cur != target:
                        tab.put(0b10 if target > cur else 0b11, 2)
                        cur += 1 if target > cur else -1
                tab.put(0, 1)
        declared = self.nselectors if self.nselectors is not None else len(sel_bits)
        extra = 0
        if self.phase is not None:
            data_at = w.n + 15 + sum(j + 1 for j in sel_bits) + tab.n
            extra = (self.phase - data_at) % 32
            declared += extra
        w.put(declared, 15)
        if sel_bits or extra:
            sb = sel_bits + [0] * extra
            w.put_array([(1 << (j + 1)) - 2 for j in sb], [j + 1 for j in sb])   # j ones, then a zero
        for v, n in zip(tab.v, tab.w):
            w.put_array(v, n)
        # symbols, 50 per group, each group with its selector's table
        cds = [codes(l) for l in lengths]
        syms = np.asarray(self.syms, dtype=np.int64)
        g = np.arange(nsym) // 50
        tsel = np.array([sels[min(i, len(sels) - 1)] if sels else 0 for i in range(ngrp)], dtype=np.int64)
        tsel[tsel >= T] = 0
        tg = tsel[g]
        ctab = np.array([[c if c is not None else -1 for c in cd] for cd in cds], dtype=np.int64)
        ltab = np.array(lengths, dtype=np.int64)
        cv, cl = ctab[tg, syms], ltab[tg, syms]
        if (cv < 0).any():
            raise ValueError("a symbol of a selected table has no code")
        w.put_array(cv.astype(np.uint64), cl.astype(np.uint8))


@dataclass
class Stream:
    blocks: list
    level: int = 9
    combined: int = None      # footer's combined CRC; computed by default

    def write(self, w):
        w.put(int.from_bytes(b"BZh", "big"), 24)
        w.put(ord("0") + self.level, 8)
        crcs = []
        for b in self.blocks:
            b.write(w)
            crcs.append(b.block_crc())
        w.put(END_MAGIC, 48)
        w.put(combine(crcs) if self.combined is None else self.combined, 32)
        w.put(0, (-w.n) % 8)

    def output(self):
        outs = [b.output() for b in self.blocks]
        return None if any(o is None for o in outs) else b"".join(outs)


def craft(streams, trailing=b""):
    """-> (file bytes, model output or None).  `streams` is a Stream, a Block or a list of Streams."""
    if isinstance(streams, Block):
        streams = Stream([streams])
    if isinstance(streams, Stream):
        streams = [streams]
    w = Bits()
    for s in streams:
        s.write(w)
    outs = [s.output() for s in streams]
    return w.tobytes() + bytes(trailing), (None if any(o is None for o in outs) else b"".join(outs))


def libbz2(data):
    """libbz2's decode of a whole file of concatenated streams, or None where it rejects the file: each stream through its
    own BZ2Decompressor, every one must reach its end, and nothing may follow the last (the project's rule for trailing
    bytes; `bz2.decompress` would drop a bad stream after a good one)."""
    out, rest = [], bytes(data)
    while True:
        d = bz2.BZ2Decompressor()
        try:
            out.append(d.decompress(rest))
        except (OSError, ValueError, EOFError):
            return None
        if not d.eof:
            return None
        rest = d.unused_data
        if not rest:
            return b"".join(out)


def bwt(data):
    """Rotation BWT by prefix doubling -> (L, row of the text).  A primitive text gives one LF cycle of length n."""
    s = np.frombuffer(bytes(data), dtype=np.uint8).astype(np.int64)
    n = s.size
    idx = np.arange(n)
    rank, k = s.copy(), 1
    while k < n:
        r2 = rank[(idx + k) % n]
        order = np.lexsort((r2, rank))
        a, b = rank[order], r2[order]
        new = np.empty(n, dtype=np.int64)
        new[order] = np.cumsum(np.r_[True, (a[1:] != a[:-1]) | (b[1:] != b[:-1])]) - 1
        rank = new
        if rank.max() == n - 1:
            break
        k *= 2
    order = np.argsort(rank, kind="stable")
    return s[(order - 1) % n].astype(np.uint8).tobytes(), int(np.nonzero(order == 0)[0][0])


# ---- the conformance cases ----------------------------------------------------------------------------------------
# name -> () -> (file, model output or None, expected result: "ok", "E_FORMAT" or "E_CRC").  "ok" cases are those
# libbz2 accepts, the others those it rejects; test_bz2craft_cpu.py checks both against libbz2.
CASES = {}


def _case(name, code="ok"):
    def reg(fn):
        CASES[name] = lambda: (*craft(fn()), code)
        return fn
    return reg


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _text(rng, n, k=256):
    """n bytes over k values with no two equal neighbours (no accidental RLE1 runs)."""
    x = rng.integers(0, k - 1, n)
    x[1:] = (x[0] + np.cumsum(1 + x[1:])) % k
    x[0] %= k
    return (x % k).astype(np.uint8).tobytes()


def _syms(rng, alpha, n, max_run=3):
    """n - 1 random MTF/RLE2 symbols using every non-EOB symbol, runs of at most `max_run` RUNA/RUNB, then EOB."""
    s = list(rng.permutation(alpha - 1)) + list(rng.integers(0, alpha - 1, max(0, n - alpha)))
    run = 0
    for i, v in enumerate(s):
        run = run + 1 if v <= 1 else 0
        if run > max_run:
            s[i] = 2 + int(rng.integers(0, alpha - 3)) if alpha > 3 else 2
            run = 0
    return [int(v) for v in s] + [alpha - 1]


def _used(alpha):
    return [i * 256 // (alpha - 2) for i in range(alpha - 2)]       # spread over the 16-ranges of the symbol map


def _settle(b, rng):
    """Give a block with a made-up L a key for which libbz2 has an output (no open RLE1 run at the end) and whose last
    byte does not depend on the walk length."""
    for _ in range(100):
        b.key = pick_key(b.bwt(), rng)
        b.__dict__.pop("_out", None)
        if b.output() is not None:
            return b
    raise ValueError("no key gives an output")


def _sym_block(name, alpha, n, **kw):
    """A block of random symbols over `alpha`."""
    rng = _rng(name)
    return _settle(Block(syms=_syms(rng, alpha, n), used=_used(alpha), key=0, **kw), rng)


def _text_block(name, n, key=None, **kw):
    """The true BWT of n random bytes (one LF cycle): every origin pointer gives a rotation of the text."""
    L, k = bwt(_text(_rng(name), n))
    return Block.from_bwt(L, k if key is None else key, **kw)


_L10 = [7] + [8] * 253 + [9, 10, 11, 11]      # complete, 258 symbols, codes of 10 and 11 bits on both sides of the LUT

for _m in (17, 18, 19, 20):
    def _f(_m=_m):
        name = f"huff_complete_maxlen_{_m}"
        ls = complete_lengths(21, _m)
        perm = _rng(name).permutation(21)
        return _sym_block(name, 21, 4000, lengths=[[ls[p] for p in perm], fixed_lengths(21)],
                          selectors=[g % 2 for g in range(80)])
    _case(f"huff_complete_maxlen_{_m}")(_f)


@_case("huff_all_258_symbols_at_length_20")
def _():
    return _sym_block("huff_all_258_symbols_at_length_20", 258, 6000, lengths=[[20] * 258] * 2)


@_case("huff_lengths_10_and_11_around_the_lut")
def _():
    perm = _rng("l10").permutation(258)
    return _sym_block("huff_lengths_10_and_11_around_the_lut", 258, 20000,
                      lengths=[[_L10[p] for p in perm], fixed_lengths(258)], selectors=[1, 0] * 200)


@_case("huff_incomplete_code_unused_codes_never_occur")
def _():
    ls = complete_lengths(21, 20)
    ls[0] = 2                                   # the codes under '1' are never assigned
    return _sym_block("huff_incomplete", 21, 3000, lengths=[ls[::-1], ls])


@_case("huff_oversubscribed_table_never_selected")
def _():
    return _sym_block("huff_oversub", 30, 2000, ngroups=3, lengths=[fixed_lengths(30), fixed_lengths(30), [1] * 30],
                      selectors=[0, 1] * 20)


@_case("huff_start_walks_to_1_and_20_and_back")
def _():
    return _sym_block("huff_walks", 30, 2000, starts=[20, 1], paths={(0, 0): [1, 20], (1, 0): [20, 1], (1, 29): [1, 20]},
                      selectors=[0, 1] * 20)


for _nm, _kw in {"huff_length_walks_to_21": dict(paths={(0, 3): [21]}),
                 "huff_length_walks_to_0": dict(paths={(1, 0): [0]}),
                 "huff_start_value_0": dict(starts=[0, 5]),
                 "huff_start_value_21": dict(starts=[5, 21])}.items():
    _case(_nm, "E_FORMAT")(lambda _nm=_nm, _kw=_kw: _sym_block(_nm, 30, 500, **_kw))

for _t in range(2, 7):
    _case(f"groups_T{_t}_one_byte_block")(lambda _t=_t: Block.from_bwt(b"x", 0, ngroups=_t, selectors=[_t - 1]))


@_case("groups_tables_never_selected")
def _():
    return _sym_block("groups_never", 40, 3000, ngroups=6)


def _six_tables(alpha, rng):
    out = []
    for t in range(6):
        ls = complete_lengths(alpha, 8 + 2 * t) if t else fixed_lengths(alpha)
        out.append([ls[p] for p in rng.permutation(alpha)])
    return out


@_case("groups_selectors_change_every_group_all_mtf_positions")
def _():
    rng = _rng("sel6")
    sels = [int(v) for v in rng.integers(0, 6, 400)]
    for i in range(1, len(sels)):
        if sels[i] == sels[i - 1]:
            sels[i] = (sels[i] + 1) % 6
    return _sym_block("sel6", 60, 20000, ngroups=6, selectors=sels, lengths=_six_tables(60, rng))


@_case("selector_ge_T_in_a_used_group", "E_FORMAT")
def _():
    return _sym_block("sel_bad", 30, 500, ngroups=3, selectors=[0, 1, 2, 3, 0, 1, 2, 0, 1, 2])


@_case("selector_ge_T_past_the_groups_used", "E_FORMAT")
def _():
    return _sym_block("sel_bad2", 30, 500, ngroups=3, selectors=[0, 1, 2] * 3 + [1, 2, 0, 1, 5])


def _nsel(name, count, level):
    def f():
        rng = _rng(name)
        b = _sym_block(name, 30, 500, ngroups=4, selectors=[int(v) for v in rng.integers(0, 4, count)])
        return Stream([b], level=level)
    _case(name)(f)


_nsel("nselectors_equal_to_groups_used", 10, 9)
_nsel("nselectors_groups_used_plus_1", 11, 9)
for _n in (2009, 18002, 18003, 32767):
    _nsel(f"nselectors_{_n}_level1", _n, 1)
for _n in (18003, 32767):
    _nsel(f"nselectors_{_n}_level9", _n, 9)


@_case("nselectors_fewer_than_groups", "E_FORMAT")
def _():
    return _sym_block("sel_few", 30, 500, selectors=[0, 1] * 4 + [0])


@_case("nselectors_0", "E_FORMAT")
def _():
    return _sym_block("sel_0", 30, 40, selectors=[])


@_case("bit_phases_32_blocks")
def _():
    blocks = []
    for i in range(32):
        rng = _rng(f"phase{i}")
        alpha = int(rng.integers(3, 259))
        b = _sym_block(f"phase{i}", alpha, int(rng.integers(alpha, 2 * alpha + 700)), ngroups=6,
                       lengths=_six_tables(alpha, rng) if alpha >= 21 else None, phase=i)
        b.selectors = [int(v) for v in rng.integers(0, 6, (len(b.syms) + 49) // 50)]
        blocks.append(b)
    return Stream(blocks)


@_case("eob_is_the_50th_symbol_of_a_group")
def _():
    return _sym_block("eob50", 30, 100)


@_case("eob_is_the_first_symbol_of_a_group")
def _():
    return _sym_block("eob51", 30, 101)


@_case("eob_only_block", "E_FORMAT")
def _():
    return Block(syms=[2], used=[65], key=0)


@_case("all_256_byte_values")
def _():
    return _text_block("all256", 5000)


@_case("one_used_byte_alphabet_3")
def _():
    return Block.from_bwt(b"q" * 1000, 0)


def _straddle(k):
    """The run of RUNA/RUNB symbols holds index 1024, where k_dec_chunks cuts, with k of its symbols before it (k = 19:
    a run of 19 that ends just before the cut -- 20 symbols would code more than 900 000 bytes)."""
    rng = _rng(f"straddle{k}")
    r = min(k + 1, 19) if k else 5
    head = [2 + int(v) for v in rng.integers(0, 18, 1024 - k)]
    run = [int(v) for v in rng.integers(0, 2, r)] if r < 19 else [0] * r
    tail = [2 + int(v) for v in rng.integers(0, 18, 40)]
    return _settle(Block(syms=head + run + tail + [20], used=_used(21), key=0), rng)


for _k in range(20):
    _case(f"run_straddles_chunk_cut_at_offset_{_k}")(lambda _k=_k: _straddle(_k))


def _run_block(n):
    """A block of n bytes: a few symbols, then one run to the end."""
    return Block.from_bwt(b"xyz" + b"a" * (n - 3), 1)


def _random_block(name, n):
    rng = _rng(name)
    return _settle(Block.from_bwt(rng.integers(0, 16, n).astype(np.uint8).tobytes(), 0), rng)


for _lv in (1, 9):
    _case(f"run_reaches_block_size_level{_lv}")(lambda _lv=_lv: Stream([_run_block(100000 * _lv)], _lv))
    _case(f"run_one_byte_past_block_size_level{_lv}", "E_FORMAT")(lambda _lv=_lv: Stream([_run_block(100000 * _lv + 1)], _lv))
    _case(f"nblock_exactly_block_size_level{_lv}")(lambda _lv=_lv: Stream([_random_block(f"nb{_lv}", 100000 * _lv)], _lv))
    _case(f"nblock_one_past_block_size_level{_lv}", "E_FORMAT")(
        lambda _lv=_lv: Stream([_random_block(f"nb{_lv}", 100000 * _lv + 1)], _lv))


@_case("level1_stream_with_a_150000_byte_block_then_a_level9_stream", "E_FORMAT")
def _():
    return [Stream([_random_block("mixed1", 150000)], 1), Stream([_text_block("mixed9", 3000)], 9)]


@_case("level9_stream_with_a_150000_byte_block_then_a_level1_stream")
def _():
    return [Stream([_random_block("mixed1", 150000)], 9), Stream([_text_block("mixed9", 3000)], 1)]


for _nm, _key in {"origptr_0": 0, "origptr_n_minus_1": 8999, "origptr_multiple_of_32": 32 * 77,
                  "origptr_multiple_of_2048": 2048 * 3}.items():
    _case(_nm)(lambda _key=_key: _text_block("origptr", 9000, key=_key))
_case("origptr_n", "E_FORMAT")(lambda: _text_block("origptr", 9000, key=9000))


def _multicycle(kind, rand):
    if kind == "aba_key1":
        return Block.from_bwt(b"aba", 1, rand=rand)
    rng = _rng(kind)
    L = rng.integers(0, 256, 20000).astype(np.uint8)
    if kind == "sorted_L":                      # P = identity: n cycles of length 1
        L.sort()
        return Block.from_bwt(L.tobytes(), int(rng.integers(0, L.size)), rand=rand)
    b = Block.from_bwt(L.tobytes(), 0, rand=rand)
    P = lf(b.L)
    for key in rng.permutation(L.size):         # a key whose cycle length does not divide n: the n-th step matters
        t = int(key)
        for _ in range(L.size):
            t = int(P[t])
        b.key = int(key)
        b.__dict__.pop("_out", None)
        if L[t] != L[key] and b.output() is not None:
            return b
    raise ValueError("no key")


for _kind in ("aba_key1", "sorted_L", "random_L"):
    for _r in (0, 1):
        _case(f"ibwt_multicycle_{_kind}" + ("_randomised" if _r else ""))(lambda _kind=_kind, _r=_r: _multicycle(_kind, _r))


def _rle1_block(x):
    L, k = bwt(x)
    return Block.from_bwt(L, k)


_case("rle1_count_bytes_0_251_252_255")(lambda: _rle1_block(b"abcd" + b"eeee\x00" + b"ffff\xfb" + b"gggg\xfc" + b"hhhh\xff" + b"xyz"))
_case("rle1_three_equal_bytes_end_the_block")(lambda: _rle1_block(b"hello" + b"zzz"))


@_case("rle1_block_ends_after_four_equal_bytes_without_a_count", "E_FORMAT")
def _():
    b = _rle1_block(b"hello" + b"zzzz")
    b.crc = crc32(b"hellozzzz")                 # the CRC of those nine bytes: the open run is the only defect
    return b
_case("rle1_count_byte_is_the_last_byte")(lambda: _rle1_block(b"hello" + b"zzzz\x07"))


@_case("rle1_runs_end_at_every_thread_and_tile_phase")
def _():
    """k_rle1_inv: 32 bytes per thread, 8 KiB tiles.  One block whose runs end at every phase mod 32, then blocks whose
    run ends around the tile edge."""
    rng = _rng("rle1phase")
    blocks = []
    x = bytearray(_text(rng, 64 * 33))
    for j in range(32):
        e = 64 * j + j + 40                     # last of the four equal bytes; the count byte follows
        x[e - 3:e + 1] = bytes([x[e - 4] ^ 0x55]) * 4
        x[e + 1] = int(rng.integers(0, 256))
        x[e + 2] = x[e] ^ 0xAA
    blocks.append(_rle1_block(bytes(x)))
    for d in range(-6, 6):
        y = bytearray(_text(rng, 8192 + 64))
        e = 8192 + d
        y[e - 3:e + 1] = bytes([y[e - 4] ^ 0x55]) * 4
        y[e + 1] = 200
        y[e + 2] = y[e] ^ 0xAA
        blocks.append(_rle1_block(bytes(y)))
    return Stream(blocks)


@_case("crc_wrong_block_crc", "E_CRC")
def _():
    b = _text_block("crc", 3000)
    b.crc = b.block_crc() ^ 1
    return Stream([b], combined=combine([b.crc ^ 1]))


@_case("crc_wrong_combined_crc_in_the_second_stream", "E_CRC")
def _():
    b = _text_block("crc2", 3000)
    return [Stream([_text_block("crc1", 2000)]), Stream([b], combined=b.block_crc() ^ 0x80000000)]
