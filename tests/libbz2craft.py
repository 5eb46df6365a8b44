"""A compact model of libbz2 1.0.8's encoder, and inputs built to sit at the edges of its four rules.

With BZ2B200_LIBBZ2 the engine writes the bytes bzip2 1.0.8 writes.  libbz2 differs from the reference in four places
(DESIGN.md §10); this module restates them with the stages both share, for small inputs:
  1. block planning: every maximal run is cut greedily from its own start into chunks of at most 255 bytes (RLE1 size:
     the length below 4, else 5); a block ends right after the first chunk at which its RLE1 length reaches
     B = 100000 * level - 19, and the chunking is never restarted at a block start;
  2. the origin pointer of a periodic block (u^k) is the row where libbz2's fallbackSort leaves rotation 0 among the k
     equal rotations (fallback_origin; libbz2 runs fallbackSort on every periodic block except the few that mainSort
     finishes within its work budget: periodic_main_sort);
  3. the initial tables partition the alphabet by exact MTF symbol counts (EOB once);
  4. code lengths come from BZ2_hbMakeCodeLengths (maxLen 17): a binary heap whose tie order is part of the output.
The BWT is a numpy prefix doubling over cyclic rotations, the rest is plain Python: fine up to a few hundred KB.

Builders return (name, level, data, edge) with `edge` a key of edges_reached(); the CPU test checks the model against
bz2.compress and that every edge is reached, the GPU test compares the engine's libbz2 mode with bz2.compress on them.
"""
import bz2
import ctypes
import ctypes.util

import numpy as np

_CRC_TAB = []
for _i in range(256):
    _c = _i << 24
    for _ in range(8):
        _c = ((_c << 1) ^ 0x04C11DB7) & 0xFFFFFFFF if _c & 0x80000000 else (_c << 1) & 0xFFFFFFFF
    _CRC_TAB.append(_c)


def crc32(data):
    """bzip2's block CRC (MSB first, polynomial 0x04C11DB7)."""
    c = 0xFFFFFFFF
    tab = _CRC_TAB
    for x in data:
        c = ((c << 8) & 0xFFFFFFFF) ^ tab[(c >> 24) ^ x]
    return c ^ 0xFFFFFFFF


def libbz2_version():
    """BZ2_bzlibVersion() of the libbz2 Python's bz2 module links, or None when it cannot be found."""
    for name in (ctypes.util.find_library("bz2"), "libbz2.so.1.0", "libbz2.so.1"):
        if not name:
            continue
        try:
            lib = ctypes.CDLL(name)
        except OSError:
            continue
        lib.BZ2_bzlibVersion.restype = ctypes.c_char_p
        return lib.BZ2_bzlibVersion().decode()
    return None


# ---- rule 1: chunks and blocks -------------------------------------------------------------------------------------
def chunks(x):
    """(start, end) of every chunk: maximal runs cut greedily from their own start into pieces of at most 255 bytes."""
    a = np.frombuffer(bytes(x), dtype=np.uint8)
    if a.size == 0:
        return []
    starts = np.flatnonzero(np.r_[True, a[1:] != a[:-1]])
    ends = np.r_[starts[1:], a.size]
    out = []
    for s, e in zip(starts.tolist(), ends.tolist()):
        while e - s > 255:
            out.append((s, s + 255))
            s += 255
        out.append((s, e))
    return out


def chunk_size(n):
    return n if n < 4 else 5


def plan(x, level):
    """libbz2's blocks as input spans [(s, e)]."""
    B = 100000 * level - 19
    blocks, cur, acc = [], 0, 0
    for s, e in chunks(x):
        acc += chunk_size(e - s)
        if acc >= B:
            blocks.append((cur, e))
            cur, acc = e, 0
    if cur < len(x):
        blocks.append((cur, len(x)))
    return blocks


def rle1(x):
    out = bytearray()
    for s, e in chunks(x):
        if e - s < 4:
            out += x[s:e]
        else:
            out += bytes([x[s]]) * 4 + bytes([e - s - 4])
    return bytes(out)


def combined_crc(x, level):
    comb = 0
    for s, e in plan(x, level):
        comb = (((comb << 1) | (comb >> 31)) & 0xFFFFFFFF) ^ crc32(x[s:e])
    return comb


def stored_combined_crc(stream):
    """The combined CRC in a .bz2 stream's footer (the footer magic is found at its bit offset from the end)."""
    v = int.from_bytes(stream, "big")
    for pad in range(8):
        w = v >> pad
        if (w >> 32) & ((1 << 48) - 1) == 0x177245385090:
            return w & 0xFFFFFFFF
    raise ValueError("no footer")


# ---- rule 2: BWT and origin pointer ---------------------------------------------------------------------------------
def bwt(block):
    """(bwt bytes, origin pointer, class size of rotation 0) of the cyclic rotations of `block`."""
    n = len(block)
    if n == 0:
        return b"", 0, 0
    a = np.frombuffer(bytes(block), dtype=np.uint8).astype(np.int64)
    rank = a.copy()
    h = 1
    while True:
        r2 = np.roll(rank, -h)
        order = np.lexsort((r2, rank))
        k1, k2 = rank[order], r2[order]
        new = np.empty(n, dtype=bool)
        new[0] = True
        new[1:] = (k1[1:] != k1[:-1]) | (k2[1:] != k2[:-1])
        rank = np.empty(n, dtype=np.int64)
        rank[order] = np.cumsum(new) - 1
        if rank.max() == n - 1 or 2 * h >= n:
            break
        h *= 2
    order = np.argsort(rank, kind="stable")
    out = a[(order - 1) % n].astype(np.uint8).tobytes()
    size = int(np.count_nonzero(rank == rank[0]))
    orig = int(np.count_nonzero(rank < rank[0])) if size == 1 else fallback_origin(block)
    return out, orig, size


def fallback_origin(block):
    """Row of rotation 0 after libbz2's fallbackSort: a Manber-Myers doubling whose buckets are split by a 3-way
    quicksort (pivot first / middle / last by a linear-congruential r % 3) and an insertion sort below 10 entries.
    Among equal rotations the order is an artefact of exactly these steps."""
    n = len(block)
    fmap = [0] * n
    ftab = [0] * 257
    for c in block:
        ftab[c] += 1
    for i in range(1, 257):
        ftab[i] += ftab[i - 1]
    for i in range(n):
        j = block[i]
        ftab[j] -= 1
        fmap[ftab[j]] = i
    bh = [False] * (n + 65)
    for i in range(256):
        bh[ftab[i]] = True
    for i in range(32):
        bh[n + 2 * i], bh[n + 2 * i + 1] = True, False
    eclass = [0] * n

    def simple(lo, hi):
        if hi - lo > 3:
            for i in range(hi - 4, lo - 1, -1):
                tmp = fmap[i]
                ec = eclass[tmp]
                j = i + 4
                while j <= hi and ec > eclass[fmap[j]]:
                    fmap[j - 4] = fmap[j]
                    j += 4
                fmap[j - 4] = tmp
        for i in range(hi - 1, lo - 1, -1):
            tmp = fmap[i]
            ec = eclass[tmp]
            j = i + 1
            while j <= hi and ec > eclass[fmap[j]]:
                fmap[j - 1] = fmap[j]
                j += 1
            fmap[j - 1] = tmp

    def qsort3(lo0, hi0):
        r, stack = 0, [(lo0, hi0)]
        while stack:
            lo, hi = stack.pop()
            if hi - lo < 10:
                if lo != hi:
                    simple(lo, hi)
                continue
            r = (r * 7621 + 1) % 32768
            med = eclass[fmap[(lo, (lo + hi) >> 1, hi)[r % 3]]]
            un_lo = lt_lo = lo
            un_hi = gt_hi = hi
            while True:
                while un_lo <= un_hi:
                    d = eclass[fmap[un_lo]] - med
                    if d == 0:
                        fmap[un_lo], fmap[lt_lo] = fmap[lt_lo], fmap[un_lo]
                        lt_lo += 1
                        un_lo += 1
                        continue
                    if d > 0:
                        break
                    un_lo += 1
                while un_lo <= un_hi:
                    d = eclass[fmap[un_hi]] - med
                    if d == 0:
                        fmap[un_hi], fmap[gt_hi] = fmap[gt_hi], fmap[un_hi]
                        gt_hi -= 1
                        un_hi -= 1
                        continue
                    if d < 0:
                        break
                    un_hi -= 1
                if un_lo > un_hi:
                    break
                fmap[un_lo], fmap[un_hi] = fmap[un_hi], fmap[un_lo]
                un_lo += 1
                un_hi -= 1
            if gt_hi < lt_lo:
                continue
            k = min(lt_lo - lo, un_lo - lt_lo)
            fmap[lo:lo + k], fmap[un_lo - k:un_lo] = fmap[un_lo - k:un_lo], fmap[lo:lo + k]
            k = min(hi - gt_hi, gt_hi - un_hi)
            fmap[un_lo:un_lo + k], fmap[hi - k + 1:hi + 1] = fmap[hi - k + 1:hi + 1], fmap[un_lo:un_lo + k]
            a = lo + un_lo - lt_lo - 1
            b = hi - (gt_hi - un_hi) + 1
            if a - lo > hi - b:
                stack += [(lo, a), (b, hi)]
            else:
                stack += [(b, hi), (lo, a)]

    H = 1
    while True:
        j = 0
        for i in range(n):
            if bh[i]:
                j = i
            eclass[(fmap[i] - H) % n] = j
        not_done, i = 0, 0
        while i < n:                                        # buckets [l, r]: a set bit, then clear bits
            l = i
            i += 1
            while i < n and not bh[i]:
                i += 1
            r = i - 1
            if r > l:
                not_done += r - l + 1
                qsort3(l, r)
                cc = -1
                for q in range(l, r + 1):
                    if eclass[fmap[q]] != cc:
                        bh[q] = True
                        cc = eclass[fmap[q]]
        H *= 2
        if H > n or not_done == 0:
            break
    return fmap.index(0)


# ---- shared: MTF / RLE2 ---------------------------------------------------------------------------------------------
def mtf_rle2(bw):
    """(MTF symbols with EOB, used byte values)."""
    used = sorted(set(bw))
    seq = {v: i for i, v in enumerate(used)}
    lst = list(range(len(used)))
    out, z = [], 0

    def flush(z):
        z -= 1
        while True:
            out.append(1 if z & 1 else 0)
            if z < 2:
                break
            z = (z - 2) // 2

    for c in bw:
        j = seq[c]
        if lst[0] == j:
            z += 1
            continue
        if z:
            flush(z)
            z = 0
        p = lst.index(j)
        del lst[p]
        lst.insert(0, j)
        out.append(p + 1)
    if z:
        flush(z)
    out.append(len(used) + 1)
    return out, used


def n_groups(nmtf):
    return 2 if nmtf < 200 else 3 if nmtf < 600 else 4 if nmtf < 1200 else 5 if nmtf < 2400 else 6


# ---- rule 3: initial partition --------------------------------------------------------------------------------------
def initial_lengths(mtfv, alpha):
    nG = n_groups(len(mtfv))
    mf = np.bincount(np.asarray(mtfv), minlength=alpha).tolist()
    ln = [[15] * alpha for _ in range(nG)]
    n_part, rem_f, gs = nG, len(mtfv), 0
    while n_part > 0:
        t_freq, ge, a_freq = rem_f // n_part, gs - 1, 0
        while a_freq < t_freq and ge < alpha - 1:
            ge += 1
            a_freq += mf[ge]
        if ge > gs and n_part != nG and n_part != 1 and (nG - n_part) % 2 == 1:
            a_freq -= mf[ge]
            ge -= 1
        for v in range(alpha):
            ln[n_part - 1][v] = 0 if gs <= v <= ge else 15
        n_part -= 1
        gs = ge + 1
        rem_f -= a_freq
    return ln


# ---- rule 4: BZ2_hbMakeCodeLengths ----------------------------------------------------------------------------------
def code_lengths(freq, alpha, max_len=17, stats=None):
    """Code lengths of BZ2_hbMakeCodeLengths.  stats (a dict) counts 'retries' (builds over max_len) and 'ties'
    (pops that chose between two equal weights)."""
    weight = [0] * (2 * alpha + 2)
    parent = [0] * (2 * alpha + 2)
    for i in range(alpha):
        weight[i + 1] = (freq[i] if freq[i] else 1) << 8
    while True:
        heap = [0] * (alpha + 2)
        n_heap, n_nodes = 0, alpha
        weight[0], parent[0] = 0, -2

        def up(z):
            tmp = heap[z]
            while weight[tmp] < weight[heap[z >> 1]]:
                heap[z] = heap[z >> 1]
                z >>= 1
            heap[z] = tmp

        def down(z):
            tmp = heap[z]
            while True:
                y = z << 1
                if y > n_heap:
                    break
                if y < n_heap and weight[heap[y + 1]] < weight[heap[y]]:
                    y += 1
                if weight[tmp] < weight[heap[y]]:
                    break
                heap[z] = heap[y]
                z = y
            heap[z] = tmp

        for i in range(1, alpha + 1):
            parent[i] = -1
            n_heap += 1
            heap[n_heap] = i
            up(n_heap)
        while n_heap > 1:
            if stats is not None and n_heap >= 3 and min(weight[heap[2]], weight[heap[3]]) == weight[heap[1]]:
                stats["ties"] = stats.get("ties", 0) + 1
            n1 = heap[1]
            heap[1] = heap[n_heap]
            n_heap -= 1
            down(1)
            n2 = heap[1]
            heap[1] = heap[n_heap]
            n_heap -= 1
            down(1)
            n_nodes += 1
            parent[n1] = parent[n2] = n_nodes
            w1, w2 = weight[n1], weight[n2]
            weight[n_nodes] = ((w1 & 0xFFFFFF00) + (w2 & 0xFFFFFF00)) | (1 + max(w1 & 0xFF, w2 & 0xFF))
            parent[n_nodes] = -1
            n_heap += 1
            heap[n_heap] = n_nodes
            up(n_heap)
        lens, too_long = [], False
        for i in range(1, alpha + 1):
            j, k = 0, i
            while parent[k] >= 0:
                k = parent[k]
                j += 1
            lens.append(j)
            too_long |= j > max_len
        if not too_long:
            return lens
        if stats is not None:
            stats["retries"] = stats.get("retries", 0) + 1
        for i in range(1, alpha + 1):
            weight[i] = (1 + (weight[i] >> 8) // 2) << 8


# ---- block and stream -----------------------------------------------------------------------------------------------
class _Bits:
    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def put(self, nbits, v):
        self.acc = (self.acc << nbits) | v
        self.n += nbits
        while self.n >= 8:
            self.n -= 8
            self.out.append((self.acc >> self.n) & 0xFF)
        self.acc &= (1 << self.n) - 1

    def bytes(self):
        return bytes(self.out) + (bytes([(self.acc << (8 - self.n)) & 0xFF]) if self.n else b"")


def block_stats(block):
    """What one RLE1 block does in the model: origin, class size, nMTF, heap retries and ties."""
    st = {}
    _encode_block(_Bits(), block, 0, st)
    return st


def _encode_block(W, block, bcrc, st):
    bw, orig, csize = bwt(block)
    mtfv, used = mtf_rle2(bw)
    alpha = len(used) + 2
    nG = n_groups(len(mtfv))
    st.update(origin=orig, class_size=csize, nmtf=len(mtfv), groups=nG)
    ln = initial_lengths(mtfv, alpha)
    arr = np.asarray(mtfv)
    starts = np.arange(0, len(mtfv), 50)
    for _ in range(4):
        costs = np.stack([np.add.reduceat(np.asarray(ln[t])[arr], starts) for t in range(nG)])
        sel = np.argmin(costs, axis=0).tolist()                  # first minimum wins
        rf = np.zeros((nG, alpha), dtype=np.int64)
        for g, s in enumerate(starts.tolist()):
            np.add.at(rf[sel[g]], arr[s:s + 50], 1)
        ln = [code_lengths(rf[t].tolist(), alpha, 17, st) for t in range(nG)]
    W.put(24, 0x314159); W.put(24, 0x265359); W.put(32, bcrc); W.put(1, 0); W.put(24, orig)
    in16 = [any(16 * i <= v < 16 * i + 16 for v in used) for i in range(16)]
    for f in in16:
        W.put(1, int(f))
    uset = set(used)
    for i in range(16):
        if in16[i]:
            for v in range(16 * i, 16 * i + 16):
                W.put(1, int(v in uset))
    W.put(3, nG)
    W.put(15, len(sel))
    pos = list(range(nG))
    for s in sel:
        j = pos.index(s)
        del pos[j]
        pos.insert(0, s)
        W.put(j + 1, (1 << (j + 1)) - 2)
    codes = []
    for t in range(nG):
        L = ln[t]
        cur = L[0]
        W.put(5, cur)
        for v in range(alpha):
            while cur < L[v]:
                W.put(2, 2)
                cur += 1
            while cur > L[v]:
                W.put(2, 3)
                cur -= 1
            W.put(1, 0)
        c, code = {}, 0
        for l in range(min(L), max(L) + 1):
            for v in range(alpha):
                if L[v] == l:
                    c[v] = (l, code)
                    code += 1
            code <<= 1
        codes.append(c)
    for g, s in enumerate(starts.tolist()):
        ct = codes[sel[g]]
        for v in mtfv[s:s + 50]:
            W.put(*ct[v])


def compress(x, level, stats=None):
    """The .bz2 stream libbz2 1.0.8 writes for `x` at `level` (stats: a list that receives block_stats per block)."""
    W = _Bits()
    for ch in b"BZh":
        W.put(8, ch)
    W.put(8, ord("0") + level)
    comb = 0
    for s, e in plan(x, level):
        st = {}
        c = crc32(x[s:e])
        _encode_block(W, rle1(x[s:e]), c, st)
        if stats is not None:
            stats.append(st)
        comb = (((comb << 1) | (comb >> 31)) & 0xFFFFFFFF) ^ c
    W.put(24, 0x177245); W.put(24, 0x385090); W.put(32, comb)
    return W.bytes()


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _no_runs(rng, n, avoid=()):
    """n random bytes without two equal neighbours (every byte is its own 1-byte chunk)."""
    a = rng.integers(0, 256, n, dtype=np.int64)
    for i in range(n):
        while (i and a[i] == a[i - 1]) or a[i] in avoid:
            a[i] = (a[i] + 1 + (i % 7)) % 256
    return bytes(a.astype(np.uint8).tolist())


def small_inputs():
    """Single-block inputs the model compresses byte for byte at every level."""
    rng = np.random.default_rng(3)
    words = [bytes(rng.choice(list(b"etaoinshrdlu "), int(rng.integers(1, 9))).tolist()) for _ in range(300)]
    return [
        ("empty", b""), ("one byte", b"a"), ("hello", b"hello world\n"), ("aaaaa", b"aaaaa"),
        ("ab x300", b"ab" * 300), ("0..255 x3", bytes(range(256)) * 3),
        ("word text", b" ".join(words[int(i)] for i in rng.integers(0, 300, 1500))),
        ("random 3000", bytes(rng.integers(0, 256, 3000, dtype=np.uint8).tolist())),
        ("two letters", bytes(rng.choice(list(b"ab"), 4000).tolist())),
        ("mixed runs", b"x" * 1000 + b"y" * 7 + b"z" * 300 + b"q" * 255 + b"r" * 256 + b"s" * 4 + b"t" * 3),
    ]


def planner_inputs():
    """Multi-block inputs at -1 and -2 for the combined-CRC check: random bytes with runs of 4 to 5000 bytes."""
    rng = np.random.default_rng(11)
    out = []
    for k, level in enumerate((1, 1, 2, 2, 1, 2)):
        buf = bytearray()
        target = [250_000, 900_000, 700_000, 1_500_000, 99_981 * 3, 200_000 * 2 + 17][k]
        p_run = [0.002, 0.001, 0.0005, 0.0005, 0.00005, 0.001][k]
        while len(buf) < target:
            if rng.random() < p_run:
                buf += bytes([int(rng.integers(0, 4))]) * int(rng.choice([4, 5, 254, 255, 256, 259, 510, 511, 1000, 5000]))
            else:
                buf.append(int(rng.integers(0, 256)))
        out.append(("planner %d -%d" % (k, level), level, bytes(buf[:target])))
    return out


def _cut_inputs():
    """Level-1 inputs whose first cut falls where an edge needs it.  A prefix of P one-byte chunks brings the block to
    RLE1 length P; the chunk that follows decides where the block ends and how long it is."""
    B = 100000 - 19
    rng = np.random.default_rng(21)
    out = []

    def build(name, edge, P, chunk_byte, chunk_len, tail):
        pre = _no_runs(rng, P, avoid=(chunk_byte,))
        rest = _no_runs(rng, tail, avoid=(chunk_byte,))
        out.append((name, 1, pre + bytes([chunk_byte]) * chunk_len + rest, edge))

    for d in range(5):                                           # a 5-byte group ends the block at B + d
        build("group to B+%d" % d, "len B+%d" % d, B + d - 5, 7, 40, 30_000)
    for k in (1, 2, 3):                                          # a chunk of k literals ends the block
        build("short chunk %d at cut" % k, "short chunk at cut", B - 1, 9, k, 30_000)
    build("run 2000 across cut", "cut inside long run", B - 20, 5, 2000, 30_000)
    build("run 257 at cut", "short chunk at cut", B - 1 - 5, 6, 257, 30_000)   # 255-byte group, then a 2-byte chunk
    out.append(("last block B-1", 1, _no_runs(rng, B - 1), "len B-1"))
    out.append(("last block one chunk", 1, _no_runs(rng, B, avoid=(3,)) + bytes([3]) * 200, "last block one chunk"))
    return out


def _nmtf_inputs():
    """Single blocks whose nMTF (EOB included) is exactly 199/200, 599/600, 1199/1200 and 2399/2400: random bytes over
    128 values, lengthened until the model hits the count."""
    out = []
    for target in (199, 200, 599, 600, 1199, 1200, 2399, 2400):
        rng = np.random.default_rng(target)
        base = bytes(rng.integers(0, 128, target + 200, dtype=np.uint8).tolist())
        for n in range(max(1, target - 80), target + 200):
            bw, _, _ = bwt(rle1(base[:n]))
            if len(mtf_rle2(bw)[0]) == target:
                out.append(("nMTF %d" % target, 9, base[:n], "nmtf %d" % target))
                break
        else:
            raise AssertionError("no prefix reaches nMTF %d" % target)
    return out


def _heap_inputs():
    """A block where a code-length build goes past 17 bits and the halving retry runs (byte counts halving from one
    value to the next, every value present: the rare ones hang a depth-8 subtree under a long chain), and one with
    many equal weights."""
    rng = np.random.default_rng(5)
    p = 0.5 ** np.arange(256)
    p /= p.sum()
    skew = bytes(rng.choice(256, 500_000, p=p).astype(np.uint8).tolist()) + bytes(range(256))
    ties = bytes(rng.integers(0, 256, 2000, dtype=np.uint8).tolist())
    return [("heap retry", 9, skew, "heap retry"), ("heap ties", 9, ties, "heap ties")]


def _periodic_inputs():
    """Periodic blocks (u^k): short periods, periods near the block length, periods made by RLE1."""
    rng = np.random.default_rng(8)
    u = _no_runs(rng, 2999)
    return [
        ("period 2", 9, b"ab" * 3000, "period short"),
        ("period 3", 1, b"xyz" * 20000, "period short"),
        ("period n/2", 9, u + u, "period near n"),
        ("period n/3", 9, u[:1500] * 3, "period near n"),
        ("rle1 period 10", 9, (b"a" * 10 + b"b" * 10) * 500, "period from rle1"),
        ("zero fill 255000", 9, bytes(255 * 1000), "period from rle1"),
        ("zero fill 306000", 9, bytes(255 * 1200), "period from rle1"),
        ("zero fill 153000", 9, bytes(255 * 600), "period from rle1"),
    ]


def periodic_main_sort():
    """Periodic blocks of 10000 bytes or more with a few long periods: libbz2's mainSort finishes them within its work
    budget (the other periodic blocks exhaust it and go to fallbackSort), and mainSort leaves rotation 0 at another row
    of its class than fallbackSort.  The engine follows fallbackSort, so on these blocks the streams differ in the 24-bit
    origin pointer only (the BWT text of equal rotations is the same whichever row is chosen) and decode to the same
    bytes.  (name, level, data)."""
    rng = np.random.default_rng(8)
    u = _no_runs(rng, 5000)
    return [("period 4000 x3", 9, u[:4000] * 3), ("period 2000 x5", 9, u[:2000] * 5)]


def long_runs():
    """A run of one byte value over three blocks or more at every level: its interior blocks are (c c c c 251)^k."""
    out = []
    for level in range(1, 10):
        jb = -(-(100000 * level - 19) // 5)
        out.append(("zeros x3 blocks -%d" % level, level, bytes(255 * jb * 3 + 1000)))
    out.append(("0xff x3.5 blocks -1", 1, b"\xff" * (255 * 20000 * 3 + 127 * 255 + 3) + b"tail"))
    return out


def crafted():
    """(name, level, data, edge) of every crafted input."""
    return _cut_inputs() + _nmtf_inputs() + _heap_inputs() + _periodic_inputs()


def edges_reached(level, data):
    """The set of edge names this input reaches in the model."""
    B = 100000 * level - 19
    got = set()
    blocks = plan(data, level)
    ch = chunks(data)
    ends = {e: (s, e) for s, e in ch}
    for k, (s, e) in enumerate(blocks):
        L = len(rle1(data[s:e]))
        last = k == len(blocks) - 1
        if not last:
            if B <= L <= B + 4:
                got.add("len B+%d" % (L - B))
            cs, ce = ends[e]
            if ce - cs < 4:
                got.add("short chunk at cut")
            if e < len(data) and data[e - 1] == data[e]:
                a, b = e, e
                while a > 0 and data[a - 1] == data[e]:
                    a -= 1
                while b < len(data) and data[b] == data[e]:
                    b += 1
                if b - a > 255:
                    got.add("cut inside long run")
        else:
            if L == B - 1:
                got.add("len B-1")
            if len(blocks) > 1 and len([c for c in ch if s <= c[0] < e]) == 1:
                got.add("last block one chunk")
    if len(blocks) == 1 and len(data) <= 900_000:
        st = block_stats(rle1(data))
        got.add("nmtf %d" % st["nmtf"])
        if st.get("retries"):
            got.add("heap retry")
        if st.get("ties"):
            got.add("heap ties")
    for s, e in blocks:
        r = rle1(data[s:e])
        if len(r) > 200_000:
            continue
        _, _, size = bwt(r)
        if size > 1:
            period = len(r) // size
            if period <= 8:
                got.add("period short")
            if period >= len(r) // 3:
                got.add("period near n")
            if r != data[s:e]:
                got.add("period from rle1")
    return got


def reference(data, level):
    """What every path of the libbz2 mode must produce."""
    return bz2.compress(data, level)
