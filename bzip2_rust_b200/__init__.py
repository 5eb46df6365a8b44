"""bzip2_rust_b200 -- B200-native bzip2 compression engine (host-side mirror of the reference API).

Python is only the test/bench harness language here.  The product is ``libbz2b200.so``
(hand-written CUDA for sm_100a behind the C ABI in ``include/bz2b200.h``); this module binds
that ABI with ctypes and mirrors the reference's function names for the compression path:

    compress_block(block, block_crc) -> (bytes, padding)     compress_block.rs:24
    bwt_encode(block) -> (key, bwt)                           bwt_sort.rs:27
    rle2_mtf_encode(bwt) -> (symbols, freq, symbol_map)       rle2_mtf.rs:23
    huf_encode(symbols, freq, symbol_map) -> (bytes, nbits)   huffman.rs:79
    compress(data, level) / decompress(data)                  compress.rs:40 / decompress.rs:38

There is no CPU fallback: importing works anywhere, but every operation raises if the CUDA
library is missing or no GPU is usable.  Nothing in here imports ``oracle/``.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libbz2b200.so")

OK, E_ARG, E_CAP, E_CUDA, E_NOMEM, E_FORMAT, E_CRC = 0, -1, -2, -3, -4, -5, -6
MAX_BLOCK = 900000
LIBBZ2 = 0x100        # BZ2B200_LIBBZ2: OR into a level for libbz2 1.0.8's exact bytes instead of the reference's


def _lvl(level, libbz2):
    """The `level` argument of the C ABI: libbz2=True selects libbz2-identical output (BZ2B200_LIBBZ2)."""
    return int(level) | LIBBZ2 if libbz2 else level

_ERRNAMES = {E_ARG: "bad argument", E_CAP: "output buffer too small", E_CUDA: "CUDA error",
             E_NOMEM: "out of memory", E_FORMAT: "malformed stream", E_CRC: "CRC mismatch"}

# every symbol include/bz2b200.h declares
EXPORTS = [
    "bz2b200_create", "bz2b200_destroy", "bz2b200_trim", "bz2b200_last_error", "bz2b200_version", "bz2b200_launch_count",
    "bz2b200_compress_blocks", "bz2b200_compress_stream", "bz2b200_compress_stream_dev",
    "bz2b200_compress_bound", "bz2b200_stream_plan", "bz2b200_compress_range", "bz2b200_merge_streams",
    "bz2b200_crc32", "bz2b200_rle1_split", "bz2b200_bwt_encode", "bz2b200_bwt_encode_batch",
    "bz2b200_mtf_rle2", "bz2b200_huffman", "bz2b200_bwt_decode", "bz2b200_decompress_stream",
    "bz2b200_set_timing", "bz2b200_get_timing", "bz2b200_get_bwt_stats", "bz2b200_kernel_stats",
    "bz2b200_reset_kernel_stats", "bz2b200_stream_plan_dev", "bz2b200_compress_range_dev",
    "bz2b200_shard_plan_dev", "bz2b200_shard_compress_dev", "bz2b200_shift_bits_dev", "bz2b200_shard_scan_dev",
    "bz2b200_create_multi", "bz2b200_destroy_multi", "bz2b200_last_error_multi", "bz2b200_multi_devices",
    "bz2b200_multi_context", "bz2b200_compress_stream_multi", "bz2b200_decompress_stream_multi", "bz2b200_multi_stats",
    "bz2b200_zstream_open", "bz2b200_zstream_write", "bz2b200_zstream_close",
    "bz2b200_dstream_open", "bz2b200_dstream_write", "bz2b200_dstream_close", "bz2b200_recover",
    "bz2b200_rstream_open", "bz2b200_rstream_write", "bz2b200_rstream_close",
]


class Bz2B200Error(RuntimeError):
    def __init__(self, rc, detail=""):
        self.rc = rc
        RuntimeError.__init__(self, "bz2b200: %s (%d) %s" % (_ERRNAMES.get(rc, "error"), rc, detail))


_lib = None
SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)     # bz2b200_sink
REC_FOOTER, REC_NO_MAGIC = 1, 2


class RecEntry(C.Structure):
    """bz2b200_rec_entry: one block or footer found by bz2b200_recover."""
    _fields_ = [("bit", C.c_uint64), ("end_bit", C.c_uint64), ("out_off", C.c_uint64), ("out_len", C.c_uint32),
                ("crc", C.c_uint32), ("status", C.c_int32), ("flags", C.c_uint32)]

    def __repr__(self):
        return "RecEntry(bit=%d, end_bit=%d, out_off=%d, out_len=%d, crc=%#010x, status=%d, flags=%d)" % (
            self.bit, self.end_bit, self.out_off, self.out_len, self.crc, self.status, self.flags)


REC_REPORT = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(RecEntry), C.c_uint32)   # bz2b200_rec_report


def load_library():
    """Loads libbz2b200.so.  Raises (loudly) when the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("BZ2B200_LIB", SO_PATH)               # A/B builds of the same CUDA library (tools/ab_build.sh)
    if not os.path.exists(path):
        raise ImportError("libbz2b200.so is missing: run `python -m bzip2_rust_b200.build` "
                          "(there is no CPU fallback)")
    L = C.CDLL(path)
    vp, u8p, u32p, u64p, szp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)
    L.bz2b200_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.bz2b200_destroy.argtypes = [vp]
    L.bz2b200_destroy.restype = None
    L.bz2b200_trim.argtypes = [vp]
    L.bz2b200_last_error.argtypes = [vp]
    L.bz2b200_last_error.restype = C.c_char_p
    L.bz2b200_version.restype = C.c_char_p
    L.bz2b200_launch_count.argtypes = [vp]
    L.bz2b200_launch_count.restype = C.c_uint64
    L.bz2b200_compress_blocks.argtypes = [vp, C.c_int, vp, u32p, u32p, vp, vp, u64p]
    L.bz2b200_compress_stream.argtypes = [vp, u8p, C.c_size_t, C.c_int, u8p, C.c_size_t, szp]
    L.bz2b200_compress_stream_dev.argtypes = [vp, u8p, C.c_size_t, C.c_int, u8p, C.c_size_t, szp]
    L.bz2b200_compress_bound.argtypes = [C.c_size_t]
    L.bz2b200_compress_bound.restype = C.c_size_t
    L.bz2b200_stream_plan.argtypes = [vp, u8p, C.c_size_t, C.c_int, u64p, C.c_uint32, C.POINTER(C.c_uint32)]
    L.bz2b200_compress_range.argtypes = [vp, u8p, C.c_size_t, C.c_int, u64p, C.c_uint32, C.c_uint32, C.c_uint32,
                                         u8p, C.c_size_t, C.POINTER(C.c_uint64), u32p]
    L.bz2b200_stream_plan_dev.argtypes = L.bz2b200_stream_plan.argtypes
    L.bz2b200_compress_range_dev.argtypes = L.bz2b200_compress_range.argtypes
    L.bz2b200_shard_plan_dev.argtypes = [vp, u8p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int, C.c_size_t, C.c_size_t,
                                         szp, C.POINTER(C.c_uint32)]
    L.bz2b200_shard_scan_dev.argtypes = [vp, u8p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int]
    L.bz2b200_shard_compress_dev.argtypes = [vp, u8p, C.c_size_t, C.POINTER(C.c_uint64), u32p]
    L.bz2b200_shift_bits_dev.argtypes = [vp, u8p, C.c_uint64, C.c_int, u8p]
    L.bz2b200_merge_streams.argtypes = [C.c_int, C.c_int, vp, u64p, vp, u32p, u8p, C.c_size_t, szp]
    L.bz2b200_crc32.argtypes = [vp, u8p, C.c_size_t, C.POINTER(C.c_uint32)]
    L.bz2b200_rle1_split.argtypes = [vp, u8p, C.c_size_t, C.c_int, u8p, C.c_size_t, u64p, u64p, u32p,
                                     C.c_uint32, C.POINTER(C.c_uint32)]
    L.bz2b200_bwt_encode.argtypes = [vp, u8p, C.c_uint32, u8p, C.POINTER(C.c_uint32)]
    L.bz2b200_bwt_encode_batch.argtypes = [vp, C.c_int, vp, u32p, vp, u32p]
    L.bz2b200_mtf_rle2.argtypes = [vp, u8p, C.c_uint32, vp, C.POINTER(C.c_uint32), u32p, vp, C.POINTER(C.c_int)]
    L.bz2b200_huffman.argtypes = [vp, vp, C.c_uint32, u32p, vp, C.c_int, u8p, C.c_size_t, C.POINTER(C.c_uint64),
                                  u8p, u8p, C.POINTER(C.c_int)]
    L.bz2b200_bwt_decode.argtypes = [vp, C.c_uint32, u8p, C.c_uint32, u8p]
    L.bz2b200_decompress_stream.argtypes = [vp, u8p, C.c_size_t, u8p, C.c_size_t, szp]
    L.bz2b200_set_timing.argtypes = [vp, C.c_int]
    L.bz2b200_set_timing.restype = None
    L.bz2b200_get_timing.argtypes = [vp, C.POINTER(C.c_float * 8)]
    L.bz2b200_get_bwt_stats.argtypes = [vp, C.POINTER(C.c_uint64 * 8)]
    L.bz2b200_kernel_stats.argtypes = [vp, C.c_int, C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64),
                                       C.POINTER(C.c_uint64)]
    L.bz2b200_reset_kernel_stats.argtypes = [vp]
    L.bz2b200_reset_kernel_stats.restype = None
    L.bz2b200_create_multi.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.bz2b200_destroy_multi.argtypes = [vp]
    L.bz2b200_destroy_multi.restype = None
    L.bz2b200_last_error_multi.argtypes = [vp]
    L.bz2b200_last_error_multi.restype = C.c_char_p
    L.bz2b200_multi_devices.argtypes = [vp]
    L.bz2b200_multi_context.argtypes = [vp, C.c_int]
    L.bz2b200_multi_context.restype = vp
    L.bz2b200_compress_stream_multi.argtypes = [vp, u8p, C.c_size_t, C.c_int, u8p, C.c_size_t, szp]
    L.bz2b200_decompress_stream_multi.argtypes = [vp, u8p, C.c_size_t, u8p, C.c_size_t, szp]
    L.bz2b200_multi_stats.argtypes = [vp, C.POINTER(C.c_uint64 * 8)]
    L.bz2b200_zstream_open.argtypes = [vp, C.c_int, SINK, vp, C.POINTER(vp)]
    L.bz2b200_zstream_write.argtypes = [vp, u8p, C.c_size_t]
    L.bz2b200_zstream_close.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bz2b200_dstream_open.argtypes = [vp, SINK, vp, C.POINTER(vp)]
    L.bz2b200_dstream_write.argtypes = [vp, u8p, C.c_size_t]
    L.bz2b200_dstream_close.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.bz2b200_recover.argtypes = [vp, u8p, C.c_size_t, SINK, vp, C.POINTER(RecEntry), C.c_uint32,
                                  C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
    L.bz2b200_rstream_open.argtypes = [vp, SINK, REC_REPORT, vp, C.POINTER(vp)]
    L.bz2b200_rstream_write.argtypes = [vp, u8p, C.c_size_t]
    L.bz2b200_rstream_close.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    _lib = L
    return L


def _np_u8(data):
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data, dtype=np.uint8)
    return np.frombuffer(bytes(data), dtype=np.uint8)


class Engine:
    """One GPU context (``bz2b200_ctx``)."""

    def __init__(self, device=-1):
        self._L = load_library()
        h = C.c_void_p()
        rc = self._L.bz2b200_create(device, C.byref(h))
        if rc != OK:
            raise Bz2B200Error(rc, "bz2b200_create: no usable CUDA device (there is no CPU fallback)")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.bz2b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != OK:
            raise Bz2B200Error(rc, self._L.bz2b200_last_error(self._h).decode())

    def trim(self):
        """Frees the device workspaces (grow-only otherwise)."""
        self._chk(self._L.bz2b200_trim(self._h))

    @property
    def launches(self):
        return int(self._L.bz2b200_launch_count(self._h))

    # ---- stage seams ------------------------------------------------------------------
    def bwt_encode(self, block):
        """bwt_encode (bwt_sort.rs:27) -> (key, bwt bytes)."""
        (r,) = self.bwt_encode_batch([block])
        return r

    def bwt_encode_batch(self, blocks):
        arrs = [_np_u8(b) for b in blocks]
        n = len(arrs)
        if n == 0:
            return []
        lens = np.array([a.size for a in arrs], dtype=np.uint32)
        outs = [np.empty(a.size, dtype=np.uint8) for a in arrs]
        inp = (C.c_void_p * n)(*[a.ctypes.data for a in arrs])
        outp = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
        keys = np.zeros(n, dtype=np.uint32)
        self._chk(self._L.bz2b200_bwt_encode_batch(self._h, n, inp, lens.ctypes.data, outp, keys.ctypes.data))
        return [(int(keys[i]), outs[i].tobytes()) for i in range(n)]

    def bwt_stats(self):
        st = (C.c_uint64 * 8)()
        self._L.bz2b200_get_bwt_stats(self._h, C.byref(st))
        return dict(blocks=st[0], rounds=st[2], list_sum=st[3], ref_sais_blocks=st[4], ref_sais_blocks_total=st[5],
                    blocks_total=st[6], big_sum=st[7])

    def rle2_mtf_encode(self, bwt):
        """rle2_mtf_encode (rle2_mtf.rs:23) -> (symbols u16[m] incl. EOB, freq u32[256], symbol map u16[<=17])."""
        a = _np_u8(bwt)
        sym = np.zeros(a.size + 1, dtype=np.uint16)
        freq = np.zeros(256, dtype=np.uint32)
        smap = np.zeros(17, dtype=np.uint16)
        m, nmap = C.c_uint32(), C.c_int()
        self._chk(self._L.bz2b200_mtf_rle2(self._h, a.ctypes.data, a.size, sym.ctypes.data, C.byref(m),
                                           freq.ctypes.data, smap.ctypes.data, C.byref(nmap)))
        return sym[:m.value].copy(), freq, smap[:nmap.value].copy()

    def huf_encode(self, sym, freq, symmap):
        """huf_encode (huffman.rs:79) on an empty BitPacker -> (bytes, nbits, info)."""
        sym = np.ascontiguousarray(sym, dtype=np.uint16)
        freq = np.ascontiguousarray(freq, dtype=np.uint32)
        symmap = np.ascontiguousarray(symmap, dtype=np.uint16)
        m = sym.size
        cap = m * 3 + 8192
        out = np.zeros(cap, dtype=np.uint8)
        lengths = np.zeros((6, 258), dtype=np.uint8)
        G = (m + 49) // 50
        sel = np.zeros(max(G, 1), dtype=np.uint8)
        bits, nt = C.c_uint64(), C.c_int()
        self._chk(self._L.bz2b200_huffman(self._h, sym.ctypes.data, m, freq.ctypes.data, symmap.ctypes.data,
                                          symmap.size, out.ctypes.data, cap, C.byref(bits), lengths.ctypes.data,
                                          sel.ctypes.data, C.byref(nt)))
        nb = (bits.value + 7) // 8
        return out[:nb].tobytes(), int(bits.value), dict(table_count=nt.value, selectors=sel[:G].tobytes(),
                                                         lengths=lengths)

    def compress_blocks(self, blocks, crcs):
        """Batched compress_block (compress_block.rs:24) -> list of (bytes, padding)."""
        arrs = [_np_u8(b) for b in blocks]
        n = len(arrs)
        if n == 0:
            return []
        lens = np.array([a.size for a in arrs], dtype=np.uint32)
        crc = np.array(crcs, dtype=np.uint32)
        caps = np.array([a.size + a.size // 2 + 4096 for a in arrs], dtype=np.uint64)
        outs = [np.zeros(int(c), dtype=np.uint8) for c in caps]
        inp = (C.c_void_p * n)(*[a.ctypes.data for a in arrs])
        outp = (C.c_void_p * n)(*[o.ctypes.data for o in outs])
        bits = np.zeros(n, dtype=np.uint64)
        self._chk(self._L.bz2b200_compress_blocks(self._h, n, inp, lens.ctypes.data, crc.ctypes.data, outp,
                                                  caps.ctypes.data, bits.ctypes.data))
        res = []
        for i in range(n):
            b = int(bits[i])
            res.append((outs[i][:(b + 7) // 8].tobytes(), (8 - b % 8) % 8))
        return res

    def compress_block(self, block, block_crc):
        return self.compress_blocks([block], [block_crc])[0]

    def crc32(self, data):
        a = _np_u8(data)
        c = C.c_uint32()
        self._chk(self._L.bz2b200_crc32(self._h, a.ctypes.data, a.size, C.byref(c)))
        return c.value

    def rle1_split(self, data, level=9, libbz2=False):
        """RLE1Block iterator (rle1.rs:245-264) for the whole input -> list of (crc, block bytes, in_start, in_end)."""
        a = _np_u8(data)
        cap_blocks = (a.size * 5 // 4) // (level * 100000 - 19 - 8) + 4      # RLE1 can turn 4 input bytes into 5
        cap = a.size + a.size // 4 + 1024
        out = np.zeros(cap, dtype=np.uint8)
        roff = np.zeros(cap_blocks + 1, dtype=np.uint64)
        ioff = np.zeros(cap_blocks + 1, dtype=np.uint64)
        crc = np.zeros(cap_blocks, dtype=np.uint32)
        nb = C.c_uint32()
        self._chk(self._L.bz2b200_rle1_split(self._h, a.ctypes.data, a.size, _lvl(level, libbz2), out.ctypes.data, cap,
                                             roff.ctypes.data, ioff.ctypes.data, crc.ctypes.data, cap_blocks,
                                             C.byref(nb)))
        return [(int(crc[i]), out[int(roff[i]):int(roff[i + 1])].tobytes(), int(ioff[i]), int(ioff[i + 1]))
                for i in range(nb.value)]

    # ---- whole stream ----------------------------------------------------------------
    def compress(self, data, level=9, libbz2=False):
        """compress (compress.rs:40): returns the .bz2 stream for `data` at block size `level`.  libbz2=True: the
        bytes bzip2 1.0.8 writes (`bz2.compress(data, level)`) instead of the reference's."""
        a = _np_u8(data)
        cap = int(self._L.bz2b200_compress_bound(a.size))
        out = np.empty(cap, dtype=np.uint8)
        n = C.c_size_t()
        self._chk(self._L.bz2b200_compress_stream(self._h, a.ctypes.data, a.size, _lvl(level, libbz2), out.ctypes.data, cap,
                                                  C.byref(n)))
        return out[:n.value].tobytes()

    def compress_dev(self, d_in_ptr, n, level, d_out_ptr, out_cap, libbz2=False):
        """Device-resident variant: raw device pointers (e.g. torch tensor .data_ptr()). Returns length."""
        ln = C.c_size_t()
        self._chk(self._L.bz2b200_compress_stream_dev(self._h, d_in_ptr, n, _lvl(level, libbz2), d_out_ptr, out_cap,
                                                      C.byref(ln)))
        return ln.value

    # ---- sharding helpers (SURVEY 8e) --------------------------------------------------
    def stream_plan(self, data, level=9, dev_ptr=None, libbz2=False):
        """Block start offsets of the whole stream (n+1 entries, last = len).  `dev_ptr` = the data already on
        this GPU (raw device pointer), otherwise `data` is uploaded window by window."""
        n = data if dev_ptr is not None else _np_u8(data).size
        cap = (n * 5 // 4) // (level * 100000 - 19 - 8) + 8
        starts = np.zeros(cap + 1, dtype=np.uint64)
        nb = C.c_uint32()
        if dev_ptr is not None:
            self._chk(self._L.bz2b200_stream_plan_dev(self._h, dev_ptr, n, _lvl(level, libbz2), starts.ctypes.data, cap,
                                                      C.byref(nb)))
        else:
            a = _np_u8(data)
            self._chk(self._L.bz2b200_stream_plan(self._h, a.ctypes.data, a.size, _lvl(level, libbz2), starts.ctypes.data, cap,
                                                  C.byref(nb)))
        return starts[:nb.value + 1].copy()

    def compress_range(self, data, level, starts, first, count, dev_ptr=None, dev_out=None, dev_out_cap=0,
                       libbz2=False):
        """Blocks [first, first+count) of the stream as a bit string -> (bytes | None, nbits, crcs)."""
        nblocks = len(starts) - 1
        level = _lvl(level, libbz2)
        starts = np.ascontiguousarray(starts, dtype=np.uint64)
        crcs = np.zeros(max(count, 1), dtype=np.uint32)
        bits = C.c_uint64()
        if dev_ptr is not None:
            self._chk(self._L.bz2b200_compress_range_dev(self._h, dev_ptr, data, level, starts.ctypes.data, nblocks,
                                                         first, count, dev_out, dev_out_cap, C.byref(bits),
                                                         crcs.ctypes.data))
            return None, int(bits.value), crcs[:count].copy()
        a = _np_u8(data)
        span = int(starts[first + count] - starts[first])
        cap = int(self._L.bz2b200_compress_bound(span))
        out = np.empty(cap, dtype=np.uint8)
        self._chk(self._L.bz2b200_compress_range(self._h, a.ctypes.data, a.size, level, starts.ctypes.data, nblocks,
                                                 first, count, out.ctypes.data, cap, C.byref(bits), crcs.ctypes.data))
        return out[:(bits.value + 7) // 8].tobytes(), int(bits.value), crcs[:count].copy()

    def shard_scan(self, d_win_ptr, win_lo, win_len, n_total, level, libbz2=False):
        """Per-position scans of a window (needs no hand-off; a following shard_plan on the same window reuses them)."""
        self._chk(self._L.bz2b200_shard_scan_dev(self._h, d_win_ptr, win_lo, win_len, n_total, _lvl(level, libbz2)))

    def shard_plan(self, d_win_ptr, win_lo, win_len, n_total, level, start, stop_at, libbz2=False):
        """Plans the blocks starting in [start, stop_at) -> (next_start, nblocks); raises E_CAP if the window is short."""
        nxt, nb = C.c_size_t(), C.c_uint32()
        self._chk(self._L.bz2b200_shard_plan_dev(self._h, d_win_ptr, win_lo, win_len, n_total, _lvl(level, libbz2),
                                                 start, stop_at,
                                                 C.byref(nxt), C.byref(nb)))
        return nxt.value, nb.value

    def shard_compress(self, nblocks, d_out_ptr, out_cap):
        """Compresses the blocks of the preceding shard_plan -> (nbits, crcs)."""
        crcs = np.zeros(max(nblocks, 1), dtype=np.uint32)
        bits = C.c_uint64()
        self._chk(self._L.bz2b200_shard_compress_dev(self._h, d_out_ptr, out_cap, C.byref(bits), crcs.ctypes.data))
        return int(bits.value), crcs[:nblocks].copy()

    def shift_bits(self, d_src_ptr, nbits, phase, d_dst_ptr):
        self._chk(self._L.bz2b200_shift_bits_dev(self._h, d_src_ptr, nbits, phase, d_dst_ptr))

    def bwt_decode(self, key, bwt):
        a = _np_u8(bwt)
        out = np.empty(a.size, dtype=np.uint8)
        self._chk(self._L.bz2b200_bwt_decode(self._h, key, a.ctypes.data, a.size, out.ctypes.data))
        return out.tobytes()

    def decompress(self, data, max_out=None):
        a = _np_u8(data)
        cap = max_out or max(a.size * 64, 1 << 20)
        while True:
            out = np.empty(cap, dtype=np.uint8)
            n = C.c_size_t()
            rc = self._L.bz2b200_decompress_stream(self._h, a.ctypes.data, a.size, out.ctypes.data, cap,
                                                   C.byref(n))
            if rc == E_CAP and max_out is None and cap < (1 << 34):
                cap *= 4
                continue
            self._chk(rc)
            return out[:n.value].tobytes()

    def recover(self, data, out=None):
        """Block recovery (bz2b200_recover): decodes every intact block of a possibly damaged .bz2 input.  The intact
        bytes go to `out.write` in input order (out=None: a report-only scan, nothing is downloaded).  Returns
        (total_out, [RecEntry, ...]): one entry per block candidate and footer, see include/bz2b200.h."""
        a = _np_u8(data)
        err = []
        cb = SINK()                                             # a NULL sink: report only
        if out is not None:
            def sink(_user, p, n):
                try:
                    out.write(C.string_at(p, n))
                    return 0
                except BaseException as e:                      # an exception must not unwind through the C library
                    err.append(e)
                    return 1
            cb = SINK(sink)
        cap = a.size // 20_000 + 256                # room for small blocks; the bound that always suffices is ~6x the input
        ents = (RecEntry * cap)()
        nent, total = C.c_uint32(), C.c_uint64()
        rc = self._L.bz2b200_recover(self._h, a.ctypes.data, a.size, cb, None, ents, cap, C.byref(nent), C.byref(total))
        if err:
            raise err[0]
        if rc == E_CAP:                             # the sink has every byte; a report-only scan fetches all entries
            cap = nent.value
            ents = (RecEntry * cap)()
            rc = self._L.bz2b200_recover(self._h, a.ctypes.data, a.size, SINK(), None, ents, cap, C.byref(nent),
                                         C.byref(C.c_uint64()))
        self._chk(rc)
        return total.value, list(ents[:nent.value])

    def set_timing(self, level=1):
        """0 = off, 1 = per-stage events, 2 = also CUDA events around every kernel launch."""
        self._L.bz2b200_set_timing(self._h, int(level))

    def kernel_stats(self):
        """-> {kernel name: (ms, launches, algorithmic bytes)} accumulated since the last reset."""
        out = {}
        i = 0
        while True:
            name = C.create_string_buffer(64)
            ms, ln, by = C.c_double(), C.c_uint64(), C.c_uint64()
            if self._L.bz2b200_kernel_stats(self._h, i, name, C.byref(ms), C.byref(ln), C.byref(by)) != OK:
                break
            if ln.value:
                out[name.value.decode()] = (ms.value, ln.value, by.value)
            i += 1
        return out

    def reset_kernel_stats(self):
        self._L.bz2b200_reset_kernel_stats(self._h)

    def timing(self):
        ms = (C.c_float * 8)()
        self._L.bz2b200_get_timing(self._h, C.byref(ms))
        names = ["rle1_crc_split", "bwt", "mtf_rle2", "huffman", "bitpack", "total"]
        return {k: float(ms[i]) for i, k in enumerate(names)}


class ZStream:
    """Streaming compression (bz2b200_zstream_*): write() input in pieces; finished .bz2 bytes go to `out.write`.

        with ZStream(engine, fileobj, level=9) as z:
            for piece in pieces: z.write(piece)

    libbz2=True: the stream bzip2 1.0.8 writes for the concatenated input.
    """

    def __init__(self, engine, out, level=9, libbz2=False):
        self._L = engine._L
        self._eng = engine
        self._out = out
        self._err = None

        def sink(_user, data, n):
            try:
                self._out.write(C.string_at(data, n))
                return 0
            except Exception as e:          # an exception must not unwind through the C library
                self._err = e
                return 1

        self._cb = SINK(sink)               # keep the callback object alive as long as the stream
        h = C.c_void_p()
        rc = self._L.bz2b200_zstream_open(engine._h, _lvl(level, libbz2), self._cb, None, C.byref(h))
        if rc != OK:
            if self._err is not None:
                raise self._err             # the sink failed on the stream header
            raise Bz2B200Error(rc, "bz2b200_zstream_open")
        self._h = h
        self.total_in = self.total_out = 0

    def write(self, data):
        a = _np_u8(data)
        rc = self._L.bz2b200_zstream_write(self._h, a.ctypes.data, a.size)
        if rc != OK:
            raise Bz2B200Error(rc, self._L.bz2b200_last_error(self._eng._h).decode())

    def close(self):
        if self._h is None:
            return
        ti, to = C.c_uint64(), C.c_uint64()
        rc = self._L.bz2b200_zstream_close(self._h, C.byref(ti), C.byref(to))
        self._h = None
        self.total_in, self.total_out = ti.value, to.value
        if self._err is not None:
            raise self._err
        if rc != OK:
            raise Bz2B200Error(rc, self._L.bz2b200_last_error(self._eng._h).decode())

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


class DStream:
    """Streaming decompression (bz2b200_dstream_*): write() .bz2 input in pieces; checked output goes to `out.write`
    (called on a library thread, in order).  out=None is test mode (bzip2 -t): every check runs, nothing is downloaded,
    total_out still counts the decoded bytes.

        with DStream(engine, fileobj) as d:
            for piece in pieces: d.write(piece)
    """

    def __init__(self, engine, out=None):
        self._L = engine._L
        self._eng = engine
        self._out = out
        self._err = None
        self._h = None
        self.total_in = self.total_out = 0
        self._cb = SINK()                   # a NULL sink: test mode
        if out is not None:
            def sink(_user, data, n):
                try:
                    self._out.write(C.string_at(data, n))
                    return 0
                except BaseException as e:  # an exception must not unwind through the C library
                    self._err = e
                    return 1
            self._cb = SINK(sink)           # keep the callback object alive as long as the stream
        h = C.c_void_p()
        rc = self._L.bz2b200_dstream_open(engine._h, self._cb, None, C.byref(h))
        if rc != OK:
            raise Bz2B200Error(rc, "bz2b200_dstream_open")
        self._h = h

    def _raise(self, rc):
        if self._err is not None:
            raise self._err
        raise Bz2B200Error(rc, self._L.bz2b200_last_error(self._eng._h).decode())

    def write(self, data):
        a = _np_u8(data)
        rc = self._L.bz2b200_dstream_write(self._h, a.ctypes.data, a.size)
        if rc != OK:
            self._raise(rc)

    def close(self):
        if self._h is None:
            return
        ti, to = C.c_uint64(), C.c_uint64()
        rc = self._L.bz2b200_dstream_close(self._h, C.byref(ti), C.byref(to))
        self._h = None
        self.total_in, self.total_out = ti.value, to.value
        if self._err is not None or rc != OK:
            self._raise(rc)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


class RStream:
    """Streaming block recovery (bz2b200_rstream_*): write() a possibly damaged .bz2 input in pieces; the bytes of its
    intact blocks go to `out.write` (out=None: report only, nothing is downloaded), its entries (RecEntry, as
    Engine.recover lists them) to `on_entries(list)` or, when that is None, to `.entries`.  Both callbacks run on one
    library thread, in input order; a batch's entries come after its bytes.  close() sets total_in, total_out and nent.

        with RStream(engine, fileobj) as r:
            for piece in pieces: r.write(piece)
        r.entries
    """

    def __init__(self, engine, out=None, on_entries=None):
        self._L = engine._L
        self._eng = engine
        self._err = None
        self._h = None
        self.entries = []
        self.total_in = self.total_out = self.nent = 0
        self._cb = SINK()                   # a NULL sink: report only
        if out is not None:
            def sink(_user, data, n):
                try:
                    out.write(C.string_at(data, n))
                    return 0
                except BaseException as e:  # an exception must not unwind through the C library
                    self._err = self._err or e
                    return 1
            self._cb = SINK(sink)           # keep the callback objects alive as long as the stream
        take = on_entries if on_entries is not None else self.entries.extend

        def report(_user, p, n):
            try:
                arr = (RecEntry * n).from_buffer_copy(C.string_at(p, n * C.sizeof(RecEntry)))
                take(list(arr))
                return 0
            except BaseException as e:
                self._err = self._err or e
                return 1
        self._rep = REC_REPORT(report)
        h = C.c_void_p()
        rc = self._L.bz2b200_rstream_open(engine._h, self._cb, self._rep, None, C.byref(h))
        if rc != OK:
            raise Bz2B200Error(rc, "bz2b200_rstream_open")
        self._h = h

    def _raise(self, rc):
        if self._err is not None:
            raise self._err
        raise Bz2B200Error(rc, self._L.bz2b200_last_error(self._eng._h).decode())

    def write(self, data):
        a = _np_u8(data)
        rc = self._L.bz2b200_rstream_write(self._h, a.ctypes.data, a.size)
        if rc != OK:
            self._raise(rc)

    def close(self):
        if self._h is None:
            return
        ti, to, ne = C.c_uint64(), C.c_uint64(), C.c_uint64()
        rc = self._L.bz2b200_rstream_close(self._h, C.byref(ti), C.byref(to), C.byref(ne))
        self._h = None
        self.total_in, self.total_out, self.nent = ti.value, to.value, ne.value
        if self._err is not None or rc != OK:
            self._raise(rc)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


class MultiEngine:
    """compress (compress.rs:40-136) on several GPUs of this process: ``bz2b200_mctx``.  `devices` = list of CUDA
    device ids (an id may repeat: several ranks then share one GPU, which is how the single-GPU tests drive it)."""

    def __init__(self, devices):
        self._L = load_library()
        ids = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        rc = self._L.bz2b200_create_multi(len(devices), ids, C.byref(h))
        if rc != OK:
            raise Bz2B200Error(rc, "bz2b200_create_multi: no usable CUDA device (there is no CPU fallback)")
        self._h = h
        self.n = len(devices)

    def close(self):
        if getattr(self, "_h", None):
            self._L.bz2b200_destroy_multi(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def compress_into(self, in_ptr, n, level, out_ptr, out_cap):
        """Raw host pointers (page-locked for full overlap) -> compressed length."""
        ln = C.c_size_t()
        rc = self._L.bz2b200_compress_stream_multi(self._h, in_ptr, n, level, out_ptr, out_cap, C.byref(ln))
        if rc != OK:
            raise Bz2B200Error(rc, self._L.bz2b200_last_error_multi(self._h).decode())
        return ln.value

    def compress(self, data, level=9, libbz2=False):
        a = _np_u8(data)
        cap = int(self._L.bz2b200_compress_bound(a.size))
        out = np.empty(cap, dtype=np.uint8)
        n = self.compress_into(a.ctypes.data, a.size, _lvl(level, libbz2), out.ctypes.data, cap)
        return out[:n].tobytes()

    def decompress_into(self, in_ptr, n, out_ptr, out_cap):
        """decompress (decompress.rs:38) on the ranks: raw host pointers (page-locked for full overlap) -> length."""
        ln = C.c_size_t()
        rc = self._L.bz2b200_decompress_stream_multi(self._h, in_ptr, n, out_ptr, out_cap, C.byref(ln))
        if rc != OK:
            raise Bz2B200Error(rc, self._L.bz2b200_last_error_multi(self._h).decode())
        return ln.value

    def decompress(self, data, max_out=None):
        """The decompressed bytes of `data`; without `max_out`, a too-small first guess is retried once at the exact size
        the failed call reports."""
        a = _np_u8(data)
        cap = max_out if max_out is not None else max(a.size * 8, 1 << 20)
        out = np.empty(cap, dtype=np.uint8)
        ln = C.c_size_t()
        rc = self._L.bz2b200_decompress_stream_multi(self._h, a.ctypes.data, a.size, out.ctypes.data, cap, C.byref(ln))
        if rc == E_CAP and max_out is None:
            cap = ln.value
            out = np.empty(max(cap, 1), dtype=np.uint8)
            rc = self._L.bz2b200_decompress_stream_multi(self._h, a.ctypes.data, a.size, out.ctypes.data, cap,
                                                         C.byref(ln))
        if rc != OK:
            raise Bz2B200Error(rc, self._L.bz2b200_last_error_multi(self._h).decode())
        return out[:ln.value].tobytes()

    def stats(self):
        st = (C.c_uint64 * 8)()
        self._L.bz2b200_multi_stats(self._h, C.byref(st))
        return dict(h2d_bytes=int(st[0]), d2h_bytes=int(st[1]))

    def launches(self):
        return sum(int(self._L.bz2b200_launch_count(self._L.bz2b200_multi_context(self._h, r))) for r in range(self.n))


_default = None


def default_engine():
    global _default
    if _default is None:
        _default = Engine()
    return _default


def compress(data, level=9, libbz2=False):
    return default_engine().compress(data, level, libbz2=libbz2)


def decompress(data):
    return default_engine().decompress(data)


def compress_block(block, block_crc):
    return default_engine().compress_block(block, block_crc)


def bwt_encode(block):
    return default_engine().bwt_encode(block)


def rle2_mtf_encode(bwt):
    return default_engine().rle2_mtf_encode(bwt)


def merge_streams(level, parts, libbz2=False):
    """Host-side ordered merge (bitwriter.rs:77-132): parts = [(bytes, nbits, [block crcs])]."""
    level = _lvl(level, libbz2)
    L = load_library()
    n = len(parts)
    bufs = [np.frombuffer(p[0], dtype=np.uint8) for p in parts]
    crcs = [np.array(p[2], dtype=np.uint32) for p in parts]
    pp = (C.c_void_p * n)(*[b.ctypes.data for b in bufs])
    cp = (C.c_void_p * n)(*[c.ctypes.data for c in crcs])
    bits = np.array([p[1] for p in parts], dtype=np.uint64)
    nc = np.array([c.size for c in crcs], dtype=np.uint32)
    cap = sum(b.size for b in bufs) + 64
    out = np.empty(cap, dtype=np.uint8)
    ln = C.c_size_t()
    rc = L.bz2b200_merge_streams(level, n, pp, bits.ctypes.data, cp, nc.ctypes.data, out.ctypes.data, cap,
                                 C.byref(ln))
    if rc != OK:
        raise Bz2B200Error(rc)
    return out[:ln.value].tobytes()
