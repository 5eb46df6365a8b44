"""tests/bz2craft.py, the hand-built .bz2 writer, against libbz2 itself: every conformance case that is meant to decode
decodes under libbz2 to the writer's model output, and every case meant to fail is rejected by libbz2.  This keeps the
generator honest; test_decode_conformance_gpu.py then holds the GPU decoder to the same cases."""
import bz2

import numpy as np
import pytest

import bz2craft as bc


@pytest.mark.parametrize("name", list(bc.CASES))
def test_case_agrees_with_libbz2(name):
    data, want, code = bc.CASES[name]()
    got = bc.libbz2(data)
    if code == "ok":
        assert want is not None and got == want
    else:
        assert got is None


def test_crc_is_bzip2s():
    def slow(data):
        c = 0xFFFFFFFF
        for b in data:
            c ^= b << 24
            for _ in range(8):
                c = ((c << 1) ^ 0x04C11DB7) & 0xFFFFFFFF if c & 0x80000000 else (c << 1) & 0xFFFFFFFF
        return c ^ 0xFFFFFFFF
    for d in (b"", b"a", b"hello world", bytes(range(256)) * 3):
        assert bc.crc32(d) == slow(d)


def test_model_matches_a_real_encoder():
    """A text RLE1-coded and BWT'd as an encoder does it, then written field by field, decodes under libbz2 to the text."""
    data = bytes(np.random.default_rng(3).integers(97, 101, 3000, dtype=np.uint8))
    x = bytearray()                               # RLE1 as the encoder applies it
    i = 0
    while i < len(data):
        j = i
        while j < len(data) and j - i < 255 + 4 and data[j] == data[i]:
            j += 1
        run = j - i
        x += data[i:i + min(run, 4)]
        if run >= 4:
            x.append(run - 4)
        i = j
    L, key = bc.bwt(bytes(x))
    assert bc.ibwt(L, key) == bytes(x)
    s, want = bc.craft(bc.Block.from_bwt(L, key))
    assert want == data and bz2.decompress(s) == data == bz2.decompress(bz2.compress(data))


def test_writer_fields():
    """Bit phases land where asked; an empty second-level word of the symbol map, several streams and a stored CRC that
    differs from the data are written as given; trailing bytes follow the last footer."""
    L, key = bc.bwt(b"the writer's fields, one by one")
    for ph in (0, 1, 17, 31):
        b = bc.Block.from_bwt(L, key, phase=ph)
        s, want = bc.craft(b)
        assert bz2.decompress(s) == want
    s, want = bc.craft(bc.Block.from_bwt(L, key, extra_l1=(0, 15)))
    assert bz2.decompress(s) == want
    two = [bc.Stream([bc.Block.from_bwt(L, key)], level=1), bc.Stream([bc.Block.from_bwt(L, key)], level=9)]
    s, want = bc.craft(two, trailing=b"xyz")
    assert s.endswith(b"xyz") and bc.libbz2(s) is None and bc.libbz2(s[:-3]) == want == 2 * bc.ibwt(L, key)
    s, _ = bc.craft(bc.Block.from_bwt(L, key, crc=1234))
    assert bc.libbz2(s) is None
