"""bz2b200_recover without a GPU: bad arguments are argument errors, the symbol is bound, and the recovery tests' libbz2
oracle (tests/test_recover_gpu.py) agrees with bzip2recover + bzip2 -t where the system has them."""
import bz2
import ctypes as C
import shutil

import numpy as np
import pytest

import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus
from test_recover_gpu import bzip2recover_pieces, flip, libbz2_block, magics


@pytest.fixture(scope="module")
def lib():
    from bzip2_rust_b200 import build
    build.build()
    return bz.load_library()


def test_null_and_empty_arguments_are_argument_errors(lib):
    s = np.frombuffer(bz2.compress(b"hello world\n" * 100), dtype=np.uint8)
    ents = (bz.RecEntry * 4)()
    nent, total = C.c_uint32(7), C.c_uint64(7)
    p = s.ctypes.data
    assert lib.bz2b200_recover(None, p, s.size, bz.SINK(), None, ents, 4, C.byref(nent), C.byref(total)) == bz.E_ARG
    h = C.c_void_p(1)        # never dereferenced: every argument check runs before the context is used
    assert lib.bz2b200_recover(h, None, s.size, bz.SINK(), None, ents, 4, C.byref(nent), C.byref(total)) == bz.E_ARG
    assert lib.bz2b200_recover(h, p, 0, bz.SINK(), None, ents, 4, C.byref(nent), C.byref(total)) == bz.E_ARG
    assert lib.bz2b200_recover(h, p, s.size, bz.SINK(), None, None, 4, C.byref(nent), C.byref(total)) == bz.E_ARG
    assert lib.bz2b200_recover(h, p, s.size, bz.SINK(), None, ents, 4, None, C.byref(total)) == bz.E_ARG
    assert lib.bz2b200_recover(h, p, s.size, bz.SINK(), None, ents, 4, C.byref(nent), None) == bz.E_ARG


def test_recover_is_bound(lib):
    assert "bz2b200_recover" in bz.EXPORTS and hasattr(lib, "bz2b200_recover")
    assert C.sizeof(bz.RecEntry) == 40
    assert callable(bz.Engine.recover)


def _oracle_pieces(d):
    """Intact blocks the oracle predicts when no magic is damaged: the bits from each block magic to the next magic,
    wrapped and decoded by libbz2."""
    m = magics(d)
    out = []
    for i, (b, foot) in enumerate(m):
        if foot:
            continue
        e = m[i + 1][0] if i + 1 < len(m) else len(d) * 8
        got = libbz2_block(d, b, e)
        if got is not None:
            out.append(got)
    return out


@pytest.mark.skipif(not (shutil.which("bzip2recover") and shutil.which("bzip2")), reason="no bzip2recover / bzip2")
def test_oracle_agrees_with_bzip2recover():
    data = b"".join(corpus.text(300_000, 50 + i).tobytes() + corpus.random_bytes(100_000, 60 + i).tobytes()
                    for i in range(4))
    s = bz2.compress(data, 1)
    blocks = [b for b, foot in magics(s) if not foot]
    assert len(blocks) > 10
    cases = [flip(s, blocks[3] + 2000), flip(flip(s, blocks[0] + 48 + 9), blocks[7] + 5000),
             s[:(blocks[5] + 3000) // 8] + s[(blocks[5] + 3000) // 8 + 1:]]
    for d in cases:
        assert _oracle_pieces(d) == bzip2recover_pieces(d)
