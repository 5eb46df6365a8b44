"""bz2b200_rstream without a GPU: NULL handles and arguments are argument errors, and the binding is complete."""
import ctypes as C
import re
import os

import pytest

import bzip2_rust_b200 as bz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from bzip2_rust_b200 import build
    build.build()
    return bz.load_library()


def test_null_arguments_are_argument_errors(lib):
    h = C.c_void_p()
    assert lib.bz2b200_rstream_open(None, bz.SINK(), bz.REC_REPORT(), None, C.byref(h)) == bz.E_ARG
    ctx = C.c_void_p(1)      # never dereferenced: the argument checks run before the context is used
    assert lib.bz2b200_rstream_open(ctx, bz.SINK(), bz.REC_REPORT(), None, None) == bz.E_ARG
    buf = (C.c_uint8 * 4)()
    assert lib.bz2b200_rstream_write(None, buf, 4) == bz.E_ARG
    t = C.c_uint64()
    assert lib.bz2b200_rstream_close(None, C.byref(t), C.byref(t), C.byref(t)) == bz.E_ARG


def test_rstream_is_bound(lib):
    for name in ("bz2b200_rstream_open", "bz2b200_rstream_write", "bz2b200_rstream_close"):
        assert name in bz.EXPORTS and hasattr(lib, name)
    assert callable(bz.RStream.write) and callable(bz.RStream.close)
    assert bz.RStream.__enter__ and bz.RStream.__exit__


def test_window_bound_is_shared_with_the_dstream():
    """The rstream and the dstream read one look-ahead constant, and it exceeds the longest block span."""
    text = open(os.path.join(ROOT, "bzip2_rust_b200", "csrc", "pump.cuh")).read()
    m = re.search(r"constexpr size_t DEC_LOOK = (\d+)u << (\d+);", text)
    look = int(m.group(1)) << int(m.group(2))
    assert look * 8 > 20 * (bz.MAX_BLOCK + 64) + (1 << 19)
    for f in ("dstream.cu", "recover.cu"):
        src = open(os.path.join(ROOT, "bzip2_rust_b200", "csrc", f)).read()
        assert '#include "pump.cuh"' in src and "LOOK = " not in src
