"""bz2b200_dstream_* without a GPU: NULL handles are argument errors, not crashes, and the CLI decodes through the
streaming decoder only."""
import ctypes as C
import os

import pytest

import bzip2_rust_b200 as bz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from bzip2_rust_b200 import build
    build.build()
    return bz.load_library()


def test_null_handles_are_argument_errors(lib):
    h = C.c_void_p()
    assert lib.bz2b200_dstream_open(None, bz.SINK(), None, C.byref(h)) == bz.E_ARG
    assert lib.bz2b200_dstream_open(None, bz.SINK(lambda u, d, n: 0), None, None) == bz.E_ARG
    assert lib.bz2b200_dstream_write(None, None, 0) == bz.E_ARG
    assert lib.bz2b200_dstream_write(None, b"BZh9", 4) == bz.E_ARG
    assert lib.bz2b200_dstream_close(None, None, None) == bz.E_ARG
    ti, to = C.c_uint64(7), C.c_uint64(7)
    assert lib.bz2b200_dstream_close(None, C.byref(ti), C.byref(to)) == bz.E_ARG


def test_dstream_is_bound(lib):
    for sym in ("bz2b200_dstream_open", "bz2b200_dstream_write", "bz2b200_dstream_close"):
        assert sym in bz.EXPORTS and hasattr(lib, sym)
    assert callable(bz.DStream)


def test_cli_has_no_whole_file_decode():
    """-d and -t read the archive in pieces into a DStream; nothing in the CLI decodes a whole file in one call."""
    src = open(os.path.join(ROOT, "tools", "bz2b200_cli.py")).read()
    assert "DStream(" in src and ".decompress(" not in src
