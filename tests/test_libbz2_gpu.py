"""BZ2B200_LIBBZ2: with the flag ORed into the level, every path that produces a stream writes the bytes libbz2 1.0.8
writes -- the one-call host and device paths, the zstream, the multi context, and plan + range + merge.  The oracle is
bz2.compress itself (the libbz2 Python's bz2 module links).  Without the flag nothing changes (the existing suites)."""
import bz2
import ctypes as C
import io
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

import bzip2_rust_b200 as bz
import libbz2craft as lc
from bzip2_rust_b200 import corpus

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = [sys.executable, os.path.join(ROOT, "tools", "bz2b200_cli.py")]


def test_records_libbz2_version():
    print("BZ2_bzlibVersion() = %s" % lc.libbz2_version())


@pytest.mark.parametrize("name", [c[0] for c in lc.crafted()])
def test_crafted_input_at_its_level(engine, name):
    _, level, data, _ = next(c for c in lc.crafted() if c[0] == name)
    assert engine.compress(data, level, libbz2=True) == bz2.compress(data, level), name


def test_planner_inputs(engine):
    for name, level, data in lc.planner_inputs():
        assert engine.compress(data, level, libbz2=True) == bz2.compress(data, level), name


@pytest.mark.parametrize("level", range(1, 10))
def test_small_inputs_every_level(engine, level):
    for name, data in lc.small_inputs():
        assert engine.compress(data, level, libbz2=True) == bz2.compress(data, level), (name, level)


@pytest.mark.parametrize("name", [r[0] for r in lc.long_runs()])
def test_long_constant_runs(engine, name):
    """Every interior block of a run of one byte value is (c c c c 251)^k: a periodic block whose origin pointer is the
    row libbz2's fallbackSort leaves rotation 0 in, at every level."""
    _, level, data = next(r for r in lc.long_runs() if r[0] == name)
    assert len(lc.plan(data, level)) >= 3
    assert engine.compress(data, level, libbz2=True) == bz2.compress(data, level), name


def test_periodic_blocks_that_main_sort_finishes(engine):
    """The documented gap (tests/libbz2craft.py periodic_main_sort): the stream has the same length, decodes to the
    input, and differs from libbz2's only inside the block's origin pointer."""
    for name, level, data in lc.periodic_main_sort():
        got, want = engine.compress(data, level, libbz2=True), bz2.compress(data, level)
        assert len(got) == len(want) and bz2.decompress(got) == data, name
        diff = np.flatnonzero(np.frombuffer(got, np.uint8) != np.frombuffer(want, np.uint8))
        assert diff.size and diff.min() >= 14 and diff.max() <= 17, (name, diff[:16])


CORPUS = {
    "text": lambda n: corpus.text(n, 71),
    "mixed": lambda n: corpus.mixed(n, 72),
    "markov": lambda n: corpus.markov(n, 73),
    "random_bytes": lambda n: corpus.random_bytes(n, 74),
    "repetitive": lambda n: corpus.repetitive(n, 75),
}


@pytest.mark.parametrize("kind", sorted(CORPUS))
def test_corpus_sizes(engine, kind):
    for n in (0, 1, 4096, 1_000_000, 20_000_000):
        data = CORPUS[kind](n).tobytes() if n else b""
        for level in (1, 5, 9):
            assert engine.compress(data, level, libbz2=True) == bz2.compress(data, level), (kind, n, level)


@pytest.fixture(scope="module")
def data40():
    return np.concatenate([corpus.text(16_000_000, 81), corpus.repetitive(12_000_000, 82),
                           corpus.random_bytes(4_000_000, 83), corpus.markov(8_000_000, 84)])


@pytest.fixture(scope="module")
def want40(data40):
    return {lv: bz2.compress(data40.tobytes(), lv) for lv in (9, 2)}


_E2E_CHILD = r"""
import sys, bz2
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import numpy as np
import bzip2_rust_b200 as bz
data = np.fromfile(sys.argv[2], dtype=np.uint8)
eng = bz.Engine(0)
for lv in (9, 2):
    assert eng.compress(data, lv, libbz2=True) == open(sys.argv[2] + ".%d.bz2" % lv, "rb").read(), lv
print("ok")
"""


@pytest.mark.parametrize("knob", [("BZ2B200_E2E_WINDOWS", "3"), ("BZ2B200_CHAIN_TABLES", "0")])
def test_one_call_path_knobs(data40, want40, tmp_path, knob):
    """Knobs read once per process, set in a child: three windows per call, and the block chain without its speculative
    tables (every link evaluated by the walking warp)."""
    p = tmp_path / "in.bin"
    data40.tofile(str(p))
    for lv, w in want40.items():
        (tmp_path / ("in.bin.%d.bz2" % lv)).write_bytes(w)
    env = dict(os.environ, **{knob[0]: knob[1]})
    r = subprocess.run([sys.executable, "-c", _E2E_CHILD, ROOT, str(p)], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr[-3000:]


def test_zstream_small_windows_random_pieces(engine, data40, want40, monkeypatch):
    rng = np.random.default_rng(9)
    monkeypatch.setenv("BZ2B200_ZSTREAM_WINDOW_MB", "1")
    data = data40.tobytes()
    for lv, want in want40.items():
        out = io.BytesIO()
        with bz.ZStream(engine, out, lv, libbz2=True) as z:
            pos = 0
            while pos < len(data):
                k = int(rng.integers(1, 3_000_000))
                z.write(data[pos:pos + k])
                pos += k
        assert out.getvalue() == want, lv


def test_compress_dev(engine, data40, want40):
    d_in = torch.from_numpy(data40).cuda()
    cap = int(bz.load_library().bz2b200_compress_bound(data40.size))
    d_out = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda")
    for lv, want in want40.items():
        n = engine.compress_dev(d_in.data_ptr(), data40.size, lv, d_out.data_ptr(), cap, libbz2=True)
        assert d_out[:n].cpu().numpy().tobytes() == want, lv


def test_plan_range_merge(engine, data40, want40):
    data = data40.tobytes()
    for lv, want in want40.items():
        starts = engine.stream_plan(data, lv, libbz2=True)
        nb = len(starts) - 1
        cuts = [0, nb // 3, nb // 3 + 1, nb]
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            raw, bits, crcs = engine.compress_range(data, lv, starts, a, b - a, libbz2=True)
            parts.append((raw, bits, crcs))
        assert bz.merge_streams(lv, parts, libbz2=True) == want, lv


def test_plan_range_merge_device_resident(engine, data40, want40):
    d_in = torch.from_numpy(data40).cuda()
    for lv, want in want40.items():
        starts = engine.stream_plan(data40.size, lv, dev_ptr=d_in.data_ptr(), libbz2=True)
        assert list(starts) == [s for s, _ in lc.plan(data40.tobytes(), lv)] + [data40.size], lv
        nb = len(starts) - 1
        parts = []
        for a, b in ((0, nb // 2), (nb // 2, nb)):
            span = int(starts[b] - starts[a])
            cap = int(bz.load_library().bz2b200_compress_bound(span)) & ~3
            d_out = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda")
            _, bits, crcs = engine.compress_range(data40.size, lv, starts, a, b - a, dev_ptr=d_in.data_ptr(),
                                                  dev_out=d_out.data_ptr(), dev_out_cap=cap, libbz2=True)
            parts.append((d_out[:(bits + 7) // 8].cpu().numpy().tobytes(), bits, crcs))
        assert bz.merge_streams(lv, parts, libbz2=True) == want, lv


def test_rle1_split_follows_the_libbz2_planner(engine):
    for name, level, data in lc.planner_inputs()[:3] + [(r[0], r[1], r[2]) for r in lc.long_runs()[:2]]:
        got = engine.rle1_split(data, level, libbz2=True)
        want = lc.plan(data, level)
        assert [(a, b) for _, _, a, b in got] == want, name
        for crc, blk, a, b in got:
            assert blk == lc.rle1(data[a:b]) and crc == lc.crc32(data[a:b]), (name, a)


def test_multi_context(data40, want40, monkeypatch):
    n = torch.cuda.device_count()
    for per, world in ((1, 2), (3, 2), (2, 3)):
        monkeypatch.setenv("BZ2B200_MULTI_WINDOWS", str(per))
        m = bz.MultiEngine([r % n for r in range(world)])
        try:
            for lv, want in want40.items():
                assert m.compress(data40, lv, libbz2=True) == want, (per, world, lv)
        finally:
            m.close()


def test_cli(tmp_path):
    data = corpus.mixed(3_000_000, 91).tobytes()
    (tmp_path / "f").write_bytes(data)
    r = subprocess.run(CLI + ["--libbz2", "-6", "-c", "f"], cwd=str(tmp_path), stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr
    assert r.stdout == bz2.compress(data, 6)
    bzip2 = shutil.which("bzip2") or ("/usr/bin/bzip2" if os.path.exists("/usr/bin/bzip2") else None)
    if bzip2:
        ref = subprocess.run([bzip2, "-c", "-6", "f"], cwd=str(tmp_path), stdout=subprocess.PIPE, timeout=600).stdout
        assert r.stdout == ref


def test_bad_flag_level_combinations_return_e_arg(engine):
    L = bz.load_library()
    buf = np.zeros(4096, np.uint8)
    out = np.zeros(1 << 16, np.uint8)
    ln = C.c_size_t()
    for lv in (0x100, 0x10A, 0x1FF, 0x200 | 9, 0x300 | 9, 0x10000 | 9, -1, 0x80000000 - 0x100 + 9, 10, 0x109 + 0x100):
        rc = L.bz2b200_compress_stream(engine._h, buf.ctypes.data, buf.size, C.c_int(lv if lv < 2**31 else lv - 2**32),
                                       out.ctypes.data, out.size, C.byref(ln))
        assert rc == bz.E_ARG, hex(lv)
        h = C.c_void_p()
        assert L.bz2b200_zstream_open(engine._h, lv, bz.SINK(lambda u, d, n: 0), None, C.byref(h)) == bz.E_ARG, hex(lv)
        assert L.bz2b200_merge_streams(lv, 0, None, None, None, None, out.ctypes.data, out.size, C.byref(ln)) == bz.E_ARG
    for lv in range(1, 10):
        assert L.bz2b200_compress_stream(engine._h, buf.ctypes.data, buf.size, lv | 0x100, out.ctypes.data, out.size,
                                         C.byref(ln)) == bz.OK


def test_default_launch_count_is_pinned(engine):
    """text100m at -9, HBM resident (one bench.py step): the default path issues 71 launches per call, as its parent did
    (bench.py --steps 10 counted 710 for both); the mode swaps two Huffman kernels for its own and adds none."""
    data = corpus.text(100_000_000, 2)
    d_in = torch.from_numpy(data).cuda()
    cap = int(bz.load_library().bz2b200_compress_bound(data.size))
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    counts = []
    for lib in (False, True):
        a = engine.launches
        engine.compress_dev(d_in.data_ptr(), data.size, 9, d_out.data_ptr(), cap, libbz2=lib)
        counts.append(engine.launches - a)
    assert counts == [71, 71], counts


def test_default_mode_unchanged_after_libbz2_calls(engine, ref):
    """The mode is per call: a default call after libbz2 calls on the same context is the reference's stream."""
    data = corpus.mixed(2_000_000, 96).tobytes()
    engine.compress(data, 9, libbz2=True)
    assert engine.compress(data, 9) == ref.compress_stream(data, 9, ref.SPEC_FAST)
