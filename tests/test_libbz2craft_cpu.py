"""The libbz2 model of tests/libbz2craft.py, checked on the CPU against the libbz2 Python's bz2 module links: byte for
byte on small inputs, the block planner through the combined CRC of multi-block streams, and every crafted input at the
edge it was built for.  The GPU side (tests/test_libbz2_gpu.py) holds the engine's BZ2B200_LIBBZ2 mode to the same
bytes."""
import bz2

import pytest

import libbz2craft as lc

EDGES = (["cut inside long run", "short chunk at cut", "len B-1"] + ["len B+%d" % d for d in range(5)] +
         ["last block one chunk"] + ["nmtf %d" % n for n in (199, 200, 599, 600, 1199, 1200, 2399, 2400)] +
         ["heap retry", "heap ties", "period short", "period near n", "period from rle1"])


def test_libbz2_version_is_recorded():
    v = lc.libbz2_version()
    print("BZ2_bzlibVersion() = %s" % v)
    assert v is None or v.startswith("1.0."), v


@pytest.mark.parametrize("level", [1, 5, 9])
def test_model_equals_libbz2_on_small_inputs(level):
    for name, data in lc.small_inputs():
        assert lc.compress(data, level) == bz2.compress(data, level), "%s at -%d" % (name, level)


@pytest.mark.parametrize("name", [n for n, _, _ in lc.planner_inputs()])
def test_planner_matches_libbz2_combined_crc(name):
    _, level, data = next(p for p in lc.planner_inputs() if p[0] == name)
    stream = bz2.compress(data, level)
    assert lc.combined_crc(data, level) == lc.stored_combined_crc(stream), name
    # and the first block's CRC, stored right after the first block magic
    s, e = lc.plan(data, level)[0]
    assert lc.crc32(data[s:e]) == int.from_bytes(stream[10:14], "big"), name


def test_planner_inputs_are_multi_block():
    assert sum(len(lc.plan(d, lv)) > 1 for _, lv, d in lc.planner_inputs()) >= 4


def test_rle1_block_bounds():
    """A non-final block is B to B + 4 RLE1 bytes, and its start is a chunk boundary."""
    for _, level, data, _ in lc.crafted():
        B = 100000 * level - 19
        bounds = {s for s, _ in lc.chunks(data)}
        blocks = lc.plan(data, level)
        for s, e in blocks[:-1]:
            assert B <= len(lc.rle1(data[s:e])) <= B + 4
            assert s in bounds and e in bounds


@pytest.mark.parametrize("edge", EDGES)
def test_edge_is_reached(edge):
    hits = [name for name, level, data, want in lc.crafted() if want == edge and edge in lc.edges_reached(level, data)]
    assert hits, "no crafted input reaches %r" % edge


@pytest.mark.parametrize("name", [c[0] for c in lc.crafted() if len(c[2]) <= 5000])
def test_model_equals_libbz2_on_small_crafted(name):
    _, level, data, _ = next(c for c in lc.crafted() if c[0] == name)
    assert lc.compress(data, level) == bz2.compress(data, level), name


def first_origin(stream):
    """The 24-bit origin pointer of the first block (stream bits 105..128)."""
    return int.from_bytes(stream[4:18], "big") >> (112 - 105) & 0xFFFFFF


@pytest.mark.parametrize("name", [c[0] for c in lc.crafted() if c[3].startswith("period")])
def test_model_equals_libbz2_on_periodic_blocks(name):
    """Among the k equal rotations of u^k libbz2 stores the row its fallbackSort leaves rotation 0 in."""
    _, level, data, _ = next(c for c in lc.crafted() if c[0] == name)
    s, e = lc.plan(data, level)[0]
    _, orig, size = lc.bwt(lc.rle1(data[s:e]))
    assert size > 1 and orig == first_origin(bz2.compress(data, level)), name


@pytest.mark.parametrize("name", [n for n, lv, _ in lc.long_runs() if lv <= 2])
def test_model_origin_of_long_runs(name):
    """The first block of a long run of one byte value is the block every interior block repeats."""
    _, level, data = next(r for r in lc.long_runs() if r[0] == name)
    s, e = lc.plan(data, level)[0]
    assert lc.fallback_origin(lc.rle1(data[s:e])) == first_origin(bz2.compress(data, level)), name


@pytest.mark.parametrize("name", [n for n, _, _ in lc.periodic_main_sort()])
def test_periodic_blocks_that_main_sort_finishes(name):
    """The documented gap: on these blocks libbz2's mainSort, not its fallbackSort, decides the row, and the model (like
    the engine) differs from libbz2 in the origin pointer only."""
    _, level, data = next(p for p in lc.periodic_main_sort() if p[0] == name)
    mine, theirs = lc.compress(data, level), bz2.compress(data, level)
    assert len(mine) == len(theirs) and first_origin(mine) != first_origin(theirs)
    diff = [i for i in range(len(mine)) if mine[i] != theirs[i]]
    assert min(diff) >= 14 and max(diff) <= 17, diff                  # bits 105..128: the origin field
    assert bz2.decompress(mine) == data
