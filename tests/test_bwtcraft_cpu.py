"""The crafted BWT blocks and the list model of tests/bwtcraft.py, checked on the CPU: the model's BWT and key against
the oracle's SPEC_FAST bwt_encode, and every edge of the coverage table reached by at least one crafted block."""
import numpy as np
import pytest

import bwtcraft as bc
from inputs import small_cases

EDGES = bc.coverage_table()


def _same_as_oracle(ref, block, name):
    m = bc.model_of(block)
    k, b, _ = ref.bwt_encode(block, ref.SPEC_FAST)
    assert m["bwt"] == b, "%s: model BWT differs from the oracle" % name
    assert m["key"] == k, "%s: model key %d, oracle %d" % (name, m["key"], k)


def test_geometry_is_read_from_the_sources():
    g = bc.geometry()
    assert g["LCAP"] <= g["RT"] and g["SCAP"] < g["LCAP"] and 2 * g["LCAP"] <= g["LW"], g
    assert g["LTILE"] == g["LW"] - g["LCAP"] and g["CH"] > 0, g


@pytest.mark.parametrize("name", [n for n, _ in bc.crafted()])
def test_model_matches_oracle_on_crafted_block(ref, name):
    _same_as_oracle(ref, dict(bc.crafted())[name], name)


def test_model_matches_oracle_on_small_cases(ref):
    for name, data in small_cases():
        _same_as_oracle(ref, data, name)


def test_model_matches_oracle_on_lengths_1_to_70(ref):
    rng = np.random.default_rng(5)
    for n in range(1, 71):
        _same_as_oracle(ref, bytes(rng.integers(97, 100, n, dtype=np.uint8)), "random abc n=%d" % n)
        _same_as_oracle(ref, (b"ab" * n)[:n], "ab n=%d" % n)


def test_model_lists_shrink_and_stop():
    """Lists only lose rotations, hold only groups of two or more, and are empty once h >= n."""
    for name, blk in bc.crafted():
        m = bc.model_of(blk)
        prev = len(blk)
        for r in m["rounds"]:
            assert r["h"] < len(blk), name
            assert r["loc"] + r["big"] <= prev, name
            assert all(z > 1 for _, z, _ in r["loc_groups"] + r["big_groups"]), name
            assert sum(z for _, z, _ in r["loc_groups"]) == r["loc"] and sum(z for _, z, _ in r["big_groups"]) == r["big"]
            prev = r["loc"] + r["big"]
    st = bc.batch_stats([bc.model_of(b) for _, b in bc.crafted()])
    assert st["rounds"] >= 17 and st["big_sum"] < st["list_sum"], st


@pytest.mark.parametrize("edge", [e for e, _ in EDGES])
def test_edge_is_reached(edge):
    pred = dict(EDGES)[edge]
    hits = [name for name, blk in bc.crafted() if pred(bc.model_of(blk), len(blk))]
    assert hits, "no crafted block reaches: %s" % edge
