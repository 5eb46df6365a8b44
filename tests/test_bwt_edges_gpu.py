"""CUDA BWT on crafted blocks at the group-size and tile edges of the suffix sort (tests/bwtcraft.py).

Every batch is checked twice: each block's bytes and key against the oracle's SPEC_FAST bwt_encode, and bwt_stats()
rounds / list_sum / big_sum against the list model.  The second check catches what the bytes cannot show: a group sent
down the wrong path, or a resolved rotation kept in a list for another round.
"""
import hashlib
import json
import os
import subprocess
import sys

import pytest

import bwtcraft as bc
from bzip2_rust_b200 import corpus

pytestmark = pytest.mark.gpu

N_MAX = 900_000
_ORACLE = {}


def _oracle(ref, block):
    if block not in _ORACLE:
        _ORACLE[block] = ref.bwt_encode(block, ref.SPEC_FAST)[:2]
    return _ORACLE[block]


def _check(engine, ref, named):
    """One bwt_encode_batch of [(name, block)]; returns the outputs."""
    got = engine.bwt_encode_batch([b for _, b in named])
    st = engine.bwt_stats()
    for (name, blk), (key, bwt) in zip(named, got):
        k, b = _oracle(ref, blk)
        assert bwt == b, "%s: BWT bytes differ (n=%d)" % (name, len(blk))
        assert key == k, "%s: key %d, oracle %d" % (name, key, k)
    want = bc.batch_stats([bc.model_of(b) for _, b in named])
    assert {k: st[k] for k in want} == want, "list stats of %s" % ", ".join(n for n, _ in named[:4])
    return got


def _full_size():
    p3 = bytearray(b"abc" * (N_MAX // 3))
    p3[-1] = ord("d")
    return [("zeros", bytes(N_MAX)), ("ab", b"ab" * (N_MAX // 2)), ("period3_last_changed", bytes(p3)),
            ("random", corpus.random_bytes(N_MAX, 61).tobytes())]


@pytest.mark.parametrize("name", [n for n, _ in bc.crafted()])
def test_crafted_block_alone(engine, ref, name):
    _check(engine, ref, [(name, dict(bc.crafted())[name])])


@pytest.mark.parametrize("order", ["forwards", "reversed"])
def test_all_crafted_blocks_in_one_batch(engine, ref, order):
    named = list(bc.crafted())
    _check(engine, ref, named if order == "forwards" else named[::-1])


@pytest.mark.parametrize("count", [5, 33, 129])
def test_batches_across_interleave_groups(engine, ref, count):
    """Block counts that are not multiples of the interleave groups (4, 32, 128): tiny blocks, crafted blocks that
    finish in different rounds, and one full-size text block that sets the stride, at a different place each time."""
    tiny = [p for p in bc.crafted() if len(p[1]) <= 8]
    rest = [p for p in bc.crafted() if 8 < len(p[1]) < N_MAX]
    seen = {}

    def spread(p):                                  # one block of each round count first, then the next of each
        r = len(bc.model_of(p[1])["rounds"])
        seen[r] = seen.get(r, 0) + 1
        return seen[r], r

    rest.sort(key=spread)
    pool = [p for pair in zip(tiny, rest) for p in pair] + rest[len(tiny):]
    named = [pool[i % len(pool)] for i in range(count - 1)]
    at = {5: 0, 33: 16, 129: 128}[count]
    named.insert(at, ("text_900000", corpus.text(N_MAX, 62).tobytes()))
    assert len({len(bc.model_of(b)["rounds"]) for _, b in named}) >= 3
    _check(engine, ref, named)


@pytest.mark.parametrize("name", [n for n, _ in _full_size()])
def test_full_size_block(engine, ref, name):
    _check(engine, ref, [(name, dict(_full_size())[name])])


def test_crafted_batch_after_full_size_batch(engine, ref):
    """The workspaces only grow and the look-back state is reused: a batch after three full-size blocks."""
    _check(engine, ref, _full_size()[:2] + _full_size()[3:])
    _check(engine, ref, list(bc.crafted()))


_KNOB_RUN = """
import hashlib, json, sys
sys.path[:0] = [%r, %r]
import bwtcraft as bc
import bzip2_rust_b200 as bz
eng = bz.Engine()
got = eng.bwt_encode_batch([b for _, b in bc.crafted()])
h = hashlib.sha256()
for key, bwt in got:
    h.update(key.to_bytes(4, "little") + bwt)
st = eng.bwt_stats()
print(json.dumps(dict(sha=h.hexdigest(), rounds=st["rounds"], list_sum=st["list_sum"], big_sum=st["big_sum"])))
"""


@pytest.mark.parametrize("env", [
    {"BZ2B200_REFINE_GROUP": "1"}, {"BZ2B200_REFINE_GROUP": "3"},
    {"BZ2B200_SWEEP_GROUP": "1"}, {"BZ2B200_SWEEP_GROUP": "5"},
    {"BZ2B200_SWEEP_GROUP_STREAM": "1"}, {"BZ2B200_SWEEP_GROUP_STREAM": "7"},
    {"BZ2B200_SWEEP_IPT0": "8", "BZ2B200_SWEEP_IPT1": "8"},
], ids=lambda e: ",".join("%s=%s" % kv for kv in e.items()))
def test_interleave_knobs_give_the_same_output(engine, ref, env):
    """The knobs are read once per process, so each setting runs in a process of its own."""
    named = list(bc.crafted())
    got = _check(engine, ref, named)
    h = hashlib.sha256()
    for key, bwt in got:
        h.update(key.to_bytes(4, "little") + bwt)
    want = dict(sha=h.hexdigest(), **bc.batch_stats([bc.model_of(b) for _, b in named]))
    tests = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-c", _KNOB_RUN % (tests, os.path.dirname(tests))], env=dict(os.environ, **env),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1]) == want, env
