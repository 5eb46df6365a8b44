"""Decode rate of the stream bench.py compresses in its `e2e` leg, so that compress and decompress rates compare.

    python tools/bench_decode.py --gpus 1 2 4 8 [--steps K] [--warmup W] [--size-mb 100] [--dstream] [--recover]
                                 [--rstream]

Workload for world N: corpus.text(size_mb * 10^6, seed 2 + r) for r < N, concatenated, compressed at -9.  Pinned host
buffers; W warm-up calls, then K calls timed with a host clock around each call (a call returns when its output is in
host memory).  N = 1 times bz2b200_decompress_stream, N > 1 bz2b200_decompress_stream_multi on devices
0..N-1 (modulo the visible devices: `distinct_gpus` says how many GPUs the ranks really had).  The output is compared
with the input after the timed calls.  One JSON line per world size.

--dstream adds two arms for world 1, timed in turn with the one-call arm (one-call, dstream, test mode, one-call, ...)
on the same workload: "decode_dstream" writes the pinned compressed stream into a bz2b200_dstream in pieces of 16 MiB
and its sink memmoves every piece into a pinned output buffer at a running offset; "decode_test" does the same in test
mode (no sink, nothing downloaded).  Both are timed with a host clock from open to close.  The dstream's output is
compared with the input after the timed calls, and test mode's total_out with the input's size.  They print one JSON
line each after the one-call arm's.

--recover adds three bz2b200_recover arms for world 1, timed in turn with the one-call arm in the same way:
"recover_report" with a NULL sink (nothing downloaded), "recover_sink" with the dstream arm's pinned memmove sink, and
"recover_damaged" with that sink on a copy of the stream with one bit flipped in every 100th block (blocks 0, 100, ...,
inside their Huffman data), and "recover_damaged_report" on that copy with a NULL sink.  The damaged arm's output is
compared with the input minus the input slices of the damaged blocks (Engine.stream_plan), the report-only arms'
totals with the expected sizes.  When bzip2recover and bzip2 are installed, one more line times the CPU way on the damaged
copy: bzip2recover, then bzip2 -dc of every piece, one after the other ("cpu_bzip2recover"); otherwise that line says
"not measured".

--rstream adds three bz2b200_rstream arms for world 1, timed in turn with "recover_report" and "recover_sink" (added
too when --recover is not given) on the same bytes: "rstream_report" (NULL sink), "rstream_sink" (the dstream arm's
pinned memmove sink) and "rstream_damaged" (that sink, on the damaged copy of --recover).  Each writes the pinned stream
in pieces of 16 MiB and is timed with a host clock from open to close; its report callback counts the entries, which
must match the count close returns.  Outputs and totals are verified as in the recovery arms.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bzip2_rust_b200 as bz  # noqa: E402
from bzip2_rust_b200 import corpus  # noqa: E402


def gpu_info():
    """Name, power limit and max SM clock of GPU 0 (a query: no setting is changed)."""
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
                           timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                          # the numbers are then unlabelled: say so
        return {"gpu": "unknown (%s)" % type(e).__name__}


def pinned(n):
    return torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True).numpy()


def run(world, args, eng, info):
    per = args.size_mb * 1_000_000
    data = np.concatenate([corpus.text(per, 2 + r) for r in range(world)])
    s = eng.compress(data, 9)
    h_in = pinned(len(s))
    h_in[:len(s)] = np.frombuffer(s, dtype=np.uint8)
    h_out = pinned(data.size + 64)
    in_ptr, out_ptr, cap = h_in.ctypes.data, h_out.ctypes.data, h_out.size
    ndev = torch.cuda.device_count()
    m = None
    arms = []
    if world == 1 and args.dstream:
        arms = dstream_arms(eng, h_in, len(s), data.size)
    if world == 1 and (args.recover or args.rstream):
        rarms = recover_arms(eng, h_in, len(s), data)
        arms += rarms if args.recover else rarms[:2]
        if args.rstream:
            arms += rstream_arms(eng, h_in, len(s), data, rarms[-1])
    if world == 1:
        L, ln = eng._L, C.c_size_t()

        def call():
            rc = L.bz2b200_decompress_stream(eng._h, in_ptr, len(s), out_ptr, cap, C.byref(ln))
            if rc != bz.OK:
                raise bz.Bz2B200Error(rc, L.bz2b200_last_error(eng._h).decode())
            return ln.value
    else:
        m = bz.MultiEngine([r % ndev for r in range(world)])

        def call():
            return m.decompress_into(in_ptr, len(s), out_ptr, cap)
    for _ in range(args.warmup):
        call()
        for arm in arms:
            arm["call"]()
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        n = call()
        times.append(time.perf_counter() - t0)
        for arm in arms:
            t0 = time.perf_counter()
            arm["n"] = arm["call"]()
            arm["times"].append(time.perf_counter() - t0)
    ok = n == data.size and np.array_equal(h_out[:n], data)
    st = m.stats() if m else {"h2d_bytes": len(s), "d2h_bytes": n}
    if m:
        m.close()
    ms = 1e3 * float(np.median(times))
    rec = {"metric": "decode", "world": world, "distinct_gpus": min(world, ndev), "decompressed_MBps": data.size / 1e6 / (ms / 1e3),
           "ms_per_call": ms, "ms_min": 1e3 * min(times), "ms_max": 1e3 * max(times), "steps": args.steps,
           "compressed_bytes": len(s), "decompressed_bytes": int(data.size), "h2d_bytes": st["h2d_bytes"],
           "d2h_bytes": st["d2h_bytes"], "verified": bool(ok),
           "library": os.environ.get("BZ2B200_LIB", "bzip2_rust_b200/libbz2b200.so")}
    rec.update(info)
    print(json.dumps(rec), flush=True)
    for arm in arms:
        want = arm.get("want", data)
        a_ok = arm["n"] == want.size and (arm["out"] is None or np.array_equal(arm["out"][:want.size], want))
        ms = 1e3 * float(np.median(arm["times"]))
        r = {"metric": arm["metric"], "world": 1, "distinct_gpus": 1, "decompressed_MBps": data.size / 1e6 / (ms / 1e3),
             "ms_per_call": ms, "ms_min": 1e3 * min(arm["times"]), "ms_max": 1e3 * max(arm["times"]), "steps": args.steps,
             "piece_bytes": PIECE, "compressed_bytes": len(s), "decompressed_bytes": int(data.size),
             "verified": bool(a_ok), "library": rec["library"]}
        r.update({k: arm[k] for k in ("damaged_blocks", "blocks", "window_bytes") if k in arm})
        r.update(info)
        print(json.dumps(r), flush=True)
        ok = ok and a_ok
    if world == 1 and args.recover:
        print(json.dumps(cpu_recover_reference(rarms[-1]["input"], info)), flush=True)
    return ok


PIECE = 16 << 20


def dstream_arms(eng, h_in, n_in, n_out):
    """The dstream and test-mode arms: each a dict with `call` (-> total_out), `times`, `out` (pinned, or None)."""
    L = eng._L
    in_ptr = h_in.ctypes.data
    out = pinned(n_out + 64)
    out_ptr, pos = out.ctypes.data, [0]

    def sink(_user, data, n):
        if pos[0] + n > out.size:
            return 1
        C.memmove(out_ptr + pos[0], data, n)
        pos[0] += n
        return 0
    cb = bz.SINK(sink)

    def stream(test):
        pos[0] = 0
        h, ti, to = C.c_void_p(), C.c_uint64(), C.c_uint64()
        rc = L.bz2b200_dstream_open(eng._h, bz.SINK() if test else cb, None, C.byref(h))
        if rc == bz.OK:
            for off in range(0, n_in, PIECE):
                rc = L.bz2b200_dstream_write(h, in_ptr + off, min(PIECE, n_in - off))
                if rc != bz.OK:
                    break
            rc2 = L.bz2b200_dstream_close(h, C.byref(ti), C.byref(to))
            rc = rc if rc != bz.OK else rc2
        if rc != bz.OK:
            raise bz.Bz2B200Error(rc, L.bz2b200_last_error(eng._h).decode())
        return to.value
    return [{"metric": "decode_dstream", "call": lambda: stream(False), "times": [], "out": out, "cb": cb, "n": 0},
            {"metric": "decode_test", "call": lambda: stream(True), "times": [], "out": None, "n": 0}]


def recover_arms(eng, h_in, n_in, data):
    """The recovery arms (see the module doc): each a dict like dstream_arms' plus `want` (the expected output)."""
    L = eng._L
    s = h_in[:n_in].tobytes()
    total, ents = eng.recover(s)
    blocks = [e.bit for e in ents if not e.flags & bz.REC_FOOTER]
    starts = eng.stream_plan(data, 9)
    assert total == data.size and len(blocks) == len(starts) - 1
    h_dmg = pinned(n_in)
    h_dmg[:n_in] = h_in[:n_in]
    lost = range(0, len(blocks), 100)
    for k in lost:
        bit = blocks[k] + 2000
        h_dmg[bit // 8] ^= 0x80 >> (bit % 8)
    keep = np.ones(data.size, dtype=bool)
    for k in lost:
        keep[int(starts[k]):int(starts[k + 1])] = False
    cap = len(ents) + 64
    ent = (bz.RecEntry * cap)()

    def arm(metric, buf, want, sink):
        """One arm; with `sink`, its own pinned output buffer that the sink memmoves into at a running offset."""
        a = {"metric": metric, "times": [], "out": None, "n": 0, "want": want}
        cb = bz.SINK()
        if sink:
            out = pinned(want.size + 64)
            out_ptr, pos = out.ctypes.data, [0]

            def put(_user, p, n):
                if pos[0] + n > out.size:
                    return 1
                C.memmove(out_ptr + pos[0], p, n)
                pos[0] += n
                return 0
            cb = bz.SINK(put)
            a.update(out=out, cb=cb, pos=pos)

        def call():
            if sink:
                a["pos"][0] = 0
            nent, tot = C.c_uint32(), C.c_uint64()
            rc = L.bz2b200_recover(eng._h, buf.ctypes.data, n_in, cb, None, ent, cap, C.byref(nent), C.byref(tot))
            if rc != bz.OK:
                raise bz.Bz2B200Error(rc, L.bz2b200_last_error(eng._h).decode())
            return tot.value
        a["call"] = call
        return a
    dmg_report = arm("recover_damaged_report", h_dmg, data[keep], False)
    damaged = arm("recover_damaged", h_dmg, data[keep], True)
    for a in (dmg_report, damaged):
        a.update(damaged_blocks=len(lost), blocks=len(blocks))
    damaged["input"] = h_dmg[:n_in].tobytes()
    return [arm("recover_report", h_in, data, False), arm("recover_sink", h_in, data, True), dmg_report, damaged]


def memmove_sink(n):
    """A pinned output buffer of n bytes and a sink that memmoves into it at a running offset: (out, cb, pos)."""
    out = pinned(n)
    out_ptr, pos = out.ctypes.data, [0]

    def put(_user, p, k):
        if pos[0] + k > out.size:
            return 1
        C.memmove(out_ptr + pos[0], p, k)
        pos[0] += k
        return 0
    return out, bz.SINK(put), pos


def rstream_arms(eng, h_in, n_in, data, damaged):
    """The streaming recovery arms (see the module doc), like recover_arms'."""
    L = eng._L
    h_dmg = pinned(n_in)
    h_dmg[:n_in] = np.frombuffer(damaged["input"], dtype=np.uint8)

    def arm(metric, buf, want, sink):
        a = {"metric": metric, "times": [], "out": None, "n": 0, "want": want,
             "window_bytes": int(os.environ.get("BZ2B200_RSTREAM_WINDOW", 64 << 20))}
        cb, pos, counted = bz.SINK(), [0], [0]
        if sink:
            out, cb, pos = memmove_sink(want.size + 64)
            a["out"] = out

        def rep(_user, _p, k):
            counted[0] += k
            return 0
        rcb = bz.REC_REPORT(rep)
        a["cbs"] = (cb, rcb)                                # alive as long as the arm

        def call():
            pos[0] = counted[0] = 0
            h, ti, to, ne = C.c_void_p(), C.c_uint64(), C.c_uint64(), C.c_uint64()
            rc = L.bz2b200_rstream_open(eng._h, cb, rcb, None, C.byref(h))
            if rc == bz.OK:
                for off in range(0, n_in, PIECE):
                    rc = L.bz2b200_rstream_write(h, buf.ctypes.data + off, min(PIECE, n_in - off))
                    if rc != bz.OK:
                        break
                rc2 = L.bz2b200_rstream_close(h, C.byref(ti), C.byref(to), C.byref(ne))
                rc = rc if rc != bz.OK else rc2
            if rc != bz.OK:
                raise bz.Bz2B200Error(rc, L.bz2b200_last_error(eng._h).decode())
            if ne.value != counted[0] or ti.value != n_in:
                return -1                                   # fails verification
            return to.value
        a["call"] = call
        return a
    dmg = arm("rstream_damaged", h_dmg, damaged["want"], True)
    dmg.update(damaged_blocks=damaged["damaged_blocks"], blocks=damaged["blocks"])
    return [arm("rstream_report", h_in, data, False), arm("rstream_sink", h_in, data, True), dmg]


def cpu_recover_reference(damaged, info):
    """bzip2recover + bzip2 -dc of each piece on the damaged copy, timed once with a host clock (the CPU reference)."""
    import shutil
    import tempfile
    rec = {"metric": "cpu_bzip2recover"}
    rec.update(info)
    if not (os.path.exists("/usr/bin/bzip2recover") and shutil.which("bzip2")):
        rec["ms_per_call"] = "not measured (no bzip2recover / bzip2 on this host)"
        return rec
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "damaged.bz2")
        open(f, "wb").write(damaged)
        t0 = time.perf_counter()
        subprocess.run(["/usr/bin/bzip2recover", f], cwd=td, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        n = 0
        for p in sorted(x for x in os.listdir(td) if x.startswith("rec")):
            r = subprocess.run(["bzip2", "-dc", os.path.join(td, p)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            if r.returncode == 0:
                n += len(r.stdout)
        rec["ms_per_call"] = 1e3 * (time.perf_counter() - t0)
        rec["recovered_bytes"] = n
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--gpus", type=int, nargs="+", default=[1])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--size-mb", type=int, default=100)
    ap.add_argument("--dstream", action="store_true", help="also time the streaming decoder and its test mode (world 1)")
    ap.add_argument("--recover", action="store_true", help="also time block recovery, intact and damaged (world 1)")
    ap.add_argument("--rstream", action="store_true", help="also time streaming recovery against block recovery (world 1)")
    args = ap.parse_args()
    if args.steps < 1 or min(args.gpus) < 1:
        ap.error("--steps and --gpus must be at least 1")
    info = gpu_info()
    eng = bz.Engine(0)
    ok = all([run(w, args, eng, info) for w in args.gpus])
    eng.close()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
