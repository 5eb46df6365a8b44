"""Decode rate of the stream bench.py compresses in its `e2e` leg, so that compress and decompress rates compare.

    python tools/bench_decode.py --gpus 1 2 4 8 [--steps K] [--warmup W] [--size-mb 100]

Workload for world N: corpus.text(size_mb * 10^6, seed 2 + r) for r < N, concatenated, compressed at -9.  Pinned host
buffers; W warm-up calls, then K calls timed with a host clock around each call (a call returns when its output is in
host memory).  N = 1 times bz2b200_decompress_stream, N > 1 bz2b200_decompress_stream_multi on devices
0..N-1 (modulo the visible devices: `distinct_gpus` says how many GPUs the ranks really had).  The output is compared
with the input after the timed calls.  One JSON line per world size.
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
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        n = call()
        times.append(time.perf_counter() - t0)
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
    return ok


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--gpus", type=int, nargs="+", default=[1])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--size-mb", type=int, default=100)
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
