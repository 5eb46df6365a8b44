"""Cost of libbz2-identical output (BZ2B200_LIBBZ2) against the default output, on one GPU.

    python tools/bench_libbz2.py [--mb 100] [--level 9] [--reps 7] [--warmup 2] [--out FILE]

Input: text100m (corpus.text(100 MB, seed 2), bench.py's N = 1 workload) resident in HBM; bz2b200_compress_stream_dev
in both modes, alternated call by call after the warm-up, median of --reps calls each.  Then one call per mode with
per-kernel CUDA events (bz2b200_set_timing(ctx, 2)) for the kernels the mode changes.  Prints one JSON record (and
writes it to --out): times, per-kernel times, compressed sizes, whether the libbz2-mode stream equals
bz2.compress(data, level), and the GPU name and power limit read in the same process."""
import argparse
import bz2
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bzip2_rust_b200 as bz
from bzip2_rust_b200 import corpus

CHANGED = ["k_rle_chain", "k_rle_emit", "k_bwt_out", "k_huf_init", "k_huf_init_libbz2", "k_huf_lengths",
           "k_huf_lengths_libbz2", "k_huf_select"]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=int, default=100)
    ap.add_argument("--level", type=int, default=9)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    data = corpus.text(a.mb * 1_000_000, 2)
    d_in = torch.from_numpy(data).cuda()
    eng = bz.Engine(0)
    cap = int(bz.load_library().bz2b200_compress_bound(data.size))
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")

    def call(lib):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        z = eng.compress_dev(d_in.data_ptr(), data.size, a.level, d_out.data_ptr(), cap, libbz2=lib)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, z

    for _ in range(a.warmup):
        call(False)
        call(True)
    times = {"default": [], "libbz2": []}
    size = {}
    for _ in range(a.reps):
        for key, lib in (("default", False), ("libbz2", True)):
            ms, z = call(lib)
            times[key].append(ms)
            size[key] = int(z)
    same = d_out[:size["libbz2"]].cpu().numpy().tobytes() == bz2.compress(data.tobytes(), a.level)
    kernels = {}
    for key, lib in (("default", False), ("libbz2", True)):
        eng.set_timing(2)
        eng.reset_kernel_stats()
        call(lib)
        ks = eng.kernel_stats()
        eng.set_timing(0)
        kernels[key] = {k: [round(v[0], 4), v[1]] for k, v in ks.items() if k in CHANGED}
        kernels[key]["all_kernels_ms"] = round(sum(v[0] for v in ks.values()), 3)
    med = {k: statistics.median(v) for k, v in times.items()}
    rec = {
        "workload": "text100m level %d, HBM resident, bz2b200_compress_stream_dev" % a.level if a.mb == 100 else
                    "text %d MB level %d, HBM resident" % (a.mb, a.level),
        "gpu": gpu_info(),
        "reps": a.reps, "warmup": a.warmup,
        "median_ms": {k: round(v, 3) for k, v in med.items()},
        "all_ms": {k: [round(x, 3) for x in v] for k, v in times.items()},
        "ratio_libbz2_over_default": round(med["libbz2"] / med["default"], 4),
        "bytes": size,
        "libbz2_mode_equals_bz2_compress": same,
        "kernels_ms_launches": kernels,
    }
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
