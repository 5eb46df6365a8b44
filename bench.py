#!/usr/bin/env python
"""bench.py -- compress MB/s at -9, byte-identical to the reference (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our CUDA engine
    python bench.py --impl reference --gpus N ...            # the reference algorithm (CPU oracle port) on host cores

One "step" = one whole-stream compression of the workload:
  N = 1  : `text100m` (BASELINE config 2: 100 MB synthetic text-like corpus, level 9)
  N > 1  : ONE stream of N x 100 MB; rank r compresses the blocks that start in its 100 MB slice.  The block
           chain is handed from rank to rank as one number (no data-path collective: blocks never exchange
           data); the ordered merge ORs pre-shifted bit strings on rank 0.                     -> "weak" scaling
`value`  : input and output resident in HBM (bz2b200_compress_stream_dev / bz2b200_shard_*_dev, one process per GPU)
`e2e`    : the same through host buffers: pinned host input, H2D + kernels + D2H of the .bz2 bytes inside the timed
           region.  N = 1: bz2b200_compress_stream.  N > 1: ONE call of the library's multi-GPU entry point
           bz2b200_compress_stream_multi from rank 0 (one host thread + one context per GPU inside the library, the
           block chain handed over through host memory, no NCCL / barrier / Python inside the step); the other ranks'
           processes idle on a host (gloo) barrier meanwhile.
Prints ONE JSON line on rank 0.

--dump-outputs DIR writes the .bz2 stream of the last timed step to DIR as .npy files (see dump_stream), so that two
builds can be compared output for output: the inputs are seeded, identical from run to run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree, which may be read-only

METRIC = "compress_MBps_level9_byte_identical"
UNIT = "MB/s"
DUMP_WINDOW = 64 << 10                  # --dump-outputs: bytes per sampled window of the stream
DUMP_WINDOWS = 128                      # 8 MiB of stream bytes, 32 MiB as float32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size-mb", type=int, default=100, help="input MB per GPU")
    ap.add_argument("--level", type=int, default=9)
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--cpu-sample-mb", type=int, default=0, help="cpu_baseline sample size (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the stream of the last timed step to DIR (.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_stream(out_dir, stream):
    """Writes a compressed stream (uint8 array) for output-to-output comparison of two builds:
        stream_length.npy   float64 [1]     its length in bytes
        stream_offsets.npy  float64 [k]     where each row of stream_bytes starts in the stream
        stream_bytes.npy    float32 [k, w]  byte values
    A stream of at most DUMP_WINDOWS * DUMP_WINDOW bytes is written whole, as one row.  A longer one is sampled as
    DUMP_WINDOWS windows of DUMP_WINDOW bytes: its first (stream header, first block) and its last (footer with the
    combined CRC), and the others at offsets drawn from a fixed seed."""
    os.makedirs(out_dir, exist_ok=True)
    n = int(stream.size)
    if n <= DUMP_WINDOWS * DUMP_WINDOW:
        offs = np.zeros(1, dtype=np.int64)
        rows = stream[None, :]
    else:
        mid = np.sort(np.random.default_rng(0).integers(0, n - DUMP_WINDOW + 1, size=DUMP_WINDOWS - 2))
        offs = np.concatenate([[0], mid, [n - DUMP_WINDOW]]).astype(np.int64)
        rows = stream[offs[:, None] + np.arange(DUMP_WINDOW)]
    np.save(os.path.join(out_dir, "stream_length.npy"), np.array([n], dtype=np.float64))
    np.save(os.path.join(out_dir, "stream_offsets.npy"), offs.astype(np.float64))
    np.save(os.path.join(out_dir, "stream_bytes.npy"), rows.astype(np.float32))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                  "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
        except Exception:
            return
        self._p = p
        for line in p.stdout:
            self.rows.append([c.strip() for c in line.strip().split(",")])
            if self._stop.is_set():
                break

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        time.sleep(0.3)

    def stop(self):
        self._stop.set()
        try:
            self._p.terminate()
        except Exception:
            pass
        if self._t:
            self._t.join(timeout=3)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 6:
                try:
                    sm.append(float(r[0]))
                    mx.append(float(r[1]))
                except ValueError:
                    continue
                for k, nm in enumerate(names):
                    if r[2 + k].lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_rate(data, level, sample_mb, threads):
    """The reference algorithm (oracle port of compress.rs:40 with the native comparison-sort BWT) on host cores."""
    from oracle import pyref
    pyref.build()
    if sample_mb <= 0:
        sample_mb = max(2, min(len(data) // (1 << 20), int(threads * 1.8)))     # ~2 blocks per thread
    sample = data[:sample_mb << 20].tobytes()
    t0 = time.perf_counter()
    out, st = pyref.compress_stream(sample, level, pyref.SPEC, threads=threads, want_stats=True)
    dt = time.perf_counter() - t0
    # Huffman (weight, syms) ties between distinct nodes, and those at list lengths 21..49 where rustc 1.65's
    # sort_unstable is not pinned by the reference's tests (SURVEY D.3): 0 means the sample never enters that window
    cpu_reference_rate.ties = {"tie_events": int(st["tie_events"]), "tie_events_unpinned": int(st["tie_unpinned"])}
    return len(sample) / 1e6 / dt, dt, len(sample), len(out)


def bzip2_cli_rate(data, level):
    """/usr/bin/bzip2 -<level>, one thread, on a bounded sample: libbz2's own encoder (a different byte stream) as a sanity
    reference for the CPU numbers."""
    import shutil
    exe = shutil.which("bzip2")
    if not exe:
        return None
    sample = data[:16_000_000].tobytes()
    t0 = time.perf_counter()
    p = subprocess.run([exe, "-%d" % level, "-c"], input=sample, stdout=subprocess.PIPE)
    dt = time.perf_counter() - t0
    if p.returncode != 0:
        return None
    return {"value": len(sample) / 1e6 / dt, "unit": UNIT, "cores": 1, "sample": "first 16 MB of the workload, /usr/bin/bzip2 -%d" % level}


def ref_path_accounting(eng, data, level, limit=48):
    """SURVEY 8c: #blocks native / sais-valid / sais-divergent.  The device counts the blocks the reference's selector
    (bwt_sort.rs:29) sends to SA-IS; here (outside any timed region) the oracle's bug-for-bug EXACT mode runs on exactly
    those blocks (the first `limit` of them): where its BWT and origin pointer equal the true ones the reference's bytes
    are ours ("sais_valid"); where only the origin pointer differs the block is fully periodic and the reference names
    another row of the same class of equal rotations -- a valid block, 24 bits different from ours
    ("sais_valid_other_origin", SURVEY D.2); where the BWT differs the reference's block does not decode
    ("sais_divergent")."""
    from oracle import pyref
    blocks = eng.rle1_split(data, level)
    flagged = [b for _, b, _, _ in blocks if len(b) > 5000 and pyref.lms_count(b) <= 1499]
    valid = other = div = 0
    for b in flagged[:limit]:
        k1, w1, _ = pyref.bwt_encode(b, pyref.EXACT)
        k2, w2, _ = pyref.bwt_encode(b, pyref.SPEC_FAST)
        if (k1, w1) == (k2, w2):
            valid += 1
        elif w1 == w2:
            other += 1
        else:
            div += 1
    return {"blocks": len(blocks), "native": len(blocks) - len(flagged), "sais": len(flagged),
            "sais_checked": min(limit, len(flagged)), "sais_valid": valid, "sais_valid_other_origin": other,
            "sais_divergent": div}


def workload_config(level, per, total, world):
    return {"workload": "text100m level %d (BASELINE config 2)%s" % (level, "" if world == 1 else
                                                                      " x%d as one stream, blocks sharded" % world),
            "level": level, "input_bytes_per_gpu": per, "input_bytes_total": total,
            "l2": "inputs + workspaces (>4 GB) exceed the 126 MB L2; no explicit flush",
            "parallelism": "blocks x%d, no collective on the data path" % world}


def run_reference(args):
    """The reference's CPU path (C restatement, all host threads) on the SAME configuration as the b200 arm: one step =
    the whole N x 100 MB stream at level 9 (rank r's segment is corpus.text(seed 2 + r), as in the b200 arm)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from bzip2_rust_b200 import corpus
    from oracle import pyref
    pyref.build()
    threads = os.cpu_count() or 1
    world = args.gpus
    per = args.size_mb * 1_000_000
    total = per * world
    # K steps of the whole workload when that fits ~150 s of host time, otherwise a bounded leading sample per step
    rate_guess = 2.6e6 * threads                               # bytes / s of the port (measured: 42 MB/s on 16 cores)
    budget = 150.0 / max(1, args.steps)
    want = total if not args.cpu_sample_mb else min(total, args.cpu_sample_mb << 20)
    nbytes = int(min(want, max(16_000_000, budget * rate_guess)))
    segs, have, r = [], 0, 0
    while have < nbytes:
        seg = corpus.text(per, 2 + r)[:nbytes - have]
        segs.append(seg)
        have += seg.size
        r += 1
    data = np.concatenate(segs)
    raw = data.tobytes()
    steps = max(1, args.steps)
    warm = 1 if args.warmup > 0 else 0
    for _ in range(warm):
        pyref.compress_stream(raw[:max(1, len(raw) // 8)], args.level, pyref.SPEC, threads=threads)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = pyref.compress_stream(raw, args.level, pyref.SPEC, threads=threads)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_stream(args.dump_outputs, np.frombuffer(out, dtype=np.uint8))
    dt = float(np.mean(times))
    value = len(raw) / 1e6 / dt
    sample = ("the whole workload (%d bytes)" % len(raw)) if len(raw) == total else "first %d bytes of the workload" % len(raw)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.level, per, total, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%s per step, C restatement of the reference (native comparison-sort BWT), %d pthreads "
                                   "over blocks; the Rust toolchain is absent, so this is the port, not the Rust binary"
                                   % (sample, threads)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "bzip2_cli_single_thread": bzip2_cli_rate(data, args.level),
    }
    print(json.dumps(line))
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    # Only the JSON line may reach stdout: NCCL / torchrun chatter written to fd 1 goes to stderr instead.
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        return _main(args, real_stdout)
    finally:
        os.dup2(real_stdout, 1)


def _main(args, real_stdout):

    import torch
    import bzip2_rust_b200 as bz
    from bzip2_rust_b200 import corpus

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    N = args.gpus
    dist = None
    host_group = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")            # host-only barrier: no kernel spins on a GPU while rank 0 drives it
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", local if world > 1 else 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")

    level = args.level
    per = args.size_mb * 1_000_000
    # ---- synthetic input: rank r generates segment r, NCCL all_gather builds the whole stream on every GPU ----
    seg = corpus.text(per, 2 + rank)
    d_seg = torch.from_numpy(seg).to(dev)
    if world > 1:
        parts = [torch.empty_like(d_seg) for _ in range(world)]
        dist.all_gather(parts, d_seg)
        d_in = torch.cat(parts)
        del parts
    else:
        d_in = d_seg
    total = d_in.numel()
    h_in = None
    if rank == 0:
        h_in = torch.empty(total, dtype=torch.uint8).pin_memory()
        h_in.copy_(d_in)
    torch.cuda.synchronize()

    eng = bz.Engine(local if world > 1 else 0)
    L = bz.load_library()
    my_lo, my_hi = rank * per, (total if rank == world - 1 else (rank + 1) * per)
    cap = int(L.bz2b200_compress_bound(total if world == 1 else per + (64 << 20)))
    d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
    h_out = torch.empty(int(L.bz2b200_compress_bound(total)), dtype=torch.uint8).pin_memory() if rank == 0 else None
    if world > 1:
        # block-chain hand-off between neighbouring ranks of the HBM-resident measurement: a mailbox in shared host
        # memory, slot r = (sequence number, first block start of rank r, sequence number the receiver has consumed)
        box_path = "/dev/shm/bz2b200_bench_%s.chain" % os.environ.get("MASTER_PORT", "0")
        if rank == 0:
            with open(box_path, "wb") as f:
                f.truncate(24 * (world + 1))
        dist.barrier()
        box = np.memmap(box_path, dtype=np.int64, mode="r+", shape=(world + 1, 3))    # seq, value, ack
        if rank == 0:
            box[:] = 0
        dist.barrier()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def host_barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=host_group)

    out_len = C.c_size_t()
    state = {"seq": 0}

    def chain_recv():
        """-> first block start of this rank (the previous rank's last block end)."""
        state["seq"] += 1
        if rank == 0:
            return 0
        seq = state["seq"]
        deadline = time.perf_counter() + 60.0
        while int(box[rank, 0]) != seq:                        # written last by the sender, after the value
            if time.perf_counter() > deadline:
                raise RuntimeError("chain hand-off timed out on rank %d" % rank)
        v = int(box[rank, 1])
        box[rank, 2] = seq                                     # the slot may be reused
        return v

    def chain_send(nxt):
        if rank < world - 1:
            deadline = time.perf_counter() + 60.0
            while int(box[rank + 1, 2]) != state["seq"] - 1:   # the receiver has not read the previous step's value yet
                if time.perf_counter() > deadline:
                    raise RuntimeError("chain hand-off: rank %d never acknowledged" % (rank + 1))
            box[rank + 1, 1] = nxt
            box[rank + 1, 0] = state["seq"]                    # x86 keeps the two stores in order

    def step_dev():
        """HBM-resident.  N > 1: scan own slice, take the chain from rank-1, pass it on, compress own blocks."""
        if world == 1:
            state["dev_len"] = eng.compress_dev(d_in.data_ptr(), total, level, d_out.data_ptr(), cap)
            return
        look = 4 << 20                                         # look-ahead for the last block of the slice
        win_hi = min(total, my_hi + look)
        eng.shard_scan(d_in.data_ptr() + my_lo, my_lo, win_hi - my_lo, total, level)     # parallel on all ranks
        start = chain_recv()
        while True:
            try:
                nxt, nb = eng.shard_plan(d_in.data_ptr() + my_lo, my_lo, win_hi - my_lo, total, level, start, my_hi)
                break
            except bz.Bz2B200Error as e:                       # a block spans more input than the look-ahead
                if e.rc != bz.E_CAP or win_hi >= total:
                    raise
                look *= 8
                win_hi = min(total, my_hi + look)
        chain_send(nxt)
        bits, crcs = eng.shard_compress(nb, d_out.data_ptr(), cap)
        state["dev_bits"], state["dev_crcs"] = bits, crcs

    multi = None
    if world > 1 and rank == 0:
        multi = bz.MultiEngine(list(range(world)))             # the library's own scheduler: one thread + context per GPU

    def step_e2e():
        """Host buffers; copies inside the timed region (rank 0 only).  -> (h2d bytes, d2h bytes)"""
        if world == 1:
            rc = L.bz2b200_compress_stream(eng._h, h_in.data_ptr(), total, level, h_out.data_ptr(), h_out.numel(),
                                           C.byref(out_len))
            if rc != 0:
                raise RuntimeError("compress_stream failed: %d %s" % (rc, L.bz2b200_last_error(eng._h)))
            return total, out_len.value
        state["merged_len"] = multi.compress_into(h_in.data_ptr(), total, level, h_out.data_ptr(), h_out.numel())
        st = multi.stats()
        return st["h2d_bytes"], st["d2h_bytes"]

    # ---- warm-up ----
    eng.set_timing(2)
    for _ in range(max(args.warmup, 3)):
        step_dev()
    barrier()
    if rank == 0:
        for _ in range(2 if world > 1 else 1):
            step_e2e()
    host_barrier()
    eng.reset_kernel_stats()

    # ---- timed: HBM-resident value ----
    sampler = ClockSampler(local if world > 1 else 0)
    sampler.start()
    barrier()
    launches0 = eng.launches
    t0 = time.perf_counter()
    dev_ms = []
    for _ in range(args.steps):
        step_dev()
        dev_ms.append(eng.timing()["total"])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    barrier()
    launches = eng.launches - launches0
    kstats = eng.kernel_stats()
    stage = eng.timing()
    bst_timed = eng.bwt_stats()                                # of the last timed step (later calls overwrite the per-batch fields)
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    dt_max = float(tt.item())
    launches = int(lt.item())
    value = total / 1e6 * args.steps / dt_max

    # ---- timed: end to end through host buffers (the library call a user makes) ----
    eng.set_timing(1)
    host_barrier()
    h2d = d2h = 0
    e2e_dt = 0.0
    e2e_launches = 0
    if rank == 0:
        l0 = multi.launches() if multi else eng.launches
        t0 = time.perf_counter()
        for _ in range(args.steps):
            h2d, d2h = step_e2e()
        torch.cuda.synchronize()
        e2e_dt = time.perf_counter() - t0
        e2e_launches = (multi.launches() if multi else eng.launches) - l0
    host_barrier()
    clocks = sampler.stop()
    if rank != 0:
        dist.barrier()                                         # rank 0 verifies (it uses its engine) before everybody leaves
        dist.destroy_process_group()
        return 0
    e2e_value = total / 1e6 * args.steps / e2e_dt
    h2d_total, d2h_total = int(h2d), int(d2h)

    if args.dump_outputs:
        # N = 1: the stream of the last HBM-resident step (the one `value` times).  N > 1: those steps leave each rank's
        # blocks on its own GPU, so the whole stream rank 0 holds is the one of the last multi-GPU call.
        if world == 1:
            dump_stream(args.dump_outputs, d_out[:state["dev_len"]].cpu().numpy())
        else:
            dump_stream(args.dump_outputs, h_out[:state["merged_len"]].numpy())

    # ---- verification outside the timed region ----
    verified = None
    oracle_checked = None
    if not args.no_verify:
        import bz2
        raw = h_in.numpy().tobytes()
        if world == 1:
            stream = h_out[:out_len.value].numpy().tobytes()
            dev_stream = d_out[:state["dev_len"]].cpu().numpy().tobytes()
            verified = (stream == dev_stream) and (bz2.decompress(stream) == raw)
            clen = out_len.value
        else:
            stream = h_out[:state["merged_len"]].numpy().tobytes()
            verified = bz2.decompress(stream) == raw
            # and the multi-GPU stream is the same bytes one GPU produces for the whole input
            verified = verified and (eng.compress(h_in.numpy(), level) == stream)
            clen = state["merged_len"]
        # byte identity against the CPU oracle on a sample of the LAST segment (seed 2 + N - 1): the full-size identity
        # tests live in tests/test_fullsize_gpu.py, this keeps every bench run honest about "byte_identical"
        from oracle import pyref
        k = min(per, 6_000_000)
        sample = h_in.numpy()[total - per:total - per + k]
        oracle_checked = eng.compress(sample, level) == pyref.compress_stream(sample.tobytes(), level, pyref.SPEC_FAST,
                                                                              threads=os.cpu_count() or 1)
    else:
        clen = out_len.value if world == 1 else state.get("merged_len", 0)

    # ---- roofline of the dominant kernel (CUDA events around every launch, same timed region) ----
    peak, peak_src = measured_peak()
    roof = None
    ksum = sum(v[0] for v in kstats.values()) or 1.0
    if kstats:
        name, (ms, ln, by) = max(kstats.items(), key=lambda kv: kv[1][0])
        achieved = (by / ln) / (ms / ln * 1e-3) / 1e9 if ln and ms > 0 else 0.0
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get(name)
            except Exception:
                traffic = None
        roof = {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "launches": ln, "avg_ms": ms / ln, "algorithmic_bytes_per_launch": by / ln,
                "share_of_kernel_time": ms / ksum}
    top = sorted(kstats.items(), key=lambda kv: -kv[1][0])[:8]

    # ---- CPU baseline: the reference algorithm on this box's host cores, bounded sample ----
    threads = os.cpu_count() or 1
    cpu_rate, cpu_dt, cpu_bytes, _ = cpu_reference_rate(h_in.numpy(), level, args.cpu_sample_mb, threads)

    bst = eng.bwt_stats()
    # device-side count over every block the engine has seen; the oracle classifies the flagged ones (none on this corpus)
    ref_path = {"blocks": int(bst["blocks_total"]), "native": int(bst["blocks_total"] - bst["ref_sais_blocks_total"]),
                "sais": int(bst["ref_sais_blocks_total"]), "sais_valid": 0, "sais_divergent": 0}
    if ref_path["sais"] and not args.no_verify:
        acc = ref_path_accounting(eng, h_in.numpy()[:min(total, 200_000_000)], level)
        ref_path.update({"sais_checked": acc["sais_checked"], "sais_valid": acc["sais_valid"],
                         "sais_divergent": acc["sais_divergent"]})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": N, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dt_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": workload_config(level, per, total, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total,
                "ms_per_step": e2e_dt / args.steps * 1e3, "gpu_launches": int(e2e_launches),
                "api": "bz2b200_compress_stream" if world == 1 else "bz2b200_compress_stream_multi (rank 0 drives all %d GPUs)" % world},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": {"value": cpu_rate, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "first %.0f MB of the same workload in %.1f s: C restatement of the reference "
                                   "(native comparison-sort BWT), %d pthreads over blocks" % (cpu_bytes / 1e6, cpu_dt, threads),
                         "huffman_ties": getattr(cpu_reference_rate, "ties", None)},
        "device_ms_per_step": float(np.mean(dev_ms)),
        "stage_ms": stage,
        "top_kernels": [{"kernel": k, "ms": v[0] / args.steps, "launches": v[1] // args.steps,
                         "GBps_algorithmic": (v[2] / 1e9) / (v[0] * 1e-3) if v[0] > 0 else 0.0} for k, v in top],
        # every kernel of the timed region: ms per step, launches per step, algorithmic GB/s and its fraction of the HBM peak
        "kernels": [[k, round(v[0] / args.steps, 4), v[1] // args.steps,
                     round((v[2] / 1e9) / (v[0] * 1e-3), 1) if v[0] > 0 else 0.0,
                     round((v[2] / 1e9) / (v[0] * 1e-3) / peak, 4) if v[0] > 0 else 0.0]
                    for k, v in sorted(kstats.items(), key=lambda kv: -kv[1][0])],
        # "byte_identical" in the metric name rests on tests/test_fullsize_gpu.py (whole stream == oracle); in THIS run:
        # libbz2 round trip of the produced stream, device path == host path (N > 1: multi-GPU == one GPU), and a
        # sample of the last segment == the CPU oracle
        "verified_roundtrip_libbz2": verified,
        "verified_oracle_sample": oracle_checked,
        # blocks (since the engine was created) that the reference's path selector (bwt_sort.rs:29) would have sent to its
        # SA-IS fallback, counted on the device: 0 means the reference's output is well defined for the whole workload
        "ref_path": ref_path,
        # prefix doubling of the last timed step: rounds after the 8-byte sort, unresolved-list entries summed over the rounds
        # per input byte, and the part of them that took the global (BIG group) path instead of the shared-memory refinement
        "bwt": {"rounds": int(bst_timed["rounds"]), "list_sum_per_n": round(bst_timed["list_sum"] / max(1, per), 4),
                "big_path_share": round(bst_timed["big_sum"] / max(1, bst_timed["list_sum"]), 4)},
        "compressed_bytes": int(clen),
    }
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if multi:
        multi.close()
    if world > 1:
        dist.barrier()
        try:
            os.unlink(box_path)
        except OSError:
            pass
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
