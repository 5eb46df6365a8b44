#!/usr/bin/env python
"""bz2b200 -- command line front end with the reference's flag surface (src/tools/cli.rs:113-303).

    bz2b200_cli.py [-1..-9|--fast|--best] [-z|-d|-t] [-k] [-f] [-c] [-q] [-v] FILE...
    bz2b200_cli.py --recover [-f] [-c] [-q] FILE.bz2...

Only block size (-1..-9), mode (-z/-d/-t) and the file list change the output, exactly as in the reference
(compress.rs:50-55 reads only files[0] and block_size; this tool also accepts several files and stdin/stdout, which
the reference advertises in its help text but does not implement, cli.rs:331-333).
Compression writes FILE.bz2 (compress.rs:59-60); decompression strips ".bz2" (the reference appends ".txt", an
author's test convenience, decompress.rs:67-70 -- not reproduced).  Input files are ALWAYS kept, as in the reference
(cli.rs:314 "-k --keep ... ALWAYS KEEPS"; compress.rs never reads keep_input_files): -k is accepted and changes nothing.
Decoding verifies every block CRC and the combined CRC (the reference only logs mismatches, decompress.rs:376-402) and
accepts concatenated streams.  All work happens on the GPU through libbz2b200.
--recover writes the bytes of every intact block of a damaged archive to FILE.recovered (FILE.bz2 -> FILE.recovered)
and prints one line per damaged block and per gap (input bits no block or footer accounts for) to stderr, with the
input bit range and the output offset where the lost bytes would have been; it exits 0 when everything was intact,
2 otherwise.
"""
import argparse
import mmap
import os
import sys

GAP_BITS = 80 + 7 + 32          # a footer, its padding and the next stream's header lie between two streams' blocks


def recover(bz, eng, name, a):
    """--recover for one file -> exit status (0: every block and stream intact)."""
    oname = (name[:-4] if name.endswith(".bz2") else name) + ".recovered"
    to_stdout = a.stdout or name == "-"
    if not to_stdout and os.path.exists(oname) and not a.force:
        sys.stderr.write("bz2b200: output file %s already exists (use -f)\n" % oname)
        return 1
    import numpy as np
    mm = None
    if name == "-":
        src = sys.stdin.buffer.read()
    else:
        with open(name, "rb") as f:
            if os.fstat(f.fileno()).st_size:
                mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)     # the input is not copied into host memory
        src = mm
    size = len(src) if src is not None else 0
    if size == 0:
        sys.stderr.write("bz2b200: %s: empty file\n" % name)
        return 2
    view = np.frombuffer(src, dtype=np.uint8)
    err = None
    dst = sys.stdout.buffer if to_stdout else open(oname, "wb")
    try:
        total, ents = eng.recover(view, dst)                       # the sink writes as blocks decode
    except BaseException as e:
        err = e.with_traceback(None)        # its frames would hold views of the map, which must be closed first
    finally:
        if dst is not sys.stdout.buffer:
            dst.close()
    del view
    if mm is not None:
        mm.close()
    if err is not None:
        raise err
    nbits = size * 8
    lines, cursor = [], 0
    for i, e in enumerate(ents):
        if e.bit - cursor > GAP_BITS:
            lines.append("lost input bits [%d, %d), output offset %d" % (cursor, e.bit, e.out_off))
        end = e.end_bit or (ents[i + 1].bit if i + 1 < len(ents) else nbits)
        if e.status != 0 and not e.flags & bz.REC_FOOTER:
            lines.append("damaged block at input bits [%d, %d), output offset %d (%s)"
                         % (e.bit, end, e.out_off, "CRC mismatch" if e.status == bz.E_CRC else "does not parse"))
        cursor = max(cursor, end)
    if nbits - cursor > GAP_BITS:
        lines.append("lost input bits [%d, %d), output offset %d" % (cursor, nbits, total))
    # complete: nothing lost, and the input ends with an intact footer (a truncated last stream has none)
    complete = not lines and bool(ents) and all(e.status == 0 for e in ents) and bool(ents[-1].flags & bz.REC_FOOTER)
    if not a.quiet:
        for ln in lines:
            sys.stderr.write("bz2b200: %s: %s\n" % (name, ln))
        sys.stderr.write("bz2b200: %s: %d bytes recovered from %d blocks%s\n"
                         % (name, total, sum(1 for e in ents if e.out_len), "" if complete else ", the archive is damaged"))
    return 0 if complete else 2

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main(argv=None):
    ap = argparse.ArgumentParser(prog="bz2b200", add_help=True, description=__doc__,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    for lv in range(1, 10):
        ap.add_argument("-%d" % lv, dest="level", action="store_const", const=lv, help="block size %d00k" % lv)
    ap.add_argument("--fast", dest="level", action="store_const", const=1)
    ap.add_argument("--best", dest="level", action="store_const", const=9)
    ap.add_argument("-z", "--compress", dest="mode", action="store_const", const="z")
    ap.add_argument("-d", "--decompress", dest="mode", action="store_const", const="d")
    ap.add_argument("-t", "--test", dest="mode", action="store_const", const="t")
    ap.add_argument("--recover", dest="mode", action="store_const", const="r",
                    help="write the intact blocks of damaged archives to FILE.recovered and report the losses")
    ap.add_argument("-k", "--keep", action="store_true", help="keep input files (always the case, as in the reference)")
    ap.add_argument("-f", "--force", action="store_true", help="overwrite existing output files")
    ap.add_argument("-c", "--stdout", action="store_true", help="write to standard output")
    ap.add_argument("-q", "--quiet", action="store_true")
    ap.add_argument("-v", "--verbose", action="count", default=0)
    ap.add_argument("-s", "--small", action="store_true", help="accepted and ignored (as in the reference)")
    ap.add_argument("-L", "--license", action="store_true", help="display software version & license")
    ap.add_argument("-V", "--version", action="store_true", help="display software version & license")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("files", nargs="*")
    a = ap.parse_args(argv)
    level = a.level or 9                      # cli.rs:90 default block size 9
    mode = a.mode or "z"

    import bzip2_rust_b200 as bz
    if a.license or a.version:
        sys.stdout.write("bz2b200, a block-sorting file compressor on B200 GPUs.  %s\n"
                         % bz.load_library().bz2b200_version().decode())
        return 0
    eng = bz.Engine(a.device)
    rc = 0
    files = a.files or ["-"]
    for name in files:
        try:
            if mode == "r":
                rc = max(rc, recover(bz, eng, name, a))
                continue
            if mode == "z":
                # pipelined: the file is read in pieces while earlier pieces are uploaded, compressed and written
                oname = name + ".bz2"
                to_stdout = a.stdout or name == "-"
                if not to_stdout and os.path.exists(oname) and not a.force:
                    sys.stderr.write("bz2b200: output file %s already exists (use -f)\n" % oname)
                    rc = 1
                    continue
                src = sys.stdin.buffer if name == "-" else open(name, "rb")
                dst = sys.stdout.buffer if to_stdout else open(oname, "wb")
                try:
                    with bz.ZStream(eng, dst, level) as z:
                        while True:
                            piece = src.read(16 << 20)
                            if not piece:
                                break
                            z.write(piece)
                finally:
                    if src is not sys.stdin.buffer:
                        src.close()
                    if dst is not sys.stdout.buffer:
                        dst.close()                       # the input file stays (reference: "ALWAYS KEEPS")
                if a.verbose and not a.quiet:
                    sys.stderr.write("  %s: %d -> %d bytes (%.3f:1)\n" % (name, z.total_in, z.total_out,
                                                                         z.total_in / max(1, z.total_out)))
                continue
            # pipelined in bounded memory: the archive is read in pieces while earlier pieces are decoded and their
            # checked bytes written; -t decodes and checks on the GPU without downloading anything
            oname = name[:-4] if name.endswith(".bz2") else name + ".out"
            to_stdout = a.stdout or name == "-"
            if mode == "d" and not to_stdout and os.path.exists(oname) and not a.force:
                sys.stderr.write("bz2b200: output file %s already exists (use -f)\n" % oname)
                rc = 1
                continue
            src = sys.stdin.buffer if name == "-" else open(name, "rb")
            dst = None
            if mode == "d":
                dst = sys.stdout.buffer if to_stdout else open(oname, "wb")
            ok = False
            try:
                with bz.DStream(eng, dst) as ds:
                    while True:
                        piece = src.read(16 << 20)
                        if not piece:
                            break
                        ds.write(piece)
                ok = True
            finally:
                if src is not sys.stdin.buffer:
                    src.close()
                if dst is not None and dst is not sys.stdout.buffer:
                    dst.close()                           # the input file stays (reference: "ALWAYS KEEPS")
                    if not ok:
                        os.remove(oname)                  # as bzip2 does: no partial output file after an error
            if mode == "t" and not a.quiet:
                sys.stderr.write("%s: ok\n" % name)
            if a.verbose and not a.quiet:
                sys.stderr.write("  %s: %d -> %d bytes (%.3f:1)\n" % (name, ds.total_in, ds.total_out,
                                                                     ds.total_in / max(1, ds.total_out)))
        except (OSError, bz.Bz2B200Error) as e:
            sys.stderr.write("bz2b200: %s: %s\n" % (name, e))
            rc = 2
    return rc


if __name__ == "__main__":
    sys.exit(main())
