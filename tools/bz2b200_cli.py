#!/usr/bin/env python
"""bz2b200 -- command line front end with the reference's flag surface (src/tools/cli.rs:113-303).

    bz2b200_cli.py [-1..-9|--fast|--best] [-z|-d|-t] [-k] [-f] [-c] [-q] [-v] FILE...

Only block size (-1..-9), mode (-z/-d/-t) and the file list change the output, exactly as in the reference
(compress.rs:50-55 reads only files[0] and block_size; this tool also accepts several files and stdin/stdout, which
the reference advertises in its help text but does not implement, cli.rs:331-333).
Compression writes FILE.bz2 (compress.rs:59-60); decompression strips ".bz2" (the reference appends ".txt", an
author's test convenience, decompress.rs:67-70 -- not reproduced).  Input files are ALWAYS kept, as in the reference
(cli.rs:314 "-k --keep ... ALWAYS KEEPS"; compress.rs never reads keep_input_files): -k is accepted and changes nothing.
Decoding verifies every block CRC and the combined CRC (the reference only logs mismatches, decompress.rs:376-402) and
accepts concatenated streams.  All work happens on the GPU through libbz2b200.
"""
import argparse
import os
import sys

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
