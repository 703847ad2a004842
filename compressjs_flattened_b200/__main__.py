"""Command line of the bzip2 path, with the flags and defaults of the reference's bin/compressjs
(NPM/bin/compressjs:7-33,58,163-180):

  python -m compressjs_flattened_b200 -d|-z [-1 .. -9] [-b <bits>] [-t bzip2] [infile] [outfile]
  python -m compressjs_flattened_b200 -d --list [--multistream] [infile]
  python -m compressjs_flattened_b200 -d --range START:LEN [--index FILE] [--multistream] [infile] [outfile]
  python -m compressjs_flattened_b200 -d --grep PATTERN [--grep PATTERN ...] [--ignore-case] [--line-number] [--count]
      [--multistream] [infile] [outfile]

  -z  compress (the default), stream flavour: the input is read piece by piece (bz2b200_zstream_*), level 7 by default
  -d  decompress the FIRST stream of the input, stream flavour (bz2b200_dstream_*); --multistream decodes all of them
      (an extension: the reference's command line never passes the flag, NPM/bin/compressjs:166)
  -b  with -d: extract the single block whose signature starts at bit <bits> (Bzip2.decompressBlock)
  --recover  write what survives of a damaged file (every block that decodes and matches its CRC, all streams); one line per
      damaged region on stderr; exit status 0 when everything was intact, 2 when anything was lost
  --list  print the block index (Bzip2Index.to_text: one line per block, stream, level, bit range, output range, CRC) to
      stdout; with --multistream it covers every stream
  --range START:LEN  write the decompressed bytes [START, START+LEN), clipped like a slice, decoding only the blocks that
      hold them; --index FILE takes the index from --list output, otherwise it is built first (a full decode).  A negative
      START (counted from the end, like a slice) must be written --range=START:LEN, since -1 .. -9 are flags
  --grep PATTERN  write the lines of the decompressed output that contain PATTERN (a fixed string, UTF-8; repeat the flag
      for several), searched on the GPU (Bzip2Engine.search), like bzgrep -F; --ignore-case folds ASCII letters,
      --line-number puts "N:" (1-based) before each line, --count prints the number of matching lines instead.  Exit
      status 0 when a line matched, 1 when none did, as with grep
Usage errors (flags that contradict each other) exit with status 1.
If <infile> is omitted, reads from stdin; if <outfile> is omitted, writes to stdout.  Needs a CUDA device: no CPU fallback."""
import argparse
import sys

from .bzip2 import MATCH_FIRST_IN_LINE, NO_SIGNATURE, Bzip2Index, Err


def main(argv=None, engine=None):
    ap = argparse.ArgumentParser(prog="compressjs_flattened_b200", usage="%(prog)s -d|-z [infile] [outfile]", description=__doc__,
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("-d", "--decompress", action="store_true", help="Decompress stdin to stdout")
    ap.add_argument("-z", "--compress", action="store_true", help="Compress stdin to stdout")
    ap.add_argument("-b", "--block", type=int, default=-1, metavar="<n>", help="Extract a single block, starting at <n> bits.")
    ap.add_argument("-t", dest="type", default="bzip2", metavar="<compressor>", help="Select compressor type (only bzip2 is on this path)")
    ap.add_argument("--multistream", action="store_true", help="with -d: decode every concatenated stream")
    ap.add_argument("--chunk-mb", type=int, default=64, help="input collected before its blocks are compressed")
    for lv in range(1, 10):
        ap.add_argument(f"-{lv}", dest=f"l{lv}", action="store_true",
                        help="Fastest/largest compression" if lv == 1 else "Slowest/smallest compression" if lv == 9 else argparse.SUPPRESS)
    ap.add_argument("infile", nargs="?", default=None)
    ap.add_argument("outfile", nargs="?", default=None)
    ap.add_argument("--recover", action="store_true", help="write the intact blocks of a damaged file, report the damage")
    ap.add_argument("--list", action="store_true", help="with -d: print the block index")
    ap.add_argument("--range", default=None, metavar="START:LEN", help="with -d: write only these decompressed bytes")
    ap.add_argument("--index", default=None, metavar="FILE", help="with --range: the block index (--list output)")
    ap.add_argument("--grep", action="append", default=None, metavar="PATTERN", help="with -d: write the lines that contain PATTERN")
    ap.add_argument("--ignore-case", action="store_true", help="with --grep: ASCII letters match either case")
    ap.add_argument("--line-number", action="store_true", help="with --grep: prefix each line with its 1-based number and ':'")
    ap.add_argument("--count", action="store_true", help="with --grep: print the number of matching lines")
    a = ap.parse_args(argv)
    for flag, on in (("--ignore-case", a.ignore_case), ("--line-number", a.line_number), ("--count", a.count)):
        if on and not a.grep:
            print(f"{flag} can only be used with --grep", file=sys.stderr)
            return 1
    for flag, on, verb in (("--list", a.list, "listing"), ("--range", a.range is not None, "reading a range"), ("--grep", bool(a.grep), "searching")):
        if not on:
            continue
        if a.compress:
            print(f"{flag} can only be used without -z", file=sys.stderr)
            return 1
        if a.block >= 0:
            print(f"{flag} and --block can't be used together", file=sys.stderr)
            return 1
        if a.recover:
            print(f"{flag} and --recover can't be used together", file=sys.stderr)
            return 1
        if any(getattr(a, f"l{lv}") for lv in range(1, 10)):
            print(f"Compression level has no effect when {verb}.", file=sys.stderr)
            return 1
        a.decompress = True
    if a.list and a.range is not None:
        print("--list and --range can't be used together", file=sys.stderr)
        return 1
    for flag, on in (("--list", a.list), ("--range", a.range is not None)):
        if on and a.grep:
            print(f"{flag} and --grep can't be used together", file=sys.stderr)
            return 1
    if a.index is not None and a.range is None:
        print("--index can only be used with --range", file=sys.stderr)
        return 1
    if a.range is not None:
        try:
            start, length = (int(v) for v in a.range.split(":"))
        except ValueError:
            print(f"--range takes START:LEN, not {a.range}", file=sys.stderr)
            return 1
    if a.recover:
        if a.compress:
            print("--recover can only be used without -z", file=sys.stderr)
            return 1
        if a.block >= 0:
            print("--recover and --block can't be used together", file=sys.stderr)
            return 1
        if any(getattr(a, f"l{lv}") for lv in range(1, 10)):
            print("Compression level has no effect when recovering.", file=sys.stderr)
            return 1
        a.decompress = True
    if not a.decompress:
        a.compress = True
    if a.decompress and a.compress:
        print("Must specify either -d or -z.", file=sys.stderr)
        return 1
    if a.compress and a.block >= 0:
        print("--block can only be used with decompression", file=sys.stderr)
        return 1
    level = None
    for lv in range(1, 10):
        if getattr(a, f"l{lv}"):
            if level:
                print(f"Can't specify both -{level} and -{lv}", file=sys.stderr)
                return 1
            level = lv
    if level and a.decompress:
        print("Compression level has no effect when decompressing.", file=sys.stderr)
        return 1
    level = level or 7   # NPM/bin/compressjs:58
    if a.type.lower() not in ("bzip", "bzip2"):
        print(f"Unknown compressor on this path: {a.type} (only bzip2; SURVEY.md section 8)", file=sys.stderr)
        return 1
    if engine is None:
        from .bzip2 import Bzip2 as engine
    Bzip2 = engine
    src = open(a.infile, "rb") if a.infile else sys.stdin.buffer
    dst = open(a.outfile, "wb") if a.outfile else sys.stdout.buffer
    status = 0
    try:
        if a.recover:
            data, regions = Bzip2.recover(src.read())
            dst.write(data)
            names = {v: k for k, v in vars(Err).items() if isinstance(v, int)}
            for r in regions:
                if r.status:
                    sig = " (no signature)" if r.flags & NO_SIGNATURE else ""
                    print(f"bits {r.bit_begin}-{r.bit_end}: {r.kind_name}{sig} {names.get(r.status, r.status)}", file=sys.stderr)
                    status = 2
        elif a.list:
            dst.write(Bzip2.index(src.read(), a.multistream).to_text().encode())
        elif a.range is not None:
            data = src.read()
            if a.index is not None:
                with open(a.index) as fh:
                    index = Bzip2Index.from_text(fh.read())
            else:
                index = Bzip2.index(data, a.multistream)
            dst.write(Bzip2.decompressRange(data, index, start, length))
        elif a.grep:
            r = Bzip2.search(src.read(), a.grep, ignore_case=a.ignore_case, max_matches=0 if a.count else None, multistream=a.multistream,
                             lines=not a.count)
            if a.count:
                dst.write(f"{r.total_lines}\n".encode())
            elif a.line_number:
                numbers = r.matches["line"][(r.matches["flags"] & MATCH_FIRST_IN_LINE) != 0]
                dst.write(b"".join(b"%d:%s\n" % (int(n) + 1, ln) for n, ln in zip(numbers, r.lines.split(b"\n"))))
            else:
                dst.write(r.lines)
            status = 0 if r.total_lines else 1
        elif a.decompress and a.block >= 0:
            dst.write(Bzip2.decompressBlock(src.read(), a.block))
        elif a.decompress:
            Bzip2.decompressStream(src, dst, a.multistream)
        else:
            Bzip2.compressStream(src, dst, level, chunk_bytes=a.chunk_mb << 20)
    finally:
        if a.infile:
            src.close()
        if a.outfile:
            dst.close()
        else:
            dst.flush()
    return status


if __name__ == "__main__":
    sys.exit(main())
