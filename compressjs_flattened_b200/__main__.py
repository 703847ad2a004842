"""Command line of the bzip2 path, with the flags and defaults of the reference's bin/compressjs
(NPM/bin/compressjs:7-33,58,163-180):

  python -m compressjs_flattened_b200 -d|-z [-1 .. -9] [-b <bits>] [-t bzip2] [infile] [outfile]
  python -m compressjs_flattened_b200 -z [-1 .. -9] --index-out FILE [infile] [outfile]
  python -m compressjs_flattened_b200 -z --append FILE [--index FILE] [--index-out FILE] [infile]
  python -m compressjs_flattened_b200 -d --list [--multistream] [infile]
  python -m compressjs_flattened_b200 -d --range START:LEN [--index FILE] [--multistream] [infile] [outfile]
  python -m compressjs_flattened_b200 -d --line-index [--multistream] [infile]
  python -m compressjs_flattened_b200 -d --lines FIRST:COUNT [--index FILE] [--multistream] [infile] [outfile]
  python -m compressjs_flattened_b200 -d --grep PATTERN [--grep PATTERN ...] [--ignore-case] [--line-number] [--count]
      [--multistream] [infile] [outfile]

  -z  compress (the default), stream flavour: the input is read piece by piece (bz2b200_zstream_*), level 7 by default
  --index-out FILE  with -z: also write the line index of the stream being written (the --line-index text) to FILE, built
      while compressing, with no decode; --range and --lines take it as --index.  The stream itself is unchanged
  --append FILE  with -z: append infile (or stdin) to the bzip2 file FILE in place, recompressing only the last block of its
      last stream (Bzip2Engine.append): FILE then holds what compressing the old and the new bytes together gives, at FILE's
      level.  --index takes FILE's line index (--line-index or --index-out output; without it one is built first, a full
      decode), --index-out writes the new one (it may be the same file).  The new tail is written to a temporary file next to
      FILE first; FILE is changed only once that has succeeded, so an error leaves it as it was
  -d  decompress the FIRST stream of the input, stream flavour (bz2b200_dstream_*); --multistream decodes all of them
      (an extension: the reference's command line never passes the flag, NPM/bin/compressjs:166)
  -b  with -d: extract the single block whose signature starts at bit <bits> (Bzip2.decompressBlock)
  --recover  write what survives of a damaged file (every block that decodes and matches its CRC, all streams); one line per
      damaged region on stderr; exit status 0 when everything was intact, 2 when anything was lost
  --list  print the block index (Bzip2Index.to_text: one line per block, stream, level, bit range, output range, CRC) to
      stdout; with --multistream it covers every stream
  --range START:LEN  write the decompressed bytes [START, START+LEN), clipped like a slice, decoding only the blocks that
      hold them; --index FILE takes the index from --list output, otherwise it is built first (a full decode).  A negative
      START (counted from the end, like a slice) must be written --range=START:LEN, since -1 .. -9 are flags; a line index
      (--line-index or --index-out output) is accepted as --index too
  --grep PATTERN  write the lines of the decompressed output that contain PATTERN (a fixed string, UTF-8; repeat the flag
      for several), searched on the GPU (Bzip2Engine.search), like bzgrep -F; --ignore-case folds ASCII letters,
      --line-number puts "N:" (1-based) before each line, --count prints the number of matching lines instead.  Exit
      status 0 when a line matched, 1 when none did, as with grep
  --line-index  print the line index (Bzip2LineIndex.to_text: the --list columns plus the '\n' bytes of every block, under a
      "# lines" total) to stdout; with --multistream it covers every stream
  --lines FIRST:COUNT  write COUNT lines from line FIRST (1-based, the numbers --grep --line-number prints), clipped to the
      output, decoding only the blocks that hold them; --index FILE takes the index from --line-index output, otherwise it
      is built first (a full decode)
Usage errors (flags that contradict each other) exit with status 1.
If <infile> is omitted, reads from stdin; if <outfile> is omitted, writes to stdout.  Needs a CUDA device: no CPU fallback."""
import argparse
import os
import shutil
import sys
import tempfile

from .bzip2 import MATCH_FIRST_IN_LINE, NO_SIGNATURE, Bzip2Index, Bzip2LineIndex, Err


def _append_in_place(engine, path, src, index, chunk_bytes):
    """engine.append of src to the file at `path`: the tail goes to a temporary file next to it, and only once the append
    has succeeded is the file overwritten from `keep`, truncated and synced.  Returns the new line index."""
    fd, tmp = tempfile.mkstemp(prefix=".append-", dir=os.path.dirname(os.path.abspath(path)))
    try:
        with os.fdopen(fd, "w+b") as t:
            keep, _, index = engine.append(path, src, index, sink=t, chunk_bytes=chunk_bytes)
            t.seek(0)
            with open(path, "r+b") as fh:
                fh.seek(keep)
                shutil.copyfileobj(t, fh, 1 << 20)
                fh.truncate()
                fh.flush()
                os.fsync(fh.fileno())
    finally:
        os.unlink(tmp)
    return index


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
    ap.add_argument("--index", default=None, metavar="FILE",
                    help="with --range: the block index (--list output) or a line index; with --lines: the line index")
    ap.add_argument("--index-out", default=None, metavar="FILE", help="with -z: write the line index of the stream to FILE")
    ap.add_argument("--append", default=None, metavar="FILE", help="with -z: append the input to the bzip2 file FILE in place")
    ap.add_argument("--line-index", action="store_true", help="with -d: print the line index")
    ap.add_argument("--lines", default=None, metavar="FIRST:COUNT", help="with -d: write COUNT lines from line FIRST (1-based)")
    ap.add_argument("--grep", action="append", default=None, metavar="PATTERN", help="with -d: write the lines that contain PATTERN")
    ap.add_argument("--ignore-case", action="store_true", help="with --grep: ASCII letters match either case")
    ap.add_argument("--line-number", action="store_true", help="with --grep: prefix each line with its 1-based number and ':'")
    ap.add_argument("--count", action="store_true", help="with --grep: print the number of matching lines")
    a = ap.parse_args(argv)
    not_z = (("-d", a.decompress), ("--list", a.list), ("--range", a.range is not None), ("--grep", bool(a.grep)),
             ("--line-index", a.line_index), ("--lines", a.lines is not None), ("--recover", a.recover), ("-b", a.block >= 0))
    for opt in ("--append", "--index-out"):
        if getattr(a, opt[2:].replace("-", "_")) is None:
            continue
        for flag, on in not_z:
            if on:
                print(f"{opt} can only be used with -z, not with {flag}", file=sys.stderr)
                return 1
    if a.append is not None:
        if any(getattr(a, f"l{lv}") for lv in range(1, 10)):
            print("--append keeps the level of the file it appends to: a compression level has no effect", file=sys.stderr)
            return 1
        if a.outfile is not None:
            print("--append changes FILE in place and takes no outfile", file=sys.stderr)
            return 1
    for flag, on in (("--ignore-case", a.ignore_case), ("--line-number", a.line_number), ("--count", a.count)):
        if on and not a.grep:
            print(f"{flag} can only be used with --grep", file=sys.stderr)
            return 1
    modes = (("--list", a.list, "listing"), ("--range", a.range is not None, "reading a range"), ("--grep", bool(a.grep), "searching"),
             ("--line-index", a.line_index, "listing lines"), ("--lines", a.lines is not None, "reading lines"))
    for flag, on, verb in modes:
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
    chosen = [flag for flag, on, _ in modes if on]
    if len(chosen) > 1:
        print(f"{chosen[0]} and {chosen[1]} can't be used together", file=sys.stderr)
        return 1
    if a.index is not None and a.range is None and a.lines is None and a.append is None:
        print("--index can only be used with --range", file=sys.stderr)
        return 1
    if a.range is not None:
        try:
            start, length = (int(v) for v in a.range.split(":"))
        except ValueError:
            print(f"--range takes START:LEN, not {a.range}", file=sys.stderr)
            return 1
    if a.lines is not None:
        try:
            first, count = (int(v) for v in a.lines.split(":"))
        except ValueError:
            first = 0
        if first < 1:
            print(f"--lines takes FIRST:COUNT with FIRST from 1, not {a.lines}", file=sys.stderr)
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
                    text = fh.read()
                index = Bzip2LineIndex.from_text(text).blocks if text.startswith(Bzip2LineIndex.HEADER) else Bzip2Index.from_text(text)
            else:
                index = Bzip2.index(data, a.multistream)
            dst.write(Bzip2.decompressRange(data, index, start, length))
        elif a.line_index:
            dst.write(Bzip2.lineIndex(src.read(), a.multistream).to_text().encode())
        elif a.lines is not None:
            data = src.read()
            if a.index is not None:
                with open(a.index) as fh:
                    text = fh.read()
                if text.startswith(Bzip2Index.HEADER):
                    print(f"--lines needs a line index (--line-index output), and {a.index} is a block index", file=sys.stderr)
                    return 1
                index = Bzip2LineIndex.from_text(text)
            else:
                index = Bzip2.lineIndex(data, a.multistream)
            dst.write(b"".join(Bzip2.decompressLines(data, index, [(first - 1, count)])))
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
        elif a.append is not None:
            index = None
            if a.index is not None:
                with open(a.index) as fh:
                    text = fh.read()
                if text.startswith(Bzip2Index.HEADER):
                    print(f"--append needs a line index (--line-index or --index-out output), and {a.index} is a block index", file=sys.stderr)
                    return 1
                index = Bzip2LineIndex.from_text(text)
            index = _append_in_place(Bzip2, a.append, src, index, a.chunk_mb << 20)
            if a.index_out is not None:
                with open(a.index_out, "w") as fh:
                    fh.write(index.to_text())
        elif a.index_out is not None:
            _, index = Bzip2.compressStream(src, dst, level, chunk_bytes=a.chunk_mb << 20, index=True)
            with open(a.index_out, "w") as fh:
                fh.write(index.to_text())
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
