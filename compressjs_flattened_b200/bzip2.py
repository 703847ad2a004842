"""Host-side mirror of the reference's `Bzip2` object (BJ = /root/reference/Bzip2_joined_.js).

    Bzip2.compressFile(input, output=None, props=None)        BJ:2199-2249
    Bzip2.decompressFile(input, output=None, multistream=False)  BJ:1769-1796
    Bzip2.decompressBlock(input, bitpos, output=None)         BJ:1797-1818
    Bzip2.table(input, callback, multistream=False)           BJ:1823-1863

Random access (no counterpart in the reference): Bzip2Engine.index, decompressRanges, decompressRange and open.
Lines by number (no counterpart in the reference): Bzip2Engine.lineIndex, decompressLines and lineSpans.
The same line index while compressing, with no decode: Bzip2Engine.compressIndexed and compressStream(..., index=True).
Appending to a stream and its line index, recompressing only the last block: Bzip2Engine.append.
Search (bzgrep -F, no counterpart in the reference): Bzip2Engine.search.

Same names, argument meaning and error behaviour as the JavaScript API; the work is done by
the CUDA library behind include/bz2b200.h.  Coercions follow Util.coerceInputStream /
coerceOutputStream (BJ:178-272):
  input : bytes-like / list of ints / object with readByte() (-1 at EOF)
  output: None -> returns a new bytes object (the JS returns a fresh Uint8Array);
          int  -> expected size, TypeError('outputsize does not match decoded input') if wrong;
          bytearray/memoryview -> filled in place, same size check;
          object with writeByte(b) -> bytes pushed one at a time, flush() called if present,
          the object itself is returned.
Errors: `Bzip2Error` (a TypeError, like the JS `_throw`, BJ:1384-1391) carrying `.errorCode`;
a bad level raises ValueError('Invalid block size multiplier') (JS: Error, BJ:2208).
"""
import builtins
import ctypes as C
import io
import mmap
import os
from collections import namedtuple

import numpy as np

from . import _native

EOF = -1


class Bzip2Error(TypeError):
    def __init__(self, code, message):
        super().__init__(message)
        self.errorCode = code


class Err:  # BJ:1365-1375
    OK = 0
    LAST_BLOCK = -1
    NOT_BZIP_DATA = -2
    UNEXPECTED_INPUT_EOF = -3
    UNEXPECTED_OUTPUT_EOF = -4
    DATA_ERROR = -5
    OUT_OF_MEMORY = -6
    OBSOLETE_INPUT = -7
    END_OF_BLOCK = -8


REGION_HEADER, REGION_BLOCK, REGION_END, REGION_UNKNOWN = 0, 1, 2, 3   # bz2b200_region.kind
REGION_KINDS = ("HEADER", "BLOCK", "END", "UNKNOWN")
NO_SIGNATURE = 1   # bz2b200_region.flags: a block parsed where its predecessor ends (its signature is damaged)

# One region of Bzip2Engine.recover: input bits [bit_begin, bit_end), its kind (and kind_name), status (0 or an Err code),
# where its bytes are in the recovered data, the stored CRC, the stream (END regions before it) and flags.
Region = namedtuple("Region", "bit_begin bit_end kind kind_name status out_offset out_bytes crc stream flags")


# bz2b200_block_entry (include/bz2b200.h), field for field
INDEX_DTYPE = np.dtype([("bit_begin", "<u8"), ("bit_end", "<u8"), ("out_offset", "<u8"), ("out_bytes", "<u4"), ("crc", "<u4"),
                        ("stream", "<u4"), ("level", "<u4")])
assert INDEX_DTYPE.itemsize == C.sizeof(_native.BlockEntry)
LEVEL9_BLOCK = 900_000

# bz2b200_match (include/bz2b200.h), field for field
MATCH_DTYPE = np.dtype([("offset", "<u8"), ("line", "<u8"), ("line_begin", "<u8"), ("line_end", "<u8"), ("pattern", "<u4"), ("flags", "<u4")])
assert MATCH_DTYPE.itemsize == C.sizeof(_native.Match)
SEARCH_IGNORE_CASE = 1   # bz2b200_search flags
MATCH_FIRST_IN_LINE = 1  # bz2b200_match.flags: the first match of its line
SEARCH_MAX_PATTERNS = SEARCH_MAX_LEN = 256

# Bzip2Engine.search: matches (numpy array of MATCH_DTYPE, sorted by offset then pattern), the exact totals whatever
# max_matches cut, the decoded size, and the lines (bytes, or None when not asked for)
SearchResult = namedtuple("SearchResult", "matches total_matches total_lines out_bytes lines")


def _patterns(patterns):
    """bytes / str (one pattern) or an iterable of them -> list of bytes, within the limits of bz2b200_search"""
    if isinstance(patterns, (bytes, bytearray, memoryview, str)):
        patterns = [patterns]
    pats = [p.encode() if isinstance(p, str) else bytes(p) for p in patterns]
    if not 1 <= len(pats) <= SEARCH_MAX_PATTERNS:
        raise ValueError(f"search takes 1..{SEARCH_MAX_PATTERNS} patterns, not {len(pats)}")
    for i, p in enumerate(pats):
        if not 1 <= len(p) <= SEARCH_MAX_LEN:
            raise ValueError(f"pattern {i}: length must be 1..{SEARCH_MAX_LEN}, not {len(p)}")
    return pats   # the largest block a stream can have: the buffer of Bzip2Engine.open


def _level(props):
    """the level of compressFile's props (BJ:2204-2210): a number 1..9, 9 when props is not a number"""
    level = props if isinstance(props, (int, float)) and not isinstance(props, bool) else 9
    if level < 1 or level > 9 or int(level) != level:
        raise ValueError("Invalid block size multiplier")
    return int(level)


def _line_index_call(owner, fn, *args):
    """fn(*args, entries, newlines, count, total_lines) -> a Bzip2LineIndex of what it returned; errors through owner._raise"""
    ptr, nlp, n, lines = C.POINTER(_native.BlockEntry)(), C.POINTER(C.c_uint32)(), C.c_size_t(), C.c_uint64()
    rc = fn(*args, C.byref(ptr), C.byref(nlp), C.byref(n), C.byref(lines))
    if rc:
        owner._raise(rc)
    try:
        raw = _native.take_bytes(C.cast(ptr, C.POINTER(C.c_uint8)), n.value * INDEX_DTYPE.itemsize)
        nl = _native.take_bytes(C.cast(nlp, C.POINTER(C.c_uint8)), n.value * 4)
    finally:
        owner._L.bz2b200_free(ptr)
        owner._L.bz2b200_free(nlp)
    return Bzip2LineIndex(Bzip2Index(np.frombuffer(raw, dtype=INDEX_DTYPE)), np.frombuffer(nl, dtype=np.uint32), lines.value)


def _compress_indexed(owner, fn, handle, input, props, *extra):
    """fn = bz2b200_compress_indexed or bz2b200_pool_compress_indexed on `handle` (extra: the arguments after the level)
    -> (stream bytes, Bzip2LineIndex)"""
    level = _level(props)
    a = _coerce_input(input)
    out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
    index = _line_index_call(owner, fn, handle, a.ctypes.data, a.size, level, *extra, C.byref(out), C.byref(n))
    return owner._take(out, n.value), index


def _search(owner, fn, handle, input, patterns, ignore_case, max_matches, multistream, lines, *extra):
    """fn = bz2b200_search or bz2b200_pool_search on `handle` (extra: the arguments between max_matches and the
    results), its arguments checked and packed and its results unpacked into a SearchResult; errors through owner._raise"""
    pats = _patterns(patterns)
    if max_matches is None:
        max_matches = (1 << 64) - 1
    elif max_matches < 0:
        raise ValueError("max_matches must not be negative")
    max_matches = min(int(max_matches), (1 << 64) - 1)
    a = _coerce_input(input)
    packed = np.frombuffer(b"".join(pats), dtype=np.uint8)
    lens = np.array([len(p) for p in pats], dtype=np.uint32)
    mp, nm, tot = C.POINTER(_native.Match)(), C.c_size_t(), _native.SearchTotals()
    lp, nl = C.POINTER(C.c_uint8)(), C.c_size_t()
    rc = fn(handle, a.ctypes.data, a.size, int(bool(multistream)), packed.ctypes.data, lens.ctypes.data, len(pats),
            SEARCH_IGNORE_CASE if ignore_case else 0, int(max_matches), *extra, C.byref(mp), C.byref(nm), C.byref(tot),
            C.byref(lp) if lines else None, C.byref(nl) if lines else None)
    if rc:
        owner._raise(rc)
    try:
        raw = _native.take_bytes(C.cast(mp, C.POINTER(C.c_uint8)), nm.value * MATCH_DTYPE.itemsize)
    finally:
        owner._L.bz2b200_free(mp)
    text = owner._take(lp, nl.value) if lines else None
    return SearchResult(np.frombuffer(raw, dtype=MATCH_DTYPE), tot.matches, tot.lines, tot.out_bytes, text)


class Bzip2Index:
    """The blocks of a bzip2 file (Bzip2Engine.index): `entries` is a numpy structured array with the layout of
    bz2b200_block_entry -- bit_begin, bit_end, out_offset, out_bytes, crc, stream, level -- one row per block in stream order."""
    HEADER = "# bzip2 block index v1"
    _TEXT_FIELDS = ("stream", "level", "bit_begin", "bit_end", "out_offset", "out_bytes", "crc")

    def __init__(self, entries):
        self.entries = np.ascontiguousarray(entries, dtype=INDEX_DTYPE)

    @property
    def total(self):
        """decompressed bytes the index covers"""
        if not len(self.entries):
            return 0
        last = self.entries[-1]
        return int(last["out_offset"]) + int(last["out_bytes"])

    def __len__(self):
        return len(self.entries)

    def to_text(self):
        """One line per block under a header line: stream, level, bit_begin, bit_end, out_offset, out_bytes, crc (hex), tab-separated."""
        return "\n".join([self.HEADER] + ["\t".join(r) for r in self._text_rows()]) + "\n"

    def _text_rows(self):
        for e in self.entries:
            yield [str(int(e[f])) for f in self._TEXT_FIELDS[:-1]] + [f"{int(e['crc']):08x}"]

    @classmethod
    def from_text(cls, text):
        """The inverse of to_text; ValueError on anything else."""
        lines = text.splitlines()
        if not lines or lines[0] != cls.HEADER:
            raise ValueError(f"not a block index: the first line must be {cls.HEADER!r}")
        return cls(_parse_rows(lines[1:], 2, cls._TEXT_FIELDS)[0])


def _parse_rows(lines, first_no, fields):
    """tab-separated rows of `fields` (those of Bzip2Index._TEXT_FIELDS, then optionally "newlines", a u32), numbered from
    line first_no -> (the block columns as an INDEX_DTYPE array, the newlines column as uint32 or None); ValueError on
    anything else"""
    rows, extra = [], []
    for no, line in enumerate(lines, first_no):
        parts = line.split("\t")
        if len(parts) != len(fields):
            raise ValueError(f"line {no}: {len(parts)} fields, expected {len(fields)}")
        vals = []
        for name, p in zip(fields, parts):
            digits = "0123456789abcdefABCDEF" if name == "crc" else "0123456789"
            if not p or any(ch not in digits for ch in p):
                raise ValueError(f"line {no}: bad {name} {p!r}")
            v = int(p, 16 if name == "crc" else 10)
            if v >= 1 << ((INDEX_DTYPE[name].itemsize if name in INDEX_DTYPE.names else 4) * 8):
                raise ValueError(f"line {no}: {name} {p} out of range")
            vals.append(v)
        rec = dict(zip(fields, vals))
        rows.append(tuple(rec[f] for f in INDEX_DTYPE.names))
        extra.append(rec.get("newlines", 0))
    return np.array(rows, dtype=INDEX_DTYPE), (np.array(extra, dtype=np.uint32) if "newlines" in fields else None)


class Bzip2LineIndex:
    """The blocks of a bzip2 file and the '\n' bytes of each (Bzip2Engine.lineIndex): `blocks` is a Bzip2Index,
    `newlines` a uint32 array with one count per block, `total_lines` the number of lines of the decompressed output (the
    '\n' bytes, plus one when the output does not end with '\n') and `total` its bytes."""
    HEADER = "# bzip2 line index v1"
    _TEXT_FIELDS = Bzip2Index._TEXT_FIELDS + ("newlines",)

    def __init__(self, blocks, newlines, total_lines):
        self.blocks = blocks if isinstance(blocks, Bzip2Index) else Bzip2Index(blocks)
        self.newlines = np.ascontiguousarray(newlines, dtype=np.uint32)
        self.total_lines = int(total_lines)
        if len(self.newlines) != len(self.blocks):
            raise ValueError(f"{len(self.newlines)} newline counts for {len(self.blocks)} blocks")

    @property
    def total(self):
        """decompressed bytes the index covers"""
        return self.blocks.total

    def __len__(self):
        return len(self.blocks)

    def to_text(self):
        """The header line, "# lines <total_lines>", then one line per block: the columns of Bzip2Index.to_text and the
        block's '\n' bytes, tab-separated."""
        rows = (r + [str(int(k))] for r, k in zip(self.blocks._text_rows(), self.newlines))
        return "\n".join([self.HEADER, f"# lines {self.total_lines}"] + ["\t".join(r) for r in rows]) + "\n"

    @classmethod
    def from_text(cls, text):
        """The inverse of to_text; ValueError on anything else, and on counts that do not add up (a count above its
        block's bytes, or total_lines other than the '\n' bytes, or those + 1 when the last line has no '\n')."""
        lines = text.splitlines()
        if not lines or lines[0] != cls.HEADER:
            raise ValueError(f"not a line index: the first line must be {cls.HEADER!r}")
        head = lines[1].split(" ") if len(lines) > 1 else []
        if len(head) != 3 or head[:2] != ["#", "lines"] or not head[2].isascii() or not head[2].isdigit():
            raise ValueError("line 2: expected '# lines <total_lines>'")
        entries, newlines = _parse_rows(lines[2:], 3, cls._TEXT_FIELDS)
        ix = cls(entries, newlines, int(head[2]))
        nl = int(newlines.sum(dtype=np.uint64))
        if (newlines > entries["out_bytes"]).any():
            raise ValueError("a block's newlines exceed its bytes")
        if ix.total_lines not in ((nl, nl + 1) if nl and ix.total else (1,) if ix.total else (0,)):
            raise ValueError(f"# lines {ix.total_lines} does not match {nl} '\\n' bytes in {ix.total} bytes")
        return ix


class _RangeReader(io.RawIOBase):
    """Raw side of Bzip2Engine.open: every readinto is one decompressRanges call."""

    def __init__(self, eng, data, index):
        super().__init__()
        self._eng, self._data, self._index = eng, data, index
        self._total, self._pos = index.total, 0

    def readable(self):
        return True

    def seekable(self):
        return True

    def tell(self):
        return self._pos

    def seek(self, offset, whence=io.SEEK_SET):
        base = {io.SEEK_SET: 0, io.SEEK_CUR: self._pos, io.SEEK_END: self._total}.get(whence)
        if base is None:
            raise ValueError(f"invalid whence ({whence})")
        if base + offset < 0:
            raise ValueError(f"negative seek position {base + offset}")
        self._pos = base + offset
        return self._pos

    def readinto(self, b):
        mv = memoryview(b).cast("B")
        n = max(0, min(len(mv), self._total - self._pos))
        if n:
            mv[:n] = self._eng.decompressRange(self._data, self._index, self._pos, n)
            self._pos += n
        return n

    def readall(self):
        data = self._eng.decompressRange(self._data, self._index, self._pos, max(0, self._total - self._pos))
        self._pos += len(data)
        return data


def _coerce_input(inp):
    """Util.coerceInputStream (BJ:178-220): drain any source into a contiguous uint8 array."""
    if hasattr(inp, "readByte"):
        out = bytearray()
        while True:
            ch = inp.readByte()
            if ch == EOF:
                break
            out.append(ch)
        return np.frombuffer(bytes(out), dtype=np.uint8)
    if isinstance(inp, np.ndarray):
        return np.ascontiguousarray(inp, dtype=np.uint8).reshape(-1)
    if isinstance(inp, (bytes, bytearray, memoryview)):
        return np.frombuffer(inp, dtype=np.uint8)
    return np.asarray(list(inp), dtype=np.uint8)


def _map_path(input):
    """a path -> the file's bytes, memory-mapped read-only (b"" for an empty file); anything else as it is"""
    if isinstance(input, (str, os.PathLike)):
        with builtins.open(input, "rb") as fh:
            size = os.fstat(fh.fileno()).st_size
            return np.frombuffer(mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ), dtype=np.uint8) if size else b""
    return input


def _deliver(data, output):
    """Util.coerceOutputStream + BufferStream.getBuffer (BJ:222-272)."""
    if output is None or output is False:
        return bytes(data)
    if hasattr(output, "writeByte"):
        for b in data:
            output.writeByte(b)
        if hasattr(output, "flush"):
            output.flush()
        return output
    if isinstance(output, int):
        if output != len(data):
            raise TypeError("outputsize does not match decoded input")
        return bytes(data)
    mv = memoryview(output)
    if len(mv) != len(data):
        raise TypeError("outputsize does not match decoded input")
    mv[:] = data
    return output


class Bzip2Engine:
    """One CUDA context (one GPU).  `Bzip2` below is the process-wide default instance."""

    def __init__(self, device=0, library=None):
        self._lib = library or _native.default_library()
        self._L = self._lib.L
        self._ctx = C.c_void_p()
        rc = self._L.bz2b200_create(device, C.byref(self._ctx))
        if rc:
            raise RuntimeError(f"bz2b200_create(device={device}) failed ({rc}): no usable CUDA device; "
                               "this package has no CPU fallback")
        self.Err = Err

    def close(self):
        if self._ctx:
            self._L.bz2b200_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- error mapping (BJ:1376-1391) --
    def _raise(self, rc):
        if rc == _native.E_LEVEL:
            raise ValueError("Invalid block size multiplier")
        msg = self._L.bz2b200_strerror(rc).decode()
        if rc in (_native.E_CUDA, _native.E_ARG):
            raise RuntimeError(msg + ": " + self._L.bz2b200_last_error(self._ctx).decode())
        detail = self._L.bz2b200_last_error(self._ctx).decode()
        raise Bzip2Error(rc, msg + (": " + detail if detail else ""))  # _throw(status, optDetail), BJ:1384-1391

    def _take(self, ptr, n):
        data = _native.take_bytes(ptr, n)
        self._L.bz2b200_free(ptr)
        return data

    # -- the four methods of the reference object --
    def compressFile(self, input, output=None, props=None):
        level = _level(props)
        a = _coerce_input(input)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_compress(self._ctx, a.ctypes.data, a.size, level, C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return _deliver(self._take(out, n.value), output)

    def compressIndexed(self, input, props=None):
        """compressFile that also returns the stream's line index, computed while compressing (no decode):
        (stream bytes, Bzip2LineIndex), the index equal to lineIndex(stream).  The stream is compressFile's."""
        return _compress_indexed(self, self._L.bz2b200_compress_indexed, self._ctx, input, props)

    # -- the stream flavour (SURVEY 8f N2; what NPM/bin/compressjs:163-180 does with {readByte}/{writeByte} streams) --
    @staticmethod
    def _reader(source, piece):
        if hasattr(source, "read"):
            return source.read
        if hasattr(source, "readByte"):
            def read(n):
                out = bytearray()
                while len(out) < n:
                    ch = source.readByte()
                    if ch == EOF:
                        break
                    out.append(ch)
                return bytes(out)
            return read
        view, pos = memoryview(_coerce_input(source)), [0]

        def read(n):
            b = view[pos[0]:pos[0] + n].tobytes()
            pos[0] += len(b)
            return b
        return read

    def _pump(self, kind, handle, source, sink, piece, finished=None):
        """read pieces, feed them, hand on what comes back; the C stream object does the work (csrc/stream_abi.inl).
        finished: called with the handle after finish succeeded, before the handle is closed; the result is then
        (what is returned without it, what finished returned)"""
        L = self._L
        feed, finish = getattr(L, f"bz2b200_{kind}_feed"), getattr(L, f"bz2b200_{kind}_finish")
        read = self._reader(source, piece)
        collected = bytearray() if sink is None else None

        def put(ptr, n):
            data = self._take(ptr, n) if n else b""
            if not data:
                return
            if collected is not None:
                collected.extend(data)
            elif hasattr(sink, "write"):
                sink.write(data)
            else:
                for x in data:
                    sink.writeByte(x)

        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        try:
            while True:
                data = read(piece)
                if not data:
                    break
                a = np.frombuffer(data, dtype=np.uint8)
                rc = feed(handle, a.ctypes.data, a.size, C.byref(out), C.byref(n))
                if rc:
                    self._raise(rc)
                put(out, n.value)
                if len(data) < piece:
                    break
            rc = finish(handle, C.byref(out), C.byref(n))
            if rc:
                self._raise(rc)
            put(out, n.value)
            extra = finished(handle) if finished else None
        finally:
            getattr(L, f"bz2b200_{kind}_close")(handle)
        if sink is None:
            result = bytes(collected)
        else:
            if hasattr(sink, "flush"):
                sink.flush()
            result = sink
        return (result, extra) if finished else result

    def compressStream(self, source, sink=None, props=None, chunk_bytes=64 << 20, piece_bytes=None, index=False):
        """Stream flavour of compressFile: the source is read piece by piece and whole blocks are compressed as soon as the
        bytes after them (their halo) have arrived, so neither the input nor the output is ever held in full.
        Byte-identical to compressFile on the concatenated input.  source: .read(n) -> bytes, {readByte}, or bytes-like;
        sink: .write(bytes), {writeByte}, or None (the stream is returned as bytes).  index=True: returns (what it
        returns otherwise, the stream's Bzip2LineIndex), built while compressing as compressIndexed builds it."""
        level = _level(props)
        h = C.c_void_p()
        open_ = self._L.bz2b200_zstream_open_indexed if index else self._L.bz2b200_zstream_open
        rc = open_(self._ctx, level, int(chunk_bytes), C.byref(h))
        if rc:
            self._raise(rc)
        finished = (lambda handle: _line_index_call(self, self._L.bz2b200_zstream_index, handle)) if index else None
        return self._pump("zstream", h, source, sink, int(piece_bytes or max(1, chunk_bytes // 4)), finished)

    def append(self, stream, source, index=None, sink=None, chunk_bytes=64 << 20, piece_bytes=None):
        """Append the bytes of `source` to the last stream of `stream`, recompressing only its last block: returns (keep,
        tail, Bzip2LineIndex).  The new stream is stream[:keep] + tail; for a stream written from input A (by this library
        or the reference) it is byte for byte compressFile(A + B) at the stream's level, and the index is that of the new
        stream (include/bz2b200.h, bz2b200_zstream_open_append).  stream: bytes-like, or a path, which is memory-mapped as
        open() maps it; only its last block and footer are read.  source: what compressStream takes.  sink: as for
        compressStream, the tail goes there and the sink is returned in its place.  index: the Bzip2LineIndex of `stream`
        (compressIndexed, compressStream(..., index=True), lineIndex or a previous append); without it one is built first
        with lineIndex(stream, multistream=True): that is a full decode of the stream."""
        if isinstance(index, Bzip2Index):
            raise TypeError("append needs a line index (Bzip2LineIndex: compressIndexed, lineIndex), not a block index")
        a = _coerce_input(_map_path(stream))
        if index is None:
            index = self.lineIndex(a, multistream=True)
        ix = index.blocks.entries
        h, keep = C.c_void_p(), C.c_uint64()
        rc = self._L.bz2b200_zstream_open_append(self._ctx, a.ctypes.data, a.size, ix.ctypes.data, index.newlines.ctypes.data, len(ix),
                                                 index.total_lines, int(chunk_bytes), C.byref(h), C.byref(keep))
        if rc:
            self._raise(rc)
        finished = lambda handle: _line_index_call(self, self._L.bz2b200_zstream_index, handle)  # noqa: E731
        tail, li = self._pump("zstream", h, source, sink, int(piece_bytes or max(1, chunk_bytes // 4)), finished)
        return keep.value, tail, li

    def decompressStream(self, source, sink=None, multistream=False, chunk_bytes=16 << 20, piece_bytes=None):
        """Stream flavour of decompressFile: blocks are decoded as soon as they are complete; the bytes of the blocks before
        an error have been delivered when it is raised (like the reference, which writes as it goes)."""
        h = C.c_void_p()
        rc = self._L.bz2b200_dstream_open(self._ctx, int(bool(multistream)), int(chunk_bytes), C.byref(h))
        if rc:
            self._raise(rc)
        return self._pump("dstream", h, source, sink, int(piece_bytes or max(1, chunk_bytes // 4)))

    def decompressFile(self, input, output=None, multistream=False):
        a = _coerce_input(input)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_decompress(self._ctx, a.ctypes.data, a.size, int(bool(multistream)), C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return _deliver(self._take(out, n.value), output)

    def decompressBlock(self, input, pos, output=None):
        a = _coerce_input(input)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_decompress_block(self._ctx, a.ctypes.data, a.size, int(pos), C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return _deliver(self._take(out, n.value), output)

    def table(self, input, callback, multistream=False):
        a = _coerce_input(input)
        pos, sz, n = C.POINTER(C.c_uint64)(), C.POINTER(C.c_uint32)(), C.c_size_t()
        rc = self._L.bz2b200_table(self._ctx, a.ctypes.data, a.size, int(bool(multistream)), C.byref(pos), C.byref(sz), C.byref(n))
        if rc:
            self._raise(rc)
        try:
            for i in range(n.value):
                callback(int(pos[i]), int(sz[i]))
        finally:
            self._L.bz2b200_free(pos)
            self._L.bz2b200_free(sz)

    def recover(self, input):
        """What survives of a damaged file (bzip2recover, without stopping at damage): the input is read as a sequence of
        streams; returns (data, regions).  data = the bytes of every block that decodes and matches its CRC, in input
        order; regions = list of Region tiling the input bits (include/bz2b200.h, bz2b200_recover).  Damage is reported in
        the regions, never raised: only CUDA or argument errors raise."""
        a = _coerce_input(input)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        regs, nr = C.POINTER(_native.Region)(), C.c_size_t()
        rc = self._L.bz2b200_recover(self._ctx, a.ctypes.data, a.size, C.byref(out), C.byref(n), C.byref(regs), C.byref(nr))
        if rc:
            self._raise(rc)
        try:
            regions = [Region(r.bit_begin, r.bit_end, r.kind, REGION_KINDS[r.kind], r.status, r.out_offset, r.out_bytes, r.crc,
                              r.stream, r.flags) for r in (regs[i] for i in range(nr.value))]
        finally:
            self._L.bz2b200_free(regs)
        return self._take(out, n.value), regions

    # -- random access (include/bz2b200.h, bz2b200_index / bz2b200_decompress_ranges) --
    def index(self, input, multistream=False):
        """The block index of `input` (a Bzip2Index): the same walk as table(), and the same errors."""
        a = _coerce_input(input)
        ptr, n = C.POINTER(_native.BlockEntry)(), C.c_size_t()
        rc = self._L.bz2b200_index(self._ctx, a.ctypes.data, a.size, int(bool(multistream)), C.byref(ptr), C.byref(n))
        if rc:
            self._raise(rc)
        try:
            raw = _native.take_bytes(C.cast(ptr, C.POINTER(C.c_uint8)), n.value * INDEX_DTYPE.itemsize)
        finally:
            self._L.bz2b200_free(ptr)
        return Bzip2Index(np.frombuffer(raw, dtype=INDEX_DTYPE))

    def decompressRanges(self, input, index, ranges):
        """The bytes of every (start, length) of the decompressed output, as a list in request order.  Each range is clipped
        to the output the way slicing clips output[start:start + length].  One call decodes every block that covers a
        range, once, and nothing else; the stream CRC is not checked (include/bz2b200.h).  index: a Bzip2Index or a
        Bzip2LineIndex (its blocks are used)."""
        if isinstance(index, Bzip2LineIndex):
            index = index.blocks
        a = _coerce_input(input)
        ix = index.entries
        total = index.total
        se = [slice(int(s), int(s) + int(ln)).indices(total)[:2] for s, ln in ranges]
        starts = np.array([s for s, _ in se], dtype=np.uint64)
        lens = np.array([max(0, e - s) for s, e in se], dtype=np.uint64)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_decompress_ranges(self._ctx, a.ctypes.data, a.size, ix.ctypes.data, len(ix), starts.ctypes.data,
                                               lens.ctypes.data, len(se), C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        data = self._take(out, n.value)
        ends = np.cumsum(lens, dtype=np.uint64).tolist()
        return [data[e - int(ln):e] for e, ln in zip(ends, lens.tolist())]

    def decompressRange(self, input, index, start, length):
        """decompressRanges for one range: output[start:start + length]"""
        return self.decompressRanges(input, index, [(start, length)])[0]

    def open(self, input, index=None, multistream=False):
        """A seekable, read-only binary file over the decompressed bytes of `input` (bytes-like, or a path, which is
        memory-mapped).  Every read decodes only the blocks it needs.  index: a Bzip2Index or a Bzip2LineIndex (what
        compressIndexed returns); without it one is built first: that is a full decode of the input.  The buffer holds one level-9 block, so small sequential reads do not decode a block each;
        read() to the end is one call."""
        a = _coerce_input(_map_path(input))
        if index is None:
            index = self.index(a, multistream)
        elif isinstance(index, Bzip2LineIndex):
            index = index.blocks
        return io.BufferedReader(_RangeReader(self, a, index), buffer_size=LEVEL9_BLOCK)

    # -- lines by number (include/bz2b200.h, bz2b200_line_index / bz2b200_decompress_lines) --
    def lineIndex(self, input, multistream=False):
        """The block index of `input` with the '\n' bytes of every block (a Bzip2LineIndex).  The input is decoded as
        decompressFile decodes it, with the same errors; the '\n' bytes are counted on the GPU.  A stream compressed here
        can have the same index without a decode: compressIndexed."""
        a = _coerce_input(input)
        return _line_index_call(self, self._L.bz2b200_line_index, self._ctx, a.ctypes.data, a.size, int(bool(multistream)))

    def _lines(self, input, index, requests, want_bytes):
        """bz2b200_decompress_lines over the clipped requests -> (bytes or None, (k, 2) uint64 spans)"""
        a = _coerce_input(input)
        ix = index.blocks.entries
        se = [slice(int(f), int(f) + int(k)).indices(index.total_lines)[:2] for f, k in requests]
        firsts = np.array([f for f, _ in se], dtype=np.uint64)
        counts = np.array([max(0, e - f) for f, e in se], dtype=np.uint64)
        spans = np.zeros((len(se), 2), dtype=np.uint64)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_decompress_lines(self._ctx, a.ctypes.data, a.size, ix.ctypes.data, index.newlines.ctypes.data, len(ix), index.total_lines,
                                              firsts.ctypes.data, counts.ctypes.data, len(se), C.byref(out) if want_bytes else None,
                                              C.byref(n) if want_bytes else None, spans.ctypes.data)
        if rc:
            self._raise(rc)
        return (self._take(out, n.value) if want_bytes else None), spans

    def decompressLines(self, input, index, requests):
        """The lines of every (first, count) of the decompressed output, 0-based, as a list of bytes in request order.  A
        request is clipped the way slicing clips lines[first:first + count]; the bytes are as in the output (a last line
        without '\n' comes back without one).  index: a Bzip2LineIndex.  One call decodes every block that holds a
        requested line, once, and nothing else (include/bz2b200.h)."""
        data, spans = self._lines(input, index, requests, True)
        ends = np.cumsum(spans[:, 1], dtype=np.uint64).tolist()
        return [data[e - int(ln):e] for e, ln in zip(ends, spans[:, 1].tolist())]

    def lineSpans(self, input, index, requests):
        """The byte (start, length) of every (first, count) of decompressLines, as a (k, 2) uint64 array: what
        decompressRanges takes.  Decodes what decompressLines decodes and returns no bytes."""
        return self._lines(input, index, requests, False)[1]

    def debug_set_line_tile(self, nbytes):
        """tests only: bytes per newline-directory tile (a multiple of 256 up to 8192; 0 restores the default)"""
        rc = self._L.bz2b200_debug_set_line_tile(self._ctx, nbytes)
        if rc:
            self._raise(rc)

    # -- search (include/bz2b200.h, bz2b200_search) --
    def search(self, input, patterns, ignore_case=False, max_matches=None, multistream=False, lines=False):
        """Every occurrence of every fixed-string pattern in the decompressed output, found on the GPU where the decode
        leaves the bytes (what bzgrep -F does).  patterns: one bytes / str (UTF-8) or an iterable of them, 1..256 patterns
        of 1..256 bytes (ValueError otherwise).  ignore_case folds ASCII A-Z only.  Returns a SearchResult: `matches`
        holds the first max_matches (None: all) in (offset, pattern) order; total_matches and total_lines count them all.
        lines=True also returns the distinct lines holding a returned match, each ending in '\n' (grep -F's output).
        Decode errors raise Bzip2Error as decompressFile does."""
        return _search(self, self._L.bz2b200_search, self._ctx, input, patterns, ignore_case, max_matches, multistream, lines)

    def debug_set_search_tile(self, nbytes):
        """tests only: bytes per search tile (a multiple of 256 up to 8192; 0 restores the default)"""
        rc = self._L.bz2b200_debug_set_search_tile(self._ctx, nbytes)
        if rc:
            self._raise(rc)

    # -- extras used by bench.py / tests --
    def stats(self):
        st = _native.Stats()
        self._L.bz2b200_last_stats(self._ctx, C.byref(st))
        return st

    def compress_device(self, d_in_ptr, n, level, d_out_ptr, out_cap):
        olen = C.c_size_t()
        rc = self._L.bz2b200_compress_device(self._ctx, d_in_ptr, n, level, d_out_ptr, out_cap, C.byref(olen))
        if rc:
            self._raise(rc)
        return olen.value

    def decompress_device(self, d_in_ptr, n, multistream, d_out_ptr, out_cap):
        olen = C.c_size_t()
        rc = self._L.bz2b200_decompress_device(self._ctx, d_in_ptr, n, int(bool(multistream)), d_out_ptr, out_cap, C.byref(olen))
        if rc:
            self._raise(rc)
        return olen.value

    def compress_bound(self, n, level=9):
        return int(self._L.bz2b200_compress_bound(n, level))

    def debug_fetch(self, what, blk, nbytes):
        buf = np.zeros(nbytes, dtype=np.uint8)
        got = self._L.bz2b200_debug_fetch(self._ctx, what, blk, buf.ctypes.data, nbytes)
        if got < 0:
            self._raise(int(got))
        return buf[:got]

    # -- block-range shards (include/bz2b200.h, "multi-GPU") --
    def shard_begin(self, data, level, device_ptr=None, nbytes=None):
        if device_ptr is not None:
            rc = self._L.bz2b200_shard_begin(self._ctx, device_ptr, nbytes, 1, level)
        else:
            a = _coerce_input(data)
            self._shard_keep = a
            rc = self._L.bz2b200_shard_begin(self._ctx, a.ctypes.data, a.size, 0, level)
        if rc:
            self._raise(rc)

    def shard_cut(self, s_start, own_len, is_last):
        info = _native.ShardInfo()
        rc = self._L.bz2b200_shard_cut(self._ctx, s_start, own_len, int(is_last), C.byref(info))
        if rc:
            self._raise(rc)
        return info

    def shard_gtotal(self, pos):
        g = C.c_uint64()
        rc = self._L.bz2b200_shard_gtotal(self._ctx, pos, C.byref(g))
        if rc:
            self._raise(rc)
        return g.value

    def shard_cut_g(self, g_before, own_len):
        """Speculative cut walks (g_before = G of the earlier shards); shard_cut_pick chooses among them."""
        rc = self._L.bz2b200_shard_cut_g(self._ctx, g_before, own_len)
        if rc:
            self._raise(rc)

    def shard_cut_pick(self, s_start, own_len, is_last):
        """The speculated walk that started at s_start, or None (then call shard_cut)."""
        info, found = _native.ShardInfo(), C.c_int()
        rc = self._L.bz2b200_shard_cut_pick(self._ctx, s_start, own_len, int(is_last), C.byref(info), C.byref(found))
        if rc:
            self._raise(rc)
        return info if found.value else None

    def shard_compress(self, info):
        rc = self._L.bz2b200_shard_compress(self._ctx, C.byref(info))
        if rc:
            self._raise(rc)
        return info

    def shard_emit(self, info, bit_phase, to_host=True):
        """to_host: True -> bytes; False -> the segment stays in HBM, its length is returned;
        "raw" -> (pointer, length) in the library's page-locked result memory, released with free_raw."""
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_shard_emit(self._ctx, bit_phase, C.byref(info), C.byref(out) if to_host else None, C.byref(n))
        if rc:
            self._raise(rc)
        if to_host == "raw":
            return out, n.value
        return self._take(out, n.value) if to_host else n.value

    def free_raw(self, ptr):
        self._L.bz2b200_free(ptr)

    def stitch_shards(self, level, segs, infos):
        n = len(segs)
        arr = (C.c_char_p * n)(*[bytes(s) if len(s) else b"\0" for s in segs])
        inf = (_native.ShardInfo * n)(*infos)
        out, ln = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_stitch_shards(level, n, arr, inf, C.byref(out), C.byref(ln))
        if rc:
            self._raise(rc)
        return self._take(out, ln.value)

    def debug_set_block_cap(self, cap):
        """tests only: 0 restores level*100000-19"""
        rc = self._L.bz2b200_debug_set_block_cap(self._ctx, cap)
        if rc:
            self._raise(rc)

    def debug_set_batch_blocks(self, blocks):
        """tests only: blocks per batch of the per-block stages, 0 restores the automatic limit"""
        rc = self._L.bz2b200_debug_set_batch_blocks(self._ctx, blocks)
        if rc:
            self._raise(rc)

    def debug_set_ignore_block_crc(self, on):
        """tests only: decode without comparing block CRCs (what a damaged stream decodes TO)"""
        rc = self._L.bz2b200_debug_set_ignore_block_crc(self._ctx, int(bool(on)))
        if rc:
            self._raise(rc)

    def debug_set_decode_batch(self, candidates):
        """tests only: signature candidates per decode batch (0 restores the default), so that neighbours fall in different batches"""
        rc = self._L.bz2b200_debug_set_decode_batch(self._ctx, None, candidates)
        if rc:
            self._raise(rc)

    def debug_set_rle1_threads(self, threads):
        """tests only: threads per CTA of the RLE1 inverse, 512 or 1024 (0 restores the choice by block count)"""
        rc = self._L.bz2b200_debug_set_rle1_threads(self._ctx, None, threads)
        if rc:
            self._raise(rc)

    def decode_candidates(self):
        """tests only: the DecBlk of every candidate of the last batch of the last decode call"""
        sz = C.sizeof(_native.DecBlk)
        raw = self.debug_fetch(7, 0, sz * (1 << 20)).tobytes()
        return list((_native.DecBlk * (len(raw) // sz)).from_buffer_copy(raw))

    def decode_stages(self, k, nsym=None):
        """tests only: (symbols, offsets, L column) of candidate k of the last decode batch; nsym: read that many symbols
        and offsets instead of the candidate's own count (which a block that failed the size checks has set to 0)"""
        b = self.decode_candidates()[k]
        nsym = b.nsym if nsym is None else nsym
        syms = np.frombuffer(self.debug_fetch(8, k, 2 * nsym).tobytes(), dtype=np.uint16)
        offs = np.frombuffer(self.debug_fetch(9, k, 4 * (nsym + 1)).tobytes(), dtype=np.uint32)
        return syms, offs, self.debug_fetch(10, k, b.count)

    def decode_inverted(self):
        """tests only: [(candidate index, inverse-BWT output)] of the blocks the last decode batch inverted, in stream order"""
        chain = np.frombuffer(self.debug_fetch(12, 0, 4 << 20).tobytes(), dtype=np.uint32)
        cands = self.decode_candidates()
        return [(int(k), self.debug_fetch(11, p, cands[k].count).tobytes()) for p, k in enumerate(chain)]

    def debug_huffman_lengths(self, sorted_freqs, maxlen):
        """tests only: HuffmanAllocator.allocateHuffmanCodeLengths (BJ:1275-1298) run by the device copy of the allocator"""
        a = np.asarray(sorted_freqs, dtype=np.int32).copy()
        rc = self._L.bz2b200_debug_huffman_lengths(self._ctx, a.ctypes.data, a.size, int(maxlen))
        if rc:
            self._raise(rc)
        return [int(x) for x in a]

    def debug_set_pool(self, min_bytes=32_000_000, shard_bytes=0, first_halo=0, force_staging=False):
        """tests only: which inputs compressFile sends through the context's two-lane pool, and how they are cut"""
        rc = self._L.bz2b200_debug_set_pool(self._ctx, min_bytes, shard_bytes, first_halo, int(bool(force_staging)))
        if rc:
            self._raise(rc)

    def block_table(self):
        nb = self.stats().n_blocks
        raw = self.debug_fetch(0, 0, C.sizeof(_native.BlockRec) * nb)
        return (_native.BlockRec * nb).from_buffer_copy(raw.tobytes()) if nb else []

    def block_meta(self):
        nb = self.stats().n_blocks
        raw = self.debug_fetch(4, 0, C.sizeof(_native.BlockMeta) * nb)
        return (_native.BlockMeta * nb).from_buffer_copy(raw.tobytes()) if nb else []

    def block_huffman(self, k):
        """tests only: (selectors, code lengths) of block k of the last batch of the last compress call: the table index
        of every group of 50 symbols (n_sel of them) and the lengths as a (6, 260) array (n_groups x alphabet + 2 used)"""
        sel = self.debug_fetch(5, k, 1 << 15)   # raises for a block outside the batch; a block has at most 18 000 selectors
        sz = C.sizeof(_native.BlockMeta)
        meta = _native.BlockMeta.from_buffer_copy(self.debug_fetch(4, 0, sz * (k + 1))[sz * k:].tobytes())
        return sel[:meta.n_sel], self.debug_fetch(6, k, 6 * 260).reshape(6, 260)


class _Lazy:
    """`Bzip2` global of the reference (BJ:2198-2255): created on first use."""
    _eng = None

    def _get(self):
        if _Lazy._eng is None:
            _Lazy._eng = Bzip2Engine(0)
        return _Lazy._eng

    def __getattr__(self, name):
        return getattr(self._get(), name)


Bzip2 = _Lazy()
