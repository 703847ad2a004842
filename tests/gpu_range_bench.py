"""Measurement of the range reads (Bzip2Engine.index / decompressRanges / open) on the 100 MB level-9 bench stream
(gen_text(100 MB, seed 8)), written as JSON to <outdir>/range_bench.json.  Host-call times, median of --runs calls each
after a warm-up of every shape:
  (a) index against decompressFile;
  (b) 64 random 4 KiB reads: one decompressRanges call against 64 decompressBlock calls (one per covering block read);
  (c) 4 096 random 4 KiB reads in one decompressRanges call;
  (d) one 1 MB and one 16 MB range against a whole decompressFile;
  (e) the whole file read sequentially through open() in 1 MiB reads;
  (f) 10 000 random one-byte reads in one decompressRanges call, and the device time of the call against (c)'s (many tiny
      pieces: k_gather_ranges copies the pieces of its output chunk one after the other).
Every result is compared with the bytes of decompressFile.  The card's name and power limit are read in the same run
(nvidia-smi --query-gpu, read-only).
    python tests/gpu_range_bench.py <outdir> [--runs N]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from compressjs_flattened_b200.bzip2 import Bzip2Engine  # noqa: E402
from compressjs_flattened_b200.corpus import gen_text  # noqa: E402


def median_ms(fn, runs):
    fn()   # warm-up
    ts = []
    for _ in range(runs):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir", help="directory the JSON is written to")
    ap.add_argument("--runs", type=int, default=11)
    a = ap.parse_args()
    os.makedirs(a.outdir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    eng = Bzip2Engine(0)
    src = gen_text(100_000_000, 8).tobytes()
    comp = eng.compressFile(src, None, 9)
    full = eng.decompressFile(comp)
    assert full == src
    ix = eng.index(comp)
    e = ix.entries
    rng = np.random.default_rng(2026)
    res = {"gpu": gpu.strip(), "stream": "text:100000000:8:L9", "compressed_bytes": len(comp), "blocks": len(ix), "runs": a.runs}

    # (a)
    t_dec = median_ms(lambda: eng.decompressFile(comp), a.runs)
    t_ix = median_ms(lambda: eng.index(comp), a.runs)
    res["a_index"] = {"index_ms": t_ix, "decompressFile_ms": t_dec, "index_over_decompressFile": t_ix / t_dec}

    def reads(k):
        rs = [(int(s), 4096) for s in rng.integers(0, len(full) - 4096, k)]
        got = eng.decompressRanges(comp, ix, rs)
        assert got == [full[s:s + 4096] for s, _ in rs]
        return rs

    # (b) one call against one decompressBlock per block the reads touch (the only way before this call)
    rs64 = reads(64)
    st = eng.stats()
    b_stats = {"blocks_decoded": st.n_blocks, "bytes_uploaded": st.in_bytes}
    blk = [int(np.searchsorted(e["out_offset"], s, side="right")) - 1 for s, _ in rs64]

    def by_blocks():
        out = []
        for (s, ln), k in zip(rs64, blk):
            b = eng.decompressBlock(comp, int(e["bit_begin"][k]))
            o = s - int(e["out_offset"][k])
            piece = b[o:o + ln]
            if len(piece) < ln:   # the read runs into the next block
                piece += eng.decompressBlock(comp, int(e["bit_begin"][k + 1]))[:ln - len(piece)]
            out.append(piece)
        return out
    assert by_blocks() == [full[s:s + ln] for s, ln in rs64]
    t_one = median_ms(lambda: eng.decompressRanges(comp, ix, rs64), a.runs)
    t_blocks = median_ms(by_blocks, a.runs)
    res["b_64_reads_4KiB"] = dict(b_stats, decompressRanges_ms=t_one, decompressBlock_x64_ms=t_blocks, speedup=t_blocks / t_one)

    # (c)
    rs4k = reads(4096)
    st = eng.stats()
    t_4k = median_ms(lambda: eng.decompressRanges(comp, ix, rs4k), a.runs)
    res["c_4096_reads_4KiB"] = {"decompressRanges_ms": t_4k, "blocks_decoded": st.n_blocks, "bytes_uploaded": st.in_bytes,
                                "decompressFile_ms": t_dec}

    # (d)
    res["d_large_ranges"] = {"decompressFile_ms": t_dec}
    for name, ln in (("1MB", 1_000_000), ("16MB", 16_000_000)):
        s = int(rng.integers(0, len(full) - ln))
        assert eng.decompressRange(comp, ix, s, ln) == full[s:s + ln]
        st = eng.stats()
        t = median_ms(lambda: eng.decompressRange(comp, ix, s, ln), a.runs)
        res["d_large_ranges"][name] = {"ms": t, "blocks_decoded": st.n_blocks, "bytes_uploaded": st.in_bytes, "over_decompressFile": t / t_dec}

    # (e)
    def sequential():
        with eng.open(comp, ix) as f:
            n = 0
            while True:
                b = f.read(1 << 20)
                if not b:
                    return n
                n += len(b)
    with eng.open(comp, ix) as f:
        assert b"".join(iter(lambda: f.read(1 << 20), b"")) == full
    t_seq = median_ms(sequential, a.runs)
    res["e_open_sequential_1MiB_reads"] = {"ms": t_seq, "MB_per_s": len(full) / 1e3 / t_seq, "decompressFile_ms": t_dec}

    # (f)
    rs1 = [(int(s), 1) for s in rng.integers(0, len(full), 10_000)]
    assert eng.decompressRanges(comp, ix, rs1) == [full[s:s + 1] for s, _ in rs1]
    t_1 = median_ms(lambda: eng.decompressRanges(comp, ix, rs1), a.runs)
    st = eng.stats()
    eng.decompressRanges(comp, ix, rs4k)
    dev_4k = eng.stats().ms_total
    eng.decompressFile(comp)
    res["f_10000_reads_1B"] = {"decompressRanges_ms": t_1, "device_ms": st.ms_total, "blocks_decoded": st.n_blocks,
                               "device_ms_4096_reads_4KiB": dev_4k, "device_ms_decompressFile": eng.stats().ms_total}

    with open(os.path.join(a.outdir, "range_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
