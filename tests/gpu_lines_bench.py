"""Measurement of the line reads (Bzip2Engine.lineIndex / decompressLines) on the 100 MB level-9 bench stream
(gen_text(100 MB, seed 8)), written as JSON to <outdir>/lines_bench.json.  Host-call times, median of --runs calls each
after a warm-up of every shape:
  (a) lineIndex against decompressFile, and against decompressFile plus a host bytes.count(b"\\n") per block; the device
      time of the newline-directory kernels (stats ms_stage[5]) against the decode's device time (ms_total of decompressFile);
  (b) 64 and 4 096 random single-line reads in one decompressLines call, against decompressRanges over the byte spans of
      the same lines (the same covering blocks) and against decompressFile plus split(b"\\n");
  (c) one window of 1 M consecutive lines (of the bench stream twice over: it holds 527 716 lines).
Every result is compared with the lines of the source.  The card's name and power limit are read in the same run
(nvidia-smi --query-gpu, read-only).
    python tests/gpu_lines_bench.py <outdir> [--runs N]"""
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
    assert eng.decompressFile(comp) == src
    lines = [ln + b"\n" for ln in src.split(b"\n")]
    lines[-1] = lines[-1][:-1]
    if not lines[-1]:
        lines.pop()
    starts = np.concatenate([[0], np.cumsum([len(x) for x in lines])])
    li = eng.lineIndex(comp)
    offs = li.blocks.entries["out_offset"].tolist() + [len(src)]
    assert li.total_lines == len(lines) and li.newlines.tolist() == [src.count(b"\n", x, y) for x, y in zip(offs, offs[1:])]
    res = {"gpu": gpu.strip(), "stream": "text:100000000:8:L9", "compressed_bytes": len(comp), "blocks": len(li), "lines": li.total_lines,
           "runs": a.runs}

    # (a)
    t_dec = median_ms(lambda: eng.decompressFile(comp), a.runs)
    dev_dec = eng.stats().ms_total

    def dec_count():
        full = eng.decompressFile(comp)
        return [full.count(b"\n", x, y) for x, y in zip(offs, offs[1:])]
    t_dec_count = median_ms(dec_count, a.runs)
    t_ix = median_ms(lambda: eng.lineIndex(comp), a.runs)
    st = eng.stats()
    res["a_line_index"] = {"lineIndex_ms": t_ix, "decompressFile_ms": t_dec, "decompressFile_plus_count_ms": t_dec_count,
                           "lineIndex_over_decompressFile": t_ix / t_dec, "directory_device_ms": st.ms_stage[5],
                           "lineIndex_device_ms": st.ms_total, "decompressFile_device_ms": dev_dec,
                           "directory_share_of_decode_device_time": st.ms_stage[5] / dev_dec}

    rng = np.random.default_rng(2026)

    def split_all():
        return eng.decompressFile(comp).split(b"\n")

    # (b)
    for k in (64, 4096):
        reqs = [(int(f), 1) for f in rng.integers(0, len(lines), k)]
        want = [lines[f] for f, _ in reqs]
        assert eng.decompressLines(comp, li, reqs) == want
        st = eng.stats()
        spans = eng.lineSpans(comp, li, reqs)
        assert [tuple(s) for s in spans.tolist()] == [(int(starts[f]), len(lines[f])) for f, _ in reqs]
        rs = [(int(s), int(n)) for s, n in spans.tolist()]
        assert eng.decompressRanges(comp, li.blocks, rs) == want
        assert eng.stats().n_blocks == st.n_blocks
        t_l = median_ms(lambda: eng.decompressLines(comp, li, reqs), a.runs)
        dir_ms = eng.stats().ms_stage[5]
        t_r = median_ms(lambda: eng.decompressRanges(comp, li.blocks, rs), a.runs)
        t_s = median_ms(split_all, a.runs)
        res[f"b_{k}_random_lines"] = {"decompressLines_ms": t_l, "decompressRanges_same_spans_ms": t_r, "lines_over_ranges": t_l / t_r,
                                      "decompressFile_split_ms": t_s, "blocks_decoded": st.n_blocks, "directory_device_ms": dir_ms}

    # (c) the bench stream holds 527 716 lines: the window is read from the stream twice over (two streams, 1 055 431 lines)
    comp2 = comp + comp
    lines2 = lines[:-1] + [lines[-1] + lines[0]] + lines[1:]   # the first stream does not end with '\n'
    li2 = eng.lineIndex(comp2, True)
    assert li2.total_lines == len(lines2)
    first = int(rng.integers(0, len(lines2) - 1_000_000))
    reqs = [(first, 1_000_000)]
    assert eng.decompressLines(comp2, li2, reqs) == [b"".join(lines2[first:first + 1_000_000])]
    st = eng.stats()
    t_w = median_ms(lambda: eng.decompressLines(comp2, li2, reqs), a.runs)
    t_dec2 = median_ms(lambda: eng.decompressFile(comp2, None, True), a.runs)
    res["c_window_1M_lines"] = {"stream": "the bench stream twice (multistream)", "first": first, "decompressLines_ms": t_w, "bytes": st.out_bytes,
                                "blocks_decoded": st.n_blocks, "blocks": len(li2), "decompressFile_multistream_ms": t_dec2}

    with open(os.path.join(a.outdir, "lines_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
