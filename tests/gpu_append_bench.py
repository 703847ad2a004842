"""Measurement of Bzip2Engine.append, written as JSON to <outdir>/r09_append_bench.json.  For B of 1 MB and 16 MB
(gen_text, seed 9) appended to A, the 100 MB level-9 bench stream (gen_text(100 MB, seed 8)) and 1 GB (the bench input ten
times over), the median host time of --runs calls of each of these, after a warm-up, the four calls alternating so that
all see the same machine:
  append                 Bzip2Engine.append(stream of A, B, its line index)
  compressFile(A + B)    what the append replaces
  decompressRange        the bytes of A's last block, read with the index
  compressStream         of the last block's bytes plus B
The append decodes the last block and compresses it again together with B, so its cost should be about the sum of the last
two and should not grow with |A|.  In the same run, every append's result is compared with compressFile(A + B) (SHA-256)
and its index with compressIndexed(A + B)'s.  The card's name and power limit are read in the same run
(nvidia-smi --query-gpu, read-only).
    python tests/gpu_append_bench.py <outdir> [--runs N]"""
import argparse
import hashlib
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


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def alternate(fns, runs):
    """medians (ms) of every fn over `runs` rounds, one call of each per round, after one warm-up of each"""
    for f in fns:
        f()
    ts = [[] for _ in fns]
    for _ in range(runs):
        for t, f in zip(ts, fns):
            t.append(timed(f))
    return [statistics.median(t) for t in ts]


def same_index(li, ref):
    return (li.blocks.entries.tolist() == ref.blocks.entries.tolist() and li.newlines.tolist() == ref.newlines.tolist()
            and li.total_lines == ref.total_lines)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir", help="directory the JSON is written to")
    ap.add_argument("--runs", type=int, default=11)
    a = ap.parse_args()
    os.makedirs(a.outdir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    eng = Bzip2Engine(0)
    bench = gen_text(100_000_000, 8)
    res = {"gpu": gpu.strip(), "runs": a.runs, "level": 9,
           "timing": "median host time of each call, the four calls alternating, after one warm-up of each", "cases": []}
    for a_name, A in (("text:100000000:8", bench.tobytes()), ("text:100000000:8 x10", np.tile(bench, 10).tobytes())):
        S, li = eng.compressIndexed(A, 9)
        last = li.blocks.entries[-1]
        off, size = int(last["out_offset"]), int(last["out_bytes"])
        for n in (1_000_000, 16_000_000):
            B = gen_text(n, 9).tobytes()
            AB, LB = A + B, A[off:] + B   # outside the timed calls
            keep, tail, got = eng.append(S, B, li)
            want = eng.compressFile(AB, None, 9)
            assert hashlib.sha256(S[:keep] + tail).digest() == hashlib.sha256(want).digest(), (a_name, n)
            assert same_index(got, eng.compressIndexed(AB, 9)[1]), (a_name, n)
            t_app, t_full, t_range, t_stream = alternate([lambda: eng.append(S, B, li), lambda: eng.compressFile(AB, None, 9),
                                                         lambda: eng.decompressRange(S, li, off, size),
                                                         lambda: eng.compressStream(LB, None, 9)], a.runs)
            res["cases"].append({"A": a_name, "A_bytes": len(A), "A_stream_bytes": len(S), "B_bytes": n, "last_block_bytes": size,
                                 "keep": keep, "tail_bytes": len(tail), "result_equals_compressFile": True, "index_equals_compressIndexed": True,
                                 "append_ms": t_app, "compressFile_A_plus_B_ms": t_full, "decompressRange_last_block_ms": t_range,
                                 "compressStream_last_block_plus_B_ms": t_stream,
                                 "append_over_range_plus_stream": t_app / (t_range + t_stream), "append_over_compressFile": t_app / t_full})
            print(json.dumps(res["cases"][-1]), flush=True)
    with open(os.path.join(a.outdir, "r09_append_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
