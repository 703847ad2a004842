"""Measurement of Bzip2Engine.search (bz2b200_search) on the 100 MB level-9 bench stream (gen_text(100 MB, seed 8)),
written as JSON to <outdir>/search_bench.json.  Host-call times are the median of --runs calls each, after a warm-up of
every shape; device times are the medians of bz2b200_last_stats over the same calls:
  (a) one rare word: search against decompressFile, and against decompressFile plus a host bytes.find loop;
  (b) 16 and 256 patterns, with and without IGNORE_CASE;
  (c) a frequent pattern with lines=True: host time and the bytes returned (matches + lines);
  (d) the search stage (ms_stage[5]: count, scan, emit, line gather) against the decode's device time, and as a rate over
      the decoded bytes (a whole-stage rate, not a share of HBM bandwidth).
Every result is checked against a Python model on the decoded bytes (bytes.find, one byte at a time).  The card's name
and power limit are read in the same run (nvidia-smi --query-gpu, read-only).
    python tests/gpu_search_bench.py <outdir> [--runs N]"""
import argparse
import collections
import json
import os
import re
import statistics
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from compressjs_flattened_b200.bzip2 import Bzip2Engine  # noqa: E402
from compressjs_flattened_b200.corpus import gen_text  # noqa: E402
from test_search import RARE, WORDS16, model  # noqa: E402


def timed(fn, runs, eng=None):
    """(median host ms, median stats) of `runs` calls after one warm-up"""
    fn()
    ts, stats = [], []
    for _ in range(runs):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
        if eng is not None:
            st = eng.stats()
            stats.append((st.ms_total, st.ms_stage[5]))
    med = {}
    if stats:
        med = {"device_ms_total": statistics.median(s[0] for s in stats), "device_ms_search": statistics.median(s[1] for s in stats)}
    return 1e3 * statistics.median(ts), med


def find_all(data, word):
    n, i = 0, data.find(word)
    while i >= 0:
        n += 1
        i = data.find(word, i + 1)
    return n


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
    res = {"gpu": gpu.strip(), "stream": "text:100000000:8:L9", "compressed_bytes": len(comp), "decoded_bytes": len(full), "runs": a.runs}

    def search_case(pats, ignore_case=False, max_matches=None, lines=False):
        r = eng.search(comp, pats, ignore_case, max_matches, False, lines)
        want, total, nlines, text = model(full, pats, ignore_case, max_matches)
        assert np.array_equal(r.matches, want) and (r.total_matches, r.total_lines) == (total, nlines)
        assert not lines or r.lines == text
        host, dev = timed(lambda: eng.search(comp, pats, ignore_case, max_matches, False, lines), a.runs, eng)
        out = {"patterns": len(pats), "ignore_case": ignore_case, "matches": total, "lines": nlines, "host_ms": host}
        out.update(dev)
        out["search_stage_GBps_of_decoded_bytes"] = len(full) / (dev["device_ms_search"] * 1e6) if dev.get("device_ms_search") else None
        return out, r

    # decode alone, for (a) and (d)
    t_dec, dec_dev = timed(lambda: eng.decompressFile(comp), a.runs, eng)
    assert find_all(full, RARE) == model(full, [RARE])[1]
    t_find, _ = timed(lambda: find_all(eng.decompressFile(comp), RARE), a.runs)
    ra, _ = search_case([RARE])
    res["a_rare_word"] = {"word": RARE.decode(), **ra, "decompressFile_ms": t_dec, "decompressFile_plus_find_ms": t_find,
                          "search_over_decompressFile": ra["host_ms"] / t_dec}
    # (b)
    words = collections.Counter(re.findall(rb"[A-Za-z]{4,}", full[:5_000_000]))
    w256 = [w for w, _ in words.most_common(256)]
    res["b_patterns"] = [search_case(p, ic)[0] for p in (WORDS16, w256) for ic in (False, True)]
    # (c)
    rc, r = search_case([b"the"], lines=True)
    rc["bytes_returned"] = {"matches": int(r.matches.nbytes), "lines": len(r.lines)}
    res["c_frequent_with_lines"] = rc
    # (d)
    decode_dev = dec_dev["device_ms_total"]
    res["d_stage"] = {"decode_device_ms": decode_dev, "note": "search stage = count + scan + emit (+ line gather), device time; rate = decoded bytes / stage time",
                      "cases": [{"case": name, "search_stage_ms": c["device_ms_search"], "over_decode": c["device_ms_search"] / decode_dev,
                                 "GBps": c["search_stage_GBps_of_decoded_bytes"]}
                                for name, c in [("rare word", ra)] + [(f"{b['patterns']} patterns ignore_case={b['ignore_case']}", b) for b in res["b_patterns"]]
                                + [("'the' with lines", rc)]]}
    with open(os.path.join(a.outdir, "search_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
