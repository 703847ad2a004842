"""Measurement of Bzip2Pool.search (bz2b200_pool_search) against Bzip2Engine.search on one context and against
Bzip2Pool.decompressFile, written as JSON to <outdir>/pool_search_bench.json.  Two streams: the 100 MB level-9 bench stream
(gen_text(100 MB, seed 8)) and 1 GB of text (gen_text(1 GB, seed 9), level 9).  Two pools: two lanes of one device, and two
lanes on every visible device (not measured with one device).  Host-call times are the median of --runs calls each after
one warm-up call of each; device search time is the median of ms_stage[5] over the same calls (summed over the lanes for
a pool).  Every search result is checked against the Python model of tests/test_search.py.  The card's name and power
limit are read in the same run (nvidia-smi --query-gpu, read-only).
    python tests/gpu_pool_search_bench.py <outdir> [--runs N]"""
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
sys.path.insert(0, HERE)
from compressjs_flattened_b200.bzip2 import Bzip2Engine  # noqa: E402
from compressjs_flattened_b200.corpus import gen_text  # noqa: E402
from compressjs_flattened_b200.pool import Bzip2Pool  # noqa: E402
from test_search import RARE, model  # noqa: E402


def timed(fn, runs, stats=None):
    """(median host ms, median ms_stage[5]) of `runs` calls after one warm-up"""
    fn()
    ts, dev = [], []
    for _ in range(runs):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
        if stats is not None:
            dev.append(stats().ms_stage[5])
    return 1e3 * statistics.median(ts), (statistics.median(dev) if dev else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir", help="directory the JSON is written to")
    ap.add_argument("--runs", type=int, default=7)
    a = ap.parse_args()
    os.makedirs(a.outdir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    import torch
    ndev = torch.cuda.device_count()
    eng = Bzip2Engine(0)
    pools = {"1 device x 2 lanes": Bzip2Pool([0], 2)}
    if ndev >= 2:
        pools[f"{ndev} devices x 2 lanes"] = Bzip2Pool(list(range(ndev)), 2)
    res = {"gpu": gpu.strip(), "visible_devices": ndev, "runs": a.runs, "pattern": RARE.decode(), "streams": []}
    if ndev < 2:
        res["every_device"] = "not measured: one device visible"
    for name, n, seed in (("text:100000000:8:L9", 100_000_000, 8), ("text:1000000000:9:L9", 1_000_000_000, 9)):
        src = gen_text(n, seed).tobytes()
        comp = pools["1 device x 2 lanes"].compressFile(src, None, 9)
        want, total, nlines, text = model(src, [RARE])
        row = {"stream": name, "compressed_bytes": len(comp), "decoded_bytes": len(src), "matches": total}
        r = eng.search(comp, [RARE], lines=True)
        assert np.array_equal(r.matches, want) and r.lines == text
        host, dev = timed(lambda: eng.search(comp, [RARE], lines=True), a.runs, eng.stats)
        row["engine_search"] = {"host_ms": host, "device_ms_search": dev}
        for pname, pool in pools.items():
            r = pool.search(comp, [RARE], lines=True)
            assert np.array_equal(r.matches, want) and (r.total_matches, r.total_lines) == (total, nlines) and r.lines == text
            assert pool.decompressFile(comp, len(src)) == src
            s_host, s_dev = timed(lambda: pool.search(comp, [RARE], lines=True), a.runs, pool.stats)
            d_host, _ = timed(lambda: pool.decompressFile(comp, len(src)), a.runs)
            row[pname] = {"pool_search_host_ms": s_host, "pool_search_device_ms_search_summed_over_lanes": s_dev, "pool_decompressFile_host_ms": d_host,
                          "pool_search_over_engine_search": s_host / host, "pool_search_over_pool_decompressFile": s_host / d_host}
        res["streams"].append(row)
        del src, comp, want, text
    for p in pools.values():
        p.close()
    with open(os.path.join(a.outdir, "pool_search_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
