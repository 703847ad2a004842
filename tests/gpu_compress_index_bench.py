"""Measurement of the indexed compress calls (Bzip2Engine.compressIndexed, Bzip2Pool.compressIndexed), written as JSON to
<outdir>/r08_compress_index_bench.json.  Host-call times, median of --runs calls each after a warm-up, the plain and the
indexed call alternating so that both see the same machine:
  (a) compressIndexed against compressFile on the 100 MB level-9 bench input (gen_text(100 MB, seed 8)), on the default
      route (inputs of 32 MB or more run on the context's two lanes);
  (b) compressIndexed against compressFile followed by lineIndex of the stream (the only other way to that index);
  (c) (a) on one context, and there the device time of the index kernel (stats ms_stage[5], summed over batches) against
      the compress call's device time (ms_total);
  (d) (a) at 1 GB (the bench input ten times over): through the context's own two-lane route, and through a pool on
      every visible device.
Every stream is compared with compressFile's and every index with lineIndex's.  The card's name and power limit are read
in the same run (nvidia-smi --query-gpu, read-only).
    python tests/gpu_compress_index_bench.py <outdir> [--runs N]"""
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
from compressjs_flattened_b200.pool import Bzip2Pool  # noqa: E402


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t0)


def alternate(fa, fb, runs, after_b=None):
    """medians (ms) of fa and fb over `runs` alternating calls after one warm-up of each; after_b() runs after every fb
    call (outside its time) and its values are collected"""
    fa(), fb()
    ta, tb, extra = [], [], []
    for _ in range(runs):
        ta.append(timed(fa))
        tb.append(timed(fb))
        if after_b:
            extra.append(after_b())
    return statistics.median(ta), statistics.median(tb), extra


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
    src = gen_text(100_000_000, 8).tobytes()
    comp = eng.compressFile(src, None, 9)
    got, li = eng.compressIndexed(src, 9)
    ref = eng.lineIndex(comp)
    assert got == comp and same_index(li, ref)
    res = {"gpu": gpu.strip(), "input": "text:100000000:8:L9", "compressed_bytes": len(comp), "blocks": len(li), "lines": li.total_lines,
           "runs": a.runs, "timing": "median host time of each call, plain and indexed calls alternating, after one warm-up"}

    # (a) the default route (inputs of 32 MB or more take the context's two lanes)
    t_plain, t_ix, _ = alternate(lambda: eng.compressFile(src, None, 9), lambda: eng.compressIndexed(src, 9), a.runs)
    res["a_default_route"] = {"compressFile_ms": t_plain, "compressIndexed_ms": t_ix, "index_cost_share_of_compressFile": (t_ix - t_plain) / t_plain,
                              "index_kernel_ms_summed_over_lanes": eng.stats().ms_stage[5]}

    # (c) one context (the two-lane route switched off), so that ms_total is one stream's device time
    eng.debug_set_pool(min_bytes=1 << 62)

    def dev_stats():
        st = eng.stats()
        return st.ms_stage[5], st.ms_total
    t_plain, t_ix, ds = alternate(lambda: eng.compressFile(src, None, 9), lambda: eng.compressIndexed(src, 9), a.runs, dev_stats)
    dev_plain = []
    for _ in range(3):
        eng.compressFile(src, None, 9)
        dev_plain.append(eng.stats().ms_total)
    ix_ms, tot_ms = statistics.median(d[0] for d in ds), statistics.median(d[1] for d in ds)
    res["c_one_context"] = {"compressFile_ms": t_plain, "compressIndexed_ms": t_ix, "index_cost_share_of_compressFile": (t_ix - t_plain) / t_plain,
                            "index_kernel_ms": ix_ms, "compressIndexed_device_ms": tot_ms, "compressFile_device_ms": statistics.median(dev_plain),
                            "index_kernel_share_of_device_time": ix_ms / tot_ms,
                            "index_kernel_input_bytes_per_s": len(src) / (ix_ms * 1e-3) if ix_ms else None}
    eng.debug_set_pool()

    # (b)
    def plain_then_index():
        c = eng.compressFile(src, None, 9)
        return eng.lineIndex(c)
    t_two, t_ix2, _ = alternate(plain_then_index, lambda: eng.compressIndexed(src, 9), a.runs)
    res["b_against_compress_then_lineIndex"] = {"compressFile_then_lineIndex_ms": t_two, "compressIndexed_ms": t_ix2, "saved_ms": t_two - t_ix2}

    # (d) 1 GB
    big = np.tile(np.frombuffer(src, dtype=np.uint8), 10).tobytes()
    bcomp = eng.compressFile(big, None, 9)
    got, bli = eng.compressIndexed(big, 9)
    assert got == bcomp and same_index(bli, eng.lineIndex(bcomp))
    t_plain, t_ix, _ = alternate(lambda: eng.compressFile(big, None, 9), lambda: eng.compressIndexed(big, 9), a.runs)
    res["d_1GB_own_two_lanes"] = {"compressFile_ms": t_plain, "compressIndexed_ms": t_ix, "index_cost_share": (t_ix - t_plain) / t_plain,
                                  "index_kernel_ms_summed_over_lanes": eng.stats().ms_stage[5]}
    import torch
    ndev = torch.cuda.device_count()
    pool = Bzip2Pool(list(range(ndev)), 2)
    try:
        got, pli = pool.compressIndexed(big, 9)
        assert got == bcomp and same_index(pli, bli)
        t_plain, t_ix, _ = alternate(lambda: pool.compressFile(big, None, 9), lambda: pool.compressIndexed(big, 9), a.runs)
        res["d_1GB_pool"] = {"devices": ndev, "lanes_per_device": 2, "compressFile_ms": t_plain, "compressIndexed_ms": t_ix,
                             "index_cost_share": (t_ix - t_plain) / t_plain, "index_kernel_ms_summed_over_lanes": pool.stats().ms_stage[5]}
    finally:
        pool.close()

    with open(os.path.join(a.outdir, "r08_compress_index_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
