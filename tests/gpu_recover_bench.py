"""Measurement of Bzip2Engine.recover on the 100 MB level-9 bench stream (gen_text(100 MB, seed 8)), written as JSON to
<outdir>/recover_bench.json:
  - intact stream: host-call time of recover against decompressFile (the same kernels), median of --runs runs each after a
    warm-up, the two calls alternating;
  - the same stream with one bit flipped in the symbol data of every tenth block: recover time and bytes recovered;
  - the CPU figure for the same damaged file: bzip2recover (when on the PATH) plus bz2.decompress of every piece it wrote.
The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only).
    python tests/gpu_recover_bench.py <outdir> [--runs N]"""
import argparse
import bz2
import hashlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from compressjs_flattened_b200.bzip2 import Bzip2Engine  # noqa: E402
from compressjs_flattened_b200.corpus import gen_text  # noqa: E402


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return time.perf_counter() - t0, r


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
    rows = []
    eng.table(comp, lambda p, s: rows.append(p), True)
    bad = bytearray(comp)
    ends = rows[1:] + [8 * len(comp) - 88]
    for i in range(0, len(rows), 10):   # a bit in the middle of the block: its symbol data
        q = (rows[i] + ends[i]) // 2
        bad[q >> 3] ^= 0x80 >> (q & 7)
    bad = bytes(bad)
    # warm-up of every shape, then the two calls alternating on the intact stream
    assert eng.decompressFile(comp) == src
    data, _ = eng.recover(comp)
    assert data == src
    eng.recover(bad)
    t_dec, t_rec, dev_dec, dev_rec = [], [], [], []
    for _ in range(a.runs):
        t, _ = timed(lambda: eng.decompressFile(comp))
        t_dec.append(t)
        dev_dec.append(eng.stats().ms_total)
        t, _ = timed(lambda: eng.recover(comp))
        t_rec.append(t)
        dev_rec.append(eng.stats().ms_total)
    t_bad = []
    for _ in range(a.runs):
        t, (got, regions) = timed(lambda: eng.recover(bad))
        t_bad.append(t)
    lost = [r for r in regions if r.status]
    res = {
        "gpu": gpu.strip(),
        "stream": "text:100000000:8:L9", "compressed_bytes": len(comp), "blocks": len(rows), "runs": a.runs,
        "intact": {
            "decompressFile_ms_median": 1e3 * statistics.median(t_dec), "recover_ms_median": 1e3 * statistics.median(t_rec),
            "recover_over_decompressFile": statistics.median(t_rec) / statistics.median(t_dec),
            "decompressFile_device_ms_median": statistics.median(dev_dec), "recover_device_ms_median": statistics.median(dev_rec),
        },
        "damaged": {
            "flipped_blocks": len(range(0, len(rows), 10)), "recover_ms_median": 1e3 * statistics.median(t_bad),
            "bytes_recovered": len(got), "bytes_total": len(src), "blocks_recovered": eng.stats().n_blocks,
            "damaged_regions": [[r.bit_begin, r.bit_end, r.kind_name, r.status] for r in lost],
            "recovered_sha256": hashlib.sha256(got).hexdigest(),
        },
    }
    if shutil.which("bzip2recover"):
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "damaged.bz2")
            with open(path, "wb") as fh:
                fh.write(bad)
            t0 = time.perf_counter()
            subprocess.run(["bzip2recover", path], cwd=tmp, check=True, capture_output=True)
            t1 = time.perf_counter()
            saved = 0
            pieces = sorted(f for f in os.listdir(tmp) if f.startswith("rec"))
            for name in pieces:
                try:
                    saved += len(bz2.decompress(open(os.path.join(tmp, name), "rb").read()))
                except (OSError, ValueError):
                    pass
            t2 = time.perf_counter()
        res["cpu_bzip2recover"] = {"bzip2recover_ms": 1e3 * (t1 - t0), "bz2_decompress_pieces_ms": 1e3 * (t2 - t1),
                                   "total_ms": 1e3 * (t2 - t0), "pieces": len(pieces), "bytes_recovered": saved}
    else:
        res["cpu_bzip2recover"] = None
    with open(os.path.join(a.outdir, "recover_bench.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["intact"]), json.dumps({k: v for k, v in res["damaged"].items() if k != "damaged_regions"}),
          json.dumps(res["cpu_bzip2recover"]), res["gpu"])


if __name__ == "__main__":
    main()
