#!/usr/bin/env python
"""bench.py -- bzip2 level-9 compress throughput (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--level 9] [--mb 100] [--mode compress|decompress]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path (Bzip2.compressFile at level 9) over one 100 MB batch of synthetic enwik8-like text
per GPU (BASELINE.json configs[1]; at N > 1 the N ranks compress ONE N x 100 MB stream as block-range shards: weak
scaling, no collective on the data path -- per-shard scalars travel through shared memory).

  value     whole-job MB/s (MB = 1e6 uncompressed input bytes) with the input resident in HBM, timed on the device with
            CUDA events on the launching stream, max over ranks
  e2e       the same metric through the reference-facing host call (bz2b200_compress at N = 1; at N > 1
            bz2b200_pool_compress_shards over a shared-memory group): host input, H2D + kernels + D2H inside the timed
            region, which the library overlaps by cutting the stream into shards over two lanes per GPU
  parity    SHA-256 of the produced stream against the oracle's golden (tests/golden/corpus_goldens.json)
  roofline  the dominant kernels of the BWT stage (kernel-local) and the whole pipeline (SURVEY 8d figure) against the
            measured HBM copy peak (MEASURED_PEAKS.json)
  decompress  device-resident and host-call decompression of the same stream; at N > 1 ONE stream decoded by all ranks
  cpu_baseline  the CPU oracle (a C port of the reference's algorithm, oracle/) on the host cores (rank 0, N = 1 only)

--impl reference times that CPU port with all host threads on the same config/metric.
--mode decompress makes decompression the headline value of the line (compress figures are then reported alongside).
--dump-outputs DIR writes what the last timed device-resident compress and decompress steps produced (one process only):
  compress_stream.npy / decompress_output.npy   the bytes as float32: all of them up to 4 Mi bytes, else the bytes at
                                                4 Mi sorted positions drawn with seed 0 from the output's length
  compress_stream_len.npy / decompress_output_len.npy   the output length in bytes (float64)
The inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import ctypes
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from untouched (it may be read-only)

UNIT = "MB/s"
DUMP_VALUES = 4 << 20   # bytes kept per dumped output: 16 MiB as float32, 32 MiB for the two outputs


def metric_name(level, mode):
    return f"bzip2-{level} compress MB/s, byte-identical output" if mode == "compress" else f"bzip2-{level} decompress MB/s, bit-exact round trip"


def workload_desc(level, mb, n_gpus):
    cfg = {1: "BASELINE.json configs[2]", 9: "BASELINE.json configs[1]"}.get(level, "")
    return {"workload": f"bzip2 level {level} ({level * 100} KB blocks) on {mb} MB synthetic enwik8-like text per GPU "
                        f"(compressjs_flattened_b200.corpus.gen_text, seed 8; {cfg})",
            "level": level, "bytes_per_gpu": mb * 1_000_000,
            "parallelism": f"block-range shards of ONE {mb * n_gpus} MB stream over {n_gpus} GPU(s); cross-rank: first-block offset + end bit + CRC fold "
                           "per shard (scalars, shared memory), no data-path collective",
            "l2": "two distinct 100 MB input buffers alternate between steps (200 MB > 126 MB L2); per-call device state is 5.3 GB"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): clocks.sm,
    clocks.max.sm and the clocks_event_reasons.active bitmask (decoded below), every 100 ms.  Measured beside this
    bench (tests/gpu_sampler_probe.py) the loop costs nothing as long as the timed path makes no driver-lock calls."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake"}

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = "index,clocks.sm,clocks.max.sm,clocks_event_reasons.active"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for t, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 4 or not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
                mask = int(f[3], 16)
            except ValueError:
                continue
            for bit, name in self.REASONS.items():
                if mask & bit:
                    reasons.add(name)
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}
        if not sm and self.lines:  # a window shorter than the sampling period: report the sample nearest to it
            t, line = min(self.lines, key=lambda x: abs(x[0] - (t0 + t1) / 2))
            f = [x.strip() for x in line.split(",")]
            try:
                out.update({"sm_mhz": float(f[1]), "sm_max_mhz": float(f[2]), "reasons": sorted(n for b, n in self.REASONS.items() if int(f[3], 16) & b),
                            "samples": 1, "note": f"nearest sample, {abs(t - (t0 + t1) / 2) * 1e3:.0f} ms from the middle of the timed region"})
            except (ValueError, IndexError):
                pass
        return out


# dram__bytes_read.sum + dram__bytes_write.sum of one k_rs_scatter<9> launch over 100 M keys (first pass of a bench step),
# `ncu --set full`, profiles/r01_ncu_notes.md; the algorithmic figure for that launch is 1.6e9 bytes
NCU_TRAFFIC_PER_LAUNCH = 1602111488
NCU_TRAFFIC_NOTE = "ncu --set full, first scatter pass of a step (100 M keys, 1.6e9 algorithmic bytes): 850.6 MB read + 751.5 MB written"


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def goldens():
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "corpus_goldens.json")))
    except Exception:
        return {}


def cpu_baseline(level, sample_mb, threads):
    import oracle_binding as O
    from compressjs_flattened_b200.corpus import gen_text
    data = gen_text(sample_mb * 1_000_000, 8)
    O.compress(data[:5_000_000], level, O.SORT_STABLE, threads=threads)
    t0 = time.time()
    out = O.compress(data, level, O.SORT_STABLE, threads=threads)
    dt = time.time() - t0
    t1 = time.time()
    back = O.decompress(out, False, threads=threads)
    dd = time.time() - t1
    return {"value": round(sample_mb / dt, 3), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"the first {sample_mb} MB of the workload ({len(out)} bytes out), oracle/liboracle.so (C port of Bzip2_joined_.js: SA-IS BWT, same "
                      f"table optimiser), block-parallel over {threads} pthreads, {dt:.1f} s; the reference itself is single-threaded JavaScript and Node "
                      "is not installed here",
            "out_bytes": len(out), "decompress_value": round(sample_mb / dd, 3), "decompress_ok": len(back) == sample_mb * 1_000_000}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_binding as O
    from compressjs_flattened_b200.corpus import gen_text
    threads = os.cpu_count() or 1
    sample_mb = args.ref_mb or args.mb
    data = gen_text(sample_mb * 1_000_000, 8)
    comp = O.compress(data, args.level, threads=threads) if args.mode == "decompress" else None
    for _ in range(min(args.warmup, 1)):
        O.compress(data[:5_000_000], args.level, threads=threads)
    times = []
    for _ in range(args.steps):
        t0 = time.time()
        if args.mode == "decompress":
            O.decompress(comp, False, threads=threads)
        else:
            O.compress(data, args.level, threads=threads)
        times.append(time.time() - t0)
    ms = 1e3 * sum(times) / len(times)
    val = sample_mb / (ms / 1e3)
    line = {"impl": "reference", "metric": metric_name(args.level, args.mode), "value": round(val, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": workload_desc(args.level, args.mb, args.gpus),
            "cpu_baseline": {"value": round(val, 3), "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"each step = {sample_mb} MB of the workload ({'all ' + str((sample_mb * 1_000_000) // (args.level * 100000 - 19) + 1) + ' blocks of one GPU share'}) "
                                       f"through oracle/liboracle.so on {threads} pthreads "
                                       "(Node is absent, so the reference's own JS cannot run; the oracle is its C restatement)"},
            "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def dump_output(out_dir, name, d_bytes):
    """a uint8 device tensor as out_dir/<name>.npy (float32, the seeded sample described in the module docstring) and its
    length as out_dir/<name>_len.npy"""
    import numpy as np
    import torch
    n = d_bytes.numel()
    if n > DUMP_VALUES:
        idx = np.sort(np.random.default_rng(0).integers(0, n, DUMP_VALUES))
        d_bytes = d_bytes[torch.from_numpy(idx).to(d_bytes.device)]
    np.save(os.path.join(out_dir, name + ".npy"), d_bytes.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, name + "_len.npy"), np.array([n], dtype=np.float64))


def gen_range(lo, hi, seed=8):
    """bytes [lo, hi) of the synthetic corpus (chunks of 1 MB are generated independently)"""
    from compressjs_flattened_b200.corpus import CHUNK, gen_text
    c0 = lo // CHUNK
    c1 = (hi + CHUNK - 1) // CHUNK
    buf = gen_text((c1 - c0) * CHUNK, seed, first_chunk=c0)
    return buf[lo - c0 * CHUNK: hi - c0 * CHUNK]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--level", type=int, default=9)
    ap.add_argument("--mb", type=int, default=100)
    ap.add_argument("--mode", default="compress", choices=["compress", "decompress"])
    ap.add_argument("--ref-mb", type=int, default=0, help="reference arm: MB per step (0 = --mb: the whole share of one GPU)")
    ap.add_argument("--cpu-sample-mb", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-big-check", action="store_true")
    ap.add_argument("--profile-only", action="store_true", help="device-resident compress steps only (for ncu runs)")
    ap.add_argument("--e2e-only", action="store_true", help="development: only the host-call leg, printed per rank 0 as a short line")
    ap.add_argument("--lanes", type=int, default=1, help="lanes per rank of the N>1 host-call leg (measured best at 8 ranks: 1, plan [25, 75] MB)")
    ap.add_argument("--plan-first-mb", type=float, default=0.0)
    ap.add_argument("--plan-growth", type=float, default=0.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed steps to DIR (see above)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs: the b200 implementation in one process only")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from compressjs_flattened_b200 import Bzip2Engine, _native
    from compressjs_flattened_b200.corpus import gen_text
    from compressjs_flattened_b200.pool import Bzip2Pool, ShardGroup, shard_plan

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: run on the CPUs next to it before any page-locked buffer exists (-1: the platform hides the node)
    from compressjs_flattened_b200.pool import bind_thread_to_device
    cpus_before = os.sched_getaffinity(0)
    host_node = bind_thread_to_device(local)
    ctl = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        ctl = dist.new_group(backend="gloo")   # verification gathers travel host-side
    host_nodes = [host_node]
    if world > 1:
        host_nodes = [None] * world
        dist.all_gather_object(host_nodes, host_node, group=ctl)
    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("BENCH_NO_SAMPLER"):
        sampler.start()   # started early (corpus generation takes seconds): it is streaming well before the timed region
    eng = Bzip2Engine(local)
    L = eng._L
    from compressjs_flattened_b200.sharded import HostMailbox, compress_shard
    mbox = HostMailbox(rank, world, os.environ.get("MASTER_PORT", "0")) if world > 1 else None
    level = args.level
    nbytes = args.mb * 1_000_000
    chunks = args.mb
    GOLD = goldens()
    halo_mb = 2 if (world > 1 and rank < world - 1) else 0   # bytes after the slice that the last owned block may need
    # two distinct corpora (j) so consecutive steps never re-read a cached input (200 MB > L2); rank r owns
    # bytes [r*mb MB, (r+1)*mb MB) of corpus j = one block-range shard of a world*mb MB stream
    host = [gen_text(nbytes + halo_mb * 1_000_000, 8, first_chunk=j * world * chunks + rank * chunks) for j in range(2)]
    pinned = [torch.from_numpy(h).pin_memory() for h in host]
    d_in = [p.to(dev) for p in pinned]
    navail = nbytes + halo_mb * 1_000_000
    bound = eng.compress_bound(nbytes, level)
    d_out = torch.empty((bound + 3) // 4 * 4 + 64, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def dev_step(i):
        if world == 1:
            return eng.compress_device(d_in[i % 2].data_ptr(), nbytes, level, d_out.data_ptr(), d_out.numel())
        n, _, _ = compress_shard(eng, None, rank * nbytes, nbytes, level, rank == world - 1, rank=rank, world=world, group=ctl,
                                 device_ptr=d_in[i % 2].data_ptr(), nbytes=navail, to_host=False, mailbox=mbox)
        return n

    # ---------------- device-resident: `value` ----------------
    for i in range(args.warmup):
        out_len = dev_step(i)
    barrier()
    t0 = time.time()
    dev_ms, dom_ms, dom_bytes, dom_launches, launches, stage = 0.0, 0.0, 0, 0, 0, [0.0] * 5
    for i in range(args.steps):
        out_len = dev_step(i)
        st = eng.stats()
        dev_ms += st.ms_total
        dom_ms += st.dom_ms
        dom_bytes += st.dom_bytes
        dom_launches += st.dom_launches
        launches += st.kernel_launches
        for k in range(5):
            stage[k] += st.ms_stage[k]
    barrier()
    t1 = time.time()
    if world > 1:
        print(f"[bench] rank {rank}: speculated shard starts held / recut = {compress_shard.guesses[True]} / {compress_shard.guesses[False]}", file=sys.stderr, flush=True)
    wall_ms = (t1 - t0) * 1e3
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    st_last = eng.stats()
    if args.dump_outputs:   # before anything else writes d_out
        os.makedirs(args.dump_outputs, exist_ok=True)
        dump_output(args.dump_outputs, "compress_stream", d_out[:out_len])

    if args.profile_only:
        print(json.dumps({"profile_only": True, "ms_per_step": round(dev_ms / args.steps, 3), "launches_per_step": launches // args.steps}), flush=True)
        return

    # ---------------- parity of what was just timed (N = 1): the stream of corpus 0 against the oracle's golden ----------------
    parity = None
    gkey = f"text:{nbytes * world}:8:L{level}"
    if world == 1:
        n0 = eng.compress_device(d_in[0].data_ptr(), nbytes, level, d_out.data_ptr(), d_out.numel())
        sha = hashlib.sha256(d_out[:n0].cpu().numpy().tobytes()).hexdigest()
        parity = {"golden": gkey if gkey in GOLD else None, "out_bytes": int(n0),
                  "sha256_equals_oracle_golden": (sha == GOLD[gkey]["out_sha256"]) if gkey in GOLD else None}

    # ---------------- end to end through the host API: `e2e` ----------------
    out_p, out_n = ctypes.POINTER(ctypes.c_uint8)(), ctypes.c_size_t()
    pool = grp = None
    e2e_jobs = None
    if world > 1:
        # ONE stream of world*mb MB as interleaved shards: wave k holds one shard of size plan[k] per rank, rank r takes shard
        # k*world + r.  Small first wave (its upload is the only exposed one), growing waves (copies hide under kernels).
        pool = Bzip2Pool([local], args.lanes)
        grp = ShardGroup(f"bench_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}", rank, world)
        plan = shard_plan(nbytes, level, args.lanes, int(args.plan_first_mb * 1e6), args.plan_growth)
        halo = 2_000_000
        total_bytes = world * nbytes
        e2e_jobs, keep, at = [], [], 0
        for k, sz in enumerate(plan):
            base = world * at + rank * sz
            hi = min(base + sz + halo, total_bytes)
            buf = torch.from_numpy(np.ascontiguousarray(gen_range(base, hi))).pin_memory()
            keep.append(buf)
            e2e_jobs.append(dict(src=buf.numpy(), own_len=sz, base=base, index=k * world + rank))
            at += sz
        total_shards = len(plan) * world
        h2d_bytes = sum(min(j["own_len"] + level * 125_000 + 65_536, j["src"].size) for j in e2e_jobs)

    def host_call(j, src=None):
        if world > 1:
            res = pool.compress_shards(grp, e2e_jobs, total_shards, level, to_bytes=False)
            n = 0
            for seg, info, off, nb in res:
                if seg:
                    pool.free_raw(seg)
                n += nb
            return n
        ptr = pinned[j].data_ptr() if src is None else src[j]
        rc = L.bz2b200_compress(eng._ctx, ptr, nbytes, level, ctypes.byref(out_p), ctypes.byref(out_n))
        if rc:
            eng._raise(rc)
        n = out_n.value
        L.bz2b200_free(out_p)
        return n

    def timed_host(src=None):
        host_call(0, src)
        host_call(1, src)
        barrier()
        e0 = time.time()
        n = 0
        for i in range(args.steps):
            n = host_call(i % 2, src)
        barrier()
        return (time.time() - e0) * 1e3, n

    e2e_ms, e2e_out = timed_host()
    if args.e2e_only:
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if rank == 0:
            print(json.dumps({"e2e_only": True, "n_gpus": world, "lanes": args.lanes, "plan_mb": [round(x / 1e6, 1) for x in (plan if world > 1 else [])],
                              "ms_per_step": round(float(tt.item()) / args.steps, 3), "MBps": round(world * args.mb * args.steps / (float(tt.item()) / 1e3), 1)}), flush=True)
        if world > 1:
            pool.close(); grp.close(); dist.destroy_process_group()
        return
    e2e_pageable_ms = None
    if world == 1:
        e2e_pageable_ms, _ = timed_host([h.ctypes.data for h in host])
        h2d_bytes = nbytes

    # ---------------- N > 1: the ranks' segments make ONE stream; it is checked against the oracle's golden ----------------
    stitched = None
    whole_dev = None
    if world > 1:
        res = pool.compress_shards(grp, e2e_jobs, total_shards, level)
        payload = [(j["index"], seg, (int(i.next_start), int(i.bits), int(i.n_blocks), int(i.crc_fold), int(i.complete), int(i.bit_phase)))
                   for j, (seg, i, _, _) in zip(e2e_jobs, res)]
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(payload, gathered, dst=0, group=ctl)
        nwhole = torch.zeros(1, dtype=torch.int64, device=dev)
        if rank == 0:
            parts = sorted(x for g in gathered for x in g)
            whole = eng.stitch_shards(level, [p[1] for p in parts], [_native.ShardInfo(*p[2]) for p in parts])
            sha = hashlib.sha256(whole).hexdigest()
            stitched = {"bytes": len(whole), "shards": len(parts), "blocks": sum(p[2][2] for p in parts), "golden": gkey if gkey in GOLD else None,
                        "sha256_equals_oracle_golden": (sha == GOLD[gkey]["out_sha256"]) if gkey in GOLD else None}
            nwhole[0] = len(whole)
        dist.broadcast(nwhole, 0)
        whole_dev = torch.empty(int(nwhole.item()) + 64, dtype=torch.uint8, device=dev)
        if rank == 0:
            whole_dev[:len(whole)] = torch.frombuffer(bytearray(whole), dtype=torch.uint8).to(dev)
            del whole, gathered, parts
        dist.broadcast(whole_dev, 0)
        out_len = eng.compress_device(d_in[0].data_ptr(), nbytes, level, d_out.data_ptr(), d_out.numel())

    # ---------------- decompress ----------------
    dec_steps = args.steps
    dec = {}
    if world == 1:
        last_in = (args.steps - 1) % 2
        out_len = eng.compress_device(d_in[last_in].data_ptr(), nbytes, level, d_out.data_ptr(), d_out.numel())
        comp = torch.empty(out_len, dtype=torch.uint8, device=dev)
        comp.copy_(d_out[:out_len])
        d_back = torch.empty(nbytes + 64, dtype=torch.uint8, device=dev)
        eng.decompress_device(comp.data_ptr(), out_len, False, d_back.data_ptr(), d_back.numel())
        dec_ms = 0.0
        for i in range(dec_steps):
            got = eng.decompress_device(comp.data_ptr(), out_len, False, d_back.data_ptr(), d_back.numel())
            dec_ms += eng.stats().ms_total
        roundtrip_ok = bool(got == nbytes and torch.equal(d_back[:nbytes], d_in[last_in][:nbytes]))
        if args.dump_outputs:
            dump_output(args.dump_outputs, "decompress_output", d_back[:got])
        comp_host = comp.cpu().pin_memory()
        def dec_host():
            rc = L.bz2b200_decompress(eng._ctx, comp_host.data_ptr(), out_len, 0, ctypes.byref(out_p), ctypes.byref(out_n))
            if rc:
                eng._raise(rc)
            L.bz2b200_free(out_p)
            return out_n.value
        dec_host()
        torch.cuda.synchronize()
        h0 = time.time()
        for i in range(dec_steps):
            dec_host()
        dec_e2e_ms = (time.time() - h0) * 1e3
        st_dec = eng.stats()
        dec_alg = (nbytes + 10 * st_dec.rle1_bytes + 2 * out_len) / 1e9 / (dec_ms / dec_steps / 1e3)
        dec = {"value": round(args.mb * dec_steps / (dec_ms / 1e3), 2), "unit": UNIT, "ms_per_step": round(dec_ms / dec_steps, 3),
               "roundtrip_bit_exact": roundtrip_ok,
               "e2e": {"value": round(args.mb * dec_steps / (dec_e2e_ms / 1e3), 2), "unit": UNIT, "ms_per_step": round(dec_e2e_ms / dec_steps, 3),
                       "h2d_bytes_per_step": int(out_len), "d2h_bytes_per_step": nbytes, "api": "bz2b200_decompress: pinned host input, page-locked host output"},
               "roofline": {"bound": "hbm", "scope": "pipeline (SURVEY 8d: 1 + 10*rho1 + 2*rho bytes per output byte)", "achieved": round(dec_alg, 1),
                            "unit": "GB/s", "frac": round(dec_alg / peaks()[0], 4)}}
        dec_ms_max = dec_ms
    else:
        # ONE stream (world*mb MB of text) decoded by all ranks: rank r takes byte slice r of the stream (resident in HBM),
        # the state of the reference's walk travels from slice to slice through the group
        nw = whole_dev.numel() - 64
        per = (nw + world - 1) // world
        per = (per + 15) & ~15   # slices of a device-resident stream start 16-byte aligned
        lo, hi = min(rank * per, nw), min((rank + 1) * per, nw)
        job = [dict(src=whole_dev.data_ptr() + lo, on_device=True, n_readable=nw - lo, own_len=hi - lo, base=lo, index=rank)] if hi > lo else []
        first_level = level
        r0 = pool.decompress_shards(grp, job, world, nw, first_level, keep_on_device=False)   # verification pass: bytes come back
        part, off, nb_, rc_, nblk = r0[0] if r0 else (b"", 0, 0, 0, 0)
        exp = gen_range(off, off + nb_) if nb_ else np.zeros(0, dtype=np.uint8)
        ok = torch.tensor([int(rc_ == 0 and bytes(part) == exp.tobytes()), nb_, nblk], dtype=torch.int64, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.SUM)
        barrier()
        d0 = time.time()
        for i in range(dec_steps):
            pool.decompress_shards(grp, job, world, nw, first_level, keep_on_device=True)
        barrier()
        dec_ms = (time.time() - d0) * 1e3
        dec = {"unit": UNIT, "one_stream_over_ranks": True, "stream_bytes": int(nw), "decoded_bytes": int(ok[1].item()), "blocks": int(ok[2].item()),
               "all_ranks_bit_exact": bool(ok[0].item() == world and ok[1].item() == world * nbytes),
               "timing": "host wall clock around the collective call, stream resident in HBM, decoded bytes stay in HBM"}
        dec_e2e_ms = None

    # ---------------- BASELINE configs[0]: the 2 MB HTML-like buffer, compress + decompress round trip through the host API ----------------
    small = None
    if world == 1 and not args.no_cpu_baseline:
        from compressjs_flattened_b200.corpus import gen_html
        hd = gen_html(2_130_640, 5)
        hz = eng.compressFile(hd, None, 9)
        eng.decompressFile(hz)
        reps = 10
        s0 = time.time()
        for _ in range(reps):
            hz = eng.compressFile(hd, None, 9)
        s1 = time.time()
        for _ in range(reps):
            hb = eng.decompressFile(hz)
        s2 = time.time()
        gk = "html:2130640:5:L9"
        small = {"workload": "BASELINE.json configs[0]: 2 130 640 B synthetic HTML-like text (gen_html, seed 5), level 9, 3 blocks, host buffers in and out",
                 "compress_ms": round((s1 - s0) / reps * 1e3, 3), "decompress_ms": round((s2 - s1) / reps * 1e3, 3),
                 "compress_MBps": round(2.13064 / ((s1 - s0) / reps), 1), "decompress_MBps": round(2.13064 / ((s2 - s1) / reps), 1),
                 "roundtrip_bit_exact": hb == hd.tobytes(),
                 "sha256_equals_oracle_golden": (hashlib.sha256(hz).hexdigest() == GOLD[gk]["out_sha256"]) if gk in GOLD else None}

    # ---------------- reduce over ranks ----------------
    t = torch.tensor([dev_ms, wall_ms, e2e_ms, dec_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, wall_ms_max, e2e_ms_max, dec_ms_max = [float(x) for x in t.tolist()]
    if rank == 0:
        peak, peak_src = peaks()
        total_mb = world * args.mb * args.steps
        achieved = dom_bytes / 1e9 / (dom_ms / 1e3) if dom_ms > 0 else 0.0
        pipe_alg = (1 + 12 * st_last.rle1_bytes / nbytes + 22 * st_last.mtf_syms / nbytes + 3 * out_len / nbytes) * nbytes / 1e9 / (dev_ms / args.steps / 1e3)
        if world > 1:
            dec.update({"value": round(world * args.mb * dec_steps / (dec_ms_max / 1e3), 2), "ms_per_step": round(dec_ms_max / dec_steps, 3)})
        comp_line = {"value": round(total_mb / (dev_ms_max / 1e3), 2), "ms_per_step": round(dev_ms_max / args.steps, 3)}
        e2e = {"value": round(total_mb / (e2e_ms_max / 1e3), 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(e2e_out),
               "ms_per_step": round(e2e_ms_max / args.steps, 3), "input": "pinned host memory",
               "api": "bz2b200_compress (N=1; inputs >= 32 MB run as shards over two lanes of the device) / bz2b200_pool_compress_shards over a "
                      "shared-memory group (N>1): page-locked host output from the library's result pool"}
        if e2e_pageable_ms:
            e2e["pageable_input"] = {"value": round(total_mb / (e2e_pageable_ms / 1e3), 2), "ms_per_step": round(e2e_pageable_ms / args.steps, 3),
                                     "note": "the same call on a pageable numpy buffer: staged through page-locked memory by the library's helper threads"}
        line = {
            "metric": metric_name(level, args.mode), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": workload_desc(level, args.mb, world),
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_rs_scatter<9>/<8> (BWT radix-sort scatter passes)", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": NCU_TRAFFIC_PER_LAUNCH, "traffic_note": NCU_TRAFFIC_NOTE, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(dom_bytes / max(dom_launches, 1)), "launches_per_step": dom_launches // args.steps,
                         "avg_launch_ms": round(dom_ms / max(dom_launches, 1), 4), "share_of_step": round(dom_ms / dev_ms, 3) if dev_ms else None,
                         "pipeline": {"scope": "whole compress pipeline, SURVEY 8d compulsory bytes 1 + 12*rho1 + 22*mu + 3*rho per input byte",
                                      "achieved": round(pipe_alg, 1), "frac": round(pipe_alg / peak, 4)},
                         "pipeline_algorithmic_GBps": round(pipe_alg, 1)},
            "stage_ms_per_step": {k: round(v / args.steps, 3) for k, v in zip(("rle1_cut_crc", "bwt", "mtf_rle2", "huffman_emit", "stitch"), stage)},
            "wall_ms_per_step": round(wall_ms_max / args.steps, 3),
            "clocks": clocks,
            "parity": parity,
            "stitched_stream": stitched,
            "small_file": small,
            "out_bytes_per_step": int(out_len), "blocks_per_step": int(st_last.n_blocks), "sort_rounds": int(st_last.sort_rounds),
        }
        if args.mode == "compress":
            line.update(comp_line)
            line["e2e"] = e2e
            line["decompress"] = dec
        else:
            line.update({"value": dec["value"], "ms_per_step": dec["ms_per_step"]})
            line["e2e"] = dec.get("e2e") or {"value": dec["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                                             "note": "N>1: stream and result resident in HBM"}
            line["compress"] = dict(comp_line, e2e=e2e)
            line["decompress"] = dec
        line["host_numa_node"] = host_nodes   # per rank: the node its feeding thread was bound to (-1: hidden by the platform)
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, cpus_before)   # the CPU arm gets every core the process started with
            line["cpu_baseline"] = cpu_baseline(level, args.cpu_sample_mb or args.mb, os.cpu_count() or 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        pool.close()
        grp.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
