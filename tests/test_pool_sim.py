"""The shard scheduler (csrc/pool.inl) on the CPU simulator: lanes of one process, forced staging, halo growth, shards
that own no block, and two PROCESSES exchanging the per-shard scalars through a shared-memory group -- every stream
byte-identical to the oracle (and to the single-call path)."""
import multiprocessing as mp
import os

import numpy as np
import pytest

from conftest import HERE

SIM_SO = os.path.join(HERE, "sim", "libbz2b200_sim.so")


def _runny(rng, n, nsym, plong):
    out = bytearray()
    while len(out) < n:
        b = int(rng.integers(0, nsym))
        ln = int(rng.integers(4, 700)) if rng.random() < plong else int(rng.integers(1, 4))
        out += bytes([b]) * ln
    return bytes(out[:n])


def _inputs():
    rng = np.random.default_rng(21)
    from compressjs_flattened_b200.corpus import gen_text
    return {
        "text": gen_text(60_000, 4).tobytes(),
        "runny": _runny(rng, 50_000, 3, 0.4),        # blocks that read far more input than they hold: halos must grow
        "zeros": bytes(40_000),
        "rand": rng.integers(0, 256, 30_000, dtype=np.uint8).tobytes(),
        "empty": b"",
        "tiny": b"abc",
    }


@pytest.fixture(scope="module")
def sim_lib(sim_engine):
    from compressjs_flattened_b200 import _native
    return _native.Library(SIM_SO)


@pytest.mark.parametrize("name", sorted(_inputs()))
def test_context_pool_equals_oracle(sim_lib, oracle, name):
    """bz2b200_compress routed through the context's own two-lane pool (threshold lowered for the test)."""
    from compressjs_flattened_b200.bzip2 import Bzip2Engine
    data = _inputs()[name]
    eng = Bzip2Engine(0, sim_lib)
    eng.debug_set_block_cap(997)
    oracle.set_block_cap(997)
    try:
        exp, st = oracle.compress(data, 9, return_stats=True)
        for shard, halo, staging in ((4096, 0, False), (8192, 64, True), (1000, 16, False)):
            eng.debug_set_pool(0, shard, halo, staging)
            assert eng.compressFile(data, None, 9) == exp, (shard, halo, staging)
            assert eng.stats().n_blocks == st.n_blocks
    finally:
        oracle.set_block_cap(0)
        eng.close()


def test_pool_lanes_and_devices(sim_lib, oracle):
    """an explicit pool: 2 'devices' x 2 lanes, several shard sizes, levels 1 and 9 at the real block sizes; then small
    blocks in batches of 1 and 3, so that every lane stitches its segment from several batches"""
    from compressjs_flattened_b200.pool import Bzip2Pool
    from compressjs_flattened_b200.corpus import gen_text
    data = gen_text(450_000, 7).tobytes()
    pool = Bzip2Pool([0, 0], 2, library=sim_lib)
    try:
        for level, shard in ((1, 0), (1, 120_000), (9, 200_000)):
            assert pool.compressFile(data, None, level, shard_bytes=shard) == oracle.compress(data, level)
        pool.set_plan(30_000, 2.0)    # growing waves: 30, 30, 30, 30, 60, ... KB over the four lanes
        assert pool.compressFile(data, None, 1) == oracle.compress(data, 1)
        with pytest.raises(ValueError):
            pool.compressFile(data, None, 0)
        pool.set_plan(0, 0.0)
        oracle.set_block_cap(7001)
        try:
            exp = oracle.compress(data[:120_000], 9)
            for per in (1, 3):
                pool.debug(block_cap=7001, batch_blocks=per)
                assert pool.compressFile(data[:120_000], None, 9, shard_bytes=30_000) == exp, per
        finally:
            oracle.set_block_cap(0)
    finally:
        pool.close()


def _rank_main(rank, world, name, data, shard, cap, q):
    try:
        from compressjs_flattened_b200 import _native
        from compressjs_flattened_b200.pool import Bzip2Pool, ShardGroup
        lib = _native.Library(SIM_SO)
        grp = ShardGroup(name, rank, world, timeout_ms=60_000, library=lib)
        pool = Bzip2Pool([0], 2, library=lib)
        pool.debug(block_cap=cap, first_halo=32)
        total = (len(data) + shard - 1) // shard
        outs = []
        for rep in range(2):      # two collective calls on one group: epochs must not mix
            jobs = [dict(src=np.frombuffer(data[j * shard:], dtype=np.uint8), own_len=min(shard, len(data) - j * shard), base=j * shard, index=j)
                    for j in range(total) if j % world == rank]
            res = pool.compress_shards(grp, jobs, total, 9)
            outs.append([(j["index"], seg, (int(i.next_start), int(i.bits), int(i.n_blocks), int(i.crc_fold), int(i.complete), int(i.bit_phase)))
                         for j, (seg, i, _, _) in zip(jobs, res)])
        q.put((rank, outs))
        pool.close()
        grp.close()
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))


@pytest.mark.parametrize("world", [2, 3])
def test_group_of_processes_equals_oracle(sim_lib, oracle, world):
    from compressjs_flattened_b200 import _native
    from compressjs_flattened_b200.bzip2 import Bzip2Engine
    rng = np.random.default_rng(5)
    data = _runny(rng, 30_000, 4, 0.2) + bytes(rng.integers(0, 256, 20_000, dtype=np.uint8))
    shard, cap = 3000, 701
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    name = f"test_{os.getpid()}_{world}"
    procs = [ctx.Process(target=_rank_main, args=(r, world, name, data, shard, cap, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r, v in got.items():
        assert not isinstance(v, str), f"rank {r}: {v}"
    oracle.set_block_cap(cap)
    try:
        exp = oracle.compress(data, 9)
    finally:
        oracle.set_block_cap(0)
    eng = Bzip2Engine(0, sim_lib)
    for rep in range(2):
        parts = sorted(x for r in range(world) for x in got[r][rep])
        segs = [p[1] for p in parts]
        infos = [_native.ShardInfo(*p[2]) for p in parts]
        assert eng.stitch_shards(9, segs, infos) == exp


def _dead_peer_main(name, q):
    from compressjs_flattened_b200 import _native
    from compressjs_flattened_b200.pool import Bzip2Pool, ShardGroup
    lib = _native.Library(SIM_SO)
    grp = ShardGroup(name, 1, 2, timeout_ms=8_000, library=lib)
    pool = Bzip2Pool([0], 1, library=lib)
    data = np.frombuffer(b"x" * 5000, dtype=np.uint8)
    try:   # shard 0 never arrives: rank 0 joined the group and left
        pool.compress_shards(grp, [dict(src=data[2500:], own_len=2500, base=2500, index=1)], 2, 9)
        q.put("no error")
    except RuntimeError as e:
        q.put(str(e))


def test_dead_peer_is_an_error_not_a_hang(sim_lib):
    """Robustness of the shard protocol (VERDICT r1 item 9): a peer that never publishes makes the wait time out."""
    from compressjs_flattened_b200.pool import ShardGroup
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    name = f"dead_{os.getpid()}"
    p = ctx.Process(target=_dead_peer_main, args=(name, q))
    p.start()
    grp = ShardGroup(name, 0, 2, timeout_ms=8_000, library=sim_lib)   # attaches, then does nothing
    msg = q.get(timeout=120)
    p.join(timeout=30)
    grp.close()
    assert "peer" in msg


# ------------------------------------------------------------------------------------------------ decompress
def _streams(oracle):
    rng = np.random.default_rng(33)
    from compressjs_flattened_b200.corpus import gen_text
    text = gen_text(70_000, 9).tobytes()
    oracle.set_block_cap(1201)
    try:
        many = oracle.compress(text, 9)                                   # ~58 small blocks
        runny = oracle.compress(_runny(rng, 40_000, 3, 0.5), 9)
        rand = oracle.compress(rng.integers(0, 256, 9_000, dtype=np.uint8).tobytes(), 9)   # blocks larger than a slice
    finally:
        oracle.set_block_cap(0)
    return {"many": (many, False), "runny": (runny, False), "rand": (rand, False),
            "multi": (many + rand + oracle.compress(b"tail stream"), True), "first_only": (many + rand, False),
            "empty": (oracle.compress(b""), False), "tiny": (oracle.compress(b"xyz"), False)}


@pytest.mark.parametrize("name", ["many", "runny", "rand", "multi", "first_only", "empty", "tiny"])
def test_pool_decompress_slices_equal_oracle(sim_lib, oracle, name):
    """ONE stream decoded as byte slices over the lanes (walk state chained from slice to slice): slices smaller than a
    block, halos that must grow, several batches per slice, multistream hops across slices, size hint and no hint."""
    from compressjs_flattened_b200.pool import Bzip2Pool
    blob, ms = _streams(oracle)[name]
    exp = oracle.decompress(blob, ms)
    pool = Bzip2Pool([0, 0], 2, library=sim_lib)
    try:
        for slice_bytes, halo, batch, hint in ((0, 0, 0, 0), (997, 64, 0, len(exp)), (4000, 16, 3, 0), (300, 8, 2, 0)):
            pool.debug(first_halo=halo)
            pool.debug_decode_batch(batch)
            got = pool.decompressFile(blob, hint if hint else None, ms, slice_bytes=slice_bytes)
            assert got == exp, (name, slice_bytes, halo, batch)
    finally:
        pool.close()


def test_single_context_decode_in_batches(sim_lib, oracle):
    """ADVICE r1 (medium): the candidates of a stream are decoded in batches, so device memory is bounded"""
    from compressjs_flattened_b200.bzip2 import Bzip2Engine
    blob, _ = _streams(oracle)["many"]
    eng = Bzip2Engine(0, sim_lib)
    eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, 5)
    try:
        assert eng.decompressFile(blob) == oracle.decompress(blob)
        rows = []
        eng.table(blob, lambda p, s: rows.append((p, s)))
        assert rows == oracle.table(blob)
    finally:
        eng.close()


def test_pool_decompress_errors_first_in_stream_order(sim_lib, oracle):
    from compressjs_flattened_b200.bzip2 import Bzip2Error
    from compressjs_flattened_b200.pool import Bzip2Pool
    blob, _ = _streams(oracle)["many"]
    pool = Bzip2Pool([0], 3, library=sim_lib)
    cases = [blob[:len(blob) // 2], blob[:-3]]
    for at in (len(blob) // 5, len(blob) // 2, len(blob) - 30):
        b = bytearray(blob)
        b[at] ^= 0x5A
        cases.append(bytes(b))
    two = bytearray(blob)     # two damaged places: the earlier one decides
    two[len(blob) // 4] ^= 1
    two[3 * len(blob) // 4] ^= 0xFF
    cases.append(bytes(two))
    cases += [b"", b"BZ", b"BZh0" + blob[4:], b"XXXX" + blob[4:]]
    try:
        for i, bad in enumerate(cases):
            try:
                exp = ("ok", oracle.decompress(bad))
            except oracle.OracleError as e:
                exp = ("err", e.errorCode)
            try:
                got = ("ok", pool.decompressFile(bad, None, False, slice_bytes=1500))
            except Bzip2Error as e:
                got = ("err", e.errorCode)
            assert got == exp, i
    finally:
        pool.close()


def _dec_rank_main(rank, world, name, blob, slice_bytes, q):
    try:
        from compressjs_flattened_b200 import _native
        from compressjs_flattened_b200.pool import Bzip2Pool, ShardGroup
        lib = _native.Library(SIM_SO)
        grp = ShardGroup(name, rank, world, timeout_ms=60_000, library=lib)
        pool = Bzip2Pool([0], 2, library=lib)
        pool.debug(first_halo=100)
        total = (len(blob) + slice_bytes - 1) // slice_bytes
        jobs = [dict(src=np.frombuffer(blob[j * slice_bytes:], dtype=np.uint8), own_len=min(slice_bytes, len(blob) - j * slice_bytes), base=j * slice_bytes, index=j)
                for j in range(total) if j % world == rank]
        res = pool.decompress_shards(grp, jobs, total, len(blob), blob[3] - 0x30)
        q.put((rank, [(j["index"],) + r for j, r in zip(jobs, res)]))
        pool.close()
        grp.close()
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))


def test_group_of_processes_decodes_one_stream(sim_lib, oracle):
    blob, _ = _streams(oracle)["many"]
    exp = oracle.decompress(blob)
    world, slice_bytes = 2, 2500
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    name = f"dec_{os.getpid()}"
    procs = [ctx.Process(target=_dec_rank_main, args=(r, world, name, blob, slice_bytes, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r, v in got.items():
        assert not isinstance(v, str), f"rank {r}: {v}"
    parts = sorted(x for r in range(world) for x in got[r])
    out = bytearray(len(exp))
    for idx, part, off, nbytes, rc, nblk in parts:
        assert rc == 0
        out[off:off + nbytes] = part
    assert bytes(out) == exp and sum(p[3] for p in parts) == len(exp)


def test_ranked_decode_checks_the_stream_header(sim_lib, oracle):
    """the rank that holds slice 0 checks 'BZh<level>' (BJ:1408-1427); a wrong header is the stream's error, not a crash"""
    from compressjs_flattened_b200.pool import Bzip2Pool
    blob = oracle.compress(b"header check " * 300, 9)
    pool = Bzip2Pool([0], 1, library=sim_lib)
    try:
        job = lambda b: [dict(src=np.frombuffer(b, dtype=np.uint8), own_len=len(b), base=0, index=0)]
        part, off, n, rc, nblk = pool.decompress_shards(None, job(blob), 1, len(blob), 9)[0]
        assert rc == 0 and part == b"header check " * 300
        for bad, lvl in ((b"BZx9" + blob[4:], 9), (blob, 5), (b"BZ", 9)):
            res = pool.decompress_shards(None, job(bad), 1, len(bad), lvl)[0]
            assert res[3] == -2 and res[2] == 0
    finally:
        pool.close()


_BIND_CHILD = r"""
import ctypes, os, sys
L = ctypes.CDLL(sys.argv[1])
L.bz2b200_bind_thread_to_device.argtypes = [ctypes.c_int]
before = sorted(os.sched_getaffinity(0))
node = L.bz2b200_bind_thread_to_device(int(sys.argv[2]))
print(node, ",".join(map(str, before)), ",".join(map(str, sorted(os.sched_getaffinity(0)))))
"""


def _fake_sysfs(tmp_path, bus, node, cpulist):
    d = tmp_path / "bus" / "pci" / "devices" / bus
    d.mkdir(parents=True)
    (d / "numa_node").write_text(f"{node}\n")
    if node >= 0:
        nd = tmp_path / "devices" / "system" / "node" / f"node{node}"
        nd.mkdir(parents=True)
        (nd / "cpulist").write_text(cpulist + "\n")


@pytest.mark.parametrize("case", ["bind", "hidden", "foreign_cpus", "switched_off"])
def test_bind_thread_to_device(sim_engine, tmp_path, case):
    """bz2b200_bind_thread_to_device: sysfs numa_node of the device's PCI address -> the node's cpulist, intersected with the
    thread's own CPUs (made-up sysfs tree; the simulator takes the PCI address from the environment).  A hidden node (-1),
    a node with none of our CPUs, or BZ2B200_NUMA=0 leave the thread alone and return -1."""
    import subprocess
    import sys
    mine = sorted(os.sched_getaffinity(0))
    if len(mine) < 3:
        pytest.skip("needs three CPUs")
    env = dict(os.environ, BZ2B200_SYSFS=str(tmp_path), BZ2B200_SIM_BUSID="0000:1B:00.0")
    expect_node, expect_cpus = -1, mine
    if case == "bind":   # "a,b-c" with a range, plus CPUs that do not exist here
        _fake_sysfs(tmp_path, "0000:1b:00.0", 1, f"{mine[0]},{mine[1]}-{mine[2]},{mine[-1] + 900}-{mine[-1] + 910}")
        expect_node, expect_cpus = 1, sorted(set([mine[0]] + list(range(mine[1], mine[2] + 1))) & set(mine))
    elif case == "hidden":
        _fake_sysfs(tmp_path, "0000:1b:00.0", -1, "")
    elif case == "foreign_cpus":
        _fake_sysfs(tmp_path, "0000:1b:00.0", 0, f"{mine[-1] + 900}-{mine[-1] + 910}")
    else:
        _fake_sysfs(tmp_path, "0000:1b:00.0", 1, f"{mine[0]}")
        env["BZ2B200_NUMA"] = "0"
    out = subprocess.run([sys.executable, "-c", _BIND_CHILD, SIM_SO, "0"], env=env, capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    node, before, after = out.stdout.split()
    assert int(node) == expect_node
    assert [int(x) for x in before.split(",")] == mine
    assert [int(x) for x in after.split(",")] == expect_cpus


def test_shard_plan_invariants(sim_lib):
    """bz2b200_pool_plan: for every size, lane count, first-shard size and growth the shards are non-empty and add up to the
    input (a first shard of one byte once rounded the part count of the last wave down to zero: an empty plan)."""
    import ctypes as C
    arr = (C.c_size_t * 4096)()
    for n in list(range(0, 40)) + [100, 4095, 4096, 4097, 10_000, 123_457, (1 << 24) + 5, 10 ** 8, 8 * 10 ** 9]:
        for lanes in (1, 2, 3, 8):
            for first in (0, 1, 2, 7, 4096, n // 5 * 2 + 1, 25_000_000):
                for growth in (0.0, 1.0, 3.0, 1000.0):
                    k = sim_lib.L.bz2b200_pool_plan(n, 9, lanes, first, growth, arr, 4096)
                    if k < 0:   # more than 4096 shards: refused, not truncated
                        assert first and first * 4096 < n
                        continue
                    sizes = [int(arr[i]) for i in range(k)]
                    assert k >= 1 and sum(sizes) == n and (n == 0 or min(sizes) > 0), (n, lanes, first, growth, sizes[:8])


def test_context_pool_on_tiny_inputs(sim_lib, oracle):
    """bz2b200_compress through the context's own lanes for inputs of 1..9 bytes (plan_first = n / 5 * 2 + 1 = 1)."""
    from compressjs_flattened_b200.bzip2 import Bzip2Engine
    eng = Bzip2Engine(0, sim_lib)
    eng.debug_set_pool(1)
    try:
        for n in range(1, 10):
            data = bytes(range(65, 65 + n))
            assert eng.compressFile(data, None, 9) == oracle.compress(data, 9)
    finally:
        eng.debug_set_pool()


def test_object_lifecycles_leave_nothing_behind(tmp_path):
    """tests/sim/leak_check.cpp under AddressSanitizer + LeakSanitizer: three rounds of create / use / destroy of a context
    (whole-buffer calls, table, one block, a damaged stream, its own lanes), stream objects (finished and abandoned) and a
    pool.  In the simulator device memory is host memory, so a buffer the library forgets to free -- on either side -- is
    reported; the simulator's own fiber stacks are suppressed (tests/sim/lsan.supp)."""
    import shutil
    import subprocess
    if not os.environ.get("BZ2B200_SANITIZER_TESTS"):
        pytest.skip("opt-in (BZ2B200_SANITIZER_TESTS=1): builds the simulator with -fsanitize=address, ~100 s")
    if not shutil.which("g++"):
        pytest.skip("no g++")
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no libasan")
    sim = os.path.join(HERE, "sim")
    root = os.path.dirname(HERE)
    subprocess.check_call([os.path.join(sim, "build_sim.sh")], env=dict(os.environ, SIM_SANITIZE="address"))
    exe = str(tmp_path / "leak_check")
    subprocess.check_call(["g++", "-std=c++17", "-g", "-fsanitize=address", "-I" + os.path.join(root, "include"), os.path.join(sim, "leak_check.cpp"),
                           os.path.join(sim, "libbz2b200_sim_address.so"), "-Wl,-rpath," + sim, "-o", exe])
    env = dict(os.environ, ASAN_OPTIONS="detect_stack_use_after_return=0",
               LSAN_OPTIONS="suppressions=" + os.path.join(sim, "lsan.supp") + ":print_suppressions=0")
    out = subprocess.run([exe], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "3 rounds done" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
