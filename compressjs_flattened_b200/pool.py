"""Host mirror of the shard scheduler (include/bz2b200.h, "the shard scheduler"): `Bzip2.compressFile` /
`decompressFile` of ONE stream over several lanes, devices and -- through a ShardGroup -- processes of one node.

    pool = Bzip2Pool([0, 1, 2, 3])            # lanes on four GPUs of this process
    blob = pool.compressFile(data, None, 9)   # byte-identical to Bzip2.compressFile(data, None, 9)

    grp = ShardGroup("job42", rank, world)    # one process per GPU (torchrun): scalars through shared memory
    res = pool.compress_shards(grp, jobs, total_shards, 9)
"""
import ctypes as C

import numpy as np

from . import _native
from .bzip2 import Bzip2Error, _coerce_input, _compress_indexed, _deliver, _level, _search


def shard_plan(n, level=9, lanes=2, first_bytes=0, growth=0.0, library=None):
    """Shard sizes the scheduler would use for n bytes over `lanes` lanes (small first wave, growing waves)."""
    lib = library or _native.default_library()
    arr = (C.c_size_t * 4096)()
    k = lib.L.bz2b200_pool_plan(int(n), level, lanes, int(first_bytes), float(growth), arr, 4096)
    if k < 0:
        raise ValueError(f"bz2b200_pool_plan failed ({k})")
    return [int(arr[i]) for i in range(k)]


def bind_thread_to_device(device, library=None):
    """Run the calling thread on the CPUs next to `device` (bz2b200_bind_thread_to_device): call before allocating
    page-locked buffers in a one-process-per-GPU job.  Returns the NUMA node, or -1 when the platform hides it."""
    lib = library or _native.default_library()
    return int(lib.L.bz2b200_bind_thread_to_device(int(device)))


def _shard_jobs(jobs):
    """jobs (dicts {src, n_readable, own_len, base, index, on_device}) as a bz2b200_shard_job array, and the host
    arrays it points into (keep them alive for the call)."""
    arr = (_native.ShardJob * max(len(jobs), 1))()
    keep = []
    for i, j in enumerate(jobs):
        src = j["src"]
        if j.get("on_device"):
            ptr, nr = int(src), int(j["n_readable"])
        else:
            a = src if isinstance(src, np.ndarray) else _coerce_input(src)
            keep.append(a)
            ptr, nr = a.ctypes.data, int(j.get("n_readable", a.size))
        arr[i] = _native.ShardJob(ptr, nr, int(j["own_len"]), int(j["base"]), int(j["index"]), int(bool(j.get("on_device"))))
    return arr, keep


class ShardGroup:
    def __init__(self, name, rank, world, timeout_ms=120_000, library=None):
        self._lib = library or _native.default_library()
        self._g = C.c_void_p()
        rc = self._lib.L.bz2b200_group_open(str(name).encode(), rank, world, timeout_ms, C.byref(self._g))
        if rc:
            raise RuntimeError(f"bz2b200_group_open({name!r}, rank {rank} of {world}) failed ({rc})")
        self.rank, self.world = rank, world

    def close(self):
        if self._g:
            self._lib.L.bz2b200_group_close(self._g)
            self._g = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Bzip2Pool:
    def __init__(self, devices=(0,), lanes_per_device=2, library=None):
        self._lib = library or _native.default_library()
        self._L = self._lib.L
        self._p = C.c_void_p()
        devs = (C.c_int * len(devices))(*devices)
        rc = self._L.bz2b200_pool_create(devs, len(devices), lanes_per_device, C.byref(self._p))
        if rc:
            raise RuntimeError(f"bz2b200_pool_create(devices={list(devices)}) failed ({rc}): no usable CUDA device; "
                               "this package has no CPU fallback")

    def close(self):
        if self._p:
            self._L.bz2b200_pool_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _raise(self, rc):
        if rc == _native.E_LEVEL:
            raise ValueError("Invalid block size multiplier")
        msg = self._L.bz2b200_strerror(rc).decode()
        detail = self._L.bz2b200_pool_last_error(self._p).decode()
        if rc in (_native.E_CUDA, _native.E_ARG, _native.E_PEER):
            raise RuntimeError(msg + (": " + detail if detail else ""))
        raise Bzip2Error(rc, msg + (": " + detail if detail else ""))

    def _take(self, ptr, n):
        data = _native.take_bytes(ptr, n)
        self._L.bz2b200_free(ptr)
        return data

    def stats(self):
        st = _native.Stats()
        self._L.bz2b200_pool_last_stats(self._p, C.byref(st))
        return st

    def debug(self, block_cap=0, batch_blocks=0, first_halo=0, force_staging=False):
        rc = self._L.bz2b200_pool_debug(self._p, block_cap, batch_blocks, first_halo, int(bool(force_staging)))
        if rc:
            self._raise(rc)

    def set_plan(self, first_bytes=0, growth=0.0):
        rc = self._L.bz2b200_pool_set_plan(self._p, int(first_bytes), float(growth))
        if rc:
            self._raise(rc)

    def compressFile(self, input, output=None, props=None, shard_bytes=0):
        level = _level(props)
        a = _coerce_input(input)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_pool_compress(self._p, a.ctypes.data, a.size, level, shard_bytes, C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return _deliver(self._take(out, n.value), output)

    def compressIndexed(self, input, props=None, shard_bytes=0):
        """compressFile that also returns the stream's line index, built by every lane for its shards while compressing
        (no decode): (stream bytes, Bzip2LineIndex), as Bzip2Engine.compressIndexed returns them."""
        return _compress_indexed(self, self._L.bz2b200_pool_compress_indexed, self._p, input, props, int(shard_bytes))

    def compress_raw(self, ptr, nbytes, level, shard_bytes=0):
        """(pointer, length) of the stream in the library's page-locked result memory; release with free_raw."""
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_pool_compress(self._p, ptr, nbytes, level, shard_bytes, C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return out, n.value

    def free_raw(self, ptr):
        self._L.bz2b200_free(ptr)

    def decompressFile(self, input, output=None, multistream=False, slice_bytes=0):
        """Bzip2.decompressFile of ONE stream, block ranges over the lanes of the pool.  `output` given as a size (the
        reference's expected-size form, NPM/test/bzip2-basic.js:16) or a buffer doubles as the size hint."""
        a = _coerce_input(input)
        hint = output if isinstance(output, int) and not isinstance(output, bool) else (len(memoryview(output)) if isinstance(output, (bytearray, memoryview)) else 0)
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_pool_decompress(self._p, a.ctypes.data, a.size, int(bool(multistream)), int(hint), int(slice_bytes), C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return _deliver(self._take(out, n.value), output)

    def decompress_raw(self, ptr, nbytes, multistream=False, size_hint=0, slice_bytes=0):
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        rc = self._L.bz2b200_pool_decompress(self._p, ptr, nbytes, int(bool(multistream)), int(size_hint), int(slice_bytes), C.byref(out), C.byref(n))
        if rc:
            self._raise(rc)
        return out, n.value

    def search(self, input, patterns, ignore_case=False, max_matches=None, multistream=False, lines=False, slice_bytes=0):
        """Bzip2Engine.search of ONE stream, decoded and searched slice by slice over the lanes of the pool: the same
        SearchResult, field for field.  slice_bytes: bytes of stream per slice (0 = as decompressFile picks them)."""
        return _search(self, self._L.bz2b200_pool_search, self._p, input, patterns, ignore_case, max_matches, multistream, lines, int(slice_bytes))

    def debug_set_search_tile(self, nbytes):
        """tests only: bytes per search tile of every lane (a multiple of 256 up to 8192; 0 restores the default)"""
        rc = self._L.bz2b200_debug_set_pool_search_tile(self._p, nbytes)
        if rc:
            self._raise(rc)

    def debug_decode_batch(self, candidates):
        self._L.bz2b200_debug_set_decode_batch(None, self._p, candidates)

    def debug_rle1_threads(self, threads):
        rc = self._L.bz2b200_debug_set_rle1_threads(None, self._p, threads)
        if rc:
            self._raise(rc)

    def decompress_shards(self, group, jobs, total_shards, total_n, first_level, multistream=False, keep_on_device=False, to_bytes=True):
        """This process's byte slices of a stream that spans the group.  jobs: dicts {src, n_readable, own_len, base, index,
        on_device}.  Returns [(bytes | pointer | None, out_offset, n_bytes, rc, n_blocks)] per job; the stream's status is
        the first non-zero rc in slice order over ALL ranks."""
        n = len(jobs)
        arr, keep = _shard_jobs(jobs)
        res = (_native.RangeResult * max(n, 1))()
        rc = self._L.bz2b200_pool_decompress_shards(self._p, group._g if group is not None else None, arr, n, total_shards, int(total_n),
                                                    int(first_level), int(bool(multistream)), int(bool(keep_on_device)), res)
        if rc:
            self._raise(rc)
        out = []
        for i in range(n):
            r = res[i]
            if r.part and to_bytes:
                part = self._take(r.part, r.bytes)
            elif r.part:
                part = r.part
            else:
                part = b"" if (to_bytes and not keep_on_device) else None
            out.append((part, int(r.out_offset), int(r.bytes), int(r.rc), int(r.n_blocks)))
        return out

    def compress_shards(self, group, jobs, total_shards, level, keep_on_device=False, to_bytes=True):
        """jobs: list of dicts {src: bytes-like or device pointer (int), n_readable, own_len, base, index, on_device}.
        Returns a list of (segment, ShardResult): segment = bytes (to_bytes), a raw pointer, or None (keep_on_device)."""
        n = len(jobs)
        arr, keep = _shard_jobs(jobs)
        res = (_native.ShardResult * max(n, 1))()
        rc = self._L.bz2b200_pool_compress_shards(self._p, group._g if group is not None else None, arr, n, total_shards, level,
                                                  int(bool(keep_on_device)), res)
        if rc:
            self._raise(rc)
        out = []
        for i in range(n):
            r = res[i]
            if keep_on_device or not r.seg_bytes:
                seg = b"" if (to_bytes and not keep_on_device) else None
                if r.seg:
                    self._L.bz2b200_free(r.seg)
            elif to_bytes:
                seg = self._take(r.seg, r.seg_bytes)
            else:
                seg = r.seg
            info = _native.ShardInfo(r.info.next_start, r.info.bits, r.info.n_blocks, r.info.crc_fold, r.info.complete, r.info.bit_phase)
            out.append((seg, info, int(r.bit_offset), int(r.seg_bytes)))
        return out
