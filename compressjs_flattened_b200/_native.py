"""ctypes loader for libbz2b200.so (the CUDA library behind include/bz2b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device can be
opened, every entry point raises.  (tests/sim/ builds a CPU *simulation* of the kernels for
logic tests; it is loaded only by tests through `Library(path=...)`, never from here.)
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_SO = os.environ.get("BZ2B200_LIB") or os.path.join(_HERE, "libbz2b200.so")   # BZ2B200_LIB: development builds of the same CUDA library

E_LEVEL, E_CUDA, E_ARG, E_PEER = -100, -101, -102, -103


class Stats(C.Structure):
    _fields_ = [("in_bytes", C.c_uint64), ("out_bytes", C.c_uint64), ("n_blocks", C.c_uint32),
                ("sort_rounds", C.c_uint32), ("rle1_bytes", C.c_uint64), ("mtf_syms", C.c_uint64),
                ("sort_slots", C.c_uint64), ("kernel_launches", C.c_uint32), ("d1_triggered", C.c_uint32),
                ("ms_total", C.c_float), ("ms_stage", C.c_float * 8),
                ("dom_ms", C.c_float), ("dom_launches", C.c_uint32), ("dom_bytes", C.c_uint64)]


class BlockRec(C.Structure):
    _fields_ = [("s", C.c_int64), ("p", C.c_int64), ("e_true", C.c_int64), ("Ge", C.c_uint64),
                ("outR", C.c_uint32), ("n", C.c_uint32), ("crc", C.c_uint32), ("orig_ptr", C.c_uint32)]


class BlockMeta(C.Structure):
    _fields_ = [("alpha", C.c_uint32), ("m", C.c_uint32), ("used", C.c_uint32 * 8), ("n_groups", C.c_uint32),
                ("n_sel", C.c_uint32), ("bits", C.c_uint64), ("d1", C.c_uint32), ("pad", C.c_uint32)]


class DecBlk(C.Structure):
    _fields_ = [("bitpos", C.c_uint64), ("endbit", C.c_uint64), ("target_crc", C.c_uint32), ("orig_ptr", C.c_uint32),
                ("count", C.c_uint32), ("err", C.c_int32), ("kind", C.c_uint32), ("nsym", C.c_uint32)]


class ShardInfo(C.Structure):
    _fields_ = [("next_start", C.c_uint64), ("bits", C.c_uint64), ("n_blocks", C.c_uint32), ("crc_fold", C.c_uint32),
                ("complete", C.c_uint32), ("bit_phase", C.c_uint32)]


class ShardJob(C.Structure):
    _fields_ = [("src", C.c_void_p), ("n_readable", C.c_size_t), ("own_len", C.c_size_t), ("base", C.c_uint64),
                ("index", C.c_int32), ("on_device", C.c_int32)]


class ShardResult(C.Structure):
    _fields_ = [("seg", C.POINTER(C.c_uint8)), ("seg_bytes", C.c_size_t), ("info", ShardInfo), ("bit_offset", C.c_uint64),
                ("end_bit", C.c_uint64), ("blocks_through", C.c_uint64), ("crc_fold_through", C.c_uint32), ("pad", C.c_uint32)]


class RangeResult(C.Structure):
    _fields_ = [("part", C.POINTER(C.c_uint8)), ("bytes", C.c_uint64), ("out_offset", C.c_uint64), ("rc", C.c_int32), ("n_blocks", C.c_uint32)]


class Region(C.Structure):
    _fields_ = [("bit_begin", C.c_uint64), ("bit_end", C.c_uint64), ("out_offset", C.c_uint64), ("out_bytes", C.c_uint32),
                ("crc", C.c_uint32), ("status", C.c_int32), ("kind", C.c_uint32), ("stream", C.c_uint32), ("flags", C.c_uint32)]


class BlockEntry(C.Structure):
    _fields_ = [("bit_begin", C.c_uint64), ("bit_end", C.c_uint64), ("out_offset", C.c_uint64), ("out_bytes", C.c_uint32),
                ("crc", C.c_uint32), ("stream", C.c_uint32), ("level", C.c_uint32)]


class Match(C.Structure):
    _fields_ = [("offset", C.c_uint64), ("line", C.c_uint64), ("line_begin", C.c_uint64), ("line_end", C.c_uint64),
                ("pattern", C.c_uint32), ("flags", C.c_uint32)]


class SearchTotals(C.Structure):
    _fields_ = [("matches", C.c_uint64), ("lines", C.c_uint64), ("out_bytes", C.c_uint64)]


def take_bytes(ptr, n):
    """n bytes at a ctypes pointer as a bytes object (ctypes.string_at takes an int-sized length: streams above 2 GiB)"""
    if not n:
        return b""
    if n < (1 << 31):
        return C.string_at(ptr, n)
    return bytes(memoryview((C.c_ubyte * n).from_address(C.addressof(ptr.contents))))


class Library:
    """Thin typed view of the C ABI."""

    def __init__(self, path=None):
        path = path or DEFAULT_SO
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                "There is no CPU fallback.")
        L = C.CDLL(path)
        vp, u8pp, szp = C.c_void_p, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_size_t)
        L.bz2b200_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.bz2b200_destroy.argtypes = [vp]
        L.bz2b200_destroy.restype = None
        L.bz2b200_compress.argtypes = [vp, vp, C.c_size_t, C.c_int, u8pp, szp]
        L.bz2b200_decompress.argtypes = [vp, vp, C.c_size_t, C.c_int, u8pp, szp]
        L.bz2b200_decompress_block.argtypes = [vp, vp, C.c_size_t, C.c_uint64, u8pp, szp]
        L.bz2b200_table.argtypes = [vp, vp, C.c_size_t, C.c_int, C.POINTER(C.POINTER(C.c_uint64)),
                                    C.POINTER(C.POINTER(C.c_uint32)), szp]
        L.bz2b200_recover.argtypes = [vp, vp, C.c_size_t, u8pp, szp, C.POINTER(C.POINTER(Region)), szp]
        L.bz2b200_index.argtypes = [vp, vp, C.c_size_t, C.c_int, C.POINTER(C.POINTER(BlockEntry)), szp]
        L.bz2b200_decompress_ranges.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t, vp, vp, C.c_size_t, u8pp, szp]
        L.bz2b200_search.argtypes = [vp, vp, C.c_size_t, C.c_int, vp, vp, C.c_size_t, C.c_uint, C.c_uint64, C.POINTER(C.POINTER(Match)), szp,
                                     C.POINTER(SearchTotals), u8pp, szp]
        L.bz2b200_free.argtypes = [vp]
        L.bz2b200_free.restype = None
        L.bz2b200_compress_device.argtypes = [vp, vp, C.c_size_t, C.c_int, vp, C.c_size_t, szp]
        L.bz2b200_decompress_device.argtypes = [vp, vp, C.c_size_t, C.c_int, vp, C.c_size_t, szp]
        L.bz2b200_compress_bound.argtypes = [C.c_size_t, C.c_int]
        L.bz2b200_compress_bound.restype = C.c_size_t
        L.bz2b200_strerror.argtypes = [C.c_int]
        L.bz2b200_strerror.restype = C.c_char_p
        L.bz2b200_last_error.argtypes = [vp]
        L.bz2b200_last_error.restype = C.c_char_p
        L.bz2b200_last_stats.argtypes = [vp, C.POINTER(Stats)]
        L.bz2b200_debug_fetch.argtypes = [vp, C.c_int, C.c_int, vp, C.c_size_t]
        L.bz2b200_debug_fetch.restype = C.c_longlong
        L.bz2b200_debug_set_block_cap.argtypes = [vp, C.c_uint32]
        L.bz2b200_debug_set_batch_blocks.argtypes = [vp, C.c_uint32]
        L.bz2b200_debug_set_ignore_block_crc.argtypes = [vp, C.c_int]
        L.bz2b200_debug_set_search_tile.argtypes = [vp, C.c_uint32]
        L.bz2b200_debug_huffman_lengths.argtypes = [vp, vp, C.c_int, C.c_int]
        L.bz2b200_shard_begin.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_int]
        L.bz2b200_shard_cut.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(ShardInfo)]
        L.bz2b200_shard_compress.argtypes = [vp, C.POINTER(ShardInfo)]
        L.bz2b200_shard_gtotal.argtypes = [vp, C.c_uint64, C.POINTER(C.c_uint64)]
        L.bz2b200_shard_cut_g.argtypes = [vp, C.c_uint64, C.c_uint64]
        L.bz2b200_shard_cut_pick.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(ShardInfo), C.POINTER(C.c_int)]
        L.bz2b200_shard_emit.argtypes = [vp, C.c_int, C.POINTER(ShardInfo), u8pp, szp]
        L.bz2b200_stitch_shards.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_char_p), C.POINTER(ShardInfo), u8pp, szp]
        L.bz2b200_pool_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(vp)]
        L.bz2b200_pool_destroy.argtypes = [vp]
        L.bz2b200_pool_destroy.restype = None
        L.bz2b200_pool_compress.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_size_t, u8pp, szp]
        L.bz2b200_pool_set_plan.argtypes = [vp, C.c_size_t, C.c_double]
        L.bz2b200_pool_plan.argtypes = [C.c_size_t, C.c_int, C.c_int, C.c_size_t, C.c_double, C.POINTER(C.c_size_t), C.c_int]
        L.bz2b200_pool_last_stats.argtypes = [vp, C.POINTER(Stats)]
        L.bz2b200_pool_last_error.argtypes = [vp]
        L.bz2b200_pool_last_error.restype = C.c_char_p
        L.bz2b200_group_open.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
        L.bz2b200_bind_thread_to_device.argtypes = [C.c_int]
        L.bz2b200_bind_thread_to_device.restype = C.c_int
        L.bz2b200_group_close.argtypes = [vp]
        L.bz2b200_group_close.restype = None
        L.bz2b200_pool_compress_shards.argtypes = [vp, vp, C.POINTER(ShardJob), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(ShardResult)]
        L.bz2b200_pool_decompress.argtypes = [vp, vp, C.c_size_t, C.c_int, C.c_size_t, C.c_size_t, u8pp, szp]
        L.bz2b200_pool_decompress_shards.argtypes = [vp, vp, C.POINTER(ShardJob), C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int,
                                                     C.POINTER(RangeResult)]
        L.bz2b200_debug_set_decode_batch.argtypes = [vp, vp, C.c_uint32]
        L.bz2b200_debug_set_rle1_threads.argtypes = [vp, vp, C.c_uint32]
        L.bz2b200_pool_search.argtypes = [vp, vp, C.c_size_t, C.c_int, vp, vp, C.c_size_t, C.c_uint, C.c_uint64, C.c_size_t, C.POINTER(C.POINTER(Match)),
                                          szp, C.POINTER(SearchTotals), u8pp, szp]
        L.bz2b200_debug_set_pool_search_tile.argtypes = [vp, C.c_uint32]
        for name in ("zstream", "dstream"):
            getattr(L, f"bz2b200_{name}_open").argtypes = [vp, C.c_int, C.c_size_t, C.POINTER(vp)]
            getattr(L, f"bz2b200_{name}_feed").argtypes = [vp, vp, C.c_size_t, u8pp, szp]
            getattr(L, f"bz2b200_{name}_finish").argtypes = [vp, u8pp, szp]
            getattr(L, f"bz2b200_{name}_close").argtypes = [vp]
            getattr(L, f"bz2b200_{name}_close").restype = None
        L.bz2b200_pool_debug.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_size_t, C.c_int]
        L.bz2b200_debug_set_pool.argtypes = [vp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int]
        self.L = L
        self.path = path


_default = None


def default_library():
    global _default
    if _default is None:
        _default = Library()
    return _default
