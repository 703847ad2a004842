"""Kernel launches of the fixed-string search (stats().kernel_launches, the decode's launches included).

The search on one context runs the pool search's per-slice steps as a pool of one slice.  Its launch sequence is pinned
to the one it had with a driver of its own: the same kernels in the same order, with no seeded re-scan of a single
slice.  The pool search launches no more than it did then.  The counts are the same with either parse kernel and with
256-byte and default search tiles."""
import bz2

import pytest

from compressjs_flattened_b200.corpus import gen_text
from test_pool_search import blocky, text_without_runs
from test_pool_search import pe  # noqa: F401  (a fixture)
from test_search import eng  # noqa: F401  (a fixture)

TILES = (256, 0)

# (patterns, lines, max_matches): launches of a search of gen_text(40_000, 41) compressed at level 1
ONE = [((b"zzzzqq",), True, None, 23),   # no match: count and scan only
       ((b"the",), False, None, 24),     # 445 matches: emit, no lines
       ((b"the",), True, None, 28),      # lines: the scan of the piece lengths and the gather
       ((b"e", b"th"), True, None, 28),  # several patterns
       ((b"the",), True, 5, 28)]         # cut at max_matches


@pytest.mark.parametrize("patterns,lines,max_matches,launches", ONE)
def test_one_context_launches(eng, patterns, lines, max_matches, launches):  # noqa: F811
    data = gen_text(40_000, 41).tobytes()
    comp = bz2.compress(data, 1)
    for tile in TILES:
        eng.debug_set_search_tile(tile)
        try:
            r = eng.search(comp, list(patterns), False, max_matches, False, lines=lines)
        finally:
            eng.debug_set_search_tile(0)
        assert r.total_matches == sum(data.startswith(p, i) for i in range(len(data)) for p in patterns), tile
        assert eng.stats().kernel_launches == launches, tile


# (slice_bytes, lines, max_matches): the most launches of test_pool_search.py's matches-across-slices input, over every
# pool of it and both tile sizes
POOL_MAX = {(0, False, None): 25, (0, True, None): 29, (60, False, None): 1467, (60, True, None): 1515, (60, True, 5): 1455,
            (1500, False, None): 100, (1500, True, None): 116}


def test_pool_launches_no_higher(pe, oracle):  # noqa: F811
    pool, eng = pe
    data = bytes(text_without_runs(6000, 61))
    comp, cuts = blocky(oracle, data, 100)
    pats = [data[c - 3:c + 4] for c in cuts[5:40:6]] + [data[cuts[20] - 10:cuts[20] + 246], data[cuts[30] - 1:cuts[30] + 1]]
    total = eng.search(comp, pats).total_matches
    for tile in TILES:
        pool.debug_set_search_tile(tile)
        try:
            for (sb, lines, mm), most in POOL_MAX.items():
                r = pool.search(comp, pats, False, mm, False, lines=lines, slice_bytes=sb)
                assert (r.total_matches, len(r.matches)) == (total, min(total, mm or total)), (tile, sb, lines, mm)
                assert pool.stats().kernel_launches <= most, (tile, sb, lines, mm)
        finally:
            pool.debug_set_search_tile(0)
