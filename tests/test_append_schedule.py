"""Tile schedule of the append sweep (``tvbf_append_topk``), checked on the host copy of the kernel's
item -> tiles map (no GPU needed).

Appending Q shows to N needs the pairs with at least one new show.  The sweep computes the 256 x 256
tiles (row block a, column block b) with b >= max(a, N // 256) and offers every score to both shows;
tiles of column block N // 256 also hold old-old pairs when N % 256 != 0, which the kernel masks."""

import ctypes as C

import numpy as np
import pytest

SMS = 148


def _items(n_old, n_shows, sms=SMS):
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    cap = 1 << 16
    out = (C.c_int32 * (6 * cap))()
    n = lib.tvbf_debug_append_schedule(n_old, n_shows, sms, out, cap)
    assert 0 <= n <= cap
    return np.frombuffer(out, dtype=np.int32, count=6 * n).reshape(n, 6).copy()


def _tiles(n_old, n_shows):
    """tile -> how often it is computed"""
    seen = {}
    for sb, _split, _t0, _t1, r0, r1 in _items(n_old, n_shows):
        if sb < 0:
            continue
        for c in range(r0, r1):
            seen[(int(sb), c)] = seen.get((int(sb), c), 0) + 1
    return seen


@pytest.mark.parametrize("n_old", [1, 200, 255, 256, 257, 511, 3 * 256, 3 * 256 + 1, 41 * 256 - 1])
@pytest.mark.parametrize("q", [1, 255, 256, 257, 3000])
def test_every_pair_with_a_new_show_is_computed_exactly_once(n_old, q):
    n = n_old + q
    col_tiles = (n + 255) // 256
    b0 = n_old // 256
    seen = _tiles(n_old, n)
    assert all(v == 1 for v in seen.values()), "a tile is computed twice"
    # a pair (i, j), i <= j, lies in tile (i // 256, j // 256); it has a new show iff j >= n_old, so its
    # column block is >= b0: exactly the tiles on/above the diagonal with column block >= b0
    want = {(a, b) for b in range(b0, col_tiles) for a in range(0, b + 1)}
    assert set(seen) == want
    # only column block b0 holds old columns beside new ones; there the kernel drops old-old pairs
    for a, b in seen:
        if b * 256 < n_old:
            assert b == b0 and n_old % 256 != 0
    # tile count formula: b0 old row blocks x the band, plus the triangle of the new blocks
    span = col_tiles - b0
    assert len(seen) == b0 * span + span * (span + 1) // 2


def test_c3_append_of_1000_shows_computes_2_5_percent_of_the_tiles():
    seen = _tiles(100_000, 101_000)
    assert len(seen) == 390 * 5 + 15 == 1965
    full = 395 * 396 // 2
    assert len(seen) / full < 0.026


@pytest.mark.parametrize("n_old,q", [(100_000, 256), (100_000, 1000), (100_000, 5000), (80_000, 1000)])
def test_narrow_band_spreads_over_every_sm(n_old, q):
    """Round-robin items to the 74 CTA pairs: the busiest pair walks at most ~1.3x the mean tiles."""
    items = _items(n_old, n_old + q)
    clusters = SMS // 2
    load = np.zeros(clusters)
    for i, (sb, _s, _t0, _t1, r0, r1) in enumerate(items):
        if sb >= 0:
            load[i % clusters] += max(r1 - r0, 0)
    assert load.min() > 0
    assert load.max() <= 1.3 * load.mean() + 2


def test_bad_arguments_are_rejected():
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    out = (C.c_int32 * 6)()
    assert lib.tvbf_debug_append_schedule(0, 10, SMS, out, 1) < 0
    assert lib.tvbf_debug_append_schedule(10, 10, SMS, out, 1) < 0
