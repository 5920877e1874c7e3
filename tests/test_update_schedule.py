"""Tile schedule of the update sweep (``tvbf_update_topk``), checked on the host copy of the kernel's
item -> tiles map (no GPU needed).

Updating Q shows of a catalogue of N gathers their Q operand rows into ceil(Q / 256) row blocks and
sweeps every (gathered row block, column tile) of that rectangle.  A score is offered to the gathered
row's show and to the column's show unless that one is updated too (its own gathered row offers it)."""

import ctypes as C

import numpy as np
import pytest

SMS = 148


def _items(q, n, sms=SMS):
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    cap = 1 << 16
    out = (C.c_int32 * (6 * cap))()
    k = lib.tvbf_debug_update_schedule(q, n, sms, out, cap)
    assert 0 <= k <= cap
    return np.frombuffer(out, dtype=np.int32, count=6 * k).reshape(k, 6).copy()


def _tiles(q, n):
    """(gathered row block, column tile) -> how often it is computed"""
    seen = {}
    for sb, _split, _t0, _t1, r0, r1 in _items(q, n):
        if sb < 0:
            continue
        for c in range(r0, r1):
            seen[(int(sb), c)] = seen.get((int(sb), c), 0) + 1
    return seen


@pytest.mark.parametrize("n", [3000, 3001, 41 * 256 - 1, 41 * 256, 41 * 256 + 1, 100_000])
@pytest.mark.parametrize("q", [1, 255, 256, 257, 3000])
def test_every_gathered_block_and_column_tile_is_computed_exactly_once(q, n):
    seen = _tiles(q, n)
    assert all(v == 1 for v in seen.values()), "a tile is computed twice"
    assert set(seen) == {(a, b) for a in range((q + 255) // 256) for b in range((n + 255) // 256)}


def test_c3_update_of_1000_shows_computes_1564_tiles():
    assert len(_tiles(1000, 100_000)) == 4 * 391 == 1564


@pytest.mark.parametrize("q,n", [(1, 100_000), (256, 100_000), (1000, 100_000), (5000, 100_000), (1000, 80_000)])
def test_the_rectangle_spreads_over_every_sm(q, n):
    """Round-robin items to the 74 CTA pairs: the busiest pair walks at most ~1.3x the mean tiles (a
    single row block splits its 391 column tiles 66 ways: a few pairs idle, none walks more than 6)."""
    items = _items(q, n)
    clusters = SMS // 2
    load = np.zeros(clusters)
    for i, (sb, _s, _t0, _t1, r0, r1) in enumerate(items):
        if sb >= 0:
            load[i % clusters] += max(r1 - r0, 0)
    assert load.sum() == (q + 255) // 256 * ((n + 255) // 256)
    assert load.max() <= 1.3 * load.mean() + 2


@pytest.mark.parametrize("n,q,seed", [(700, 1, 0), (700, 300, 1), (513, 513, 2), (1000, 257, 3)])
def test_each_ordered_pair_with_an_updated_show_reaches_its_list_once(n, q, seed):
    """Restates the kernel's offer rule over the scheduled tiles: gathered row r (show u = U[r]) offers
    column j to u's list unless j == u, and u to j's list unless j is updated.  Every ordered pair
    (x, y), x != y, with x or y updated then reaches x's list exactly once; self never does."""
    rng = np.random.default_rng(seed)
    upd = np.sort(rng.choice(n, size=q, replace=False))
    is_upd = np.zeros(n, dtype=bool)
    is_upd[upd] = True
    got = np.zeros((n, n), dtype=np.int64)   # got[x, y]: times y was offered to x's list
    for (sb, tile), _ in _tiles(q, n).items():
        r = np.arange(sb * 256, min(sb * 256 + 256, q))
        j = np.arange(tile * 256, min(tile * 256 + 256, n))
        u = upd[r]
        uu, jj = np.meshgrid(u, j, indexing="ij")
        row_side = uu != jj
        np.add.at(got, (uu[row_side], jj[row_side]), 1)
        col_side = ~is_upd[jj]
        np.add.at(got, (jj[col_side], uu[col_side]), 1)
    want = (is_upd[:, None] | is_upd[None, :]).astype(np.int64)
    np.fill_diagonal(want, 0)
    assert np.array_equal(got, want)


def test_bad_arguments_are_rejected():
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    out = (C.c_int32 * 6)()
    assert lib.tvbf_debug_update_schedule(0, 10, SMS, out, 1) < 0
    assert lib.tvbf_debug_update_schedule(11, 10, SMS, out, 1) < 0
    assert lib.tvbf_debug_update_schedule(1, 10, 1, out, 1) < 0
