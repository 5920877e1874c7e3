"""Offer rule of the refresh sweep (``tvbf_refresh_topk``), checked on the host copy of the update
sweep's item -> tiles map (no GPU needed), and the argument checks of the C entry point that need no
device.

A refresh gathers the operand rows of G = S + A, where S holds the updated and appended shows (their
pair scores changed or are new) and A the other shows whose previous row names a removed show, and
sweeps every (gathered row block, column tile) of that rectangle.  Gathered row r (show u) offers
column j to u's list unless j == u; when u is in S it also offers u to j's list unless j is in G (j's
own gathered row offers it that pair).  A row of A feeds its own list only: its scores are unchanged."""

import ctypes as C

import numpy as np
import pytest

SMS = 148


def _tiles(q, n, sms=SMS):
    """(gathered row block, column tile) -> how often it is computed"""
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    cap = 1 << 16
    out = (C.c_int32 * (6 * cap))()
    k = lib.tvbf_debug_update_schedule(q, n, sms, out, cap)
    assert 0 <= k <= cap
    seen = {}
    for sb, _split, _t0, _t1, r0, r1 in np.frombuffer(out, dtype=np.int32, count=6 * k).reshape(k, 6):
        if sb < 0:
            continue
        for c in range(r0, r1):
            seen[(int(sb), c)] = seen.get((int(sb), c), 0) + 1
    return seen


def _offers(n, in_s, in_g):
    """got[x, y]: times the refresh sweep offers y to x's list"""
    g_rows = np.nonzero(in_g)[0]           # the gathered rows, ascending (the compaction's order)
    q = g_rows.size
    got = np.zeros((n, n), dtype=np.int64)
    seen = _tiles(q, n)
    assert all(v == 1 for v in seen.values()), "a tile is computed twice"
    assert set(seen) == {(a, b) for a in range((q + 255) // 256) for b in range((n + 255) // 256)}
    for sb, tile in seen:
        r = np.arange(sb * 256, min(sb * 256 + 256, q))
        j = np.arange(tile * 256, min(tile * 256 + 256, n))
        u = g_rows[r]
        uu, jj = np.meshgrid(u, j, indexing="ij")
        row_side = uu != jj
        np.add.at(got, (uu[row_side], jj[row_side]), 1)
        col_side = in_s[uu] & ~in_g[jj]
        np.add.at(got, (jj[col_side], uu[col_side]), 1)
    return got


# (n shows after the refresh, |S|, |A|): partial last row blocks and column tiles, S or A empty, G of
# more than one row block, G = every show
@pytest.mark.parametrize("n,n_s,n_a,seed", [
    (700, 1, 0, 0), (700, 0, 1, 1), (700, 40, 90, 2), (513, 300, 213, 3), (1000, 257, 3, 4),
    (1000, 3, 300, 5), (257, 1, 255, 6), (1537, 300, 600, 7),
])
def test_every_pair_reaches_its_list_once_and_no_other_is_offered(n, n_s, n_a, seed):
    rng = np.random.default_rng(seed)
    pick = rng.permutation(n)
    in_s = np.zeros(n, dtype=bool)
    in_s[pick[:n_s]] = True
    in_g = in_s.copy()
    in_g[pick[n_s:n_s + n_a]] = True
    got = _offers(n, in_s, in_g)
    # x in G: every column once (x's own gathered row); x outside G: every show of S once (offered by
    # that show's gathered row); no other pair, and never the show itself
    want = np.where(in_g[:, None], True, in_s[None, :]).astype(np.int64)
    np.fill_diagonal(want, 0)
    assert np.array_equal(got, want)


def test_appended_shows_at_the_end_of_a_partial_tile():
    """the appended shows are the last rows, up to the partial last column tile, and are in S"""
    n, n_app = 3001 - 2000, 45
    in_s = np.zeros(n, dtype=bool)
    in_s[n - n_app:] = True
    in_s[[0, 256, 511]] = True              # updated shows at row 0 and on block edges
    in_g = in_s.copy()
    in_g[[1, 255, 700]] = True              # rows that named a removed show
    got = _offers(n, in_s, in_g)
    want = np.where(in_g[:, None], True, in_s[None, :]).astype(np.int64)
    np.fill_diagonal(want, 0)
    assert np.array_equal(got, want)


# ---------------------------------------------------------------------------------------------- arguments
def _fake_call(**over):
    """tvbf_refresh_topk on a catalogue of 1000 shows at fake (never dereferenced) addresses; returns
    (status, error message).  Every check that runs here runs before the call touches a device."""
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    addr = iter(range(1 << 20, 1 << 30, 1 << 16))
    f = _lib.Features(n_shows=1000, n_pad=1024, k_pad=64, text_dtype=_lib.TEXT_FP16, vocab=50,
                      operand=next(addr), text_indptr=next(addr), text_indices=next(addr), text_values=next(addr),
                      genre_mode=_lib.GROUP_PACKED, genre_dim=20, meta_mode=_lib.GROUP_PACKED, meta_kind=_lib.META_MEAN3,
                      meta_groups=3, col_side=next(addr), meta_scale=next(addr))
    f.text_signed = over.pop("text_signed", 0)
    p = _lib.Params(genre_weight=0.4, text_weight=0.5, metadata_weight=0.1, min_similarity=0.1, k=20,
                    exclude_self=1, row_begin=0, row_end=1000)
    prev = _lib.TopKOut(*(next(addr) for _ in range(7)))
    out = _lib.TopKOut(*(next(addr) for _ in range(7)))
    if over.pop("alias", False):
        out.hybrid = prev.text
    args = {"removed": next(addr), "n_removed": 5, "updated": next(addr), "n_updated": 5, "n_appended": 5,
            "changed": next(addr), "workspace": next(addr)}
    args.update(over)
    rc = lib.tvbf_refresh_topk(C.byref(f), C.byref(p), args["removed"], args["n_removed"], args["updated"],
                               args["n_updated"], args["n_appended"], C.byref(prev), C.byref(out), args["changed"],
                               args["workspace"], 1 << 30, None)
    return rc, lib.tvbf_last_error().decode()


@pytest.mark.parametrize("over,needle", [
    ({"n_removed": -1}, "negative count"),
    ({"n_appended": -1}, "negative count"),
    ({"n_appended": 1000}, "must remain"),
    ({"n_updated": 996}, "appended shows in a catalogue"),
    ({"removed": None}, "NULL row list"),
    ({"updated": None}, "NULL row list"),
    ({"changed": None}, "NULL argument"),
    ({"alias": True}, "aliases the previous one"),
    ({"text_signed": 1}, "signed text"),
])
def test_bad_arguments_are_rejected_before_any_device_work(over, needle):
    rc, msg = _fake_call(**over)
    assert rc != 0
    assert needle in msg


def test_empty_row_lists_may_be_null_and_bad_counts_need_no_workspace():
    from tvbingefriend_recommendation_service_b200 import _lib

    rc, msg = _fake_call(removed=None, n_removed=0, updated=None, n_updated=0, n_appended=0, changed=None)
    assert rc != 0 and "NULL argument" in msg      # the row lists passed, the changed flags did not
    lib = _lib.load()
    f = _lib.Features(n_shows=10, n_pad=256, k_pad=64, text_dtype=_lib.TEXT_FP16, operand=1 << 20,
                      text_indptr=1 << 21, text_indices=1 << 22, text_values=1 << 23, col_side=1 << 24,
                      meta_scale=1 << 25)
    p = _lib.Params(genre_weight=0.4, text_weight=0.5, metadata_weight=0.1, min_similarity=0.1, k=20,
                    exclude_self=1, row_begin=0, row_end=10)
    for counts in ((-1, 0, 0), (0, 0, 10), (0, 11, 0), (0, 6, 5)):
        assert lib.tvbf_refresh_workspace_bytes(C.byref(f), C.byref(p), *counts) == 0
