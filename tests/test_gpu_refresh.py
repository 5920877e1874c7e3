"""Refreshing a computed catalogue (``-m gpu``): removed, updated and appended shows in one call,
``HybridTopKEngine.top_k_refresh_device`` and ``SimilarityComputer.refresh_top_k``.

Every refresh is compared with the whole job on the features after the refresh in a second, fresh
engine: indices, counts and the four fp64 score arrays must be identical bit for bit.
``changed_rows`` must equal a host comparison of every remaining row with its previous row, whose
indices are renumbered (a removed show becomes -1), plus every appended row; every row it does not
list must be byte-identical to that renumbered row."""

import itertools

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
MS = 0.1
KEYS = ("genre_features", "text_features", "platform_features", "type_features", "language_features")
FIELDS = ("indices", "counts", "hybrid", "genre", "text", "metadata")


@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


@pytest.fixture(scope="module")
def fresh():
    """computes the whole jobs the refreshes are compared with"""
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


def _catalogue(n, vocab=5000, genres=40, seed=0, nnz=30):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    return make_catalogue(n, vocab, nnz=nnz, n_genres=genres, seed=seed).features()


def _rows(feats, sel):
    out = dict(feats)
    for key in KEYS:
        a = feats[key]
        out[key] = a[sel] if not sp.issparse(a) else a[sel].tocsr()
    return out


def _stack(*parts):
    out = dict(parts[0])
    for key in KEYS:
        a = [p[key] for p in parts]
        out[key] = sp.vstack(a).tocsr() if sp.issparse(a[0]) else np.concatenate(a)
    return out


def _after(before, removed, updated, new, appended):
    """features after the refresh: the remaining shows in their old order, the updated ones with the
    rows of `new`, then `appended`"""
    n = before["genre_features"].shape[0]
    src = np.arange(n)
    src[updated] = n + np.arange(len(updated))
    sel = np.r_[np.delete(src, removed), n + len(updated) + np.arange(appended["genre_features"].shape[0])]
    return _rows(_stack(before, new, appended), sel)


def _pick(n, q, where, seed, avoid=()):
    """q rows of n outside `avoid`: random, including row 0, a 256-row block, or the last rows"""
    rng = np.random.default_rng(seed)
    free = np.setdiff1d(np.arange(n), avoid)
    if where == "random":
        return np.sort(rng.choice(free, size=q, replace=False))
    if where == "row0":
        return np.sort(np.r_[free[0], rng.choice(free[1:], size=q - 1, replace=False)])
    if where == "block":
        b = min(len(free) // 3, len(free) - q)
        return free[b:b + q]
    return free[len(free) - q:]          # "tail": the last rows, in the last partial tile


def _assert_same(got, want):
    assert np.array_equal(got.counts, want.counts)
    assert np.array_equal(got.indices, want.indices)
    for name in ("hybrid", "genre", "text", "metadata"):
        g, w = getattr(got, name), getattr(want, name)
        assert np.array_equal(np.isnan(g), np.isnan(w)), name
        m = ~np.isnan(w)
        assert np.array_equal(g[m].view(np.uint64), w[m].view(np.uint64)), name


def _check_changed(prev, top, changed, removed, n_app):
    n_old = prev.counts.shape[0]
    keep = np.delete(np.arange(n_old), removed)
    row_map = np.full(n_old, -1, dtype=np.int64)
    row_map[keep] = np.arange(keep.size)
    old = {name: getattr(prev, name)[keep] for name in FIELDS}
    idx = old["indices"]
    old["indices"] = np.where(idx >= 0, row_map[np.maximum(idx, 0)], idx).astype(idx.dtype)
    m = keep.size
    diff = (top.counts[:m] != old["counts"]) | (top.indices[:m] != old["indices"]).any(axis=1)
    for name in ("hybrid", "genre", "text", "metadata"):
        diff |= (getattr(top, name)[:m].view(np.int64) != old[name].view(np.int64)).any(axis=1)
    assert changed.dtype == np.int32
    assert np.array_equal(changed, np.r_[np.nonzero(diff)[0], m + np.arange(n_app)])
    same = np.ones(m, dtype=bool)
    same[diff] = False
    for name in FIELDS:
        assert getattr(top, name)[:m][same].tobytes() == old[name][same].tobytes(), name


def _chain(engine, cat, removed, updated, new, appended):
    """the resident catalogue after the refresh: update, then remove, then extend"""
    if len(updated):
        cat = engine.update(cat, updated, new)
    if len(removed):
        cat = engine.remove(cat, removed)
    if appended["genre_features"].shape[0]:
        cat = engine.extend(cat, appended)
    return cat


def _job(n, nr, nu, na, where="random", seed=0, vocab=5000, genres=40, complete=False):
    """(before, removed, updated, new features of the updated shows, appended features)"""
    before = _catalogue(n, vocab=vocab, genres=genres, seed=seed)
    removed = _pick(n, nr, where, seed + 1) if nr else np.zeros(0, dtype=np.int64)
    updated = _pick(n, nu, where, seed + 2, avoid=removed) if nu else np.zeros(0, dtype=np.int64)
    other = _catalogue(max(nu, 1) + na, vocab=vocab, genres=genres, seed=seed + 3)
    if complete or not nu:
        new = _rows(other, np.arange(nu))
    else:                                  # mostly small edits: the genre and text rows of a neighbour
        new = _rows(before, np.minimum(updated + 1, n - 1))
        new["platform_features"] = before["platform_features"][updated]
    appended = _rows(other, max(nu, 1) + np.arange(na))
    return before, removed, updated, new, appended


def _run(engine, fresh, job, weights=W, k=20, ms=MS, mode="mean3", incremental=True, prev_d=None, cat=None):
    """previous table -> refresh -> incremental table, compared with the whole job on the features
    after the refresh; returns (table dict, host table, changed rows, catalogue, features after)"""
    before, removed, updated, new, appended = job
    if cat is None:
        cat = engine.ingest(before, mode, weights)
        prev_d = engine.top_k_device(cat, weights, k, ms)
    prev = engine.to_host(prev_d)
    cat = _chain(engine, cat, removed, updated, new, appended)
    na = appended["genre_features"].shape[0]
    t = engine.top_k_refresh_device(cat, prev_d, removed[::-1].copy(), updated[::-1].copy(), na, weights, k, ms)
    assert t["incremental"] == incremental
    changed = t["changed_rows"].cpu().numpy()
    top = engine.to_host(t)
    after = _after(before, removed, updated, new, appended)
    _assert_same(top, fresh.compute_top_k(after, weights, k, ms, mode))
    _check_changed(prev, top, changed, removed, na)
    return t, top, changed, cat, after


# ---------------------------------------------------------------------------------------------- kinds
@pytest.mark.parametrize("kinds", [c for r in (1, 2, 3) for c in itertools.combinations("RUA", r)],
                         ids=lambda c: "".join(c))
def test_each_kind_alone_and_every_pair_and_triple(engine, fresh, kinds):
    q = 77
    job = _job(3001, q * ("R" in kinds), q * ("U" in kinds), q * ("A" in kinds), seed=len(kinds) * 10 + ord(kinds[0]))
    t, top, changed, _, _ = _run(engine, fresh, job)
    if len(kinds) > 1:
        return
    # one kind: the same table and rows as the call for that kind alone
    before, removed, updated, new, appended = job
    cat = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    cat = _chain(engine, cat, removed, updated, new, appended)
    if kinds == ("R",):
        one = engine.top_k_remove_device(cat, removed, prev_d, W, 20, MS)
        assert np.array_equal(one["changed_rows"].cpu().numpy(), changed)
    elif kinds == ("U",):
        one = engine.top_k_update_device(cat, updated, prev_d, W, 20, MS)
        assert np.array_equal(one["changed_rows"].cpu().numpy(), changed)
    else:
        one = engine.top_k_append_device(cat, 3001, prev_d, W, 20, MS)
        assert np.array_equal(np.r_[one["changed_rows"].cpu().numpy(), 3001 + np.arange(q)], changed)
    assert one["incremental"]
    _assert_same(engine.to_host(one), top)


# ---------------------------------------------------------------------------------------------- sizes
@pytest.mark.parametrize("n,q,where", [
    (1000, 1, "random"), (1000, 1, "row0"), (1000, 300, "random"), (1000, 256, "block"), (1000, 77, "tail"),
    (3001, 1, "tail"), (3001, 77, "row0"), (3001, 256, "block"), (3001, 900, "random"),
    (41000, 1, "random"), (41000, 77, "tail"), (41000, 2000, "random"),
])
def test_refresh_equals_the_whole_job(engine, fresh, n, q, where):
    _run(engine, fresh, _job(n, q, q, q, where, seed=n + q))


def test_an_updated_show_named_by_rows_that_named_a_removed_show(engine, fresh):
    before = _catalogue(3001, seed=5)
    cat = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    prev = engine.to_host(prev_d)
    x = 1500
    rows = [r for r in range(3001) if x in prev.indices[r, :prev.counts[r]]]
    assert rows
    y = int(next(j for j in prev.indices[rows[0], :prev.counts[rows[0]]] if j != x and j != rows[0]))
    other = _catalogue(6, seed=6)
    job = (before, np.array([x]), np.array([y]), _rows(other, [0]), _rows(other, np.arange(1, 6)))
    _, _, changed, _, _ = _run(engine, fresh, job, prev_d=prev_d, cat=cat)
    renumbered = np.array(rows) - (np.array(rows) > x)
    assert np.isin(renumbered, changed).all()      # a row that named the removed show always changes


# ---------------------------------------------------------------------------------------------- hubs and ties
def test_hubs(engine, fresh):
    before = _catalogue(3001, seed=8)
    cat = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    prev = engine.to_host(prev_d)
    named = np.bincount(np.concatenate([prev.indices[r, :prev.counts[r]] for r in range(3001)]), minlength=3001)
    hubs = np.argsort(named)[::-1][:4]
    other = _catalogue(10, seed=9)
    job = (before, np.sort(hubs[:2]), np.sort(hubs[2:]), _rows(other, [0, 1]), _rows(other, np.arange(2, 10)))
    _run(engine, fresh, job, prev_d=prev_d, cat=cat)


def test_duplicated_shows(engine, fresh):
    before = _catalogue(3001, seed=11)
    dup = _rows(before, np.array([0, 0, 0, 1] + list(range(4, 3001))))      # rows 1, 2 duplicate show 0
    appended = _rows(dup, [0, 0])                                            # and two more, appended
    job = (dup, np.array([1]), np.array([5]), _rows(dup, [0]), appended)
    _, top, _, _, _ = _run(engine, fresh, job)
    assert top.indices[0][0] == 1


def test_a_300_wide_plateau_reaches_the_exact_kernel(engine, fresh):
    before = _catalogue(3001, seed=12)
    plateau = _pick(3001, 300, "random", seed=13)
    sel = np.arange(3001)
    sel[plateau] = plateau[0]                     # 300 identical shows
    feats = _rows(before, sel)
    other = _catalogue(50, seed=14)
    job = (feats, plateau[1::7].copy(), plateau[3::7].copy(), _rows(other, np.arange(plateau[3::7].size)),
           _rows(feats, [plateau[0]] * 3))
    _, top, changed, _, _ = _run(engine, fresh, job)
    assert changed.size > 0
    assert top.flagged_rows > 0, "the 300-wide plateau should send rows to the exact kernel"


# ---------------------------------------------------------------------------------------------- repair stage
def test_rows_that_fail_the_rank_cut_go_to_the_second_sweep(engine, fresh):
    """every updated show replaced completely: many rows lose a neighbour below their previous k-th
    entry; the second sweep repairs them, the exact kernel gets almost none"""
    job = _job(41000, 0, 500, 0, seed=15, complete=True)
    t, top, changed, cat, _ = _run(engine, fresh, job)
    stats = t["stats"].cpu().numpy()
    assert stats[5] > 1000, stats
    assert top.flagged_rows * 10 < stats[5], stats
    g_rows = 500
    tiles = engine.refresh_tiles(cat, g_rows, int(stats[5]), W, 20, MS)
    assert tiles["sweep_tiles"] == 2 * ((41000 + 255) // 256)
    assert tiles["repair_sweep_tiles"] == (int(stats[5]) + 255) // 256 * ((41000 + 255) // 256)
    assert 0 < tiles["repair_seed_tiles"] <= tiles["repair_sweep_tiles"]
    # the same update on the update path sends those rows to the exact kernel
    before, removed, updated, new, appended = job
    c2 = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(c2, W, 20, MS)
    one = engine.top_k_update_device(engine.update(c2, updated, new), updated, prev_d, W, 20, MS)
    assert engine.to_host(one).flagged_rows >= stats[5] // 2
    _assert_same(engine.to_host(one), top)


# ---------------------------------------------------------------------------------------------- shapes
@pytest.mark.parametrize("n,q,vocab,genres,k,weights,mode,ms", [
    (3001, 100, 500, 40, 20, W, "mean3", MS),                 # folded second operand
    (3001, 100, 500, 100, 20, W, "hstack", MS),               # two-word genre masks, folded operand
    (3001, 100, 5000, 100, 20, (0.6, 0.3, 0.1), "mean3", MS),  # two-word genre masks
    (1000, 77, 5000, 40, 100, W, "mean3", MS),
    (3001, 77, 5000, 40, 20, W, "hstack", 0.45),              # high min_similarity: short rows
])
def test_refresh_equals_the_whole_job_across_shapes(engine, fresh, n, q, vocab, genres, k, weights, mode, ms):
    job = _job(n, q, q, q, seed=7 * n + q + k, vocab=vocab, genres=genres, complete=True)
    _, top, _, _, _ = _run(engine, fresh, job, weights, k, ms, mode)
    if ms > 0.4:
        assert (top.counts < k).any(), "expected short rows"


# ---------------------------------------------------------------------------------------------- chains
def _assert_catalogue_equal(a, b):
    ca, cb = a.c, b.c
    assert a.n_shows == b.n_shows and ca.k_pad == cb.k_pad
    assert bool(ca.text_signed) == bool(cb.text_signed)
    n = a.n_shows
    assert torch.equal(a.operand[:n].view(torch.int16), b.operand[:n].view(torch.int16))
    for name in ("col_side", "meta_scale", "genre_hi"):
        x, y = a.parts[name], b.parts[name]
        assert (x is None) == (y is None), name
        if x is not None:
            assert torch.equal(x[:n], y[:n]), name
    nnz = a.parts["nnz"]
    assert nnz == b.parts["nnz"]
    assert torch.equal(a.text_indptr[:n + 1], b.text_indptr[:n + 1])
    assert torch.equal(a.text_indices[:nnz], b.text_indices[:nnz])
    assert torch.equal(a.parts["values"][:nnz].view(torch.int64), b.parts["values"][:nnz].view(torch.int64))


@pytest.mark.parametrize("vocab,genres", [(5000, 40), (500, 100)])
def test_the_catalogue_chain_equals_a_fresh_ingest(engine, fresh, vocab, genres):
    job = _job(3001, 300, 200, 250, seed=21, vocab=vocab, genres=genres, complete=True)
    _, _, _, cat, after = _run(engine, fresh, job)
    _assert_catalogue_equal(cat, fresh.ingest(after, "mean3", W))


def test_refreshes_in_sequence_mixed_with_the_single_kind_calls(engine, fresh):
    n = 3001
    feats = _catalogue(n, seed=31)
    cat = engine.ingest(feats, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    for step, kind in enumerate(["refresh", "refresh", "extend", "refresh", "update", "remove", "refresh"]):
        if kind == "refresh":
            job = _job(n, 50 + step, 60, 70, "tail" if step == 3 else "random", seed=100 + step, complete=step % 2 == 0)
            job = (feats,) + job[1:]
            t, _, _, cat, feats = _run(engine, fresh, job, prev_d=prev_d, cat=cat)
            n = feats["genre_features"].shape[0]
        else:
            if kind == "extend":
                new = _catalogue(300, seed=40 + step)
                cat = engine.extend(cat, new)
                t = engine.top_k_append_device(cat, n, prev_d, W, 20, MS)
                feats = _stack(feats, new)
                n += 300
            elif kind == "update":
                r = _pick(n, 77, "random", seed=step)
                new = _catalogue(77, seed=40 + step)
                cat = engine.update(cat, r, new)
                t = engine.top_k_update_device(cat, r, prev_d, W, 20, MS)
                feats = _after(feats, np.zeros(0, dtype=np.int64), r, new, _rows(new, slice(0, 0)))
            else:
                r = _pick(n, 256, "random", seed=step)
                cat = engine.remove(cat, r)
                t = engine.top_k_remove_device(cat, r, prev_d, W, 20, MS)
                feats = _rows(feats, np.delete(np.arange(n), r))
                n -= 256
            assert t["incremental"]
            _assert_same(engine.to_host(t), fresh.compute_top_k(feats, W, 20, MS))
        prev_d = t


# ---------------------------------------------------------------------------------------------- fallbacks
def _spy(engine, monkeypatch):
    """records, per top_k_refresh_device call, whether the incremental path ran"""
    calls, real = [], engine.top_k_refresh_device

    def wrapped(*a, **kw):
        t = real(*a, **kw)
        calls.append(bool(t["incremental"]))
        return t

    monkeypatch.setattr(engine, "top_k_refresh_device", wrapped)
    return calls


@pytest.mark.parametrize("case", ["incremental", "signed_text", "fractional_genres", "exclude_self_false", "k_120"])
def test_drop_in_and_its_whole_job_fallbacks_keep_the_contract(engine, fresh, case, monkeypatch):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    before, removed, updated, new, appended = _job(3001, 100, 100, 100, seed=51, complete=True)
    if case == "signed_text":
        for f in (before, new, appended):
            t = f["text_features"].copy()
            t.data = t.data * np.where(np.random.default_rng(1).random(t.nnz) < 0.3, -1.0, 1.0)
            f["text_features"] = t
    if case == "fractional_genres":
        for f in (before, new, appended):
            f["genre_features"] = f["genre_features"].astype(np.float64) * 0.5
    after = _after(before, removed, updated, new, appended)
    kw = {"exclude_self": False} if case == "exclude_self_false" else {}
    kw["k"] = 120 if case == "k_120" else 20
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(before, **kw)
    calls = _spy(engine, monkeypatch)
    top = comp.refresh_top_k(after, prev, removed[::-1].copy(), updated, **kw)      # any order
    assert calls == {"incremental": [True], "exclude_self_false": []}.get(case, [False])
    _assert_same(top, SimilarityComputer(engine=fresh).compute_top_k(after, **kw))
    _check_changed(prev, top, top.changed_rows, removed, 100)
    same = comp.refresh_top_k(after, top, **kw)
    assert same.changed_rows.size == 0 and np.array_equal(same.indices, top.indices)


def test_the_engine_fallback_keeps_the_contract(engine, fresh):
    job = list(_job(3001, 77, 77, 77, seed=55, complete=True))
    for f in job[0], job[3], job[4]:
        t = f["text_features"].copy()
        t.data = t.data * np.where(np.random.default_rng(2).random(t.nnz) < 0.3, -1.0, 1.0)
        f["text_features"] = t
    _run(engine, fresh, tuple(job), incremental=False)


# ---------------------------------------------------------------------------------------------- validation
def test_bad_input_raises(engine):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    before = _catalogue(1000, seed=61)
    cat = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    grown = engine.extend(engine.ingest(before, "mean3", W), _catalogue(3, seed=62))
    for bad in ([3, 3], [-1], [1000], [0.5]):
        with pytest.raises(ValueError):
            engine.top_k_refresh_device(cat, prev_d, updated=bad)
        with pytest.raises(ValueError):
            engine.top_k_refresh_device(grown, prev_d, removed=bad, n_appended=3)
    with pytest.raises(ValueError):
        engine.top_k_refresh_device(cat, prev_d, removed=[4], updated=[4, 5], n_appended=1)   # overlap
    with pytest.raises(ValueError):
        engine.top_k_refresh_device(grown, prev_d, n_appended=3, k=10)                       # previous has k = 20
    with pytest.raises(ValueError):
        engine.top_k_refresh_device(grown, {**prev_d, "counts": prev_d["counts"][:-1]}, n_appended=3)
    with pytest.raises(ValueError):
        engine.top_k_refresh_device(grown, prev_d, n_appended=2)                             # 1000 + 2 != 1003
    with pytest.raises(ValueError):
        engine.top_k_refresh_device(grown, prev_d, removed=[0], n_appended=3)
    with pytest.raises(ValueError):
        engine.top_k_refresh_device(engine.ingest(_catalogue(3, seed=63), "mean3", W), prev_d,
                                    removed=np.arange(1000), n_appended=3)                   # every old show
    same = engine.top_k_refresh_device(cat, prev_d)
    assert same["changed_rows"].numel() == 0 and same["indices"] is prev_d["indices"]
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(before, k=20)
    with pytest.raises(ValueError):
        comp.refresh_top_k(before, prev, updated=[1], k=10)
    with pytest.raises(ValueError):
        comp.refresh_top_k(before, prev, removed=[1], updated=[1])
    with pytest.raises(ValueError):
        comp.refresh_top_k(_rows(before, np.arange(10)), prev, removed=[1])                  # fewer than remain
    with pytest.raises(ValueError):
        comp.refresh_top_k(_catalogue(3, seed=64), prev, removed=np.arange(1000))
