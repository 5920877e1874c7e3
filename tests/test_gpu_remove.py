"""Removing shows from a computed catalogue (``-m gpu``): ``HybridTopKEngine.remove`` +
``top_k_remove_device`` and ``SimilarityComputer.remove_top_k``.

Every removal is compared with the whole job on the remaining features in a second, fresh engine:
indices, counts and the four fp64 score arrays must be identical bit for bit.  ``changed_rows`` must
equal a host comparison of every row with its previous row, whose indices are renumbered (a removed
show becomes -1), and every row it does not list must be byte-identical to that renumbered row."""

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
    """computes the whole jobs the removals are compared with"""
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


def _remaining(feats, removed):
    n = feats["genre_features"].shape[0]
    return _rows(feats, np.delete(np.arange(n), removed))


def _pick(n, q, where, seed):
    rng = np.random.default_rng(seed)
    if where == "random":
        return np.sort(rng.choice(n, size=q, replace=False))
    if where == "row0":
        return np.sort(np.r_[0, rng.choice(np.arange(1, n), size=q - 1, replace=False)])
    if where == "block":
        b = min(n // 3, n - q)
        return np.arange(b, b + q)
    return np.arange(n - q, n)          # "tail": the last rows, in the last partial tile


def _assert_same(got, want):
    assert np.array_equal(got.counts, want.counts)
    assert np.array_equal(got.indices, want.indices)
    for name in ("hybrid", "genre", "text", "metadata"):
        g, w = getattr(got, name), getattr(want, name)
        assert np.array_equal(np.isnan(g), np.isnan(w)), name
        m = ~np.isnan(w)
        assert np.array_equal(g[m].view(np.uint64), w[m].view(np.uint64)), name


def _renumbered(prev, removed):
    """the previous rows of the remaining shows, indices renumbered (a removed show: -1)"""
    n = prev.counts.shape[0]
    keep = np.delete(np.arange(n), removed)
    row_map = np.full(n, -1, dtype=np.int64)
    row_map[keep] = np.arange(keep.size)
    out = {name: getattr(prev, name)[keep] for name in FIELDS}
    idx = out["indices"]
    out["indices"] = np.where(idx >= 0, row_map[np.maximum(idx, 0)], idx).astype(idx.dtype)
    return out


def _check_changed(prev, top, changed, removed):
    old = _renumbered(prev, removed)
    diff = (top.counts != old["counts"]) | (top.indices != old["indices"]).any(axis=1)
    for name in ("hybrid", "genre", "text", "metadata"):
        diff |= (getattr(top, name).view(np.int64) != old[name].view(np.int64)).any(axis=1)
    assert changed.dtype == np.int32
    assert np.array_equal(changed, np.nonzero(diff)[0])
    # exactly the rows whose previous row names a removed show
    named = np.zeros(top.counts.shape[0], dtype=bool)
    for r in range(named.size):
        named[r] = (old["indices"][r, :old["counts"][r]] < 0).any()
    assert np.array_equal(changed, np.nonzero(named)[0])
    keep = np.ones(top.counts.shape[0], dtype=bool)
    keep[changed] = False
    for name in FIELDS:
        assert getattr(top, name)[keep].tobytes() == old[name][keep].tobytes(), name


def _run(engine, fresh, before, removed, weights=W, k=20, ms=MS, mode="mean3", incremental=True):
    """previous table of `before` -> remove `removed` -> incremental table, compared with the whole
    job on the remaining features; returns (previous, table, changed rows, catalogue, want)"""
    cat = engine.ingest(before, mode, weights)
    prev_d = engine.top_k_device(cat, weights, k, ms)
    prev = engine.to_host(prev_d)
    rem = engine.remove(cat, removed)
    t = engine.top_k_remove_device(rem, removed, prev_d, weights, k, ms)
    assert t["incremental"] == incremental
    changed = t["changed_rows"].cpu().numpy()
    top = engine.to_host(t)
    want = fresh.compute_top_k(_remaining(before, np.sort(removed)), weights, k, ms, mode)
    _assert_same(top, want)
    _check_changed(prev, top, changed, np.sort(removed))
    return prev, top, changed, rem, want


# ---------------------------------------------------------------------------------------------- bit identity
@pytest.mark.parametrize("where", ["random", "row0", "block", "tail"])
@pytest.mark.parametrize("q", [1, 77, 256, 2000])
@pytest.mark.parametrize("n", [1000, 3001, 41000])
def test_remove_equals_the_whole_job(engine, fresh, n, q, where):
    if q >= n or (where == "row0" and q < 2):
        pytest.skip("no such selection")
    before = _catalogue(n, seed=n + q)
    _run(engine, fresh, before, _pick(n, q, where, seed=q))


@pytest.mark.parametrize("left", [1, 7])
def test_removals_that_leave_one_show_or_fewer_than_k(engine, fresh, left):
    _, top, _, _, _ = _run(engine, fresh, _catalogue(1000, seed=2), _pick(1000, 1000 - left, "random", seed=3))
    assert (top.counts <= left - 1).all()


def test_a_show_named_in_no_row_and_a_hub(engine, fresh):
    before = _catalogue(3001, seed=4)
    cat = engine.ingest(before, "mean3", W)
    prev = engine.to_host(engine.top_k_device(cat, W, 20, MS))
    named = np.bincount(np.concatenate([prev.indices[r, :prev.counts[r]] for r in range(3001)]), minlength=3001)
    lonely = int(np.nonzero(named == 0)[0][0])
    _, _, changed, _, _ = _run(engine, fresh, before, [lonely])
    assert changed.size == 0
    hub = int(np.argmax(named))
    _, _, changed, _, _ = _run(engine, fresh, before, [hub])
    assert changed.size == named[hub]


# ---------------------------------------------------------------------------------------------- ties
def test_removing_a_show_with_duplicates(engine, fresh):
    before = _catalogue(3001, seed=11)
    dup = _rows(before, np.array([0, 0, 0, 1] + list(range(4, 3001))))     # rows 1, 2 duplicate show 0
    _, top, _, _, _ = _run(engine, fresh, dup, [0])
    assert top.indices[0][0] == 1                 # the duplicates tie and keep their order


def test_a_300_wide_plateau_reaches_the_exact_kernel(engine, fresh):
    before = _catalogue(3001, seed=12)
    plateau = _pick(3001, 300, "random", seed=13)
    sel = np.arange(3001)
    sel[plateau] = plateau[0]                     # 300 identical shows
    feats = _rows(before, sel)
    _, top, changed, _, _ = _run(engine, fresh, feats, plateau[::7].copy())
    assert changed.size > 0
    assert top.flagged_rows > 0, "the 300-wide plateau should send rows to the exact kernel"


# ---------------------------------------------------------------------------------------------- shapes
@pytest.mark.parametrize("n,q,vocab,genres,k,weights,mode,ms", [
    (3001, 256, 500, 40, 20, W, "mean3", MS),                 # folded second operand
    (41000, 77, 500, 40, 20, (0.6, 0.3, 0.1), "hstack", MS),
    (3001, 300, 500, 100, 20, W, "hstack", MS),               # two-word genre masks, folded operand
    (1000, 77, 5000, 100, 100, W, "mean3", MS),
    (41000, 256, 5000, 40, 100, (0.6, 0.3, 0.1), "mean3", MS),
    (3001, 77, 5000, 40, 20, W, "mean3", 0.45),               # high min_similarity: short rows
    (3001, 257, 500, 40, 20, W, "hstack", 0.45),
])
def test_remove_equals_the_whole_job_across_shapes(engine, fresh, n, q, vocab, genres, k, weights, mode, ms):
    before = _catalogue(n, vocab=vocab, genres=genres, seed=7 * n + q)
    _, top, _, _, _ = _run(engine, fresh, before, _pick(n, q, "random", seed=q), weights, k, ms, mode)
    if ms > 0.4:
        assert (top.counts < k).any(), "expected short rows"


def test_remove_computes_few_tiles_and_rescores_only_changed_rows(engine, fresh):
    n, q = 41000, 77
    before = _catalogue(n, seed=15)
    _, top, changed, rem, want = _run(engine, fresh, before, _pick(n, q, "random", seed=16))
    a = changed.size
    tiles = engine.remove_tiles(rem, a)
    assert tiles["sweep_tiles"] == (a + 255) // 256 * ((n - q + 255) // 256)
    assert 0 < tiles["seed_tiles"] <= tiles["sweep_tiles"]
    assert engine.remove_tiles(rem, 0) == {"seed_tiles": 0, "sweep_tiles": 0}
    assert top.flagged_rows <= a
    assert 0 < top.rescored_pairs < 0.5 * want.rescored_pairs


# ---------------------------------------------------------------------------------------------- catalogue
def _assert_catalogue_equal(a, b):
    ca, cb = a.c, b.c
    assert a.n_shows == b.n_shows and ca.n_pad == cb.n_pad and ca.k_pad == cb.k_pad
    assert bool(ca.text_signed) == bool(cb.text_signed)
    assert torch.equal(a.operand.view(torch.int16), b.operand.view(torch.int16))   # padding rows zero
    for name in ("col_side", "meta_scale", "genre_hi"):
        x, y = a.parts[name], b.parts[name]
        assert (x is None) == (y is None), name
        if x is not None:
            assert torch.equal(x, y), name
    nnz = a.parts["nnz"]
    assert nnz == b.parts["nnz"]
    assert torch.equal(a.text_indptr[:a.n_shows + 1], b.text_indptr[:b.n_shows + 1])
    assert torch.equal(a.text_indices[:nnz], b.text_indices[:nnz])
    assert torch.equal(a.parts["values"][:nnz].view(torch.int64), b.parts["values"][:nnz].view(torch.int64))


@pytest.mark.parametrize("vocab,genres", [(5000, 40), (500, 100)])
def test_the_compacted_catalogue_equals_a_fresh_ingest(engine, fresh, vocab, genres):
    before = _catalogue(3001, vocab=vocab, genres=genres, seed=21)
    removed = _pick(3001, 600, "random", seed=22)     # 3001 -> 2401 shows: n_pad shrinks
    _, _, _, rem, _ = _run(engine, fresh, before, removed)
    _assert_catalogue_equal(rem, fresh.ingest(_remaining(before, removed), "mean3", W))
    # the compacted catalogue recycles correctly: its CSR describes the operand it hands over
    other = _catalogue(3001, vocab=vocab, genres=genres, seed=24)
    rec = engine.ingest(other, "mean3", W, recycle=rem)
    _assert_catalogue_equal(rec, fresh.ingest(other, "mean3", W))
    _assert_same(engine.to_host(engine.top_k_device(rec, W, 20, MS)), fresh.compute_top_k(other, W, 20, MS))


def test_the_compacted_catalogue_with_float_groups_equals_a_fresh_ingest(engine, fresh):
    before = _catalogue(1000, seed=25)
    before["genre_features"] = before["genre_features"].astype(np.float64) * 0.5
    removed = _pick(1000, 77, "random", seed=26)
    cat = engine.ingest(before, "mean3", W)
    rem = engine.remove(cat, removed)
    want = fresh.ingest(_remaining(before, removed), "mean3", W)
    assert rem.folded and want.folded
    _assert_catalogue_equal(rem, want)
    assert torch.equal(rem.parts["genre_dense"], want.parts["genre_dense"])


def test_sequences_of_removals_appends_and_updates(engine, fresh):
    n = 3001
    feats = _catalogue(n, seed=31)
    cat = engine.ingest(feats, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    for step, kind in enumerate(["remove", "extend", "remove", "update", "remove", "remove"]):
        prev = engine.to_host(prev_d)
        if kind == "remove":
            r = _pick(n, 77 if step % 4 == 0 else 256, "tail" if step == 4 else "random", seed=step)
            cat = engine.remove(cat, r)
            t = engine.top_k_remove_device(cat, r, prev_d, W, 20, MS)
            feats = _remaining(feats, r)
            n -= r.size
        elif kind == "extend":
            new = _catalogue(300, seed=40 + step)
            cat = engine.extend(cat, new)
            t = engine.top_k_append_device(cat, n, prev_d, W, 20, MS)
            feats = {key: (sp.vstack([feats[key], new[key]]).tocsr() if sp.issparse(feats[key])
                           else np.concatenate([feats[key], new[key]])) for key in KEYS}
            n += 300
        else:
            r = _pick(n, 77, "random", seed=step)
            new = _catalogue(77, seed=40 + step)
            cat = engine.update(cat, r, new)
            t = engine.top_k_update_device(cat, r, prev_d, W, 20, MS)
            upd = dict(feats)
            for key in KEYS:
                a, b = feats[key], new[key]
                perm = np.arange(n)
                perm[r] = n + np.arange(r.size)
                upd[key] = sp.vstack([a, b]).tocsr()[perm] if sp.issparse(a) else np.concatenate([a, b])[perm]
            feats = upd
        assert t["incremental"]
        top = engine.to_host(t)
        _assert_same(top, fresh.compute_top_k(feats, W, 20, MS))
        if kind == "remove":
            _check_changed(prev, top, t["changed_rows"].cpu().numpy(), r)
        prev_d = t


# ---------------------------------------------------------------------------------------------- fallbacks
def _spy(engine, monkeypatch):
    """records, per top_k_remove_device call, whether the incremental path ran"""
    calls, real = [], engine.top_k_remove_device

    def wrapped(*a, **kw):
        t = real(*a, **kw)
        calls.append(bool(t["incremental"]))
        return t

    monkeypatch.setattr(engine, "top_k_remove_device", wrapped)
    return calls


@pytest.mark.parametrize("case", ["incremental", "signed_text", "fractional_genres", "exclude_self_false", "k_120"])
def test_drop_in_and_its_whole_job_fallbacks_keep_the_contract(engine, fresh, case, monkeypatch):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    before = _catalogue(3001, seed=51)
    if case == "signed_text":
        t = before["text_features"].copy()
        t.data = t.data * np.where(np.random.default_rng(1).random(t.nnz) < 0.3, -1.0, 1.0)
        before["text_features"] = t
    if case == "fractional_genres":
        before["genre_features"] = before["genre_features"].astype(np.float64) * 0.5
    removed = _pick(3001, 256, "random", seed=52)
    after = _remaining(before, removed)
    kw = {"exclude_self": False} if case == "exclude_self_false" else {}
    kw["k"] = 120 if case == "k_120" else 20
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(before, **kw)
    calls = _spy(engine, monkeypatch)
    top = comp.remove_top_k(after, prev, removed[::-1].copy(), **kw)      # any order
    assert calls == {"incremental": [True], "exclude_self_false": []}.get(case, [False])
    _assert_same(top, SimilarityComputer(engine=fresh).compute_top_k(after, **kw))
    _check_changed(prev, top, top.changed_rows, removed)
    same = comp.remove_top_k(after, top, [], **kw)
    assert same.changed_rows.size == 0 and np.array_equal(same.indices, top.indices)


def test_the_engine_fallback_renumbers_the_previous_rows(engine, fresh):
    before = _catalogue(3001, seed=55)
    t = before["text_features"].copy()
    t.data = t.data * np.where(np.random.default_rng(2).random(t.nnz) < 0.3, -1.0, 1.0)
    before["text_features"] = t
    _run(engine, fresh, before, _pick(3001, 77, "random", seed=56), incremental=False)


# ---------------------------------------------------------------------------------------------- validation
def test_bad_rows_and_shapes_raise(engine):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    before = _catalogue(1000, seed=61)
    cat = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    rem = engine.remove(engine.ingest(before, "mean3", W), [5])
    for bad in ([3, 3], [-1], [1000], [0.5]):
        with pytest.raises(ValueError):
            engine.top_k_remove_device(rem, bad, prev_d, W, 20, MS)
        with pytest.raises(ValueError):
            engine.remove(cat, bad)
    with pytest.raises(ValueError):
        engine.top_k_remove_device(rem, [5], prev_d, W, 10, MS)        # previous has k = 20
    with pytest.raises(ValueError):
        engine.top_k_remove_device(rem, [5, 6], prev_d, W, 20, MS)     # 999 + 2 != 1000 previous rows
    with pytest.raises(ValueError):
        engine.remove(cat, np.arange(1000))
    assert engine.remove(cat, []) is cat
    same = engine.top_k_remove_device(cat, [], prev_d, W, 20, MS)
    assert same["changed_rows"].numel() == 0 and same["indices"] is prev_d["indices"]
    gone = engine.remove(engine.ingest(before, "mean3", W), [1])
    consumed = engine.ingest(before, "mean3", W)
    engine.remove(consumed, [1])
    with pytest.raises(ValueError):
        engine.remove(consumed, [2])                                   # consumed by the first removal
    assert gone.n_shows == 999
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(before, k=20)
    with pytest.raises(ValueError):
        comp.remove_top_k(_remaining(before, [1]), prev, [1], k=10)
    with pytest.raises(ValueError):
        comp.remove_top_k(_remaining(before, [1, 2]), prev, [1], k=20)
    with pytest.raises(ValueError):
        comp.remove_top_k(_rows(before, slice(0, 0)), prev, np.arange(1000), k=20)
