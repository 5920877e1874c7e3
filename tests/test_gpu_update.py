"""Updating the features of shows in a computed catalogue (``-m gpu``): ``HybridTopKEngine.update`` +
``top_k_update_device`` and ``SimilarityComputer.update_top_k``.

Every update is compared with the whole job on the updated features in a second, fresh engine:
indices, counts and the four fp64 score arrays must be identical bit for bit.  ``changed_rows`` must
equal a host comparison of all six fields of every row, and every row it does not list must be
byte-identical to the previous table.  ``flagged_rows`` / ``rescored_pairs`` are not compared."""

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
    """computes the whole jobs the updates are compared with"""
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


def _replace(feats, rows, new):
    """feats with rows[e] (sorted) taken from row e of new"""
    n = feats["genre_features"].shape[0]
    perm = np.arange(n)
    perm[rows] = n + np.arange(len(rows))
    out = dict(feats)
    for key in KEYS:
        a, b = feats[key], new[key]
        out[key] = sp.vstack([a, b]).tocsr()[perm] if sp.issparse(a) else np.concatenate([a, b])[perm]
    return out


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


def _check_changed(prev, top, changed):
    diff = (top.counts != prev.counts) | (top.indices != prev.indices).any(axis=1)
    for name in ("hybrid", "genre", "text", "metadata"):
        diff |= (getattr(top, name).view(np.int64) != getattr(prev, name).view(np.int64)).any(axis=1)
    assert changed.dtype == np.int32
    assert np.array_equal(changed, np.nonzero(diff)[0])
    keep = np.ones(prev.counts.shape[0], dtype=bool)
    keep[changed] = False
    for name in FIELDS:
        assert getattr(top, name)[keep].tobytes() == getattr(prev, name)[keep].tobytes(), name


def _run(engine, fresh, before, rows, new, weights=W, k=20, ms=MS, mode="mean3", incremental=True):
    """previous table of `before` -> update `rows` to `new` -> incremental table, compared with the
    whole job on the updated features; returns (previous, updated table, changed rows, catalogue, want)"""
    cat = engine.ingest(before, mode, weights)
    prev_d = engine.top_k_device(cat, weights, k, ms)
    prev = engine.to_host(prev_d)
    upd = engine.update(cat, rows, new)
    t = engine.top_k_update_device(upd, rows, prev_d, weights, k, ms)
    assert t["incremental"] == incremental
    changed = t["changed_rows"].cpu().numpy()
    top = engine.to_host(t)
    want = fresh.compute_top_k(_replace(before, np.sort(rows), new), weights, k, ms, mode)
    _assert_same(top, want)
    _check_changed(prev, top, changed)
    return prev, top, changed, upd, want


# ---------------------------------------------------------------------------------------------- bit identity
@pytest.mark.parametrize("where", ["random", "row0", "block", "tail"])
@pytest.mark.parametrize("q", [1, 77, 256, 2000])
@pytest.mark.parametrize("n", [1000, 3001, 41000])
def test_update_equals_the_whole_job(engine, fresh, n, q, where):
    if q > n or (where == "row0" and q < 2):
        pytest.skip("no such selection")
    before = _catalogue(n, seed=n + q)
    rows = _pick(n, q, where, seed=q)
    new = _catalogue(q, seed=10_000 + n + q)     # a second seeded catalogue of the same config
    _run(engine, fresh, before, rows, new)


def test_every_show_updated(engine, fresh):
    _run(engine, fresh, _catalogue(1000, seed=1), np.arange(1000), _catalogue(1000, seed=2))


@pytest.mark.parametrize("key", ["text_features", "genre_features", "platform_features"])
def test_single_group_edits(engine, fresh, key):
    before = _catalogue(3001, seed=3)
    rows = _pick(3001, 77, "random", seed=4)
    new = _rows(before, rows)
    new[key] = _rows(_catalogue(3001, seed=5), rows)[key]
    _run(engine, fresh, before, rows, new)


def test_a_revert_restores_the_previous_table(engine, fresh):
    before = _catalogue(3001, seed=6)
    rows = _pick(3001, 256, "random", seed=7)
    prev, top, _, upd, _ = _run(engine, fresh, before, rows, _catalogue(256, seed=8))
    mid = engine.top_k_device(upd, W, 20, MS)
    back = engine.update(upd, rows, _rows(before, rows))
    r = engine.top_k_update_device(back, rows, mid, W, 20, MS)
    assert r["incremental"]
    got = engine.to_host(r)
    _assert_same(got, prev)
    _check_changed(engine.to_host(mid), got, r["changed_rows"].cpu().numpy())
    # rows "updated" to the features they already have: nothing changes
    same = engine.update(back, rows, _rows(before, rows))
    r2 = engine.top_k_update_device(same, rows, r, W, 20, MS)
    assert r2["incremental"] and r2["changed_rows"].numel() == 0
    _assert_same(engine.to_host(r2), prev)


# ---------------------------------------------------------------------------------------------- ties
def test_a_show_turned_into_a_duplicate_and_one_without_text(engine, fresh):
    before = _catalogue(3001, seed=11)
    rows = np.array([5, 17, 2999])
    new = _rows(before, np.array([0, 1, 2]))
    new["text_features"] = new["text_features"].tolil()
    new["text_features"][2] = 0                   # show 2999 loses its text
    new["text_features"] = sp.csr_matrix(new["text_features"])
    new["text_features"].eliminate_zeros()
    _, top, _, _, _ = _run(engine, fresh, before, rows, new)
    assert top.indices[5][0] == 0                 # the duplicate of show 0 ties with it and loses on index


def test_a_300_wide_plateau_reaches_the_exact_kernel(engine, fresh):
    before = _catalogue(3001, seed=12)
    rows = _pick(3001, 300, "random", seed=13)
    new = _rows(_catalogue(10, seed=14), np.zeros(300, dtype=np.int64))
    _, top, _, _, _ = _run(engine, fresh, before, rows, new)
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
def test_update_equals_the_whole_job_across_shapes(engine, fresh, n, q, vocab, genres, k, weights, mode, ms):
    before = _catalogue(n, vocab=vocab, genres=genres, seed=7 * n + q)
    rows = _pick(n, q, "random", seed=q)
    new = _catalogue(q, vocab=vocab, genres=genres, seed=7 * n + q + 1)
    _, top, _, _, _ = _run(engine, fresh, before, rows, new, weights, k, ms, mode)
    if ms > 0.4:
        assert (top.counts < k).any(), "expected short rows"


def test_update_computes_few_tiles_and_rescores_few_pairs(engine, fresh):
    before = _catalogue(41000, seed=15)
    rows = _pick(41000, 77, "random", seed=16)
    _, top, _, upd, want = _run(engine, fresh, before, rows, _catalogue(77, seed=17))
    tiles = engine.update_tiles(upd, 77)
    assert tiles["sweep_tiles"] == 1 * 161
    assert 0 < tiles["seed_tiles"] <= 161
    assert 0 < top.rescored_pairs < 0.5 * want.rescored_pairs
    assert top.flagged_rows >= 0


# ---------------------------------------------------------------------------------------------- catalogue
def _assert_catalogue_equal(a, b):
    ca, cb = a.c, b.c
    assert a.n_shows == b.n_shows and ca.n_pad == cb.n_pad and ca.k_pad == cb.k_pad
    assert bool(ca.text_signed) == bool(cb.text_signed)
    assert torch.equal(a.operand.view(torch.int16), b.operand.view(torch.int16))
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
def test_the_updated_catalogue_equals_a_fresh_ingest(engine, fresh, vocab, genres):
    before = _catalogue(3001, vocab=vocab, genres=genres, seed=21)
    rows = _pick(3001, 300, "random", seed=22)
    new = _catalogue(300, vocab=vocab, genres=genres, seed=23, nnz=60)   # longer rows: the CSR grows
    after = _replace(before, rows, new)
    _, _, _, upd, want = _run(engine, fresh, before, rows, new)
    _assert_catalogue_equal(upd, fresh.ingest(after, "mean3", W))
    # the updated catalogue recycles correctly: its CSR describes the operand it hands over
    other = _catalogue(3001, vocab=vocab, genres=genres, seed=24)
    rec = engine.ingest(other, "mean3", W, recycle=upd)
    _assert_same(engine.to_host(engine.top_k_device(rec, W, 20, MS)), fresh.compute_top_k(other, W, 20, MS))


def test_sequences_of_updates_and_appends(engine, fresh):
    n = 3001
    feats = _catalogue(n, seed=31)
    cat = engine.ingest(feats, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    rows = _pick(n, 77, "random", seed=32)
    for step in range(4):
        prev = engine.to_host(prev_d)
        if step == 1:      # update -> extend
            new = _catalogue(256, seed=40 + step)
            cat = engine.extend(cat, new)
            t = engine.top_k_append_device(cat, n, prev_d, W, 20, MS)
            feats = {key: (sp.vstack([feats[key], new[key]]).tocsr() if sp.issparse(feats[key])
                           else np.concatenate([feats[key], new[key]])) for key in KEYS}
            n += 256
            prev = None
        else:              # updates, the last two of the same rows (extend -> update, update -> update)
            r = rows if step >= 2 else _pick(n, 77, "tail", seed=step)
            new = _catalogue(len(r), seed=40 + step)
            cat = engine.update(cat, r, new)
            t = engine.top_k_update_device(cat, r, prev_d, W, 20, MS)
            feats = _replace(feats, r, new)
        assert t["incremental"]
        top = engine.to_host(t)
        _assert_same(top, fresh.compute_top_k(feats, W, 20, MS))
        if prev is not None:
            _check_changed(prev, top, t["changed_rows"].cpu().numpy())
        prev_d = t


# ---------------------------------------------------------------------------------------------- fallbacks
def _spy(engine, monkeypatch):
    """records, per top_k_update_device call, whether the incremental path ran"""
    calls, real = [], engine.top_k_update_device

    def wrapped(*a, **kw):
        t = real(*a, **kw)
        calls.append(bool(t["incremental"]))
        return t

    monkeypatch.setattr(engine, "top_k_update_device", wrapped)
    return calls


@pytest.mark.parametrize("case", ["incremental", "signed_text", "fractional_genres", "exclude_self_false"])
def test_drop_in_and_its_whole_job_fallbacks_keep_the_contract(engine, fresh, case, monkeypatch):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    before = _catalogue(3001, seed=51)
    if case == "signed_text":
        t = before["text_features"].copy()
        t.data = t.data * np.where(np.random.default_rng(1).random(t.nnz) < 0.3, -1.0, 1.0)
        before["text_features"] = t
    rows = _pick(3001, 256, "random", seed=52)
    after = _replace(before, rows, _catalogue(256, seed=53))
    if case == "fractional_genres":
        g = after["genre_features"].astype(np.float64)
        g[rows] *= 0.5
        after["genre_features"] = g
    kw = {"exclude_self": False} if case == "exclude_self_false" else {}
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(before, **kw)
    calls = _spy(engine, monkeypatch)
    top = comp.update_top_k(after, prev, rows[::-1].copy(), **kw)      # any order
    assert calls == {"incremental": [True], "exclude_self_false": []}.get(case, [False])
    _assert_same(top, SimilarityComputer(engine=fresh).compute_top_k(after, **kw))
    _check_changed(prev, top, top.changed_rows)
    same = comp.update_top_k(after, top, [], **kw)
    assert same.changed_rows.size == 0 and np.array_equal(same.indices, top.indices)


# ---------------------------------------------------------------------------------------------- validation
def test_bad_rows_shapes_and_encodings_raise(engine):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    before = _catalogue(1000, seed=61)
    cat = engine.ingest(before, "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    for bad in ([3, 3], [-1], [1000], [0.5]):
        with pytest.raises(ValueError):
            engine.top_k_update_device(cat, bad, prev_d, W, 20, MS)
        with pytest.raises(ValueError):
            engine.update(cat, bad, _catalogue(len(bad), seed=62))
    with pytest.raises(ValueError):
        engine.top_k_update_device(cat, [1], prev_d, W, 10, MS)
    with pytest.raises(ValueError):
        engine.update(cat, [1, 2], _catalogue(3, seed=63))
    for bad in (_catalogue(2, vocab=4000, seed=64), _catalogue(2, genres=41, seed=65)):
        with pytest.raises(ValueError):
            engine.update(engine.ingest(before, "mean3", W), [7, 8], bad)
    wide = _catalogue(2, seed=66)
    wide["platform_features"] = np.hstack([wide["platform_features"], np.zeros((2, 1))])
    with pytest.raises(ValueError):
        engine.update(engine.ingest(before, "mean3", W), [7, 8], wide)
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(before, k=20)
    with pytest.raises(ValueError):
        comp.update_top_k(before, prev, [1], k=10)
    with pytest.raises(ValueError):
        comp.update_top_k(_rows(before, slice(0, 500)), prev, [1], k=20)
