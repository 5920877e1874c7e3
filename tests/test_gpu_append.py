"""Appending shows to a computed catalogue (``-m gpu``): ``HybridTopKEngine.extend`` +
``top_k_append_device`` and ``SimilarityComputer.extend_top_k``.

Every append is compared with the whole job on the concatenated features in a second, fresh engine:
indices, counts and the four fp64 score arrays must be identical bit for bit.  ``changed_rows`` must
equal a host comparison of the two tables, and every old row it does not list must be byte-identical
to the previous table.  ``flagged_rows`` / ``rescored_pairs`` are not compared."""

import numpy as np
import pytest
import scipy.sparse as sp

from helpers import assert_topk_matches

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
MS = 0.1
SYMMETRIC = 2 << 20
KEYS = ("genre_features", "text_features", "platform_features", "type_features", "language_features")


@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


@pytest.fixture(scope="module")
def fresh():
    """computes the whole jobs the appends are compared with"""
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


def _concat(a, b):
    out = dict(a)
    for key in KEYS:
        out[key] = sp.vstack([a[key], b[key]]).tocsr() if sp.issparse(a[key]) else np.concatenate([a[key], b[key]])
    return out


def _split(feats, n):
    return _rows(feats, slice(0, n)), _rows(feats, slice(n, None))


def _assert_same(got, want):
    assert np.array_equal(got.counts, want.counts)
    assert np.array_equal(got.indices, want.indices)
    for name in ("hybrid", "genre", "text", "metadata"):
        g, w = getattr(got, name), getattr(want, name)
        assert np.array_equal(np.isnan(g), np.isnan(w)), name
        m = ~np.isnan(w)
        assert np.array_equal(g[m].view(np.uint64), w[m].view(np.uint64)), name


def _check_changed(prev, top, changed):
    n_old = prev.counts.shape[0]
    diff = (top.counts[:n_old] != prev.counts) | (top.indices[:n_old] != prev.indices).any(axis=1)
    assert changed.dtype == np.int32
    assert np.array_equal(changed, np.nonzero(diff)[0])
    keep = np.ones(n_old, dtype=bool)
    keep[changed] = False
    for name in ("indices", "counts", "hybrid", "genre", "text", "metadata"):
        a, b = getattr(top, name)[:n_old][keep], getattr(prev, name)[keep]
        assert a.tobytes() == b.tobytes(), name


def _append(engine, old, new, weights=W, k=20, ms=MS, mode="mean3"):
    """previous table of `old` -> extend by `new` -> append; returns (previous, appended, changed)"""
    cat = engine.ingest(old, mode, weights)
    prev_d = engine.top_k_device(cat, weights, k, ms)
    prev = engine.to_host(prev_d)
    grown = engine.extend(cat, new)
    t = engine.top_k_append_device(grown, prev.counts.shape[0], prev_d, weights, k, ms)
    assert t["incremental"], "the append ran the whole job instead of the append sweep"
    changed = t["changed_rows"].cpu().numpy()
    return prev, engine.to_host(t), changed, grown


def _run(engine, fresh, old, new, weights=W, k=20, ms=MS, mode="mean3"):
    """an incremental append compared with the whole job"""
    prev, top, changed, grown = _append(engine, old, new, weights, k, ms, mode)
    want = fresh.compute_top_k(_concat(old, new), weights, k, ms, mode)
    _assert_same(top, want)
    _check_changed(prev, top, changed)
    return prev, top, changed, grown, want


# ---------------------------------------------------------------------------------------------- bit identity
@pytest.mark.parametrize("n_old", [1000, 3001, 41000])
@pytest.mark.parametrize("q", [1, 77, 256, 2000])
def test_append_equals_the_whole_job(engine, fresh, n_old, q):
    feats = _catalogue(n_old + q, seed=n_old + q)
    old, new = _split(feats, n_old)
    _run(engine, fresh, old, new)


@pytest.mark.parametrize("n_old,q,vocab,genres,k,weights,mode", [
    (3001, 256, 500, 40, 20, W, "mean3"),                # folded second operand
    (41000, 77, 500, 40, 20, (0.6, 0.3, 0.1), "hstack"),
    (3001, 2000, 500, 100, 20, W, "hstack"),             # two-word genre masks, folded operand
    (1000, 77, 5000, 100, 100, W, "mean3"),
    (41000, 256, 5000, 40, 100, (0.6, 0.3, 0.1), "mean3"),
    (3001, 1, 5000, 100, 20, (0.6, 0.3, 0.1), "hstack"),
    (41000, 2000, 500, 100, 100, W, "mean3"),
])
def test_append_equals_the_whole_job_across_shapes(engine, fresh, n_old, q, vocab, genres, k, weights, mode):
    feats = _catalogue(n_old + q, vocab=vocab, genres=genres, seed=7 * n_old + q)
    old, new = _split(feats, n_old)
    _run(engine, fresh, old, new, weights, k, MS, mode)


def test_append_computes_few_tiles_and_rescores_only_rows_with_new_candidates(engine, fresh):
    feats = _catalogue(41000 + 300, seed=5)
    old, new = _split(feats, 41000)
    _, top, _, grown, want = _run(engine, fresh, old, new)
    # column tiles 160 and 161 hold new shows: 160 old row blocks x 2 + the 3 tiles of the new blocks;
    # the seed pass samples the 2 new super blocks only
    tiles = engine.append_tiles(grown, 41000)
    assert tiles["sweep_tiles"] == 160 * 2 + 3
    assert 0 < tiles["seed_tiles"] <= 2 * 162
    # old rows without a new candidate keep their previous rows instead of being rescored
    assert 0 < top.rescored_pairs < 0.5 * want.rescored_pairs


# ---------------------------------------------------------------------------------------------- ties
def test_new_shows_that_duplicate_old_ones_lose_the_tie(engine, fresh):
    old = _catalogue(3001, seed=11)
    new = _rows(old, np.array([0, 5, 17, 2999, 3000, 1234]))
    prev, top, changed, _, _ = _run(engine, fresh, old, new)
    # row 3001 duplicates show 0: its best score, 1.0, is shared with show 0, the lowest index
    assert top.indices[3001][0] == 0 and top.hybrid[3001][0] == top.hybrid[3001].max()


def test_a_new_show_repeated_300_times(engine, fresh):
    old = _catalogue(3001, seed=12)
    new = _rows(_catalogue(10, seed=13), np.zeros(300, dtype=np.int64))
    _, top, _, _, _ = _run(engine, fresh, old, new)
    assert top.flagged_rows > 0, "the 300-wide plateau should send rows to the exact kernel"


def test_new_shows_without_text(engine, fresh):
    old = _catalogue(3001, seed=14)
    new = _catalogue(257, seed=15)
    t = new["text_features"].tolil()
    t[::2] = 0
    new["text_features"] = sp.csr_matrix(t)
    new["text_features"].eliminate_zeros()
    _run(engine, fresh, old, new)


# ---------------------------------------------------------------------------------------------- sequences
def test_three_appends_interleaved_with_a_symmetric_job(engine, fresh):
    feats = _catalogue(3001 + 77 + 256 + 1, seed=21)
    other = _catalogue(2500, seed=22)
    n = 3001
    cat = engine.ingest(_rows(feats, slice(0, n)), "mean3", W)
    prev_d = engine.top_k_device(cat, W, 20, MS)
    for q in (77, 256, 1):
        sym = engine.to_host(engine.top_k_device(engine.ingest(other, "mean3", W), W, 20, MS, tuning=SYMMETRIC))
        _assert_same(sym, fresh.compute_top_k(other, W, 20, MS))
        prev = engine.to_host(prev_d)
        cat = engine.extend(cat, _rows(feats, slice(n, n + q)))
        t = engine.top_k_append_device(cat, n, prev_d, W, 20, MS)
        assert t["incremental"]
        top = engine.to_host(t)
        n += q
        _assert_same(top, fresh.compute_top_k(_rows(feats, slice(0, n)), W, 20, MS))
        _check_changed(prev, top, t["changed_rows"].cpu().numpy())
        prev_d = t


# ---------------------------------------------------------------------------------------------- fallbacks
def _signed(feats, seed):
    rng = np.random.default_rng(seed)
    t = feats["text_features"].copy()
    t.data = t.data * np.where(rng.random(t.nnz) < 0.3, -1.0, 1.0)
    return {**feats, "text_features": t}


def _spy(engine, monkeypatch):
    """records, per top_k_append_device call, whether the incremental path ran"""
    calls, real = [], engine.top_k_append_device

    def wrapped(*a, **kw):
        t = real(*a, **kw)
        calls.append(bool(t["incremental"]))
        return t

    monkeypatch.setattr(engine, "top_k_append_device", wrapped)
    return calls


@pytest.mark.parametrize("case", ["signed_text", "fractional_genres", "k150", "fractional_new_only"])
def test_the_whole_job_fallbacks_keep_the_contract(engine, fresh, case, monkeypatch):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    feats = _catalogue(3001 + 256, seed=31)
    k = 150 if case == "k150" else 20
    if case == "signed_text":
        feats = _signed(feats, 1)
    if case == "fractional_genres":
        rng = np.random.default_rng(2)
        feats["genre_features"] = feats["genre_features"] * rng.random(feats["genre_features"].shape)
    if case == "fractional_new_only":
        g = feats["genre_features"].astype(np.float64)
        g[3001:] *= 0.5
        feats["genre_features"] = g
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(_rows(feats, slice(0, 3001)), k=k)
    calls = _spy(engine, monkeypatch)
    top = comp.extend_top_k(feats, prev, k=k)
    # fractional genres among the new shows only: the two parts cannot share one catalogue and the
    # drop-in runs the whole job without an append call; the others append on the whole-job path
    assert calls == ([] if case == "fractional_new_only" else [False])
    want = SimilarityComputer(engine=fresh).compute_top_k(feats, k=k)
    _assert_same(top, want)
    _check_changed(prev, top, top.changed_rows)


def test_drop_in_hstack_normalised_and_exclude_self_false(engine, fresh, monkeypatch):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    feats = _catalogue(1000 + 77, seed=41)
    comp = SimilarityComputer(0.5, 0.3, 0.2, engine=engine)
    ref = SimilarityComputer(0.5, 0.3, 0.2, engine=fresh)
    calls = _spy(engine, monkeypatch)
    for kw, path in (({"metadata_mode": "hstack", "normalize_weights": True}, [True]), ({"exclude_self": False}, [])):
        prev = comp.compute_top_k(_rows(feats, slice(0, 1000)), **kw)
        calls.clear()
        top = comp.extend_top_k(feats, prev, **kw)
        assert calls == path      # exclude_self=False: the whole job, no append
        _assert_same(top, ref.compute_top_k(feats, **kw))
        _check_changed(prev, top, top.changed_rows)
    same = comp.extend_top_k(_rows(feats, slice(0, 1000)), prev, exclude_self=False)
    assert same.changed_rows.size == 0 and np.array_equal(same.indices, prev.indices)


# ---------------------------------------------------------------------------------------------- oracle
def test_boundary_rows_match_the_oracle(engine, fresh):
    n_old, q = 3001, 300
    feats = _catalogue(n_old + q, seed=51)
    old, new = _split(feats, n_old)
    _, top, _, _, _ = _run(engine, fresh, old, new)
    n = n_old + q
    rows = np.unique(np.r_[0, n_old - 256:n_old + 3, n - 40:n].clip(0, n - 1))
    assert_topk_matches(top, feats, rows)


# ---------------------------------------------------------------------------------------------- validation
def test_mismatched_vocabulary_or_widths_raise(engine):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    old = _catalogue(1000, seed=61)
    for bad in (_catalogue(10, vocab=4000, seed=62), _catalogue(10, genres=41, seed=63)):
        with pytest.raises(ValueError):
            engine.extend(engine.ingest(old, "mean3", W), bad)
    wide = _catalogue(10, seed=64)
    wide["platform_features"] = np.hstack([wide["platform_features"], np.zeros((10, 1))])
    with pytest.raises(ValueError):
        engine.extend(engine.ingest(old, "mean3", W), wide)
    comp = SimilarityComputer(engine=engine)
    prev = comp.compute_top_k(old, k=20)
    with pytest.raises(ValueError):
        comp.extend_top_k(old, prev, k=10)
    with pytest.raises(ValueError):
        comp.extend_top_k(_rows(old, slice(0, 500)), prev, k=20)
