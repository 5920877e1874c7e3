"""The exact row kernel on rows with text (``-m gpu``): text scores come from the column-major copy of
the text that the kernel builds on every call.  Every table is checked bit for bit against
``tvbf_score_pairs`` (the K5 scorer) on the same pairs and against the float64 oracle."""

import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from oracle.compare import compare_topk
from helpers import oracle_rows

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)


@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


def _score_pairs(engine, dc, rows, idx):
    """hybrid / genre / text / metadata of every (rows[r], idx[r, e]) with idx >= 0, from tvbf_score_pairs"""
    import torch

    from tvbingefriend_recommendation_service_b200._lib import Params, check

    r, e = np.nonzero(idx >= 0)
    pairs = np.ascontiguousarray(np.stack([np.asarray(rows)[r], idx[r, e]], axis=1).astype(np.int32))
    p = Params(genre_weight=W[0], text_weight=W[1], metadata_weight=W[2], min_similarity=0.0, k=1, exclude_self=1,
               row_begin=0, row_end=dc.n_shows)
    with torch.cuda.device(engine.device):
        pd = torch.from_numpy(pairs).to(engine.device)
        out = torch.empty((len(pairs), 4), dtype=torch.float64, device=engine.device)
        check(engine.lib.tvbf_score_pairs(C.byref(dc.c), C.byref(p), pd.data_ptr(), len(pairs), out.data_ptr(),
                                          engine._stream()), "tvbf_score_pairs")
        return out.cpu().numpy()


def _check(engine, dc, feats, rows, top, k, min_similarity):
    """``top``: table row t is source row rows[t]"""
    rows = np.asarray(rows)
    got = _score_pairs(engine, dc, rows, top.indices)
    m = top.indices >= 0
    for c, name in enumerate(("hybrid", "genre", "text", "metadata")):
        assert np.array_equal(getattr(top, name)[m], got[:, c]), name
    pr, ridx, rcnt, rsc = oracle_rows(feats, rows, W, k, min_similarity)
    rep = compare_topk(ridx, rcnt, rsc[0], top.indices, top.counts, top.hybrid,
                       lambda r, js: pr.pair_scores(int(rows[r]), js), k, min_similarity)
    assert rep.ok, rep.summary() + "\n" + "\n".join(rep.failures)


def _upload(engine, feats):
    from tvbingefriend_recommendation_service_b200.engine import stage

    return engine.upload(stage(feats), W)


def _features(n, vocab, nnz, seed):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    return make_catalogue(n, vocab, nnz=nnz, seed=seed).features()


def test_many_rows_zipf_text(engine):
    """2 400 rows (more than the grid's row slots: whole batches per CTA), Zipf text whose most
    frequent terms are in most shows, with the empty-text rows of the catalogue among them"""
    feats = _features(6000, 3000, 60, 11)
    text = sp.csr_matrix(feats["text_features"])
    lens = np.diff(text.indptr)
    df = np.bincount(text.indices, minlength=3000)
    assert df.max() > 0.5 * 6000
    empty = np.flatnonzero(lens == 0)
    rows = np.unique(np.concatenate([np.arange(0, 6000, 3)[:2400 - 20], empty[:20]]))
    assert len(rows) >= 2000 and np.isin(empty[:20], rows).all() and len(empty) >= 20
    dc = _upload(engine, feats)
    top = engine.exact_rows(dc, rows, W, k=20, min_similarity=0.1)
    _check(engine, dc, feats, rows, top, 20, 0.1)


def test_wide_vocabulary(engine):
    """V = 150 000 columns: the postings have no vocabulary limit"""
    feats = _features(3000, 150_000, 40, 12)
    rows = np.arange(1, 3000, 10)
    dc = _upload(engine, feats)
    top = engine.exact_rows(dc, rows, W, k=30, min_similarity=0.0)
    _check(engine, dc, feats, rows, top, 30, 0.0)


def test_long_rows_and_empty_rows_in_one_batch(engine):
    """rows of more than 192 terms next to rows without text in the same batches (few rows: one
    row's column slices spread over many CTAs)"""
    feats = _features(2500, 4000, 300, 13)
    text = sp.csr_matrix(feats["text_features"])
    lens = np.diff(text.indptr)
    long_rows = np.flatnonzero(lens > 192)[:12]
    empty = np.flatnonzero(lens == 0)[:4]
    assert len(long_rows) == 12 and len(empty) >= 1
    rows = np.concatenate([long_rows[:6], empty, long_rows[6:]])
    dc = _upload(engine, feats)
    top = engine.exact_rows(dc, rows, W, k=20, min_similarity=0.0)
    _check(engine, dc, feats, rows, top, 20, 0.0)


def test_signed_text(engine):
    """negative text values (embeddings): products of both signs, cancellation in the sums"""
    feats = _features(3000, 2000, 40, 14)
    text = sp.csr_matrix(feats["text_features"]).copy()
    rng = np.random.default_rng(5)
    text.data *= np.where(rng.random(text.nnz) < 0.4, -1.0, 1.0)
    feats = {**feats, "text_features": text}
    rows = np.arange(0, 3000, 7)
    dc = _upload(engine, feats)
    assert dc.c.text_signed
    top = engine.exact_rows(dc, rows, W, k=20, min_similarity=0.0)
    _check(engine, dc, feats, rows, top, 20, 0.0)


@pytest.mark.parametrize("n", [1237, 3001])
def test_force_exact_ragged(engine, n):
    """force_exact sends every row to the exact kernel; N not a multiple of any tile or slice"""
    feats = _features(n, 2500, 45, 15 + n)
    dc = _upload(engine, feats)
    top = engine.to_host(engine.top_k_device(dc, W, 20, 0.1, force_exact=True))
    rows = np.arange(n)
    _check(engine, dc, feats, rows, top, 20, 0.1)
    ref = engine.to_host(engine.top_k_device(dc, W, 20, 0.1))
    for name in ("indices", "counts", "hybrid", "genre", "text", "metadata"):
        assert np.array_equal(np.nan_to_num(getattr(top, name)), np.nan_to_num(getattr(ref, name))), name
