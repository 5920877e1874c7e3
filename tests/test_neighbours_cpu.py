"""Host side of the threshold job (every neighbour at or above min_similarity), no GPU: the record
shape of ``NeighbourTable`` against ``TopK``'s, and the routing of ``top_n_per_show=None`` and of
``--all-above-threshold`` in the populate driver (the engine is stubbed)."""

import numpy as np
import pytest

from tvbingefriend_recommendation_service_b200.engine import NeighbourTable, TopK
from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue


def _tables(n=9, k=4, seed=0):
    """The same neighbours as a [n, k] TopK and as a NeighbourTable; row 2 and the last row are empty."""
    rng = np.random.default_rng(seed)
    cnt = rng.integers(1, k + 1, size=n).astype(np.int32)
    cnt[2] = cnt[n - 1] = 0
    idx = np.full((n, k), -1, np.int32)
    sc = [np.zeros((n, k)) for _ in range(4)]
    for r in range(n):
        c = int(cnt[r])
        idx[r, :c] = rng.choice(n, size=c, replace=False)
        for a in sc:
            a[r, :c] = np.sort(rng.random(c))[::-1]
    mask = np.arange(k)[None, :] < cnt[:, None]
    row_ptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    nt = NeighbourTable(row_ptr, idx[mask], *(a[mask] for a in sc), candidate_pairs=17)
    return TopK(idx, cnt, *sc), nt


def test_to_dict_equals_topk_and_omits_empty_rows():
    top, nt = _tables()
    ids = np.arange(500, 509)
    d = nt.to_dict(ids)
    assert d == top.to_dict(ids)
    assert 502 not in d and 508 not in d
    rec = d[500][0]
    assert set(rec) == {"similar_show_id", "similarity_score", "genre_score", "text_score", "metadata_score"}
    assert nt.to_dict(ids, id_key="other")[500][0]["other"] == rec["similar_show_id"]
    assert np.array_equal(nt.counts, top.counts)


def test_records_equal_topk_and_to_dict():
    top, nt = _tables()
    ids = np.arange(500, 509)
    a, b = nt.records(ids), top.records(ids)
    assert set(a) == set(b)
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    flat = [(sid, r["similar_show_id"], r["similarity_score"], r["genre_score"], r["text_score"], r["metadata_score"])
            for sid, recs in nt.to_dict(ids).items() for r in recs]
    got = list(zip(*(a[c].tolist() for c in ("show_id", "similar_show_id", "similarity_score", "genre_score",
                                              "text_score", "metadata_score"))))
    assert got == flat


def test_slice_matches_topk_slice():
    top, nt = _tables(n=11)
    ids = np.arange(100, 111)
    for b, e in ((0, 11), (2, 5), (3, 3), (9, 11)):
        s = nt.slice(b, e)
        assert s.row_begin == b and s.row_ptr[0] == 0 and len(s.row_ptr) == e - b + 1
        assert s.to_dict(ids) == top.slice(b, e).to_dict(ids)
        for key, v in s.records(ids).items():
            assert np.array_equal(v, top.slice(b, e).records(ids)[key]), key


def test_store_batches_accepts_a_neighbour_table():
    from tvbingefriend_recommendation_service_b200.scripts.populate_database import store_similarity_batches
    from tvbingefriend_recommendation_service_b200.sinks import ColumnarSimilaritySink, InMemorySimilaritySink

    top, nt = _tables(n=13)
    ids = np.arange(7, 20)
    m1, m2, col = InMemorySimilaritySink(), InMemorySimilaritySink(), ColumnarSimilaritySink()
    assert store_similarity_batches(nt, ids, m1) == store_similarity_batches(top, ids, m2) == int(top.counts.sum())
    assert m1.records == m2.records
    assert store_similarity_batches(nt, ids, col) == int(top.counts.sum())


class _Stub:
    """Records which SimilarityComputer path the driver called."""

    def __init__(self, monkeypatch):
        from tvbingefriend_recommendation_service_b200.ml import similarity_computer as sc

        self.calls = []
        top, nt = _tables(n=12)
        stub = self

        def compute_top_k(self_, features, k=20, min_similarity=0.1, **kw):
            stub.calls.append(("top_k", k, min_similarity))
            return top

        def compute_neighbours(self_, features, min_similarity=0.1, max_per_row=None, **kw):
            stub.calls.append(("neighbours", max_per_row, min_similarity))
            return nt

        monkeypatch.setattr(sc.SimilarityComputer, "compute_top_k", compute_top_k)
        monkeypatch.setattr(sc.SimilarityComputer, "compute_neighbours", compute_neighbours)
        self.top, self.nt = top, nt


def test_top_n_none_reaches_the_threshold_path(tmp_path, monkeypatch):
    from tvbingefriend_recommendation_service_b200.scripts import populate_database as pd_

    make_catalogue(12, 40, nnz=5, seed=3).save(tmp_path)
    stub = _Stub(monkeypatch)
    stats = pd_.compute_and_store_similarities(tmp_path, top_n_per_show=None, min_similarity=0.3)
    assert stub.calls == [("neighbours", None, 0.3)]
    assert stats["total_records"] == int(stub.nt.row_ptr[-1]) and stats["top_n_per_show"] is None
    stats = pd_.compute_and_store_similarities(tmp_path, top_n_per_show=7, min_similarity=0.2)
    assert stub.calls[-1] == ("top_k", 7, 0.2) and stats["top_n_per_show"] == 7
    with pytest.raises(ValueError, match="one GPU"):
        pd_.compute_and_store_similarities(tmp_path, top_n_per_show=None, device_ids=[0, 1])


def test_cli_flag_routes_and_top_n_keeps_its_meaning(tmp_path, monkeypatch):
    from tvbingefriend_recommendation_service_b200.scripts import populate_database as pd_

    make_catalogue(12, 40, nnz=5, seed=3).save(tmp_path)
    stub = _Stub(monkeypatch)
    base = ["--input-dir", str(tmp_path), "--skip-metadata", "--skip-test"]
    stats = pd_.main(base + ["--all-above-threshold", "--min-similarity", "0.25"])
    assert stub.calls == [("neighbours", None, 0.25)] and stats["total_records"] == int(stub.nt.row_ptr[-1])
    pd_.main(base)
    assert stub.calls[-1] == ("top_k", 20, 0.1)          # defaults unchanged
    pd_.main(base + ["--top-n", "5"])
    assert stub.calls[-1] == ("top_k", 5, 0.1)
