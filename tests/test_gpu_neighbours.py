"""Every neighbour at or above a threshold (``tvbf_neighbours_*``, ``HybridTopKEngine.neighbours_device``)
on the GPU (``-m gpu``): the pair set and scores against float64 models, the capped rows against the
top-k table bit for bit on every operand the symmetric sweep takes, the reference's loop without its
top-n cut, and the edges (attained thresholds, duplicate clusters, empty text, the diagonal, the
capacity retry, refusals, reused workspaces)."""

import numpy as np
import pytest
import torch

from oracle.compare import compare_topk
from oracle.reference_paths import ProductionRows, dict_to_arrays, production_loop

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
FIELDS = ("indices", "hybrid", "genre", "text", "metadata")


@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


@pytest.fixture(scope="module")
def engine_bf16():
    """bf16 text: the candidate pass runs on the catalogue's own operand (no merged / folded second one)"""
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0, text_dtype="bf16")


def _features(n, vocab, seed=0, nnz=30, genres=40, meta=(5, 3, 2)):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    return make_catalogue(n, vocab, nnz=nnz, n_genres=genres, meta=meta, seed=seed).features()


def _host(t):
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine.neighbours_to_host(t)


def _score_pairs(engine, cat, weights, rows, cols):
    """tvbf_score_pairs on the catalogue's features: float64 [n, 4] {hybrid, genre, text, metadata}"""
    import ctypes as C

    from tvbingefriend_recommendation_service_b200._lib import check

    p = engine._params(cat, weights, 1, 0.1)
    pk = torch.from_numpy(np.stack([rows, cols], axis=1).astype(np.int32)).to(engine.device)
    out4 = torch.empty((len(rows), 4), dtype=torch.float64, device=engine.device)
    check(engine.lib.tvbf_score_pairs(C.byref(cat.c), C.byref(p), pk.data_ptr(), len(rows), out4.data_ptr(),
                                      engine._stream()), "tvbf_score_pairs")
    return out4.cpu().numpy()


def _assert_rows_ordered(nt):
    row = np.repeat(np.arange(len(nt.row_ptr) - 1), np.diff(nt.row_ptr))
    same = row[1:] == row[:-1]
    h, j = nt.hybrid, nt.indices
    ok = (h[:-1] > h[1:]) | ((h[:-1] == h[1:]) & (j[:-1] < j[1:]))
    assert np.all(ok[same]), "a row is not ordered by (score descending, column ascending)"
    return row


def _capped_equals_topk(engine, cat, weights, ms, k):
    """neighbours_device(max_per_row=k) against top_k_device(k), bit for bit"""
    nt = _host(engine.neighbours_device(cat, weights, ms, max_per_row=k))
    top = engine.to_host(engine.top_k_device(cat, weights, k, ms))
    assert np.array_equal(nt.counts, top.counts)
    mask = np.arange(k)[None, :] < top.counts[:, None]
    for name in FIELDS:
        a, b = getattr(nt, name), getattr(top, name)[mask]
        if a.dtype == np.float64:
            a, b = a.view(np.int64), b.view(np.int64)
        assert np.array_equal(a, b), name
    return nt, top


# ---------------------------------------------------------------------------------------------- 1. float64 model
@pytest.mark.parametrize("vocab", [500, 5000])
@pytest.mark.parametrize("mode", ["mean3", "hstack"])
def test_pair_set_and_scores_equal_float64_model(engine, vocab, mode):
    n = 2200
    f = _features(n, vocab, seed=vocab + len(mode), nnz=20)
    cat = engine.ingest(f, mode, W)
    pr = ProductionRows(f, *W, metadata_mode=mode)
    h, g, t, m = pr.rows_block(np.arange(n))
    np.fill_diagonal(h, -np.inf)
    for tau in (0.15, 0.3, 0.5):
        nt = _host(engine.neighbours_device(cat, W, tau))
        rows = _assert_rows_ordered(nt)
        cols = nt.indices.astype(np.int64)
        got = set(zip(rows.tolist(), cols.tolist()))
        want_i, want_j = np.nonzero(h >= tau)
        want = set(zip(want_i.tolist(), want_j.tolist()))
        near = np.abs(h - tau) <= 1e-9         # the model and the device may round a pair onto either side
        diff = got ^ want
        assert all(near[i, j] for i, j in diff), sorted(diff)[:10]
        assert nt.candidate_pairs >= (len(got) // 2)
        ref = _score_pairs(engine, cat, W, rows, cols)
        for c, name in enumerate(("hybrid", "genre", "text", "metadata")):
            assert np.array_equal(getattr(nt, name).view(np.int64), ref[:, c].view(np.int64)), name
            model = (h, g, t, m)[c][rows, cols]
            assert np.max(np.abs(getattr(nt, name) - model), initial=0.0) <= 1e-12, name
        assert np.all(nt.hybrid >= tau)


# ---------------------------------------------------------------------------------------------- 2. cap == top-k
# The operand the sweep receives (engine._folded with k = 1, or the catalogue's own) and the epilogue
# width it implies (16 warps while k_pad / 64 <= 96) select the kernel instantiation; every case
# asserts which one it reaches.  41 000 shows: 161 column tiles, where top_k_device runs the
# symmetric sweep.
CASES = {   # n, vocab, seed, catalogue kwargs, bf16 engine, (text merged, groups folded, genre_hi, wide)
    "merged_folded_v10k": (41_000, 10_000, 11, {}, False, (True, True, False, True)),
    "merged_v50k": (41_000, 50_000, 12, {"nnz": 60}, False, (True, False, False, False)),
    "folded_v500": (41_000, 500, 13, {"nnz": 20}, False, (False, True, False, True)),
    "folded_g100": (41_000, 2_000, 14, {"genres": 100}, False, (False, True, False, True)),
    "g100_merged_narrow": (41_000, 50_000, 16, {"nnz": 60, "genres": 100}, False, (True, False, True, False)),
    "g100_plain_wide": (41_000, 2_000, 17, {"genres": 100}, True, (False, False, True, True)),
    "plain_wide": (41_000, 2_000, 18, {}, True, (False, False, False, True)),
    "ragged_small": (173, 800, 15, {}, False, (False, True, False, True)),
}


@pytest.mark.parametrize("case", list(CASES))
def test_capped_rows_equal_topk_table(engine, engine_bf16, case):
    n, vocab, seed, kw, bf16, (merged, folded, two_words, wide) = CASES[case]
    eng = engine_bf16 if bf16 else engine
    f = _features(n, vocab, seed=seed, **kw)
    cat = eng.ingest(f, "mean3", W)
    feats = eng._folded(cat, *W, 1) or cat.c
    assert (int(feats.text_cols) > 0) == merged
    assert bool(feats.bits_folded) == folded
    # the kG2 kernels: a second mask word that is not folded into the operand (fill_k1_params)
    assert (bool(feats.genre_hi) and not folded) == two_words
    assert (int(feats.k_pad) // 64 <= 96) == wide
    for k in (20, 100):
        nt, top = _capped_equals_topk(eng, cat, W, 0.2, k)
        print(f"{case} k={k}: rows cut by the cap {int(np.count_nonzero(top.counts == k))} of {n}")
        if n > 1000 and k == 20:
            assert (top.counts == k).any()


# ---------------------------------------------------------------------------------------------- 3. reference loop
def test_reference_loop_without_top_n_cut(engine):
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer
    from tvbingefriend_recommendation_service_b200.synthetic import make_config

    cat = make_config("C1")
    f, ids = cat.features(), cat.show_ids
    ms = 0.2
    ref = production_loop(f, ids, *W, top_n_per_show=len(ids), min_similarity=ms)
    nt = SimilarityComputer(*W, engine=engine).compute_neighbours(f, min_similarity=ms)
    got = nt.to_dict(ids)
    assert set(got) == set(ref)
    k = max(len(v) for v in ref.values())
    ridx, rcnt, rsc = dict_to_arrays(ref, ids, k)
    gidx, gcnt, gsc = dict_to_arrays(got, ids, k)
    pr = ProductionRows(f, *W)
    rep = compare_topk(ridx, rcnt, rsc[0], gidx, gcnt, gsc[0], lambda r, js: pr.pair_scores(r, js), k, ms)
    assert rep.ok, rep.summary() + "\n" + "\n".join(rep.failures)


# ---------------------------------------------------------------------------------------------- 4. edges
def test_attained_threshold_is_included(engine):
    f = _features(1500, 2000, seed=5)
    cat = engine.ingest(f, "mean3", W)
    nt = _host(engine.neighbours_device(cat, W, 0.3))
    tau = float(nt.hybrid[len(nt.hybrid) // 3])      # an exact score the float64 scorer attains
    at = _host(engine.neighbours_device(cat, W, tau))
    assert at.hybrid.min() == tau
    assert int(at.row_ptr[-1]) == int(np.count_nonzero(nt.hybrid >= tau))


def test_duplicate_cluster_lists_every_member(engine):
    f = _features(3000, 3000, seed=6)
    full = (f["genre_features"].sum(axis=1) > 0) & (f["type_features"].sum(axis=1) > 0) & \
        (np.diff(f["text_features"].indptr) > 0)
    src = int(np.nonzero(full)[0][0])                    # a show with every feature group non-zero
    members = np.r_[src, np.arange(src + 1, 3000, 23)[:119]]   # 120 shows with the features of show src
    for key in ("genre_features", "platform_features", "type_features", "language_features"):
        f[key][members] = f[key][members[0]]
    text = f["text_features"].tolil()
    for r in members[1:]:
        text.rows[r], text.data[r] = list(text.rows[members[0]]), list(text.data[members[0]])
    f["text_features"] = text.tocsr()
    cat = engine.ingest(f, "mean3", W)
    nt = _host(engine.neighbours_device(cat, W, 0.99))
    for r in members:
        b, e = int(nt.row_ptr[r]), int(nt.row_ptr[r + 1])
        cols = nt.indices[b:e]
        assert set(members.tolist()) - {int(r)} <= set(cols.tolist())
        inside = np.isin(cols, members)
        assert np.all(nt.hybrid[b:e][inside] == nt.hybrid[b])   # the whole cluster ties at the row's top score
        assert abs(nt.hybrid[b] - 1.0) <= 1e-12


def test_empty_text_rows_and_the_diagonal(engine):
    f = _features(1200, 1500, seed=7)
    text = f["text_features"].tolil()
    empty = np.arange(0, 1200, 7)
    for r in empty:
        text.rows[r], text.data[r] = [], []
    f["text_features"] = text.tocsr()
    f["genre_features"][3] = 0                           # a zero genre row as well
    cat = engine.ingest(f, "mean3", W)
    pr = ProductionRows(f, *W)
    h = pr.rows_block(np.arange(1200))[0]
    ms = 0.25
    for exclude_self in (True, False):
        nt = _host(engine.neighbours_device(cat, W, ms, exclude_self=exclude_self))
        _assert_rows_ordered(nt)
        hh = h.copy()
        if exclude_self:
            np.fill_diagonal(hh, -np.inf)
        near = np.abs(hh - ms) <= 1e-9
        assert abs(int(nt.row_ptr[-1]) - int(np.count_nonzero(hh >= ms))) <= int(near.sum())
        rows = np.repeat(np.arange(1200), np.diff(nt.row_ptr))
        self_hits = rows == nt.indices
        if exclude_self:
            assert not self_hits.any()
        else:
            assert np.array_equal(np.sort(rows[self_hits]), np.nonzero(np.diag(h) >= ms)[0])


def test_capacity_retry_and_reused_workspace(engine):
    f = _features(2500, 3000, seed=8)
    cat = engine.ingest(f, "mean3", W)
    a = engine.neighbours_device(cat, W, 0.3)
    b = engine.neighbours_device(cat, W, 0.3, capacity=1)
    c = engine.neighbours_device(cat, W, 0.3)
    assert a["candidate_pairs"] == b["candidate_pairs"] == c["candidate_pairs"] > 1
    for name in ("row_ptr",) + FIELDS:
        x, y, z = (t[name].cpu().numpy() for t in (a, b, c))
        assert x.tobytes() == y.tobytes() == z.tobytes(), name
    with pytest.raises(ValueError, match="max_pairs"):
        engine.neighbours_device(cat, W, 0.3, max_pairs=2 * a["candidate_pairs"] + 2499)
    engine.neighbours_device(cat, W, 0.3, max_pairs=2 * a["candidate_pairs"] + 2500)
    # count only: capacity 0 and no pair buffer
    import ctypes as C

    from tvbingefriend_recommendation_service_b200._lib import check

    feats = engine._folded(cat, *W, 1) or cat.c
    p = engine._params(cat, W, 1, 0.3)
    ws = torch.empty((int(engine.lib.tvbf_neighbours_workspace_bytes(C.byref(feats), C.byref(p), 0)),),
                     dtype=torch.uint8, device=engine.device)
    count = torch.full((1,), -1, dtype=torch.int64, device=engine.device)
    check(engine.lib.tvbf_neighbours_sweep(C.byref(feats), C.byref(p), None, 0, count.data_ptr(), ws.data_ptr(),
                                           ws.numel(), engine._stream()), "tvbf_neighbours_sweep")
    assert int(count.item()) == a["candidate_pairs"]


def test_refused_jobs_name_the_reason(engine):
    from tvbingefriend_recommendation_service_b200._lib import TvbfError

    f = _features(600, 800, seed=9)
    cat = engine.ingest(f, "mean3", W)
    for ms in (0.0, -0.5):
        with pytest.raises(TvbfError, match="min_similarity must be > 0"):
            engine.neighbours_device(cat, W, ms)
    with pytest.raises(TvbfError, match="non-negative"):
        engine.neighbours_device(cat, (0.4, 0.7, -0.1), 0.1)
    g = dict(f)
    g["genre_features"] = f["genre_features"] * np.linspace(0.5, 1.5, f["genre_features"].shape[1])[None, :]
    floaty = engine.ingest(g, "mean3", W)
    assert floaty.folded
    with pytest.raises(TvbfError, match="folded"):
        engine.neighbours_device(floaty, W, 0.1)


# ---------------------------------------------------------------------------------------------- 5. loose bound
def test_complete_under_a_loose_merged_bound(engine):
    n = 3000
    f = _features(n, 50_000, seed=10, nnz=60)
    cat = engine.ingest(f, "mean3", W)
    feats = engine._folded(cat, *W, 1)
    assert feats is not None and int(feats.text_cols) > 0
    h = ProductionRows(f, *W).rows_block(np.arange(n))[0]
    np.fill_diagonal(h, -np.inf)
    upper = h[np.triu_indices(n, 1)]
    # just below the densest band of exact scores above 0.2
    hist, edges = np.histogram(upper[upper > 0.2], bins=200)
    tau = float(edges[int(np.argmax(hist))]) - 1e-6
    nt = _host(engine.neighbours_device(cat, W, tau))
    rows = np.repeat(np.arange(n), np.diff(nt.row_ptr))
    got = set(zip(rows.tolist(), nt.indices.tolist()))
    wi, wj = np.nonzero(h >= tau + 1e-9)
    missing = [(i, j) for i, j in zip(wi.tolist(), wj.tolist()) if (i, j) not in got]
    assert not missing, missing[:10]
    exact = int(np.count_nonzero(upper >= tau))
    print(f"loose bound: tau={tau:.6f} candidate pairs {nt.candidate_pairs} exact pairs {exact} "
          f"({nt.candidate_pairs / max(exact, 1):.2f}x)")
    assert nt.candidate_pairs >= exact
