"""The merged text operand of the candidate pass (``-m gpu``): large vocabularies run K1 over text
columns merged by document frequency (``merge_text_cols``, ``tvbf_merge_plan``).  It changes which
pairs are rescored, never the table: every table here is compared bit for bit with the same job with
merging off (``merge_ratio = 0``, the catalogue's own operand)."""

import numpy as np
import pytest
import scipy.sparse as sp

from helpers import assert_topk_matches
from test_merge_plan import model_plan

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
MS = 0.1
SYM_OFF, SYM_ON = 1 << 20, 2 << 20
FIELDS = ("indices", "counts", "hybrid", "genre", "text", "metadata")


@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


@pytest.fixture(scope="module")
def plain():
    """the same jobs on the catalogue's own operand"""
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    eng = HybridTopKEngine(0)
    eng.merge_ratio = 0.0
    return eng


def _catalogue(n, vocab, seed=0, nnz=30, genres=40):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    return make_catalogue(n, vocab, nnz=nnz, n_genres=genres, seed=seed).features()


def _same(a, b):
    for name in FIELDS:
        x, y = getattr(a, name), getattr(b, name)
        assert x.tobytes() == y.tobytes(), name


def _merged_cols(engine):
    fc = engine._fold_owner
    return None if fc is None else int(fc["c"].text_cols)


def _plan_of_csr(engine, text, kt):
    """tvbf_merge_plan called directly on the C ABI over a host CSR"""
    import torch

    dev, vocab = engine.device, text.shape[1]
    indptr = torch.from_numpy(text.indptr.astype(np.int64)).to(dev)
    indices = torch.from_numpy(np.r_[text.indices, 0].astype(np.int32)).to(dev)   # non-NULL when empty
    plan = {"col_map": torch.empty((vocab,), dtype=torch.int32, device=dev),
            "slot_ptr": torch.empty((kt + 1,), dtype=torch.int32, device=dev),
            "slot_cols": torch.empty((vocab,), dtype=torch.int32, device=dev)}
    lib = engine.lib
    ws = torch.empty((int(lib.tvbf_merge_plan_workspace_bytes(vocab)),), dtype=torch.uint8, device=dev)
    rc = lib.tvbf_merge_plan(indptr.data_ptr(), indices.data_ptr(), text.shape[0], vocab, kt,
                             plan["col_map"].data_ptr(), plan["slot_ptr"].data_ptr(), plan["slot_cols"].data_ptr(),
                             ws.data_ptr(), ws.numel(), engine._stream())
    assert rc == 0, lib.tvbf_last_error().decode()
    return plan


# (vocab, text_cols, text): text "catalogue" is the synthetic one, "first_3000" uses only the first
# 3 000 columns (the others have no document: ascending index), "each_once" every column exactly once
# (all frequencies equal: the stable sort keeps index order), "empty" no entries at all
PLAN_CASES = [
    pytest.param(6000, None, "catalogue", id="6000"),
    pytest.param(10_000, None, "catalogue", id="10000"),
    pytest.param(50_000, 20_000, "catalogue", id="50000_rem0"),          # head 10 000, 4 columns per tail slot
    pytest.param(8000, 4000, "catalogue", id="8000_rem0"),
    pytest.param(10_000, 3001, "catalogue", id="odd_3001"),              # head 1 500, tail 1 501
    pytest.param(4097, 2, "catalogue", id="4097_one_slot_of_4096"),
    pytest.param(10_000, 4024, "first_3000", id="first_3000_of_10000"),
    pytest.param(10_000, 4024, "each_once", id="every_column_once"),
    pytest.param(10_000, 4024, "empty", id="no_text"),
]


@pytest.mark.parametrize("vocab,text_cols,text", PLAN_CASES)
def test_device_plan_is_the_numpy_model(engine, vocab, text_cols, text):
    from tvbingefriend_recommendation_service_b200.engine import merge_text_cols

    kt = merge_text_cols(vocab, 40) if text_cols is None else text_cols
    rng = np.random.default_rng(vocab + kt)
    if text == "catalogue":
        f = _catalogue(3000, vocab, seed=vocab)
        plan = engine._merge_plan(engine.ingest(f), kt)
        indices = f["text_features"].indices
    else:
        if text == "first_3000":
            x = _catalogue(3000, 3000, seed=61)["text_features"].tocsr()
            csr = sp.csr_matrix((x.data, x.indices, x.indptr), shape=(3000, vocab))
            f = _catalogue(3000, vocab, seed=62)
            f["text_features"] = csr
            plan = engine._merge_plan(engine.ingest(f), kt)
        elif text == "each_once":
            cols = np.sort(rng.permutation(vocab).reshape(2000, 5), axis=1)
            csr = sp.csr_matrix((rng.random(vocab) + 0.05, cols.reshape(-1), np.arange(0, vocab + 1, 5)),
                                shape=(2000, vocab))
            f = _catalogue(2000, vocab, seed=63)
            f["text_features"] = csr
            plan = engine._merge_plan(engine.ingest(f), kt)
        else:
            csr = sp.csr_matrix((100, vocab))
            plan = _plan_of_csr(engine, csr, kt)
        indices = csr.indices
    col_map, slot_ptr, slot_cols = model_plan(indices, vocab, kt)
    got = {key: plan[key].cpu().numpy() for key in ("col_map", "slot_ptr", "slot_cols")}
    assert np.array_equal(got["col_map"], col_map)
    assert np.array_equal(got["slot_ptr"], slot_ptr)
    assert np.array_equal(got["slot_cols"], slot_cols)
    head, tail = kt // 2, kt - kt // 2
    if (vocab - head) % tail == 0:
        assert np.all(np.diff(slot_ptr)[head:] == (vocab - head) // tail)
    # the ranking read back from the device plan: rank r >= head is entry (r - head) // tail of slot
    # head + (r - head) % tail; by descending frequency, equal frequencies by ascending column
    r = np.arange(vocab)
    pos = np.where(r < head, r, got["slot_ptr"][head + (r - head) % tail] + (r - head) // tail)
    ranking = got["slot_cols"][pos]
    df = np.bincount(indices, minlength=vocab)
    assert np.array_equal(ranking, np.argsort(-df, kind="stable"))
    if text in ("each_once", "empty"):
        assert np.array_equal(ranking, np.arange(vocab))
    elif text == "first_3000":
        assert np.array_equal(ranking[3000:], np.arange(3000, vocab))


@pytest.mark.parametrize("vocab", [6000, 10_000, 50_000])
@pytest.mark.parametrize("k", [20, 60, 100], ids=["k20", "k60", "k100"])
@pytest.mark.parametrize("tuning", [SYM_OFF, SYM_ON], ids=["one_sided", "symmetric"])
def test_merged_tables_equal_the_plain_ones(engine, plain, vocab, k, tuning):
    from tvbingefriend_recommendation_service_b200.engine import merge_text_cols

    f = _catalogue(3000, vocab, seed=vocab + k)
    engine._fold_owner = None
    top = engine.compute_top_k(f, W, k, MS, tuning=tuning)
    fc = engine._fold_owner
    kt = merge_text_cols(vocab, 40)
    assert fc is not None and int(fc["c"].text_cols) == kt
    assert bool(fc["c"].bits_folded) == (k <= 48 and kt + 40 + 32 <= engine.fold_max_k)
    want = plain.compute_top_k(f, W, k, MS, tuning=tuning)
    assert plain._fold_owner is None
    _same(top, want)
    print(f"V={vocab} k={k}: flagged merged {top.flagged_rows} plain {want.flagged_rows}, rescored pairs "
          f"{top.rescored_pairs} / {want.rescored_pairs}")
    if vocab == 10_000:
        assert_topk_matches(top, f, np.arange(0, 3000, 97), k=k)


def test_plan_tiles_reports_the_merged_depth(engine):
    f = _catalogue(3000, 10_000, seed=4)
    cat = engine.ingest(f)
    engine.top_k_device(cat, W, 20, MS)
    plan = engine.plan_tiles(cat, W, 20, MS)
    assert plan["k_pad"] == 4096 and plan["text_cols"] == 4024 and plan["folded_bits"]
    assert plan["flops"] == 2.0 * (plan["seed_tiles"] + plan["sweep_tiles"]) * plan["tile_rows"] * 256 * 4096


def test_merge_ratio_zero_keeps_the_catalogue_operand(engine):
    f = _catalogue(3000, 10_000, seed=5)
    old = engine.merge_ratio
    engine.merge_ratio = 0.0
    try:
        engine._fold_owner = None
        cat = engine.ingest(f)
        engine.top_k_device(cat, W, 20, MS)
        assert engine._fold_owner is None
        assert engine.plan_tiles(cat, W, 20, MS)["k_pad"] == 10_048
    finally:
        engine.merge_ratio = old


# ---------------------------------------------------------------------------------------------- incremental
def _rows(feats, sel):
    return {key: (a[sel].tocsr() if sp.issparse(a) else a[sel]) for key, a in feats.items()}


@pytest.mark.parametrize("kind", ["append", "update", "remove", "refresh"])
def test_incremental_paths_over_the_merged_operand(engine, plain, kind):
    """append / update / remove / refresh write their rows into the merged operand through the
    catalogue's plan; each table equals the whole job on the plain operand"""
    n, q, vocab = 3000, 150, 10_000
    before = _catalogue(n, vocab, seed=11)
    other = _catalogue(2 * q, vocab, seed=12)
    cat = engine.ingest(before)
    prev = engine.top_k_device(cat, W, 20, MS)
    assert _merged_cols(engine) == 4024
    rng = np.random.default_rng(13)
    rows = np.sort(rng.choice(n, size=q, replace=False))
    if kind == "append":
        cat = engine.extend(cat, _rows(other, np.arange(q)))
        t = engine.top_k_append_device(cat, n, prev, W, 20, MS)
        after = {key: (sp.vstack([before[key], other[key][:q]]).tocsr() if sp.issparse(before[key])
                       else np.concatenate([before[key], other[key][:q]])) for key in before}
    elif kind == "update":
        cat = engine.update(cat, rows, _rows(other, np.arange(q)))
        t = engine.top_k_update_device(cat, rows, prev, W, 20, MS)
        src = np.arange(n)
        src[rows] = n + np.arange(q)
        after = _rows({key: (sp.vstack([before[key], other[key][:q]]).tocsr() if sp.issparse(before[key])
                             else np.concatenate([before[key], other[key][:q]])) for key in before}, src)
    elif kind == "remove":
        cat = engine.remove(cat, rows)
        t = engine.top_k_remove_device(cat, rows, prev, W, 20, MS)
        after = _rows(before, np.delete(np.arange(n), rows))
    else:
        removed, updated = rows[::2], rows[1::2]
        cat = engine.update(cat, updated, _rows(other, np.arange(updated.size)))
        cat = engine.remove(cat, removed)
        cat = engine.extend(cat, _rows(other, q + np.arange(q)))
        t = engine.top_k_refresh_device(cat, prev, removed, updated, q, W, 20, MS)
        src = np.arange(n)
        src[updated] = n + np.arange(updated.size)
        both = {key: (sp.vstack([before[key], other[key]]).tocsr() if sp.issparse(before[key])
                      else np.concatenate([before[key], other[key]])) for key in before}
        after = _rows(both, np.r_[np.delete(src, removed), n + q + np.arange(q)])
    assert t["incremental"]
    assert _merged_cols(engine) == 4024
    _same(engine.to_host(t), plain.compute_top_k(after, W, 20, MS))


# ---------------------------------------------------------------------------------------------- adversary
def test_rows_whose_terms_share_one_merged_column(engine, plain):
    """Column c gets document frequency non-increasing in c, so the plan ranks columns in index order
    and 2012 + t, 4024 + t, 6036 + t, 8048 + t share operand column 2012 + t.  600 rows use two of
    those four columns: rows with disjoint pairs have text cosine 0 but a full merged dot, their lists
    fill with false candidates, and the table must still come out exact (through the exact kernel)."""
    n_bg, n_adv, vocab, head = 2400, 600, 10_000, 2012
    rng = np.random.default_rng(21)
    groups = np.array([[head + t, 2 * head + t, 3 * head + t, 4 * head + t] for t in range(10)])
    pairs = ((0, 1), (2, 3), (0, 2), (1, 3))
    adv = [np.sort(groups[i % 10][list(pairs[(i // 10) % 4])]) for i in range(n_adv)]
    a_cnt = np.bincount(np.concatenate(adv), minlength=vocab)
    base = 30 + (vocab - np.arange(vocab)) // 400
    b_cnt = base - a_cnt
    assert b_cnt.min() >= 0
    bg_rows = [[] for _ in range(n_bg)]
    for c in range(vocab):
        for r in rng.choice(n_bg, size=b_cnt[c], replace=False):
            bg_rows[r].append(c)
    rows = [np.array(sorted(r), dtype=np.int64) for r in bg_rows] + adv
    indptr = np.r_[0, np.cumsum([r.size for r in rows])]
    text = sp.csr_matrix((rng.random(indptr[-1]) + 0.05, np.concatenate(rows), indptr), shape=(n_bg + n_adv, vocab))
    f = _catalogue(n_bg + n_adv, vocab, seed=22)
    f["text_features"] = text
    df = np.diff(text.tocsc().indptr)
    assert np.all(df[:-1] >= df[1:])
    cat = engine.ingest(f)
    engine._fold_owner = None
    top = engine.to_host(engine.top_k_device(cat, W, 20, MS))
    col_map = engine._fold_owner["plan"]["col_map"].cpu().numpy()
    assert np.all(col_map[groups] == col_map[groups[:, :1]])
    want = plain.compute_top_k(f, W, 20, MS)
    _same(top, want)
    print(f"adversary: flagged merged {top.flagged_rows} plain {want.flagged_rows}")
    assert_topk_matches(top, f, np.r_[np.arange(0, n_bg, 311), n_bg + np.arange(0, n_adv, 37)])


# ---------------------------------------------------------------------------------------------- untouched
def test_signed_text_never_merges(engine):
    f = _catalogue(1500, 6000, seed=31)
    rng = np.random.default_rng(32)
    t = f["text_features"].tocsr().copy()
    t.data = rng.standard_normal(t.data.size)
    f["text_features"] = t
    engine._fold_owner = None
    top = engine.compute_top_k(f, W, 20, MS)
    assert engine._fold_owner is None
    exact = engine.compute_top_k(f, W, 20, MS, force_exact=True)
    assert np.array_equal(top.counts, exact.counts) and np.array_equal(top.indices, exact.indices)


def test_statistics_run_on_the_catalogue_operand(engine, plain):
    import ctypes as C

    f = _catalogue(3000, 6000, seed=41)
    cat = engine.ingest(f)
    engine.top_k_device(cat, W, 60, MS)               # the merged second operand now exists, without the groups
    merged = engine._fold_owner["c"]
    assert merged.text_cols > 0 and not merged.bits_folded
    a = engine.similarity_stats(cat, W)
    b = plain.similarity_stats(plain.ingest(f), W)
    for name in b:
        for key in ("mean", "std", "min", "max", "median"):
            assert a[name][key] == pytest.approx(b[name][key], rel=1e-9, abs=1e-12), (name, key)
    accum = engine._workspace(1 << 20)
    p = engine._params(cat, W, 20, MS)
    rc = engine.lib.tvbf_similarity_stats(C.byref(merged), C.byref(p), accum.data_ptr(), accum.data_ptr(),
                                          accum.numel(), engine._stream())
    assert rc != 0 and "text_cols" in engine.lib.tvbf_last_error().decode()
    engine.top_k_device(cat, W, 20, MS)               # merged text and the packed groups
    folded = engine._fold_owner["c"]
    assert folded.text_cols > 0 and folded.bits_folded
    rc = engine.lib.tvbf_similarity_stats(C.byref(folded), C.byref(p), accum.data_ptr(), accum.data_ptr(),
                                          accum.numel(), engine._stream())
    assert rc != 0 and "plain text operand" in engine.lib.tvbf_last_error().decode()
