"""GPU parity tests added in round 2 (``-m gpu``): the configurations BASELINE.md names on ALL rows,
bit-level properties of the reported float64 scores, and the premise of the certificate (the
candidate pass' upper bound) on dense / long-K / signed text.  Every call goes through the C ABI."""

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_golden
from helpers import assert_topk_matches
from oracle.compare import compare_topk
from oracle.cosine import normalize_rows
from oracle.reference_paths import ProductionRows

pytestmark = pytest.mark.gpu

SYM_OFF, SYM_ON = 1 << 20, 2 << 20


@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


# ---- BASELINE.json configs[0] / configs[1] on every row ---------------------------------------------
@pytest.mark.parametrize("tuning", [SYM_OFF, SYM_ON], ids=["one_sided", "symmetric"])
def test_golden_c1_all_rows(engine, tuning):
    """C1 (1 000 shows x 5 000 vocab): the table of the UNMODIFIED reference hot loop
    (scripts/populate_database.py:85-259, fixture made by oracle/make_golden.py), all 1 000 rows."""
    z, cat = load_golden("populate_c1")
    gw, tw, mw, k, ms = z["case0_params"].tolist()
    k = int(k)
    top = engine.compute_top_k(cat.features(), (gw, tw, mw), k, ms, tuning=tuning)
    pr = ProductionRows(cat.features(), gw, tw, mw)
    rep = compare_topk(z["case0_idx"].astype(np.int64), z["case0_cnt"], z["case0_scores"][0], top.indices,
                       top.counts, top.hybrid, lambda r, js: pr.pair_scores(r, js), k, ms)
    assert rep.ok and rep.rows == 1000, rep.summary() + "\n" + "\n".join(rep.failures)
    assert int(top.counts.sum()) == int(z["case0_total_records"])
    # scores of entries at identical positions: 1e-5 relative is the bar; float64 gives ~1e-16
    same = (z["case0_idx"] == top.indices) & (top.indices >= 0)
    for c, name in enumerate(("hybrid", "genre", "text", "metadata")):
        err = np.abs(getattr(top, name)[same] - z["case0_scores"][c][same])
        assert err.max() <= 1e-14, (name, err.max())


@pytest.mark.parametrize("fold", [True, False], ids=["folded", "popcount"])
@pytest.mark.parametrize("tuning", [SYM_OFF, SYM_ON], ids=["one_sided", "symmetric"])
def test_golden_production_shape_v500_all_rows(engine, tuning, fold):
    """The reference's production shape in miniature (500-term vocabulary, metadata widths 21 / 5 / 6):
    the table of the UNMODIFIED reference hot loop for 1 500 shows, all rows, reference defaults and a
    raw-weight case -- with the packed groups folded into the tensor-core operand (the default at this
    vocabulary) and with the popcount epilogue."""
    z, cat = load_golden("populate_v500_n1500")
    old = engine.fold_max_k
    engine.fold_max_k = old if fold else 0
    try:
        for c in range(int(z["n_cases"])):
            gw, tw, mw, k, ms = z[f"case{c}_params"].tolist()
            k = int(k)
            engine._fold_owner = None
            top = engine.compute_top_k(cat.features(), (gw, tw, mw), k, ms, tuning=tuning)
            assert (engine._fold_owner is not None) == fold
            pr = ProductionRows(cat.features(), gw, tw, mw)
            rep = compare_topk(z[f"case{c}_idx"].astype(np.int64), z[f"case{c}_cnt"], z[f"case{c}_scores"][0],
                               top.indices, top.counts, top.hybrid, lambda r, js: pr.pair_scores(r, js), k, ms)
            assert rep.ok and rep.rows == 1500, rep.summary() + "\n" + "\n".join(rep.failures)
            assert int(top.counts.sum()) == int(z[f"case{c}_total_records"])
            same = (z[f"case{c}_idx"] == top.indices) & (top.indices >= 0)
            for f_, name in enumerate(("hybrid", "genre", "text", "metadata")):
                ref = z[f"case{c}_scores"][f_][same]
                err = np.abs(getattr(top, name)[same] - ref)
                assert np.all(err <= 1e-14 * np.maximum(1.0, np.abs(ref))), (name, err.max())
    finally:
        engine.fold_max_k = old


def test_c1_through_the_populate_driver(engine, tmp_path):
    """Same fixture through the drop-in of ``compute_and_store_similarities`` (file contract, sink)."""
    from oracle.reference_paths import dict_to_arrays
    from tvbingefriend_recommendation_service_b200.scripts.populate_database import compute_and_store_similarities
    from tvbingefriend_recommendation_service_b200.sinks import InMemorySimilaritySink

    z, cat = load_golden("populate_c1")
    cat.save(tmp_path)
    sink = InMemorySimilaritySink()
    stats = compute_and_store_similarities(tmp_path, sink=sink)
    assert stats["total_records"] == int(z["case0_total_records"])
    idx, cnt, sc = dict_to_arrays(sink.records, cat.show_ids.tolist(), 20)
    pr = ProductionRows(cat.features())
    rep = compare_topk(z["case0_idx"].astype(np.int64), z["case0_cnt"], z["case0_scores"][0], idx, cnt, sc[0],
                       lambda r, js: pr.pair_scores(r, js), 20, 0.1)
    assert rep.ok and rep.rows == 1000, rep.summary() + "\n" + "\n".join(rep.failures)


def test_c2_all_rows_vs_oracle(engine):
    """C2 (20 000 shows x 5 000 vocab, BASELINE.json configs[1]): all 20 000 rows against the CPU
    restatement of the production loop (float64, per-row argsort walk)."""
    from tvbingefriend_recommendation_service_b200.synthetic import make_config

    cat = make_config("C2")
    top = engine.compute_top_k(cat.features(), (0.4, 0.5, 0.1), 20, 0.1)
    pr = ProductionRows(cat.features())
    rows = np.arange(cat.n_shows)
    ridx, rcnt, rsc = pr.topk_arrays(rows, 20, 0.1, block=256)
    rep = compare_topk(ridx, rcnt, rsc[0], top.indices, top.counts, top.hybrid,
                       lambda r, js: pr.pair_scores(int(r), js), 20, 0.1)
    assert rep.ok and rep.rows == 20000, rep.summary() + "\n" + "\n".join(rep.failures[:20])
    same = (ridx == top.indices) & (ridx >= 0)
    assert same.mean() > 0.95
    for c, name in enumerate(("hybrid", "genre", "text", "metadata")):
        err = np.abs(getattr(top, name)[same] - rsc[c][same])
        assert err.max() <= 1e-5 * np.abs(rsc[c][same]).max() and err.max() < 1e-13, (name, err.max())


# ---- reported scores: bit-level properties -------------------------------------------------------------
@pytest.mark.parametrize("w", [(0.4, 0.5, 0.1), (2.0, 3.0, 1.0), (0.3, 0.6, 0.1)])
def test_hybrid_is_the_numpy_expression_of_the_reported_components(engine, w):
    """similarity_score == gw*genre_score + tw*text_score + mw*metadata_score evaluated the way numpy
    evaluates scripts/populate_database.py:190-192 (three rounded products, two rounded sums, no
    FMA), bit for bit, from every kernel that reports scores: K5 (certified rows), K6 (repaired /
    forced-exact rows) and the single-show query."""
    from tvbingefriend_recommendation_service_b200.engine import stage
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(3000, 4000, nnz=35, seed=77)
    gw, tw, mw = w
    dc = engine.upload(stage(cat.features()), w)
    tabs = [engine.to_host(engine.top_k_device(dc, w, 20, 0.05)),
            engine.to_host(engine.top_k_device(dc, w, 20, 0.05, force_exact=True)),
            engine.exact_rows(dc, np.arange(0, 3000, 11), w, k=50, min_similarity=0.0)]
    for t in tabs:
        m = t.indices >= 0
        want = gw * t.genre[m] + tw * t.text[m] + mw * t.metadata[m]
        assert np.array_equal(t.hybrid[m], want)
    assert np.array_equal(tabs[0].indices, tabs[1].indices)
    m = tabs[0].indices >= 0
    for name in ("hybrid", "genre", "text", "metadata"):   # K5 and K6 agree bit for bit
        assert np.array_equal(getattr(tabs[0], name)[m], getattr(tabs[1], name)[m]), name


def test_no_cooperative_fallback_in_normal_operation(engine):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(1500, 512, nnz=12, seed=3)
    engine.compute_top_k(cat.features(), (0.4, 0.5, 0.1), 20, 0.1)
    assert int(engine.lib.tvbf_noncooperative_fallbacks()) == 0
    top = engine.compute_top_k(cat.features(), (0.4, 0.5, 0.1), 20, 0.1, tuning=1 << 30)   # plain launch on request
    assert_topk_matches(top, cat.features(), np.arange(0, 1500, 13))


# ---- the certificate's premise: U >= exact, on sparse, dense, long-K and signed text ----------------------
def _upper_bound_tile(engine, feats, weights, row0=0, col0=0):
    """(U, exact text part) of the 128 x 256 tile at (row0, col0): U from the raw tensor-core
    accumulators and the library's own slack constants, exact = text_weight * float64 cosine."""
    from tvbingefriend_recommendation_service_b200.engine import stage

    dc = engine.upload(stage(feats), weights)
    sl = engine.debug_slack(dc, weights)
    acc = engine.debug_gemm_tile(dc, row0, col0).cpu().numpy().astype(np.float64)
    tn = normalize_rows(sp.csr_matrix(feats["text_features"]))
    n = tn.shape[0]
    r1, c1 = min(row0 + 128, n), min(col0 + 256, n)
    exact = weights[1] * np.asarray((tn[row0:r1] @ tn[col0:c1].T).todense())
    terms = np.diff(tn.indptr)[row0:r1].astype(np.float64)[:, None]
    a = acc[:r1 - row0, :c1 - col0]
    u = sl["w_text"] * a + (sl["w_text_err"] + terms * sl["w_text_acc"]) * np.abs(a) + sl["eps"] + terms * sl["eps_term"]
    return u, exact, sl, a


def _only_text(n, text):
    z = np.zeros((n, 1))
    return {"genre_features": np.zeros((n, 2), dtype=np.int64), "text_features": text,
            "platform_features": z.copy(), "type_features": z.copy().astype(bool), "language_features": z.copy()}


def test_upper_bound_holds_on_dense_50k_text(engine):
    """Dense U(0,1) text at V = 50 000: 782 k-blocks of truncating fp32 accumulation and 50 000
    non-zero products per pair -- the regime the flat 2^-18 allowance of round 1 did not cover."""
    rng = np.random.default_rng(5)
    n, v = 256, 50_000
    text = sp.csr_matrix(rng.random((n, v)))
    w = (0.0, 1.0, 0.0)
    u, exact, sl, a = _upper_bound_tile(engine, _only_text(n, text), w)
    assert np.all(u >= exact), float((exact - u).max())
    # how much of the allowance the hardware uses: accumulated value against the float64 sum of the
    # SAME fp16 operands (isolates the accumulation error from the operand rounding)
    from tvbingefriend_recommendation_service_b200.engine import TEXT_SCALE_LOG2

    tn = normalize_rows(text).toarray()
    op = (tn * 2.0 ** TEXT_SCALE_LOG2).astype(np.float16).astype(np.float64)
    ref = op[:128] @ op[:256].T
    loss = (ref - a) / ref
    budget = 50_000 * sl["w_text_acc"] / sl["w_text"]
    print(f"dense 50k: accumulation loss max {loss.max():.3e} min {loss.min():.3e}, budget {budget:.3e}")
    assert loss.max() <= budget and loss.min() >= -budget


def test_upper_bound_holds_with_subnormal_operands(engine):
    """Rows whose normalised values fall below 2^-22 (fp16 subnormals after the 2^8 scaling): the
    relative bound does not cover them, the per-term absolute allowance must."""
    rng = np.random.default_rng(6)
    n, v = 256, 4096
    dense = rng.random((n, v)) * 1e-7        # tiny values ...
    dense[:, 0] = 1.0                         # ... beside one dominant column: x_k ~ 1e-7 after normalisation
    text = sp.csr_matrix(dense)
    u, exact, sl, a = _upper_bound_tile(engine, _only_text(n, text), (0.0, 1.0, 0.0))
    assert np.all(u >= exact), float((exact - u).max())


def test_upper_bound_holds_on_signed_text(engine):
    """Embedding-like text with negative values: cancellation makes the error large relative to the
    accumulator, so the library must switch to the absolute (Cauchy-Schwarz) bound."""
    rng = np.random.default_rng(7)
    n = 512
    text = sp.csr_matrix(rng.standard_normal((n, 96)))
    u, exact, sl, a = _upper_bound_tile(engine, _only_text(n, text), (0.0, 1.0, 0.0), 128, 256)
    assert sl["w_text_err"] == 0.0 and sl["w_text_acc"] == 0.0
    assert np.all(u >= exact), float((exact - u).max())


@pytest.mark.parametrize("tuning", [SYM_OFF, SYM_ON], ids=["one_sided", "symmetric"])
def test_signed_text_top_k_matches_oracle(engine, tuning):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(1500, 300, nnz=10, seed=8)
    f = cat.features()
    rng = np.random.default_rng(9)
    f["text_features"] = sp.csr_matrix(rng.standard_normal((1500, 64)))
    top = engine.compute_top_k(f, (0.4, 0.5, 0.1), 20, 0.1, tuning=tuning)
    assert_topk_matches(top, f)
    exact = engine.compute_top_k(f, (0.4, 0.5, 0.1), 20, 0.1, force_exact=True)
    assert np.array_equal(top.indices, exact.indices)


def test_dense_text_50k_certified_equals_exact_and_oracle(engine):
    """N = 1 024 shows of dense U(0,1) text at V = 50 000 (all cosines within ~1 % of 0.75): whatever
    the certificate lets through must equal the exact kernel and the float64 oracle."""
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    n, v = 1024, 50_000
    cat = make_catalogue(n, 64, nnz=4, seed=10)
    f = cat.features()
    rng = np.random.default_rng(11)
    dense = rng.random((n, v))
    f["text_features"] = sp.csr_matrix(dense)
    w = (0.4, 0.5, 0.1)
    top = engine.compute_top_k(f, w, 20, 0.1)
    exact = engine.compute_top_k(f, w, 20, 0.1, force_exact=True)
    assert np.array_equal(top.indices, exact.indices) and np.array_equal(top.counts, exact.counts)
    m = top.indices >= 0
    assert np.array_equal(top.hybrid[m], exact.hybrid[m])
    # float64 oracle with dense BLAS (the CSR product of 51 M entries would take minutes)
    tn = dense / np.sqrt((dense * dense).sum(axis=1))[:, None]
    g = normalize_rows(f["genre_features"])
    ms_ = [normalize_rows(f[k_]) for k_ in ("platform_features", "type_features", "language_features")]
    h = w[0] * (g @ g.T) + w[1] * (tn @ tn.T) + w[2] * (sum(m_ @ m_.T for m_ in ms_) / 3)
    np.fill_diagonal(h, -1.0)
    order = np.argsort(-h, axis=1, kind="stable")[:, :20]
    ref_scores = np.take_along_axis(h, order, axis=1)
    got_scores = np.where(m, top.hybrid, 0.0)
    assert np.abs(got_scores - ref_scores).max() < 1e-12
    gaps_ok = np.all(np.abs(np.diff(np.take_along_axis(h, np.argsort(-h, axis=1)[:, :21], axis=1), axis=1)) > 1e-10, axis=1)
    assert gaps_ok.mean() > 0.9
    assert np.array_equal(top.indices[gaps_ok], order[gaps_ok].astype(np.int32))


def test_long_k_moderately_dense_text(engine):
    """V = 50 000 with ~2 000 terms per show: long K (782 k-blocks), rows two orders of magnitude
    denser than TF-IDF, candidate pass still discriminating."""
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(1536, 50_000, nnz=2000, seed=12)
    w = (0.4, 0.5, 0.1)
    top = engine.compute_top_k(cat.features(), w, 20, 0.1)
    exact = engine.compute_top_k(cat.features(), w, 20, 0.1, force_exact=True)
    assert np.array_equal(top.indices, exact.indices) and np.array_equal(top.counts, exact.counts)
    assert top.flagged_rows < 1536      # the certificate still passes rows (not everything repaired)
    assert_topk_matches(top, cat.features(), np.arange(0, 1536, 24), w, 20, 0.1)


# ---- scripts/compute_similarities.main against the reference class' golden statistics ----------------------
@pytest.mark.parametrize("streaming", [False, True], ids=["matrices", "streaming"])
def test_compute_similarities_main_matches_golden_statistics(engine, tmp_path, caplog, streaming):
    """The driver of reference scripts/compute_similarities.py:180-262 on the files of the golden
    catalogue: with the N x N matrices (small catalogue) and with ``--max-matrix-bytes 0``, which
    forces the streaming statistics that large catalogues get (no N x N anywhere)."""
    import logging

    from tvbingefriend_recommendation_service_b200.scripts import compute_similarities as cs

    z, cat = load_golden("similarity_computer_n64")
    cat.save(tmp_path)
    gw, tw, mw = z["w1_weights"].tolist()
    argv = ["--input-dir", str(tmp_path), "--output-dir", str(tmp_path / "out"), "--genre-weight", str(gw),
            "--text-weight", str(tw), "--metadata-weight", str(mw)]
    with caplog.at_level(logging.INFO):
        sims = cs.main(argv + (["--max-matrix-bytes", "0"] if streaming else []))
    names = ("genre_similarity", "text_similarity", "metadata_similarity", "hybrid_similarity")
    if streaming:
        assert all(sims[name] is None for name in names)
        stats = sims["statistics"]
    else:
        from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

        comp = SimilarityComputer(gw, tw, mw, engine=engine)
        stats = {name: comp.get_similarity_statistics(sims[name]) for name in names}
        for name in names:
            assert np.abs(sims[name] - z[f"w1_{name}"]).max() < 1e-12
    for name in names:
        want = dict(zip(("mean", "std", "min", "max", "median"), z[f"w1_{name}_stats"].tolist()))
        got = stats[name]
        for key in ("mean", "std", "min", "max"):
            assert got[key] == pytest.approx(want[key], rel=1e-6, abs=2e-7), (name, key)
        res = got.get("median_resolution", 0.0) * 1.01 + 1e-12
        assert abs(got["median"] - want["median"]) <= res, (name, got["median"], want["median"])
        assert f"{name}:" in caplog.text       # the reference logs the five statistics per matrix (:119-131)
    assert not (tmp_path / "out").exists()     # nothing saved unless --save-similarities


# ---- device-side ingest (SURVEY.md section 8f-3) -----------------------------------------------------------
def test_ingest_equals_host_staging(engine):
    """Raw arrays classified / narrowed / packed on the GPU == the host-staged catalogue, for the dtypes
    compute_features.py writes and the variations numpy / scipy can hand over."""
    from tvbingefriend_recommendation_service_b200.engine import stage
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(2500, 700, nnz=15, seed=21)
    base = cat.features()
    ref = engine.upload(stage(base, "mean3"))
    variants = {"as written": base}
    v2 = dict(base)
    v2["genre_features"] = base["genre_features"].astype(np.float32)
    v2["platform_features"] = base["platform_features"].astype(np.int32)
    v2["type_features"] = base["type_features"].astype(np.uint8)
    t = base["text_features"].astype(np.float32).astype(np.float64)      # values exactly representable in fp32
    v2["text_features"] = sp.csr_matrix((t.data.astype(np.float32), t.indices.astype(np.int64), t.indptr.astype(np.int64)),
                                        shape=t.shape)
    base32 = dict(base)
    base32["text_features"] = t
    ref32 = engine.upload(stage(base32, "mean3"))
    variants["other dtypes"] = v2
    for name, f in variants.items():
        dc = engine.ingest(f, "mean3")
        want = ref if name == "as written" else ref32
        for i in (0, 1, 2, 3, 4, 5):          # indptr, indices, values, operand, col_side, meta_scale
            a, b = dc.keep[i].cpu().numpy(), want.keep[i].cpu().numpy()
            assert a.dtype == b.dtype and np.array_equal(a, b), (name, i)
        assert dc.c.text_signed == 0 and not dc.folded


def test_ingest_falls_back_for_inputs_the_packed_path_cannot_take(engine):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(900, 300, nnz=10, seed=22)
    f = cat.features()
    # (1) a genre value that is not 0/1 -> general float path (folded into the operand)
    g = dict(f)
    g["genre_features"] = f["genre_features"].astype(np.float64)
    g["genre_features"][5, 3] = 0.5
    dc = engine.ingest(g, "mean3")
    assert dc.folded
    assert_topk_matches(engine.compute_top_k(g, (0.4, 0.5, 0.1), 20, 0.1), g)
    # (2) two ones in a one-hot row -> general float path
    m = dict(f)
    m["platform_features"] = f["platform_features"].copy()
    m["platform_features"][7, :2] = 1.0
    assert engine.ingest(m, "mean3").folded
    assert_topk_matches(engine.compute_top_k(m, (0.4, 0.5, 0.1), 20, 0.1), m)
    # (3) CSR with unsorted indices and duplicates -> canonicalised on the host, same table
    t = f["text_features"].tocoo()
    rng = np.random.default_rng(3)
    perm = rng.permutation(t.nnz)
    rows, cols, vals = t.row[perm], t.col[perm], t.data[perm]
    rows = np.concatenate([rows, rows[:50]])
    cols = np.concatenate([cols, cols[:50]])
    vals = np.concatenate([vals * 1.0, np.zeros(50)])
    order = np.argsort(rows, kind="stable")
    indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=900))])
    messy = sp.csr_matrix((vals[order], cols[order], indptr), shape=t.shape)
    assert not messy.has_canonical_format
    u = dict(f)
    u["text_features"] = messy
    a = engine.compute_top_k(u, (0.4, 0.5, 0.1), 20, 0.1)
    b = engine.compute_top_k(f, (0.4, 0.5, 0.1), 20, 0.1)
    assert np.array_equal(a.indices, b.indices) and np.allclose(a.hybrid[a.indices >= 0], b.hybrid[b.indices >= 0], rtol=1e-14)
    # (4) negative text values are detected on the device
    s_ = dict(f)
    s_["text_features"] = sp.csr_matrix(np.random.default_rng(4).standard_normal((900, 48)))
    assert engine.ingest(s_, "mean3").c.text_signed == 1


# ---- float32 inputs (sklearn's dtype rule, SURVEY.md section 3.6 ii) ---------------------------------------
def test_float32_inputs_follow_sklearns_dtype_rule(engine):
    """With every input float32 the reference computes in float32 and returns float32 matrices; the
    drop-in computes in float64 and returns float32: values within 1e-6 of the reference's float32
    run (its own rounding), top-k equal under the comparator at that tolerance."""
    from oracle.cosine import cosine_similarity
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(700, 400, nnz=12, seed=33)
    f = cat.features()
    f32 = {"genre_features": f["genre_features"].astype(np.float32),
           "text_features": f["text_features"].astype(np.float32),
           "platform_features": f["platform_features"].astype(np.float32),
           "type_features": f["type_features"].astype(np.float32),
           "language_features": f["language_features"].astype(np.float32)}
    comp = SimilarityComputer(engine=engine)
    g = comp.compute_genre_similarity(f32["genre_features"])
    t = comp.compute_text_similarity(f32["text_features"])
    m = comp.compute_metadata_similarity(f32["platform_features"], f32["type_features"], f32["language_features"])
    for got, ref in ((g, cosine_similarity(f32["genre_features"])), (t, cosine_similarity(f32["text_features"])),
                     (m, cosine_similarity(np.hstack([f32["platform_features"], f32["type_features"],
                                                      f32["language_features"]])))):
        assert got.dtype == np.float32 and ref.dtype == np.float32
        assert np.abs(got.astype(np.float64) - ref.astype(np.float64)).max() < 2e-6
    assert comp.compute_genre_similarity(f["genre_features"]).dtype == np.float64     # mixed / float64 -> float64
    # top-k from float32 features: the float32 values are promoted exactly, scores are float64
    top = comp.compute_top_k(f32, k=20, min_similarity=0.1)
    f64 = {k_: (v.astype(np.float64) if not sp.issparse(v) else sp.csr_matrix(v, dtype=np.float64)) for k_, v in f32.items()}
    assert_topk_matches(top, f64)


# ---- multi-hot genres with 64 < G <= 128: two mask words (SURVEY.md section 3.5 "design for G up to 128") ----
@pytest.mark.parametrize("tuning", [SYM_OFF, SYM_ON], ids=["one_sided", "symmetric"])
@pytest.mark.parametrize("g", [65, 100, 128])
def test_wide_genre_masks(engine, g, tuning):
    from tvbingefriend_recommendation_service_b200.engine import stage
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(1800, 600, nnz=14, n_genres=g, seed=100 + g)
    f = cat.features()
    w = (0.4, 0.5, 0.1)
    dc = engine.ingest(f, "mean3", w)
    assert not dc.folded and dc.c.genre_hi            # packed: nothing folded into the operand
    top = engine.compute_top_k(f, w, 20, 0.1, tuning=tuning)
    assert_topk_matches(top, f)
    exact = engine.compute_top_k(f, w, 20, 0.1, force_exact=True)
    assert np.array_equal(top.indices, exact.indices) and np.array_equal(top.counts, exact.counts)
    m = top.indices >= 0
    assert np.array_equal(top.hybrid[m], exact.hybrid[m])
    # host-staged path packs the same words
    ref = engine.upload(stage(f, "mean3"), w)
    assert np.array_equal(dc.keep[4].cpu().numpy(), ref.keep[4].cpu().numpy())
    hi_a = dc.keep[6].cpu().numpy()
    bits = f["genre_features"][:, 64:].astype(np.uint64)
    want = (bits << np.arange(bits.shape[1], dtype=np.uint64)[None, :]).sum(axis=1).astype(np.uint64)
    assert np.array_equal(hi_a[:1800].view(np.uint64), want) and not hi_a[1800:].any()
    # single-show query and hstack / normalised conventions on the same catalogue
    q = engine.exact_rows(engine.ingest(f, "hstack", w), [3, 77, 1500], w, k=10, min_similarity=0.0)
    from oracle.reference_paths import ProductionRows
    pr = ProductionRows(f, *w, metadata_mode="hstack")
    for r, i in enumerate([3, 77, 1500]):
        h = pr.row(i)[0]
        h[i] = -1.0
        assert np.allclose(np.sort(h)[::-1][:10], q.hybrid[r], rtol=1e-12)


# ---- packed groups folded into the operand (small vocabularies) ---------------------------------------------
FOLD_CASES = [((0.4, 0.5, 0.1), "mean3", 40), ((21.0, 5.0, 6.0), "mean3", 21), ((0.3, 0.6, 0.1), "hstack", 40),
              ((0.5, 0.5, 0.0), "mean3", 100)]


@pytest.mark.parametrize("weights,mode,genres", FOLD_CASES, ids=["default", "raw_21_5_6", "hstack", "g100_no_meta"])
def test_upper_bound_holds_with_folded_bits(engine, weights, mode, genres):
    """tvbf_features.bits_folded: the accumulator over text + genre + metadata columns, inflated by the
    library's own slack, bounds the exact hybrid of every pair of the tile -- and tightly."""
    from oracle.reference_paths import ProductionRows
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(1024, 500, nnz=15, n_genres=genres, seed=51)
    f = cat.features()
    dc = engine.ingest(f, mode, weights)
    feats = engine._folded(dc, *[float(w) for w in weights], 20)
    assert feats is not None and feats.bits_folded == 1 and feats.k_pad == (500 + genres + 32 + 63) // 64 * 64
    sl = engine.debug_slack(dc, weights, feats=feats)
    a = engine.debug_gemm_tile(dc, 128, 256, feats=feats).cpu().numpy().astype(np.float64)
    pr = ProductionRows(f, *weights, metadata_mode=mode)
    exact = pr.rows_block(np.arange(128, 256))[0][:, 256:512]
    terms = (np.diff(sp.csr_matrix(f["text_features"]).indptr)[128:256] + genres + 3).astype(np.float64)[:, None]
    u = (sl["w_text"] + sl["w_text_err"] + terms * sl["w_text_acc"]) * a + sl["eps"] + terms * sl["eps_term"]
    assert np.all(u >= exact), float((exact - u).max())
    assert float((u - exact).max()) <= 2.5e-3 * sum(weights), float((u - exact).max())


@pytest.mark.parametrize("weights,mode,genres", FOLD_CASES, ids=["default", "raw_21_5_6", "hstack", "g100_no_meta"])
@pytest.mark.parametrize("tuning", [SYM_OFF, SYM_ON], ids=["one_sided", "symmetric"])
def test_folded_bits_give_the_same_table(engine, tuning, weights, mode, genres):
    """The folded candidate pass changes which pairs are rescored, never the certified result: the table
    equals the one of the popcount epilogue bit for bit, and the oracle's."""
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    cat = make_catalogue(3000, 400, nnz=12, n_genres=genres, seed=52)
    f = cat.features()
    ms = 0.1 * sum(weights)
    engine._fold_owner = None
    fold = engine.compute_top_k(f, weights, 20, ms, metadata_mode=mode, tuning=tuning)
    assert engine._fold_owner is not None, "the folded operand was not used"
    old = engine.fold_max_k
    engine.fold_max_k = 0
    try:
        plain = engine.compute_top_k(f, weights, 20, ms, metadata_mode=mode, tuning=tuning)
    finally:
        engine.fold_max_k = old
    for name in ("indices", "counts", "hybrid", "genre", "text", "metadata"):
        assert np.array_equal(getattr(fold, name), getattr(plain, name), equal_nan=True), name
    assert_topk_matches(fold, f, np.arange(0, 3000, 7), weights=weights, min_similarity=ms, metadata_mode=mode)


def test_folded_operand_follows_the_weights_and_the_catalogue(engine):
    """One device catalogue, several weight triples and a second catalogue in between: the folded
    columns are rewritten per triple, and a catalogue whose buffer was taken over rebuilds it."""
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    a, b = make_catalogue(2000, 300, nnz=10, seed=53), make_catalogue(2000, 300, nnz=10, seed=54)
    ca, cb = engine.ingest(a.features()), engine.ingest(b.features())
    rows = np.arange(0, 2000, 9)
    for w in ((0.4, 0.5, 0.1), (0.6, 0.3, 0.1), (0.4, 0.5, 0.1)):
        ta = engine.to_host(engine.top_k_device(ca, w, 20, 0.1))
        tb = engine.to_host(engine.top_k_device(cb, w, 20, 0.1))
        assert ca.fold is not None and cb.fold is not None
        assert_topk_matches(ta, a.features(), rows, weights=w)
        assert_topk_matches(tb, b.features(), rows, weights=w)


# ---- the threshold seed pass (per-row score histograms) ------------------------------------------------------
@pytest.mark.parametrize("vocab,mode", [(400, "folded_wide"), (6000, "popcount"), (6000, "merged")],
                         ids=["folded_wide", "popcount", "merged"])
def test_seeded_thresholds_are_lower_bounds_of_the_final_ones(engine, vocab, mode):
    """A seeded threshold must not exceed the K'-th best UPPER BOUND of the show over all columns (then
    nothing that belongs in the candidate list is ever dropped).  On the catalogue's own operand the
    bound is the exact hybrid inflated by the slack, so the K'-th best exact hybrid, inflated, is at
    least the seed.  Over the merged text operand the bound uses the merged text dot, which may exceed
    the exact cosine: the seed may then exceed the K'-th exact hybrid, never the K'-th merged bound.
    And the seed is useful (above min_similarity for almost every show)."""
    import torch

    from test_merge_plan import merged_dense
    from tvbingefriend_recommendation_service_b200.engine import stage
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    n, w, k, ms = 9000, (0.4, 0.5, 0.1), 20, 0.1
    cat = make_catalogue(n, vocab, nnz=15, seed=61)
    f = cat.features()
    old = engine.merge_ratio
    if mode == "popcount":
        engine.merge_ratio = 0.0           # at V = 6 000 the default merges the text and folds the groups
    try:
        dc = engine.upload(stage(f), w)
        theta = engine.sym_seed(dc, w, k, ms, 0, 1)
        torch.cuda.synchronize()
        plan = engine.plan_tiles(dc, w, k, ms)
        col_map = None if mode != "merged" else engine._fold_owner["plan"]["col_map"].cpu().numpy()
    finally:
        engine.merge_ratio = old
    assert plan["folded_bits"] == (mode != "popcount")
    assert plan["text_cols"] == (4024 if mode == "merged" else 0)
    th = theta.view(torch.float32)[:n].cpu().numpy().astype(np.float64)
    assert np.isfinite(th).all() and (th > ms * 0.99).mean() > 0.9
    kp = 32                                   # candidates kept for k = 20
    pr = ProductionRows(f, *w)
    rows = np.arange(0, n, 150)
    h, g, _, md = pr.rows_block(rows)
    if mode == "merged":
        x = pr.T
        xm = merged_dense(x[rows], col_map, 4024)
        slot = sp.csr_matrix((np.ones(vocab), (np.arange(vocab), col_map)), shape=(vocab, 4024))
        h = w[0] * g + w[1] * np.asarray((x @ slot) @ xm.T).T + w[2] * md
    h[np.arange(len(rows)), rows] = -1.0      # a show is not its own candidate
    kth = -np.sort(-h, axis=1)[:, kp - 1]
    assert np.all(th[rows] <= kth * (1 + 3e-3) + 1e-4), float((th[rows] - kth).max())
