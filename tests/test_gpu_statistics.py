"""Similarity statistics and the N x N variant against float64 models (``-m gpu``).

A. The streaming statistics (``similarity_stats``, ``compute_similarity_statistics``): no N x N
   matrix exists on the device; the results are compared with numpy statistics of the float64
   model matrices.  The text and hybrid maxima must be the float64 maxima bit for bit (also when
   many pairs share the largest fp16 element value), mean and std hold to the precision the
   docstring states, min is an exact 0.0 whenever an element is zero and the median lies within one
   histogram bin.  Signed text and N < 2 are refused.
B. The N x N variant (``cosine_matrix``, ``hybrid_combine``, ``matrix_stats``, ``matrix_rows_topk``)
   against numpy on the same matrices, at the tile edges of the kernels.
"""

import ctypes as C
import logging

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
TEXT_SCALE = 2.0 ** 8          # engine.TEXT_SCALE_LOG2: the operand holds x * 2^8
NAMES = ("genre_similarity", "text_similarity", "metadata_similarity", "hybrid_similarity")


# ---------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def engine():
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


def features(text, genre=None, meta_codes=None, seed=0):
    """A features dict around a text CSR: binary genres and one-hot metadata (the codes of the
    platform, type and language columns; -1 leaves a row all zero)."""
    rng = np.random.default_rng(seed)
    n = text.shape[0]
    if genre is None:
        genre = (rng.random((n, 12)) < 0.25).astype(np.int64)
    if meta_codes is None:
        meta_codes = [rng.integers(0, k, n) for k in (4, 3, 2)]

    def one_hot(codes, k):
        out = np.zeros((n, k))
        ok = codes >= 0
        out[np.nonzero(ok)[0], codes[ok]] = 1.0
        return out

    p, t, la = (one_hot(np.asarray(c), k) for c, k in zip(meta_codes, (4, 3, 2)))
    return {"genre_features": np.asarray(genre, dtype=np.int64), "text_features": sp.csr_matrix(text),
            "platform_features": p, "type_features": t.astype(bool), "language_features": la}


def random_text(rng, n, v, nnz, col0=0):
    rows = np.repeat(np.arange(n), nnz)
    cols = col0 + np.concatenate([rng.choice(v, nnz, replace=False) for _ in range(n)])
    return sp.csr_matrix((rng.random(n * nnz) + 0.05, (rows, cols)), shape=(n, col0 + v))


def model_matrices(f, weights, mode="mean3", normalize_weights=False):
    """The four float64 similarity matrices of the reference arithmetic."""
    from oracle.reference_paths import ProductionRows

    pr = ProductionRows(f, *weights, metadata_mode=mode, normalize_weights=normalize_weights)

    def gram(x):
        x = x.toarray() if sp.issparse(x) else np.asarray(x, dtype=np.float64)
        return x @ x.T

    g, t = gram(pr.G), gram(pr.T)
    md = sum(gram(m) for m in pr.M) / 3 if mode == "mean3" else gram(pr.M[0])
    return {"genre_similarity": g, "text_similarity": t, "metadata_similarity": md,
            "hybrid_similarity": pr.gw * g + pr.tw * t + pr.mw * md}, (pr.gw, pr.tw, pr.mw)


def model_stats(mat):
    from oracle.reference_paths import SimilarityComputerOracle

    return SimilarityComputerOracle.get_similarity_statistics(mat)


def score_pairs(engine, cat, weights, pairs):
    """``tvbf_score_pairs``: float64 [n, 4] (hybrid, genre, text, metadata)."""
    import torch

    from tvbingefriend_recommendation_service_b200._lib import check

    pk = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
    p = engine._params(cat, weights, 20, 0.5)
    with torch.cuda.device(engine.device):
        pd = torch.from_numpy(pk).to(engine.device)
        out = torch.empty((pk.shape[0], 4), dtype=torch.float64, device=engine.device)
        check(engine.lib.tvbf_score_pairs(C.byref(cat.c), C.byref(p), pd.data_ptr(), pk.shape[0], out.data_ptr(),
                                          engine._stream()), "tvbf_score_pairs")
        return out.cpu().numpy()


def assert_exact_maxima(engine, cat, weights, got, mats):
    """text / hybrid max: the float64 model's maximum, and bit for bit the ``tvbf_score_pairs`` score
    of the best pair (every pair within 1e-12 of the model's maximum is scored)."""
    iu = np.triu_indices(cat.n_shows, 1)
    for name, col in (("text_similarity", 2), ("hybrid_similarity", 0)):
        ut = mats[name][iu]
        top = np.nonzero(ut >= ut.max() - 1e-12)[0]
        exact = score_pairs(engine, cat, weights, np.stack([iu[0][top], iu[1][top]], axis=1))[:, col].max()
        assert got[name]["max"] == exact, (name, got[name]["max"], exact)
        assert got[name]["max"] == pytest.approx(ut.max(), rel=1e-15, abs=1e-15), name


def tied_group(n_members, center, member_cols, anchor_col):
    """Text rows of one fp16-tied group: the anchor {anchor_col: 1} and members
    {anchor_col: u_j, member_cols[j]: sqrt(1 - u_j^2)}, u_j increasing inside the fp16 rounding
    interval of ``center`` * 2^8 (the text element value of (anchor, member j) is fp16(u_j 2^8) / 2^8)."""
    c16 = float(np.float16(center * TEXT_SCALE))
    step = float(np.spacing(np.float16(c16)))
    u = np.linspace(c16 - 0.45 * step, c16 + 0.45 * step, n_members) / TEXT_SCALE
    rows = [{anchor_col: 1.0}] + [{anchor_col: uj, int(cj): float(np.sqrt(1.0 - uj * uj))}
                                   for uj, cj in zip(u, member_cols)]
    return rows, u


def csr_from_rows(rows, v):
    r, c, d = [], [], []
    for i, row in enumerate(rows):
        for col, val in sorted(row.items()):
            r.append(i), c.append(col), d.append(val)
    return sp.csr_matrix((d, (r, c)), shape=(len(rows), v))


def assert_premise_one_fp16(u):
    """The normalised text values of the members all round to ONE fp16 operand entry."""
    assert np.unique((np.asarray(u) * TEXT_SCALE).astype(np.float16)).size == 1
    assert np.unique(u).size == len(u)


# ---------------------------------------------------------------------------------------------- A1
@pytest.mark.parametrize("mode", ["mean3", "hstack"])
def test_fp16_tied_maxima_are_exact(engine, mode):
    """Show 0 = {c0: 1}; shows 1..200 = {c0: u_j, c_(1+j): sqrt(1 - u_j^2)} with u_j increasing inside
    one fp16 rounding interval around 0.9; identical genres and metadata everywhere, so the hybrid
    follows the text; 3 000 filler shows on a disjoint vocabulary score low.  Every (0, j) has the
    same fp16 element value, so the warp that sees row 0 keeps whichever it met first; the maximum
    is (0, 200)."""
    from oracle.reference_paths import ProductionRows

    rng = np.random.default_rng(5)
    n_fill, v_fill = 3000, 4000
    rows, u = tied_group(200, 0.9, np.arange(1, 201), 0)
    tied = csr_from_rows(rows, 201 + v_fill)
    fill = random_text(rng, n_fill, v_fill, 12, col0=201)
    text = sp.vstack([tied, fill]).tocsr()
    n = text.shape[0]
    pr = ProductionRows({"genre_features": np.ones((n, 1)), "text_features": text,
                         "platform_features": np.ones((n, 1)), "type_features": np.ones((n, 1)),
                         "language_features": np.ones((n, 1))})
    un = pr.T[1:201, 0].toarray().ravel()
    assert_premise_one_fp16(un)
    assert pr.T[0, 0] == 1.0 and np.all(np.diff(un) > 0)
    f = features(text, genre=np.ones((n, 3), np.int64), meta_codes=[np.zeros(n, int)] * 3)
    cat = engine.ingest(f, mode, W)
    got = engine.similarity_stats(cat, W)
    mats, w = model_matrices(f, W, mode)
    assert mats["text_similarity"][0, 200] == mats["text_similarity"][np.triu_indices(n, 1)].max() == un[-1]
    best = score_pairs(engine, cat, w, [(0, 200)])[0]
    assert got["text_similarity"]["max"] == best[2] == un[-1]
    assert got["hybrid_similarity"]["max"] == best[0]
    assert best[0] == pytest.approx(mats["hybrid_similarity"][0, 200], rel=1e-15)
    assert_exact_maxima(engine, cat, w, got, mats)


# ---------------------------------------------------------------------------------------------- A2
def planted_catalogue(seed, n, groups):
    """Random catalogue (text on columns >= 2 000) with fp16-tied groups planted: group g = (anchor
    row, member rows, center); its anchor column and the members' private columns lie below 2 000.
    Group members copy the anchor's genres and metadata.  Returns (features, [u of each group])."""
    rng = np.random.default_rng(seed)
    v_fill = 3000
    base = random_text(rng, n, v_fill, 10, col0=2000).tolil()
    genre = (rng.random((n, 12)) < 0.25).astype(np.int64)
    codes = [rng.integers(0, k, n) for k in (4, 3, 2)]
    col = 0
    us = []
    for anchor, members, center in groups:
        rows, u = tied_group(len(members), center, range(col + 1, col + 1 + len(members)), col)
        us.append(u)
        col += 1 + len(members)
        for r, row in zip([anchor, *members], rows):
            base.rows[r], base.data[r] = list(row), [row[c] for c in row]
            genre[r] = genre[anchor]
            for c in codes:
                c[r] = c[anchor]
    return features(base.tocsr(), genre=genre, meta_codes=codes), us


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("mode,norm", [("mean3", False), ("hstack", True)])
def test_randomised_fp16_ties_in_every_tile(engine, seed, mode, norm):
    """Groups of fp16-tied pairs in different 256-row tiles and in the last, partial tile (N is not
    a multiple of 256), with the members spread over the catalogue; the largest group center is
    the maximum of the text and of the hybrid."""
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    rng = np.random.default_rng(100 + seed)
    n = 256 * int(rng.integers(6, 11)) + int(rng.integers(1, 255))
    last_tile = n // 256 * 256
    perm = rng.permutation(n)
    groups, used = [], 0
    anchors = [int(rng.integers(0, 256)), int(rng.integers(256, 512)), int(rng.integers(last_tile, n))]
    for g, anchor in enumerate(anchors):
        members = [int(x) for x in perm[used:used + 40] if x not in anchors][:30]
        used += 40
        groups.append((anchor, members, 0.97 - 0.01 * (g != seed % 3) * (g + 1)))
    f, us = planted_catalogue(seed, n, groups)
    for u in us:
        assert_premise_one_fp16(u)
    weights = (1.0, 2.0, 0.5) if not norm else (0.3, 0.6, 0.1)
    got = SimilarityComputer(*weights, engine=engine).compute_similarity_statistics(f, mode, norm)
    mats, w = model_matrices(f, weights, mode, norm)
    assert_exact_maxima(engine, engine.ingest(f, mode, w), w, got, mats)


# ---------------------------------------------------------------------------------------------- A3 / A4
def _catalogue(kind, n, rng):
    v = 300
    text = random_text(rng, n, v, min(8, v))
    f = features(text, seed=int(rng.integers(1 << 30)))
    if kind == "empty_text_rows":
        t = f["text_features"].tolil()
        for r in range(0, n, 3):
            t.rows[r], t.data[r] = [], []
        f["text_features"] = t.tocsr()
    elif kind == "zero_genre_rows":
        f["genre_features"][::2] = 0
    elif kind == "zero_metadata_rows":
        for key in ("platform_features", "type_features", "language_features"):
            f[key][1::3] = 0
    elif kind == "no_text_entries":
        f["text_features"] = sp.csr_matrix((n, 5))
    return f


CASES = [(kind, n) for kind in ("random", "empty_text_rows", "zero_genre_rows", "zero_metadata_rows",
                                "no_text_entries") for n in (2, 3, 257, 3000)]


@pytest.mark.parametrize("weights", [(0.0, 1.0, 0.0), (1.0, 0.0, 0.0), (0.3, 0.6, 0.1)])
@pytest.mark.parametrize("kind,n", CASES)
def test_moments_min_max_median_against_float64(engine, kind, n, weights):
    """mean / std: text and hybrid to rel 1e-9 (exact float64 moments), genre and metadata to rel
    1e-8 (fp32 elements summed in float64); max exact; min an exact 0.0 whenever the model has a
    zero; median within one bin (odd pair counts at N = 2, 3, even ones at 257 and 3 000)."""
    rng = np.random.default_rng(n * 7 + len(kind))
    f = _catalogue(kind, n, rng)
    cat = engine.ingest(f, "hstack", weights)
    got = engine.similarity_stats(cat, weights)
    mats, w = model_matrices(f, weights, "hstack")
    iu = np.triu_indices(n, 1)
    for name in NAMES:
        ref, g = model_stats(mats[name]), got[name]
        rel = 1e-9 if name in ("text_similarity", "hybrid_similarity") else 1e-8
        assert g["exact_moments"] == {"text_mean": True, "text_std": True}, name
        assert g["mean"] == pytest.approx(ref["mean"], rel=rel, abs=1e-15), name
        # one-pass variance: sum(x^2) over the strict upper triangle is (all pairs - diagonal) / 2
        # and the variance sum(x^2) / count - mean^2; a few ulps of those sums survive the
        # cancellations when the elements (nearly) agree, so std has an absolute floor of
        # ~2^-26 sqrt(rms^2 + 2 / (N - 1)) (N = 2: one element, std 0)
        rms2 = ref["mean"] ** 2 + ref["std"] ** 2
        floor = 4 * 2.0 ** -26 * float(np.sqrt(rms2 + 2.0 / (n - 1)))
        assert g["std"] == pytest.approx(ref["std"], rel=rel, abs=floor), name
        if (mats[name][iu] == 0.0).any():
            assert g["min"] == 0.0, name
        else:
            assert g["min"] == pytest.approx(ref["min"], abs=1e-6), name
        assert g["max"] == pytest.approx(ref["max"], abs=1e-6), name
        assert abs(g["median"] - ref["median"]) <= g["median_resolution"] * 1.01, (name, g["median"], ref["median"])
    assert_exact_maxima(engine, cat, w, got, mats)


def test_median_is_zero_when_most_pairs_are_zero(engine):
    """Every show has its own text column and genre: more than half of the text and genre pairs
    (all of them) are zero, so min and median are exactly 0.0."""
    n = 301
    text = sp.csr_matrix((np.ones(n), (np.arange(n), np.arange(n))), shape=(n, n))
    genre = np.zeros((n, 40), np.int64)
    genre[np.arange(n), np.arange(n) % 40] = 1
    genre[: n // 2, 0] = 1      # still more than half of the genre pairs share nothing
    f = features(text, genre=genre)
    got = engine.similarity_stats(engine.ingest(f, "hstack", W), W)
    mats, _ = model_matrices(f, W, "hstack")
    for name in ("text_similarity", "genre_similarity"):
        ref = model_stats(mats[name])
        assert ref["median"] == 0.0
        assert got[name]["median"] == 0.0 and got[name]["min"] == 0.0, name
    assert got["text_similarity"]["max"] == 0.0 and got["text_similarity"]["mean"] == 0.0


def test_text_std_without_the_gram_matrix(engine):
    """gram_bytes_limit=0: no [V, V] Gram matrix, so text_std comes from the fp16 sweep: flagged as
    not exact, within the ~1e-5 DESIGN.md section 8 documents."""
    rng = np.random.default_rng(9)
    f = features(random_text(rng, 3000, 2048, 30))
    cat = engine.ingest(f, "hstack", W)
    got = engine.similarity_stats(cat, W, gram_bytes_limit=0)
    mats, _ = model_matrices(f, W, "hstack")
    for name in ("text_similarity", "hybrid_similarity"):
        assert got[name]["exact_moments"] == {"text_mean": True, "text_std": False}, name
        ref = model_stats(mats[name])
        assert got[name]["mean"] == pytest.approx(ref["mean"], rel=1e-9)
        assert got[name]["std"] == pytest.approx(ref["std"], rel=1e-5)


# ---------------------------------------------------------------------------------------------- A5 / A6
def signed_features(n, seed=3):
    rng = np.random.default_rng(seed)
    f = features(random_text(rng, n, 400, 12), seed=seed)
    t = f["text_features"].copy()
    t.data *= np.where(rng.random(t.nnz) < 0.35, -1.0, 1.0)
    f["text_features"] = t
    return f


def test_signed_text_is_refused_by_the_streaming_statistics(engine):
    from tvbingefriend_recommendation_service_b200._lib import TvbfError
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    f = signed_features(500)
    cat = engine.ingest(f, "hstack", W)
    assert cat.c.text_signed
    with pytest.raises(TvbfError, match="signed text"):
        engine.similarity_stats(cat, W)
    with pytest.raises(TvbfError, match="signed text"):
        SimilarityComputer(engine=engine).compute_similarity_statistics(f)


def _save(f, d):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    d.mkdir(parents=True, exist_ok=True)
    make_catalogue(f["genre_features"].shape[0], 50, nnz=5).save(d)     # shows_metadata.csv and layout
    for key, a in f.items():
        if key == "text_features":
            sp.save_npz(d / "text_features.npz", a)
        else:
            np.save(d / f"{key}.npy", a)


def test_compute_similarities_on_signed_text(engine, tmp_path, caplog, monkeypatch):
    """The streaming branch names the way out (--max-matrix-bytes); the N x N branch takes signed
    text and its statistics (``tvbf_matrix_stats_f64`` on negative values) equal the float64 model."""
    import tvbingefriend_recommendation_service_b200.ml.similarity_computer as scm
    from tvbingefriend_recommendation_service_b200.scripts import compute_similarities as cs

    monkeypatch.setattr(scm, "default_engine", lambda: engine)
    f = signed_features(400)
    _save(f, tmp_path)
    with caplog.at_level(logging.ERROR), pytest.raises(SystemExit):
        cs.main(["--input-dir", str(tmp_path), "--max-matrix-bytes", "0"])
    assert "--max-matrix-bytes" in caplog.text and "negative" in caplog.text
    sims = cs.main(["--input-dir", str(tmp_path)])
    mats, _ = model_matrices(cs.load_features(tmp_path), W, "hstack", normalize_weights=True)
    comp = scm.SimilarityComputer(engine=engine)
    assert mats["text_similarity"][np.triu_indices(400, 1)].min() < 0
    for name in NAMES:
        assert np.abs(sims[name] - mats[name]).max() <= 1e-13, name
        got, ref = comp.get_similarity_statistics(sims[name]), model_stats(mats[name])
        for q in ("mean", "std"):
            assert got[q] == pytest.approx(ref[q], rel=1e-9), (name, q)
        for q in ("min", "max", "median"):
            assert got[q] == pytest.approx(ref[q], abs=1e-13), (name, q)


def test_fewer_than_two_shows(engine):
    from tvbingefriend_recommendation_service_b200._lib import TvbfError
    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

    f = features(sp.csr_matrix(np.array([[0.5, 0.5]])))
    with pytest.raises(ValueError, match="upper triangle"):
        engine.similarity_stats(engine.ingest(f, "hstack", W), W)
    with pytest.raises(ValueError, match="upper triangle"):
        SimilarityComputer(engine=engine).compute_similarity_statistics(f)
    import torch

    with pytest.raises(TvbfError):
        engine.matrix_stats(torch.ones((1, 1), dtype=torch.float64, device=engine.device))


# ---------------------------------------------------------------------------------------------- B1
def _cosine_model(a):
    a = np.asarray(a, dtype=np.float64)
    norms = np.sqrt((a * a).sum(axis=1))
    norms[norms == 0.0] = 1.0
    x = a / norms[:, None]
    return x @ x.T


def _messy_csr(a, rng):
    """The same matrix as a CSR with duplicate entries (values split in two) and unsorted rows."""
    coo = sp.coo_matrix(a)
    half = coo.data * 0.5
    r = np.concatenate([coo.row, coo.row])
    c = np.concatenate([coo.col, coo.col])
    d = np.concatenate([half, coo.data - half])
    order = rng.permutation(r.size)
    order = order[np.argsort(r[order], kind="stable")]          # rows in order, entries shuffled
    indptr = np.concatenate([[0], np.cumsum(np.bincount(r, minlength=a.shape[0]))])
    m = sp.csr_matrix((d[order], c[order], indptr), shape=a.shape)
    assert not m.has_canonical_format or m.nnz == 0
    return m


@pytest.mark.parametrize("dim", [1, 15, 16, 17, 300])
@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 130, 1000])
def test_cosine_matrix_against_numpy(engine, n, dim):
    """Dense (signed values, zero rows), canonical CSR and CSR with duplicates / unsorted entries:
    max |kernel - model| <= (dim + 4) 2^-53 (unit rows: every term and sum by Cauchy-Schwarz)."""
    rng = np.random.default_rng(n * 1000 + dim)
    a = rng.standard_normal((n, dim))
    a[rng.random((n, dim)) < 0.5] = 0.0
    a[::7] = 0.0                                    # zero rows stay zero
    bound = (dim + 4) * 2.0 ** -53
    ref = _cosine_model(a)
    for what, x in (("dense", a), ("csr", sp.csr_matrix(a)), ("messy csr", _messy_csr(a, rng))):
        got = engine.cosine_matrix(x).cpu().numpy()
        assert got.shape == (n, n), what
        assert np.abs(got - ref).max() <= bound, (what, np.abs(got - ref).max())
        assert np.all(got[::7] == 0.0), what


# ---------------------------------------------------------------------------------------------- B2
def test_hybrid_combine_is_bit_identical_to_numpy(engine):
    import torch

    rng = np.random.default_rng(4)
    n = 3000
    g, t, m = (rng.standard_normal((n, n)) for _ in range(3))
    for wg, wt, wm in ((0.4, 0.5, 0.1), (1 / 3, 1 / 3, 1 / 3), (0.0, 1.0, 0.0), (0.3, 0.6, 0.1)):
        dev = [torch.from_numpy(x).to(engine.device) for x in (g, t, m)]
        got = engine.hybrid_combine(*dev, wg, wt, wm).cpu().numpy()
        ref = (wg * g + wt * t) + wm * m
        assert np.array_equal(got.view(np.int64), ref.view(np.int64)), (wg, wt, wm)


# ---------------------------------------------------------------------------------------------- B3
def _stats_cases():
    rng = np.random.default_rng(8)
    cases = {}
    for n in (2, 3, 4, 600, 3001):
        cases[f"random_{n}"] = rng.standard_normal((n, n))
    a = rng.standard_normal((700, 700))
    a[rng.random(a.shape) < 0.3] = 0.0
    a[rng.random(a.shape) < 0.2] = -0.0
    cases["signed_zeros"] = a
    cases["median_duplicates"] = rng.choice([-1.0, 0.25, 0.5, 0.75], size=(801, 801), p=[0.1, 0.2, 0.5, 0.2])
    cases["all_equal"] = np.full((500, 500), 0.375)
    b = rng.random((1000, 1000))
    il = np.tril_indices(1000)
    b[il] = np.where(rng.random(il[0].size) < 0.5, np.nan, 1e300)     # diagonal and lower triangle
    cases["ignored_lower"] = b
    return cases


STATS_CASES = _stats_cases()


@pytest.mark.parametrize("case", sorted(STATS_CASES))
def test_matrix_stats_against_numpy(engine, case):
    """min / max / median bit for bit (the radix select returns elements; (lo + hi) / 2 rounds as
    numpy's median does); mean / std to rel 1e-12."""
    import torch

    mat = STATS_CASES[case]
    ut = mat[np.triu_indices(mat.shape[0], 1)]
    got = engine.matrix_stats(torch.from_numpy(mat).to(engine.device))
    for q, ref in (("min", ut.min()), ("max", ut.max()), ("median", np.median(ut))):
        assert got[q] == float(ref), (case, q, got[q], ref)
    assert got["mean"] == pytest.approx(float(ut.mean()), rel=1e-12, abs=1e-15), case
    assert got["std"] == pytest.approx(float(ut.std()), rel=1e-12, abs=1e-15), case


# ---------------------------------------------------------------------------------------------- B4
def _rows_topk_model(mats, rows, k, min_similarity):
    n = mats["hybrid"].shape[0]
    idx = np.full((len(rows), k), -1, np.int32)
    cnt = np.zeros(len(rows), np.int32)
    sc = {name: np.zeros((len(rows), k)) for name in ("hybrid", "genre", "text", "metadata")}
    cols = np.arange(n)
    for e, r in enumerate(rows):
        h = mats["hybrid"][r]
        keep = (cols != r) & (h >= min_similarity)
        c = cols[keep]
        c = c[np.lexsort((c, -h[c]))][:k]
        cnt[e] = c.size
        idx[e, :c.size] = c
        for name in sc:
            sc[name][e, :c.size] = mats[name][r, c]
    return idx, cnt, sc


def _matrices(n, rng, ties):
    mats = {}
    for name in ("genre", "text", "metadata"):
        m = rng.standard_normal((n, n)) * 0.4
        if ties:
            m = np.round(m * 2) / 4          # a few distinct values: ties far wider than k
        mats[name] = (m + m.T) / 2
    h = (0.4 * mats["genre"] + 0.5 * mats["text"]) + 0.1 * mats["metadata"]
    if ties:
        z = h == 0.0
        h[z] = np.where(rng.random(int(z.sum())) < 0.5, -0.0, 0.0)     # both zeros, one score
    mats["hybrid"] = h
    return mats


@pytest.mark.parametrize("ties", [False, True])
@pytest.mark.parametrize("n", [64, 1000, 5000])
def test_matrix_rows_topk_against_numpy(engine, n, ties):
    """The service's matrix mode: (score desc, index asc), self excluded, score >= min_similarity;
    one row, more rows than 2 x SMs (CTAs loop and reuse their key scratch) and repeated rows;
    k = 1, 20, N - 1 and N + 5 up to the limit of 1 024 (k = 1 025 is refused); a negative
    threshold over negative entries.  With ties the matrices hold -0.0 as well as +0.0: one
    score, ordered by column."""
    import torch

    from tvbingefriend_recommendation_service_b200._lib import TvbfError

    rng = np.random.default_rng(n + ties)
    mats = _matrices(n, rng, ties)
    if ties:
        h = mats["hybrid"]
        assert np.signbit(h[h == 0.0]).any() and (~np.signbit(h[h == 0.0])).any()
    dev = {name: torch.from_numpy(m).to(engine.device) for name, m in mats.items()}
    row_sets = [np.array([n - 1]), rng.integers(0, n, 2 * engine.sm_count + 8),
                np.array([0, 5, 5, 0, n - 1, 5] * 3) % n]
    with pytest.raises(TvbfError, match="exceeds 1024"):
        engine.matrix_rows_topk(dev["hybrid"], dev["genre"], dev["text"], dev["metadata"], [0], 1025)
    for rows in row_sets:
        for k in sorted({1, 20, min(n - 1, 1024), min(n + 5, 1024)}):
            for ms in (0.0, -0.3, 0.2):
                got = engine.matrix_rows_topk(dev["hybrid"], dev["genre"], dev["text"], dev["metadata"], rows, k, ms)
                idx, cnt, sc = _rows_topk_model(mats, rows, k, ms)
                what = (len(rows), k, ms)
                assert np.array_equal(got.counts, cnt), what
                assert np.array_equal(got.indices, idx), what
                valid = np.arange(k)[None, :] < cnt[:, None]
                for name in sc:
                    assert np.array_equal(getattr(got, name)[valid], sc[name][valid]), (what, name)


def test_service_matrix_mode_against_numpy(engine, tmp_path):
    from tvbingefriend_recommendation_service_b200.services.content_based_service import (
        ContentBasedRecommendationService)
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    n = 1000
    rng = np.random.default_rng(12)
    cat = make_catalogue(n, 200, nnz=5, seed=12)
    cat.save(tmp_path)
    mats = _matrices(n, rng, ties=True)
    for name in ("genre", "text", "metadata"):
        np.save(tmp_path / f"{name}_similarity.npy", mats[name])
    gw, tw, mw = 0.3, 0.6, 0.3
    svc = ContentBasedRecommendationService(tmp_path, gw, tw, mw, use_blob=False, engine=engine)
    tot = gw + tw + mw
    mats["hybrid"] = (gw / tot * mats["genre"] + tw / tot * mats["text"]) + mw / tot * mats["metadata"]
    ids = cat.show_ids.tolist()
    for r, k, ms in ((0, 10, 0.0), (n - 1, 25, -0.2), (417, 1, 0.1), (3, n + 5, -1.0)):
        recs = svc.get_recommendations_from_matrix(ids[r], n=k, min_similarity=ms)
        idx, cnt, sc = _rows_topk_model(mats, [r], k, ms)
        assert len(recs) == cnt[0]
        assert [rec["show_id"] for rec in recs] == [ids[i] for i in idx[0, :cnt[0]]]
        for key, name in (("similarity_score", "hybrid"), ("genre_score", "genre"), ("text_score", "text"),
                          ("metadata_score", "metadata")):
            assert [rec[key] for rec in recs] == sc[name][0, :cnt[0]].tolist(), key
