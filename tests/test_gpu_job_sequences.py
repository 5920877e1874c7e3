"""Sequences of jobs through ONE long-lived engine (``-m gpu``).

The other GPU tests upload a fresh catalogue and run one job on it.  A service instead keeps one
engine and streams jobs through it: ``prepare(recycle=...)`` takes over the previous catalogue's
operand (un-scattering its old non-zeros) and its same-shaped buffers, ``h2d(reuse=True)`` cycles
two sets of device buffers, the engine caches one workspace, one fold buffer and one ``theta``,
and libtvbf keeps per-device state for the shared-list clear of the symmetric sweep.  Here every
job of such a sequence is compared with

  (a) the same job on a freshly uploaded catalogue in a second engine (own workspace, nothing
      recycled): indices, counts and the four fp64 score arrays bit-identical, and
  (b) the numpy oracle on a spread of rows, including the last (partial) 256-row tile.

``flagged_rows`` / ``rescored_pairs`` are not compared: the symmetric sweep's threshold refreshes
depend on timing."""

import numpy as np
import pytest
import scipy.sparse as sp

from helpers import assert_topk_matches

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
MS = 0.1
ONE_SIDED, SYMMETRIC = 1 << 20, 2 << 20
NO_SEED = 63 << 22            # symmetric sweep without a threshold seed pass (starts no list clear)


# ---------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def engine():
    """The long-lived engine every sequence runs through."""
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


@pytest.fixture(scope="module")
def fresh():
    """Reference engine: every catalogue uploaded on its own, never recycled."""
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


def catalogue(n, v, nnz=20, seed=0, genres=40, signed=False):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    f = make_catalogue(n, v, nnz=min(nnz, v), n_genres=genres, seed=seed).features()
    if signed:        # embedding-like text: about a third of the values negative
        t = f["text_features"].copy()
        t.data *= np.where(np.random.default_rng(seed + 1).random(t.nnz) < 0.3, -1.0, 1.0)
        f["text_features"] = t
    return f


def rotated(f, shift):
    """Same indptr (same nnz per row), every column index moved by ``shift`` mod V."""
    t = f["text_features"]
    r = sp.csr_matrix((t.data.copy(), (t.indices + shift) % t.shape[1], t.indptr.copy()), shape=t.shape)
    r.sort_indices()
    return dict(f, text_features=r)


def unsorted_csr(f):
    """The same matrix with every row's column indices in descending order (``ingest`` hands such
    a CSR to scipy on the host)."""
    t = f["text_features"]
    idx, dat = t.indices.copy(), t.data.copy()
    for r in range(t.shape[0]):
        b, e = t.indptr[r], t.indptr[r + 1]
        idx[b:e], dat[b:e] = idx[b:e][::-1], dat[b:e][::-1]
    return dict(f, text_features=sp.csr_matrix((dat, idx, t.indptr.copy()), shape=t.shape))


def fractional_genres(f):
    """Non-binary genre weights: the genre group is folded into the operand (``stage`` path)."""
    return dict(f, genre_features=f["genre_features"] * 0.5)


def device_buffers(cat) -> dict:
    """The per-catalogue device buffers the kernels read, by ``tvbf_features`` field."""
    import torch

    by_ptr = {t.data_ptr(): t for t in cat.keep if isinstance(t, torch.Tensor)}
    out = {"operand": cat.operand}
    for name in ("col_side", "meta_scale", "genre_hi", "text_values"):
        ptr = getattr(cat.c, name)
        if ptr:
            out[name] = by_ptr[ptr]
    return out


def assert_same_buffers(got, ref, what=""):
    import torch

    g, r = device_buffers(got), device_buffers(ref)
    assert g.keys() == r.keys(), (what, sorted(g), sorted(r))
    for name in g:
        assert g[name].shape == r[name].shape and g[name].dtype == r[name].dtype, (what, name)
        assert torch.equal(g[name], r[name]), f"{what}: {name} differs from a fresh upload"


def assert_same_tables(got, ref, what=""):
    assert got.indices.shape == ref.indices.shape, what
    assert np.array_equal(got.indices, ref.indices), f"{what}: indices"
    assert np.array_equal(got.counts, ref.counts), f"{what}: counts"
    valid = np.arange(ref.k)[None, :] < ref.counts[:, None]
    for name in ("hybrid", "genre", "text", "metadata"):
        assert np.array_equal(getattr(got, name)[valid], getattr(ref, name)[valid]), f"{what}: {name}"


def spread_rows(begin, end, count=6):
    """Rows of [begin, end) for the oracle: the first, a few inside, the last 256-row tile's first
    row and the last two rows."""
    if end <= begin:
        return np.zeros(0, np.int64)
    last_tile = begin + (end - 1 - begin) // 256 * 256
    rows = np.concatenate([[begin, end - 1, end - 2, last_tile, last_tile + 1],
                           np.linspace(begin, end - 1, count).astype(np.int64)])
    return np.unique(np.clip(rows, begin, end - 1))


def upload(eng, f, how, recycle=None):
    from tvbingefriend_recommendation_service_b200.engine import stage

    if how == "ingest":
        return eng.ingest(f, recycle=recycle)
    if how == "reuse":
        return eng.prepare(eng.h2d(stage(f), reuse=True), W, recycle=recycle)
    return eng.upload(stage(f), W, recycle=recycle)


# ---------------------------------------------------------------------------------------------- 1
CHAINS = {
    # same indptr, column indices rotated mod V: the same nnz at (mostly) other positions
    "rotated_columns": lambda: [catalogue(1000, 500, seed=11), rotated(catalogue(1000, 500, seed=11), 37),
                                rotated(catalogue(1000, 500, seed=11), 250)],
    # 1000 -> 900 shows in the same 1024-row padding: rows 900..999 must come back zero
    "fewer_shows": lambda: [catalogue(1000, 500, seed=12), catalogue(900, 500, seed=13),
                            catalogue(1000, 500, seed=14)],
    # more, then fewer non-zeros: the values buffer is not taken over
    "nnz_changes": lambda: [catalogue(1000, 500, nnz=20, seed=15), catalogue(1000, 500, nnz=30, seed=16),
                            catalogue(1000, 500, nnz=12, seed=17)],
    # second genre mask word handed over, then unused
    "genres_40_100_40": lambda: [catalogue(1000, 500, seed=18), catalogue(1000, 500, seed=19, genres=100),
                                 catalogue(1000, 500, seed=20)],
    "unsigned_to_signed": lambda: [catalogue(1000, 500, seed=21), catalogue(1000, 500, seed=22, signed=True),
                                   catalogue(1000, 500, seed=23)],
    # ingest falls back to stage(): folded genres (other operand shape), unsorted CSR
    "stage_fallbacks": lambda: [catalogue(1000, 500, seed=24), fractional_genres(catalogue(1000, 500, seed=25)),
                                unsorted_csr(catalogue(1000, 500, seed=26)), catalogue(1000, 500, seed=27)],
}


@pytest.mark.parametrize("how", ["upload", "ingest"])
@pytest.mark.parametrize("chain", sorted(CHAINS))
def test_recycled_catalogue_equals_a_fresh_upload(engine, fresh, chain, how):
    prev = None
    for step, f in enumerate(CHAINS[chain]()):
        what = f"{chain} via {how}, step {step}"
        cat = upload(engine, f, how, recycle=prev)
        ref = upload(fresh, f, how)
        assert_same_buffers(cat, ref, what)
        tuning = (SYMMETRIC if step % 2 else ONE_SIDED) if not cat.folded else 0
        got = engine.to_host(engine.top_k_device(cat, W, 20, MS, tuning=tuning))
        assert_same_tables(got, fresh.to_host(fresh.top_k_device(ref, W, 20, MS, tuning=tuning)), what)
        assert_topk_matches(got, f, spread_rows(0, cat.n_shows))
        prev = cat


# ---------------------------------------------------------------------------------------------- 2
def test_recycle_two_reused_h2d_sets_back(engine, fresh):
    """Two-deep pipeline over the two ``h2d(reuse=True)`` buffer sets: c3 is prepared while c2 is
    still in use and recycles c1, whose CSR tensors the h2d of c3 has just overwritten in place
    (same n and nnz).  c3's operand must equal a fresh upload's, and c2 must be unaffected."""
    from tvbingefriend_recommendation_service_b200.engine import stage

    f1 = catalogue(1000, 500, seed=31)
    f2 = catalogue(1200, 500, seed=32)
    f3 = rotated(f1, 101)
    assert f3["text_features"].nnz == f1["text_features"].nnz
    c1 = engine.prepare(engine.h2d(stage(f1), reuse=True), W)
    c2 = engine.prepare(engine.h2d(stage(f2), reuse=True), W)
    c3 = engine.prepare(engine.h2d(stage(f3), reuse=True), W, recycle=c1)
    assert_same_buffers(c3, fresh.upload(stage(f3), W), "c3 recycling c1")
    assert_same_buffers(c2, fresh.upload(stage(f2), W), "c2")


def test_recycle_two_reused_h2d_sets_back_tables(engine, fresh):
    """The same pipeline end to end: the tables of c2 and c3 equal fresh runs and the oracle."""
    from tvbingefriend_recommendation_service_b200.engine import stage

    f1 = catalogue(1000, 500, seed=33, signed=True)
    f2 = catalogue(1000, 500, seed=34)
    f3 = rotated(f1, 57)
    c1 = engine.prepare(engine.h2d(stage(f1), reuse=True), W)
    c2 = engine.prepare(engine.h2d(stage(f2), reuse=True), W)
    c3 = engine.prepare(engine.h2d(stage(f3), reuse=True), W, recycle=c1)
    for name, cat, f in (("c2", c2, f2), ("c3", c3, f3)):
        got = engine.to_host(engine.top_k_device(cat, W, 20, MS))
        ref = fresh.to_host(fresh.top_k_device(fresh.upload(stage(f), W), W, 20, MS))
        assert_same_tables(got, ref, name)
        assert_topk_matches(got, f, spread_rows(0, cat.n_shows))


# ---------------------------------------------------------------------------------------------- 3
POOL = [  # (n, V, nnz, genres, signed)
    (1, 64, 5, 40, False), (3, 500, 10, 40, False), (257, 3000, 20, 40, False), (700, 64, 8, 100, False),
    (1000, 500, 20, 40, True), (2600, 3000, 30, 40, False), (6000, 500, 20, 40, False),
    (6000, 64, 10, 40, False), (41_000, 500, 12, 40, False),
]
BIG = len(POOL) - 1           # symmetric by default (>= 160 column tiles)


def _sharded(eng, cat, w, k, ms, world, tuning):
    """The tile-sharded protocol with the ranks run one after the other on one GPU, each rank's
    seed reusing the engine's theta as the multi-GPU driver does."""
    import torch

    from tvbingefriend_recommendation_service_b200.engine import TopK
    from tvbingefriend_recommendation_service_b200.sharding import row_shard

    n = cat.n_shows
    theta = torch.stack([eng.sym_seed(cat, w, k, ms, r, world, tuning=tuning, reuse_theta=True).clone()
                         for r in range(world)]).amax(dim=0)
    parts = [eng.sym_sweep(cat, w, k, ms, r, world, theta.clone(), tuning=tuning) for r in range(world)]
    cand, cnt, bound = (torch.stack([p[i] for p in parts]) for i in range(3))
    tabs = [eng.to_host(eng.sym_rescore(cat, w, k, ms, cand, cnt, bound, *row_shard(n, world, r), tuning=tuning))
            for r in range(world)]
    return TopK(*(np.concatenate([getattr(t, f) for t in tabs]) for f in
                  ("indices", "counts", "hybrid", "genre", "text", "metadata")))


def _assert_same_stats(got, exp, what):
    for name, d in exp.items():
        for q, x in d.items():
            if isinstance(x, float):
                assert np.isclose(got[name][q], x, rtol=1e-9, atol=1e-12), (what, name, q)
            else:
                assert got[name][q] == x, (what, name, q)


def _assert_stats_refuse_signed(eng, cat, what):
    from tvbingefriend_recommendation_service_b200._lib import TvbfError

    assert cat.c.text_signed, what
    with pytest.raises(TvbfError, match="signed text"):
        eng.similarity_stats(cat, W)


def test_random_job_sequence_on_one_engine_refusing_signed_stats(engine, fresh):
    """30 seeded jobs of every entry point through one engine, each compared with a fresh engine and
    the oracle.  A statistics job on the signed-text catalogue of the pool must be refused
    (``TvbfError``: the streaming statistics take non-negative text only); the refusal is also
    checked after the sequence, whether or not the draw reached such a job."""
    from tvbingefriend_recommendation_service_b200._lib import TvbfError
    from tvbingefriend_recommendation_service_b200.synthetic import WEIGHT_SWEEP

    rng = np.random.default_rng(2024)
    feats, ref_cats, live = {}, {}, {}      # pool index -> features / fresh catalogue / engine catalogue
    reuse_made = []                         # engine catalogues whose CSR lives in an h2d(reuse=True) set
    last = None
    log = []
    fold_default = engine.fold_max_k
    try:
        for job in range(30):
            key = BIG if job in (6, 21) else int(rng.integers(BIG))
            if key not in feats:
                n, v, nnz, g, signed = POOL[key]
                feats[key] = catalogue(n, v, nnz, seed=100 + key, genres=g, signed=signed)
                ref_cats[key] = upload(fresh, feats[key], "upload")
            f, ref = feats[key], ref_cats[key]
            n = ref.n_shows
            if key not in live or rng.random() < 0.3:
                how = str(rng.choice(["upload", "ingest", "reuse"]))
                recycle = last if last is not None and rng.random() < 0.6 else None
                if recycle is not None:
                    live = {kk: c for kk, c in live.items() if c is not recycle}
                if how == "reuse":
                    # an h2d set is overwritten by the h2d call after next: its catalogue dies with it
                    for old in reuse_made[:-1]:
                        live = {kk: c for kk, c in live.items() if c is not old}
                    del reuse_made[:-1]
                live[key] = last = upload(engine, f, how, recycle=recycle)
                if how == "reuse":
                    reuse_made.append(last)
                log.append(f"job {job}: catalogue {key} {POOL[key]} via {how}, recycled: {recycle is not None}")
            cat = live[key]
            engine.fold_max_k = fold_default if rng.random() < 0.5 else 0
            entry = str(rng.choice(["topk", "topk", "topk", "sweep", "sharded", "exact", "stats"]))
            k = int(rng.choice([1, 20, 48, 64, 100]))
            sym = engine.sym_eligible(cat, W, k, MS) and not cat.c.genre_hi
            if entry == "sharded" and not sym:
                entry = "topk"
            if entry == "stats" and n < 2:
                entry = "exact"
            mode = int(rng.choice([0, 1, 2]))
            splits = int(rng.integers(0, 6))
            stride = int(rng.choice([0, 1, 63]))
            tuning = (mode << 20) | (stride << 22)
            log.append(f"job {job}: {entry} n={n} k={k} fold_max_k={engine.fold_max_k} mode={mode} "
                       f"splits={splits} stride={stride}")
            rows = spread_rows(0, n)
            if entry == "topk":
                try:
                    got = engine.to_host(engine.top_k_device(cat, W, k, MS, splits=splits, tuning=tuning))
                except TvbfError:
                    assert mode == 2, log[-1]           # only an explicit symmetric request may be refused
                    log.append("  refused (not eligible)")
                    continue
                exp = fresh.to_host(fresh.top_k_device(ref, W, k, MS, splits=splits, tuning=tuning))
                assert_same_tables(got, exp, log[-1])
                assert_topk_matches(got, f, rows, W, k, MS)
            elif entry == "sweep":
                triples = [WEIGHT_SWEEP[i] for i in rng.choice(len(WEIGHT_SWEEP), size=3, replace=False)]
                shared = bool(rng.random() < 0.5) and all(engine.sym_eligible(cat, w, k, MS) for w in triples) \
                    and not cat.c.genre_hi
                if key == BIG:
                    shared = None                       # the default: shared at this size
                log[-1] += f" sweep shared={shared}"
                tabs = engine.top_k_sweep_device(cat, triples, k, MS, shared=shared)
                for w, t in zip(triples, tabs):
                    got = engine.to_host(t)
                    assert_same_tables(got, fresh.to_host(fresh.top_k_device(ref, w, k, MS)), f"{log[-1]} {w}")
                    assert_topk_matches(got, f, rows[::2], w, k, MS)
            elif entry == "sharded":
                world = int(rng.choice([2, 3]))
                log[-1] += f" world={world}"
                got = _sharded(engine, cat, W, k, MS, world, stride << 22)
                assert_same_tables(got, fresh.to_host(fresh.top_k_device(ref, W, k, MS)), log[-1])
                assert_topk_matches(got, f, rows, W, k, MS)
            elif entry == "exact":
                b = int(rng.integers(0, n))
                e = min(n, b + int(rng.integers(1, 40)))
                got = engine.exact_rows(cat, np.arange(b, e), W, k, MS)
                exp = fresh.exact_rows(ref, np.arange(b, e), W, k, MS)
                assert_same_tables(got, exp, log[-1])
                got.row_begin = b
                assert_topk_matches(got, f, spread_rows(b, e, 3), W, k, MS)
            else:
                if POOL[key][4]:
                    # signed text: the streaming statistics refuse it, on a recycled catalogue as well
                    _assert_stats_refuse_signed(engine, cat, log[-1])
                    log.append("  refused (signed text)")
                    continue
                _assert_same_stats(engine.similarity_stats(cat, W), fresh.similarity_stats(ref, W), log[-1])
        # whether the seeded draw reaches a stats job on the signed catalogue or not: it is refused
        # through the long-lived engine, and the engine still computes statistics afterwards
        signed = next(i for i, entry in enumerate(POOL) if entry[4])
        cat = live.get(signed)
        if cat is None:
            feats.setdefault(signed, catalogue(*POOL[signed][:3], seed=100 + signed, genres=POOL[signed][3],
                                               signed=True))
            cat = upload(engine, feats[signed], "ingest")
        log.append(f"after the sequence: stats on signed catalogue {signed}")
        _assert_stats_refuse_signed(engine, cat, log[-1])
        f = catalogue(300, 200, seed=7)
        _assert_same_stats(engine.similarity_stats(engine.ingest(f), W),
                           fresh.similarity_stats(upload(fresh, f, "upload"), W), log[-1])
    except Exception as e:
        raise AssertionError("job log (seeded, replayable):\n" + "\n".join(log)) from e
    finally:
        engine.fold_max_k = fold_default


# ---------------------------------------------------------------------------------------------- 4
def _fresh_table(fresh, f, k):
    return fresh.to_host(fresh.top_k_device(upload(fresh, f, "upload"), W, k, MS))


def test_abandoned_seed_then_seedless_sweep(engine, fresh):
    """A seed-only call whose job is dropped leaves its shared-list clear behind.  After a one-sided
    job has written the same workspace, a symmetric job without a seed pass (no clear of its own)
    whose lists sit at the same address must clear them itself, not trust the stale clear."""
    import torch

    from tvbingefriend_recommendation_service_b200.sharding import row_shard

    k, world = 20, 2
    fx = catalogue(3000, 500, seed=41)
    fy = catalogue(2000, 500, seed=42)
    x = upload(engine, fx, "upload")
    y = upload(engine, fy, "upload")
    assert engine.plan_tiles(x, W, k, MS, rank=0, world=world, tile_sharded=True)["seed_tiles"] > 0
    ref_y = _fresh_table(fresh, fy, k)
    engine.to_host(engine.top_k_device(y, W, k, MS, tuning=ONE_SIDED))  # workspace large enough for Y's job
    engine.sym_seed(x, W, k, MS, 0, world, reuse_theta=True)           # abandoned: starts the clear
    base = engine._ws.data_ptr()
    one = engine.to_host(engine.top_k_device(y, W, k, MS, tuning=ONE_SIDED))
    assert engine._ws.data_ptr() == base                               # same workspace, same list address
    assert_same_tables(one, ref_y, "one-sided job on Y")
    theta = torch.stack([engine.sym_seed(x, W, k, MS, r, world, tuning=NO_SEED, reuse_theta=True).clone()
                         for r in range(world)]).amax(dim=0)
    assert engine._ws.data_ptr() == base
    parts = [engine.sym_sweep(x, W, k, MS, r, world, theta.clone(), tuning=NO_SEED) for r in range(world)]
    cand, cnt, bound = (torch.stack([p[i] for p in parts]) for i in range(3))
    ref = _fresh_table(fresh, fx, k)
    for r in range(world):
        b, e = row_shard(3000, world, r)
        got = engine.to_host(engine.sym_rescore(x, W, k, MS, cand, cnt, bound, b, e, tuning=NO_SEED))
        assert_same_tables(got, ref.slice(b, e), f"rank {r}")
        assert_topk_matches(got, fx, spread_rows(b, e, 3))


@pytest.mark.parametrize("streams", ["one_stream", "two_streams"])
def test_interleaved_seeded_jobs_of_two_engines(fresh, streams):
    """Two engines on one device: both seeds (each starts a list clear beside its seed pass), then
    both sweeps in the opposite order.  The sweep of the first job must not run into its clear."""
    import torch

    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    k = 20
    engines = [HybridTopKEngine(0), HybridTopKEngine(0)]
    fs = [catalogue(6000, 500, seed=51), catalogue(5000, 3000, seed=52)]
    cats = [upload(e, f, "upload") for e, f in zip(engines, fs)]
    if streams == "two_streams":
        ctx = [torch.cuda.Stream(0), torch.cuda.Stream(0)]
        for s in ctx:
            s.wait_stream(torch.cuda.current_stream(0))       # the uploads ran on the current stream
    else:
        ctx = [torch.cuda.current_stream(0)] * 2
    thetas, parts = [None, None], [None, None]
    for i in (0, 1):
        assert engines[i].plan_tiles(cats[i], W, k, MS, tile_sharded=True)["seed_tiles"] > 0
        with torch.cuda.stream(ctx[i]):
            thetas[i] = engines[i].sym_seed(cats[i], W, k, MS, 0, 1, reuse_theta=True)
    for i in (1, 0):
        with torch.cuda.stream(ctx[i]):
            parts[i] = engines[i].sym_sweep(cats[i], W, k, MS, 0, 1, thetas[i])
    for i in (0, 1):
        with torch.cuda.stream(ctx[i]):
            cand, cnt, bound = (p[None] for p in parts[i])
            got = engines[i].to_host(engines[i].sym_rescore(cats[i], W, k, MS, cand, cnt, bound, 0, cats[i].n_shows))
        assert_same_tables(got, _fresh_table(fresh, fs[i], k), f"engine {i}")
        assert_topk_matches(got, fs[i], spread_rows(0, cats[i].n_shows))
