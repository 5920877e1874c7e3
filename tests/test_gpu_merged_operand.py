"""The merged text operand against float64 models of it (``-m gpu``).

``tests/test_gpu_merge.py`` compares tables with merging on and off; an operand entry that is too
large only loosens the bound and leaves the table as it was.  Here the component itself is checked:
the bits ``tvbf_prep_csr_to_operand_mapped`` writes (``model_operand``), the plan ``tvbf_merge_plan``
builds at its edges (``model_plan``), the candidate pass' upper bound over the merged operand on the
tensor cores, the engine's second operand after every incremental operation, and the routes that
had never met a merged operand (the tile-sharded protocol, the shared weight sweep)."""

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from helpers import assert_topk_matches
from test_merge_plan import merged_dense, model_operand, model_plan

pytestmark = pytest.mark.gpu

W = (0.4, 0.5, 0.1)
MS = 0.1
SCALE = 256.0                       # 2^TEXT_SCALE_LOG2
FIELDS = ("indices", "counts", "hybrid", "genre", "text", "metadata")


# ---------------------------------------------------------------------------------------------- fixtures
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


@pytest.fixture(scope="module")
def fresh():
    """a second merging engine: second operands of freshly ingested catalogues"""
    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine

    return HybridTopKEngine(0)


def _catalogue(n, vocab, seed=0, nnz=30, genres=40):
    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    return make_catalogue(n, vocab, nnz=nnz, n_genres=genres, seed=seed).features()


def _with_text(text, seed):
    f = _catalogue(text.shape[0], text.shape[1], seed=seed, nnz=5)
    f["text_features"] = text.tocsr()
    return f


def _csr(rows, values, vocab):
    indptr = np.r_[0, np.cumsum([len(r) for r in rows])]
    return sp.csr_matrix((np.concatenate(values), np.concatenate(rows).astype(np.int64), indptr),
                         shape=(len(rows), vocab))


def _rows(feats, sel):
    return {key: (a[sel].tocsr() if sp.issparse(a) else a[sel]) for key, a in feats.items()}


def _stack(a, b):
    return {key: (sp.vstack([a[key], b[key]]).tocsr() if sp.issparse(a[key]) else np.concatenate([a[key], b[key]]))
            for key in a}


def _same(a, b, what=""):
    for name in FIELDS:
        assert getattr(a, name).tobytes() == getattr(b, name).tobytes(), (what, name)


def _bits(t: torch.Tensor) -> np.ndarray:
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def _csr_of(cat):
    """(indptr, indices, normalised fp64 values) of the catalogue's text CSR as the device holds it"""
    n = cat.n_shows
    indptr = cat.text_indptr[:n + 1].cpu().numpy().astype(np.int64)
    nnz = int(indptr[-1])
    return indptr, cat.text_indices[:nnz].cpu().numpy(), cat.parts["values"][:nnz].cpu().numpy()


def _plan_np(plan: dict):
    return tuple(plan[key].cpu().numpy().astype(np.int64) for key in ("col_map", "slot_ptr", "slot_cols"))


def _plan_dev(plan, device) -> dict:
    return {key: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device)
            for key, a in zip(("col_map", "slot_ptr", "slot_cols"), plan)}


def _mapped(engine, cat, plan: dict, k_pad, col_offset=0, bf16=False, extra=2) -> np.ndarray:
    """bits tvbf_prep_csr_to_operand_mapped writes for every row of ``cat`` into a zeroed buffer of
    ``extra`` more rows"""
    from tvbingefriend_recommendation_service_b200 import _lib

    n = cat.n_shows
    buf = torch.zeros((n + extra, k_pad), dtype=torch.int16, device=engine.device)
    rc = engine.lib.tvbf_prep_csr_to_operand_mapped(
        cat.text_indptr.data_ptr(), cat.text_indices.data_ptr(), cat.parts["values"].data_ptr(), n,
        plan["col_map"].data_ptr(), plan["slot_ptr"].data_ptr(), plan["slot_cols"].data_ptr(), buf.data_ptr(),
        k_pad, col_offset, SCALE, _lib.TEXT_BF16 if bf16 else _lib.TEXT_FP16, engine._stream())
    assert rc == 0, engine.lib.tvbf_last_error().decode()
    return _bits(buf)


def _model(cat, plan, k_pad, col_offset=0, dtype="fp16", extra=2) -> np.ndarray:
    want = model_operand(*_csr_of(cat), plan, k_pad, col_offset, SCALE, dtype)
    return np.vstack([want, np.zeros((extra, k_pad), dtype=np.uint16)])


def _subnormal(bits: np.ndarray) -> np.ndarray:
    return ((bits & 0x7C00) == 0) & ((bits & 0x03FF) != 0)


# ---------------------------------------------------------------------------------------------- operand bits
def _kernel_case(seed=91):
    """V = 10 000 over 4 024 operand columns: 1 200 ordinary rows, then rows of 0 .. 1 000 entries,
    rows whose entries all lie in one tail slot, and rows with values from 1e-9 to 1.  The plan is
    the model plan of the ordinary rows (any plan is valid input of the kernel)."""
    vocab, kt = 10_000, 4024
    rng = np.random.default_rng(seed)
    bg = _catalogue(1200, vocab, seed=seed)["text_features"].tocsr()
    bg.sort_indices()
    plan = model_plan(bg.indices, vocab, kt)
    _, slot_ptr, slot_cols = plan
    head = kt // 2
    rows = []
    for length in (0, 1, 31, 32, 33, 64, 200, 1000):
        rows.append(np.sort(rng.choice(vocab, size=length, replace=False)))
    concentrated = []
    for s in (head, head + 1, head + 700, kt - 1):            # 4, 4, 4 and 3 vocabulary columns
        cols = np.sort(slot_cols[slot_ptr[s]:slot_ptr[s + 1]])
        concentrated += [cols, cols[::2]]
    values = [rng.random(r.size) + 0.05 for r in rows + concentrated]
    wide = [np.sort(rng.choice(vocab, size=600, replace=False)) for _ in range(40)]
    values += [10.0 ** rng.uniform(-9.0, 0.0, r.size) for r in wide]
    text = sp.vstack([bg, _csr(rows + concentrated + wide, values, vocab)]).tocsr()
    return _with_text(text, seed + 1), plan, bg.shape[0] + len(rows), len(concentrated)


@pytest.fixture(scope="module")
def kernel_case(engine):
    f, plan, c0, n_conc = _kernel_case()
    cat = engine.ingest(f)
    return cat, plan, c0, n_conc


@pytest.mark.parametrize("layout", ["fp16", "offset_64_wide_k_pad", "bf16"])
def test_mapped_operand_bits_are_the_model(engine, kernel_case, layout):
    """Every byte of the buffer, the zeros included, against model_operand over the catalogue's own
    CSR and normalised values; two calls give the same bytes"""
    cat, plan, c0, n_conc = kernel_case
    kt = plan[1].size - 1
    k_pad, col_offset = {"fp16": (4032, 0), "offset_64_wide_k_pad": (4160, 64), "bf16": (4032, 0)}[layout]
    bf16 = layout == "bf16"
    dplan = _plan_dev(plan, engine.device)
    got = _mapped(engine, cat, dplan, k_pad, col_offset, bf16)
    want = _model(cat, plan, k_pad, col_offset, "bf16" if bf16 else "fp16")
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} entries differ, first (row, column): {bad[:5].tolist()}"
    assert np.array_equal(_mapped(engine, cat, dplan, k_pad, col_offset, bf16), got)
    text = got[:, col_offset:col_offset + kt]
    # the concentrated rows: one operand column each, the sum of all their entries
    conc = text[c0:c0 + n_conc]
    assert np.all(np.count_nonzero(conc, axis=1) == 1)
    if not bf16:
        # the wide rows: fp16 subnormals, and slot sums whose every entry is a subnormal but the sum is not
        ip, ix, vals = _csr_of(cat)
        row = np.repeat(np.arange(cat.n_shows), np.diff(ip))
        key = row * kt + plan[0][ix]
        biggest, total = np.zeros(cat.n_shows * kt), np.zeros(cat.n_shows * kt)
        np.maximum.at(biggest, key, vals * SCALE)
        np.add.at(total, key, vals * SCALE)
        crossing = int(np.count_nonzero((biggest < 2.0 ** -14) & (total >= 2.0 ** -14)))
        subnormal = int(np.count_nonzero(_subnormal(text)))
        print(f"wide values: {subnormal} subnormal entries, {crossing} sums of subnormals that are normal")
        assert subnormal > 0 and crossing > 0


def test_mapped_operand_fills_one_slot_of_4096_columns(engine):
    """V = 4 097 over 2 operand columns: the head keeps the most frequent column, the one tail slot
    takes the other 4 096.  A unit row over all of them merges to 4 096 / 64 = 64, times 2^8."""
    vocab = 4097
    rng = np.random.default_rng(92)
    rows = [np.r_[0, np.sort(rng.choice(np.arange(1, vocab), size=20, replace=False))] for _ in range(300)]
    rows.append(np.arange(1, vocab))
    values = [rng.random(r.size) + 0.05 for r in rows[:-1]] + [np.ones(vocab - 1)]
    cat = engine.ingest(_with_text(_csr(rows, values, vocab), 93))
    plan = engine._merge_plan(cat, 2)
    want_plan = model_plan(_csr_of(cat)[1], vocab, 2)
    for got_a, want_a in zip(_plan_np(plan), want_plan):
        assert np.array_equal(got_a, want_a)
    assert list(want_plan[1]) == [0, 1, vocab]
    got = _mapped(engine, cat, plan, 64)
    assert np.array_equal(got, _model(cat, want_plan, 64))
    assert got[300, 1] == np.float16(64 * SCALE).view(np.uint16) and got[300, 0] == 0


@pytest.mark.parametrize("k", [20, 60], ids=["folded", "popcount"])
def test_engine_second_operand_is_the_model(engine, k):
    """The buffer the candidate pass runs on, as top_k_device left it: text columns equal the model
    through the engine's plan; every other column without a folded group, and every padding row, is
    zero"""
    f = _catalogue(3000, 10_000, seed=94)
    cat = engine.ingest(f)
    engine._fold_owner = None
    engine.top_k_device(cat, W, k, MS)
    fc = engine._fold_owner
    ff = fc["c"]
    kt, k_pad = int(ff.text_cols), int(ff.k_pad)
    assert kt == 4024 and k_pad == (4096 if k == 20 else 4032) and bool(ff.bits_folded) == (k == 20)
    got = _bits(fc["operand"])
    assert got.shape == (int(ff.n_pad), k_pad)
    want = model_operand(*_csr_of(cat), _plan_np(fc["plan"]), k_pad, 0, SCALE)
    assert np.array_equal(got[:3000, :kt], want[:, :kt])
    groups = np.zeros(k_pad, dtype=bool)
    if ff.bits_folded:
        groups[int(ff.fold_col0):int(ff.fold_col0) + int(ff.genre_dim) + 32] = True
        assert got[:3000, groups].any()
    assert not got[:3000, kt:][:, ~groups[kt:]].any()
    assert not got[3000:].any()


# ---------------------------------------------------------------------------------------------- bound
def _check_bound(engine, f, k, tiles, weights=W, tight=False):
    """Upper bound of the candidate pass over the merged operand, every pair of every tile:
    U >= exact (the hybrid when the groups are folded, w_text * the text cosine otherwise), and the
    raw accumulators equal the float64 product of the model operand within the accumulation budget.
    Returns (operand bits, rows x operand columns merged in float64) for further checks."""
    from oracle.reference_paths import ProductionRows

    dc = engine.ingest(f)
    gw, tw, mw = (float(w) for w in weights)
    feats = engine._folded(dc, gw, tw, mw, k)
    fc = engine._fold_owner
    assert feats is not None and feats.text_cols > 0 and fc["c"] is feats
    kt, k_pad, folded = int(feats.text_cols), int(feats.k_pad), bool(feats.bits_folded)
    sl = engine.debug_slack(dc, weights, feats=feats)
    pr = ProductionRows(f, *weights)
    x = pr.T
    n = dc.n_shows
    plan = _plan_np(fc["plan"])
    op_bits = model_operand(*_csr_of(dc), plan, k_pad, 0, SCALE)
    buf = _bits(fc["operand"])[:n]
    assert np.array_equal(buf[:, :kt], op_bits[:, :kt])
    op_bits[:, kt:] = buf[:, kt:]                  # the folded groups as the engine wrote them
    op = op_bits.view(np.float16).astype(np.float64)
    xm = merged_dense(x, plan[0], kt)
    nnz = np.diff(x.indptr)
    acc_unit = sl["w_text_acc"] / sl["w_text"]
    for r0, c0, pair in tiles:
        r1, c1 = min(r0 + (256 if pair else 128), n), min(c0 + 256, n)
        rows, cols = np.arange(r0, r1), np.arange(c0, c1)
        a = engine.debug_gemm_tile(dc, r0, c0, pair=pair, feats=feats).cpu().numpy().astype(np.float64)
        a = a[:r1 - r0, :c1 - c0]
        h, _, t, _ = pr.rows_block(rows)
        h, t = h[:, c0:c1], t[:, c0:c1]
        if folded:
            terms = (nnz[rows] + int(dc.c.genre_dim) + 3).astype(np.float64)[:, None]
            u = (sl["w_text"] + sl["w_text_err"] + terms * sl["w_text_acc"]) * a + sl["eps"] + terms * sl["eps_term"]
            exact = h
        else:
            terms = nnz[rows].astype(np.float64)[:, None]
            u = sl["w_text"] * a + (sl["w_text_err"] + terms * sl["w_text_acc"]) * np.abs(a) + sl["eps"] \
                + terms * sl["eps_term"]
            exact = tw * t
        tile = (r0, c0, pair)
        assert np.all(u >= exact), (tile, float((exact - u).max()))
        if tight:
            same = np.abs(xm[rows] @ xm[cols].T - t) <= 1e-12      # pairs without a cross term
            assert same.mean() > 0.5, tile
            assert float((u - exact)[same].max()) <= 2.5e-3 * sum(weights), (tile, float((u - exact)[same].max()))
        # the accumulators against the float64 product of the same fp16 operand rows
        ref = op[rows] @ op[cols].T
        t_op = np.count_nonzero(op_bits[rows], axis=1).astype(np.float64)[:, None]
        tol = t_op * acc_unit * ref + t_op * sl["eps_term"] / sl["w_text"]
        err = np.abs(a - ref)
        assert np.all(err <= tol), (tile, float((err - tol).max()))
    return op_bits, xm


TILES_3000 = [(128, 256, False), (256, 2816, True), (2944, 2816, False)]    # 2816: the partial last column tile


def test_bound_merged_and_folded(engine):
    f = _catalogue(3000, 10_000, seed=71)
    _check_bound(engine, f, 20, TILES_3000, tight=True)
    assert engine._fold_owner["c"].bits_folded and engine._fold_owner["c"].text_cols == 4024


@pytest.mark.parametrize("vocab,n,k", [(10_000, 3000, 60), (50_000, 500, 100)], ids=["v10k_k60", "v50k_k100"])
def test_bound_merged_popcount(engine, vocab, n, k):
    f = _catalogue(n, vocab, seed=72)
    tiles = TILES_3000 if n == 3000 else [(128, 0, False), (0, 256, True)]
    _check_bound(engine, f, k, tiles)
    ff = engine._fold_owner["c"]
    assert not ff.bits_folded and ff.text_cols == (4024 if vocab == 10_000 else 20_000)


def test_bound_merged_with_subnormal_operands(engine):
    """250 rows at V = 10 000 whose vocabulary columns rank in index order (every used column has
    the same document frequency), so columns 2 017, 4 029 and 6 041 share tail slot 2 017.  Three
    rows put a dominant head column and three equal entries into that slot (a merged entry of 1.5);
    five rows put a dominant head column and about 1e-7 into one or two of the same columns, fp16
    subnormals after the 2^8 scale.  The rest fill every column below 6 042 up to the same
    frequency."""
    vocab, n, df, head = 10_000, 250, 8, 2012
    slot = [head + 5, 2 * head + 5, 3 * head + 5]
    rng = np.random.default_rng(73)
    special = [np.r_[10 + i, slot] for i in range(3)]
    special += [np.r_[20 + i, np.array(slot)[[i % 3, (i + 1) % 3][:1 + i % 2]]] for i in range(5)]
    special = [np.sort(r) for r in special]
    special_vals = [np.where(np.isin(r, slot), 1.0, 1.0) for r in special[:3]]
    special_vals += [np.where(np.isin(r, slot), rng.uniform(0.3e-7, 1.2e-7, r.size), 1.0) for r in special[3:]]
    cnt = np.bincount(np.concatenate(special), minlength=vocab)
    fill = np.where(np.arange(vocab) <= slot[-1], df, 0) - cnt
    assert fill.min() >= 0
    bg = [[] for _ in range(n - len(special))]
    for c in np.nonzero(fill)[0]:
        for r in rng.choice(len(bg), size=fill[c], replace=False):
            bg[r].append(c)
    bg = [np.array(sorted(r), dtype=np.int64) for r in bg]
    text = _csr(special + bg, special_vals + [rng.random(r.size) + 0.05 for r in bg], vocab)
    f = _with_text(text, 74)
    op_bits, xm = _check_bound(engine, f, 60, [(0, 0, False), (0, 0, True)], weights=(0.0, 1.0, 0.0))
    col_map = _plan_np(engine._fold_owner["plan"])[0]
    assert np.all(col_map[slot] == slot[0]) and np.all(col_map[:head] == np.arange(head))
    text_bits = op_bits[:, :4024]
    assert _subnormal(text_bits[3:8]).any()
    assert (text_bits[:3, slot[0]].view(np.float16) > SCALE).all()
    assert np.allclose(xm[:3, slot[0]], 1.5)


def _adversary(rng):
    """test_gpu_merge.py::test_rows_whose_terms_share_one_merged_column: columns ranked in index order,
    600 rows whose two terms share one merged column with another row's two"""
    n_bg, n_adv, vocab, head = 2400, 600, 10_000, 2012
    groups = np.array([[head + t, 2 * head + t, 3 * head + t, 4 * head + t] for t in range(10)])
    pairs = ((0, 1), (2, 3), (0, 2), (1, 3))
    adv = [np.sort(groups[i % 10][list(pairs[(i // 10) % 4])]) for i in range(n_adv)]
    a_cnt = np.bincount(np.concatenate(adv), minlength=vocab)
    b_cnt = 30 + (vocab - np.arange(vocab)) // 400 - a_cnt
    assert b_cnt.min() >= 0
    bg_rows = [[] for _ in range(n_bg)]
    for c in range(vocab):
        for r in rng.choice(n_bg, size=b_cnt[c], replace=False):
            bg_rows[r].append(c)
    rows = [np.array(sorted(r), dtype=np.int64) for r in bg_rows] + adv
    return _csr(rows, [rng.random(r.size) + 0.05 for r in rows], vocab), groups


def test_bound_on_rows_that_share_one_merged_column(engine):
    text, groups = _adversary(np.random.default_rng(21))
    f = _with_text(text, 22)
    _check_bound(engine, f, 20, [(2432, 2432, False), (2560, 2816, True), (0, 2560, False)])
    col_map = _plan_np(engine._fold_owner["plan"])[0]
    assert np.all(col_map[groups] == col_map[groups[:, :1]])


# ---------------------------------------------------------------------------------------------- incremental
def _check_second(engine, fresh, cat, feats_now, plan):
    """(a) text columns of rows [0, n) = the model of the catalogue's current CSR through ``plan``,
    (b) folded group columns = those of a freshly ingested catalogue, (c) rows [n, n_pad) zero"""
    fc = engine._fold_owner
    assert fc is not None and cat.fold is fc
    ff = fc["c"]
    n, kt, k_pad = cat.n_shows, int(ff.text_cols), int(ff.k_pad)
    got = _bits(fc["operand"])
    assert got.shape == (int(ff.n_pad), k_pad) and int(ff.n_shows) == n
    want = model_operand(*_csr_of(cat), plan, k_pad, 0, SCALE)
    bad = np.argwhere(got[:n, :kt] != want[:, :kt])
    assert bad.size == 0, f"(a) {len(bad)} text entries differ, first (row, column): {bad[:5].tolist()}"
    dc = fresh.ingest(feats_now)
    fresh_feats = fresh._folded(dc, *W, 20)
    assert fresh_feats.bits_folded and int(fresh_feats.fold_col0) == kt
    g = slice(kt, kt + int(ff.genre_dim) + 32)
    assert np.array_equal(got[:n, g], _bits(fresh._fold_owner["operand"])[:n, g]), "(b) group columns"
    assert not got[n:].any(), "(c) rows past the last show"


def _same_plan(fc, plan0):
    for key, t in plan0.items():
        assert torch.equal(fc["plan"][key], t), key


@pytest.mark.parametrize("kind", ["extend", "update", "remove", "refresh", "extend_grown"])
def test_second_operand_through_incremental_paths(engine, fresh, kind):
    n, vocab = 3000, 10_000
    before = _catalogue(n, vocab, seed=81)
    other = _catalogue(300, vocab, seed=82)
    engine._fold_owner = None
    cat = engine.ingest(before)
    prev = engine.top_k_device(cat, W, 20, MS)
    fc0 = engine._fold_owner
    assert int(fc0["c"].text_cols) == 4024 and fc0["c"].bits_folded and int(fc0["c"].n_pad) == 3072
    plan0 = {key: t.clone() for key, t in fc0["plan"].items()}
    plan = _plan_np(plan0)
    rng = np.random.default_rng(83)
    rows = np.sort(rng.choice(n, size=150, replace=False))
    assert np.unique(rows // 256).size >= 8                    # spread over the 256-row tiles
    if kind == "extend":
        cat = engine.extend(cat, _rows(other, np.arange(60)))
        now = _stack(before, _rows(other, np.arange(60)))
    elif kind == "update":
        cat = engine.update(cat, rows, _rows(other, np.arange(150)))
        src = np.arange(n)
        src[rows] = n + np.arange(150)
        now = _rows(_stack(before, _rows(other, np.arange(150))), src)
    elif kind == "remove":
        cat = engine.remove(cat, rows)
        now = _rows(before, np.delete(np.arange(n), rows))
    elif kind == "refresh":
        removed, updated = rows[::2], rows[1::2]
        cat = engine.update(cat, updated, _rows(other, np.arange(updated.size)))
        cat = engine.remove(cat, removed)
        cat = engine.extend(cat, _rows(other, 100 + np.arange(60)))
        t = engine.top_k_refresh_device(cat, prev, removed, updated, 60, W, 20, MS)
        assert t["incremental"]
        src = np.arange(n)
        src[updated] = n + np.arange(updated.size)
        both = _stack(before, other)
        now = _rows(both, np.r_[np.delete(src, removed), n + 100 + np.arange(60)])
    else:
        cat = engine.extend(cat, _rows(other, np.arange(200)))           # 3 200 shows: n_pad grows
        assert cat.fold is None and int(cat.c.n_pad) > 3072
        t = engine.top_k_append_device(cat, n, prev, W, 20, MS)
        assert t["incremental"]
        now = _stack(before, _rows(other, np.arange(200)))
        fc = engine._fold_owner
        assert fc is not fc0 and int(fc["c"].n_pad) == int(cat.c.n_pad)
        plan = model_plan(_csr_of(cat)[1], vocab, 4024)
        for got_a, want_a in zip(_plan_np(fc["plan"]), plan):
            assert np.array_equal(got_a, want_a)
    assert cat.n_shows == now["genre_features"].shape[0]
    if kind != "extend_grown":
        _same_plan(engine._fold_owner, plan0)
    _check_second(engine, fresh, cat, now, plan)


# ---------------------------------------------------------------------------------------------- routes
def _sharded(eng, cat, w, k, ms, world):
    """The tile-sharded protocol with the ranks run one after the other on one GPU, each rank's
    seed reusing the engine's theta as the multi-GPU driver does (test_gpu_job_sequences.py)."""
    from tvbingefriend_recommendation_service_b200.engine import TopK
    from tvbingefriend_recommendation_service_b200.sharding import row_shard

    n = cat.n_shows
    theta = torch.stack([eng.sym_seed(cat, w, k, ms, r, world, reuse_theta=True).clone()
                         for r in range(world)]).amax(dim=0)
    parts = [eng.sym_sweep(cat, w, k, ms, r, world, theta.clone()) for r in range(world)]
    cand, cnt, bound = (torch.stack([p[i] for p in parts]) for i in range(3))
    tabs = [eng.to_host(eng.sym_rescore(cat, w, k, ms, cand, cnt, bound, *row_shard(n, world, r)))
            for r in range(world)]
    return TopK(*(np.concatenate([getattr(t, name) for t in tabs]) for name in FIELDS))


@pytest.fixture(scope="module")
def sharded_case():
    return _catalogue(3000, 10_000, seed=101)


@pytest.mark.parametrize("k", [20, 100], ids=["k20_folded", "k100_popcount"])
@pytest.mark.parametrize("world", [2, 3])
def test_tile_sharded_protocol_over_the_merged_operand(engine, plain, sharded_case, world, k):
    f = sharded_case
    cat = engine.ingest(f)
    engine._fold_owner = None
    got = _sharded(engine, cat, W, k, MS, world)
    plan = engine.plan_tiles(cat, W, k, MS, rank=0, world=world, tile_sharded=True)
    assert plan["text_cols"] == 4024 and plan["folded_bits"] == (k == 20) and plan["seed_tiles"] > 0
    assert engine._fold_owner is cat.fold
    _same(got, plain.compute_top_k(f, W, k, MS), f"world {world} k {k}")
    assert_topk_matches(got, f, np.r_[np.arange(0, 3000, 97), 2999], k=k)


def test_shared_weight_sweep_leaves_the_merged_operand_alone(engine, plain):
    """The shared sweep runs on the catalogue's own operand; right after a merged job on the same
    engine it must give the plain tables and leave the second operand untouched"""
    from tvbingefriend_recommendation_service_b200.synthetic import WEIGHT_SWEEP

    f = _catalogue(3000, 10_000, seed=102)
    cat = engine.ingest(f)
    engine._fold_owner = None
    engine.top_k_device(cat, W, 20, MS)
    fc = engine._fold_owner
    assert fc is not None and int(fc["c"].text_cols) == 4024
    before = fc["operand"].clone()
    triples = [WEIGHT_SWEEP[i] for i in (0, 1, 2)]
    assert all(engine.sym_eligible(cat, w, 20, MS) for w in triples)
    tabs = engine.top_k_sweep_device(cat, triples, 20, MS, shared=True)
    torch.cuda.synchronize()
    assert engine._fold_owner is fc and cat.fold is fc
    assert torch.equal(fc["operand"].view(torch.int16), before.view(torch.int16))
    pc = plain.ingest(f)
    for w, t in zip(triples, tabs):
        _same(engine.to_host(t), plain.to_host(plain.top_k_device(pc, w, 20, MS)), w)
