"""The merged text operand of the candidate pass (host side, no GPU): the rule that picks its width,
a numpy model of the merge plan ``tvbf_merge_plan`` builds on the device (``tests/test_gpu_merge.py``
compares the two), and the bound the candidate pass relies on: for non-negative rows the dot product
of the merged rows is at least the exact text cosine."""

import ctypes as C

import numpy as np
import pytest

from tvbingefriend_recommendation_service_b200.engine import merge_text_cols


def model_plan(indices: np.ndarray, vocab: int, text_cols: int):
    """(col_map, slot_ptr, slot_cols) as tvbf_merge_plan defines them: columns ranked by descending
    document frequency, ties by ascending column; the text_cols // 2 first ranks keep a column of their
    own, the others are dealt round-robin by rank over the remaining columns."""
    df = np.bincount(indices, minlength=vocab)
    order = np.lexsort((np.arange(vocab), -df))
    head = text_cols // 2
    tail = text_cols - head
    rank = np.arange(vocab)
    slot_of_rank = np.where(rank < head, rank, head + (rank - head) % tail)
    col_map = np.empty(vocab, dtype=np.int64)
    col_map[order] = slot_of_rank
    slot_cols = np.concatenate([order[slot_of_rank == s] for s in range(text_cols)])
    slot_ptr = np.r_[0, np.cumsum(np.bincount(slot_of_rank, minlength=text_cols))]
    return col_map, slot_ptr, slot_cols


def merged_dense(x, col_map: np.ndarray, text_cols: int) -> np.ndarray:
    """rows of the CSR ``x`` with the columns of every slot summed (float64)"""
    coo = x.tocoo()
    out = np.zeros((x.shape[0], text_cols))
    np.add.at(out, (coo.row, col_map[coo.col]), coo.data)
    return out


# ---------------------------------------------------------------------------------------------- rule
@pytest.mark.parametrize("vocab,genres,want", [
    (500, 21, 500),               # P80k: the plain fold fits, no merge
    (4000, 40, 4000),             # exactly at the fold limit with the packed groups
    (4100, 40, 4024),             # just above: merged to what fits beside the groups
    (10_000, 40, 4024),           # C3 / C4: 0.40 V
    (50_000, 40, 20_000),         # C5: ceil(0.4 V) is wider than the fold limit allows
    (4060, 1, 4060),              # 4063 columns: merging would not narrow the 64-padded operand
])
def test_text_columns_follow_the_rule(vocab, genres, want):
    assert merge_text_cols(vocab, genres) == want


def test_either_knob_at_zero_switches_merging_off():
    assert merge_text_cols(10_000, 40, fold_max_k=4096, ratio=0.0) == 10_000
    assert merge_text_cols(10_000, 40, fold_max_k=0, ratio=0.4) == 10_000
    assert merge_text_cols(10_000, 40, fold_max_k=4096, ratio=0.3) == 4024
    assert merge_text_cols(10_000, 40, fold_max_k=2048, ratio=0.3) == 3000
    assert merge_text_cols(10_000, 40, fold_max_k=4096, ratio=1.0) == 10_000


def test_no_operand_column_takes_more_than_4096_vocabulary_columns():
    kt = merge_text_cols(20_000_000, 40, ratio=1e-6)
    assert kt == 20_000_000                         # would be 10 000 per column: not merged
    kt = merge_text_cols(2_000_000, 40, ratio=1e-6)
    head = kt // 2
    assert kt < 2_000_000 and -(-(2_000_000 - head) // (kt - head)) <= 4096


# ---------------------------------------------------------------------------------------------- plan
@pytest.mark.parametrize("vocab,text_cols", [(5000, 4024), (10_000, 4024), (10_000, 3), (7, 2), (600, 599)])
def test_plan_maps_every_column_and_keeps_the_head_apart(vocab, text_cols):
    rng = np.random.default_rng(vocab + text_cols)
    indices = np.minimum(rng.zipf(1.3, size=20 * vocab) - 1, vocab - 1)   # skewed frequencies, many ties
    col_map, slot_ptr, slot_cols = model_plan(indices, vocab, text_cols)
    assert col_map.min() >= 0 and col_map.max() < text_cols
    assert np.array_equal(np.sort(slot_cols), np.arange(vocab))          # every column in exactly one slot
    assert slot_ptr[0] == 0 and slot_ptr[-1] == vocab and np.all(np.diff(slot_ptr) >= 1)
    for s in range(text_cols):
        assert np.all(col_map[slot_cols[slot_ptr[s]:slot_ptr[s + 1]]] == s)
    head = text_cols // 2
    df = np.bincount(indices, minlength=vocab)
    order = np.lexsort((np.arange(vocab), -df))
    assert np.array_equal(col_map[order[:head]], np.arange(head))        # the head: distinct, own columns
    assert np.all(np.diff(slot_ptr)[:head] == 1)
    sizes = np.diff(slot_ptr)[head:]
    assert sizes.max() - sizes.min() <= 1                                # the tail is dealt evenly
    assert np.all(df[order][:-1] >= df[order][1:])


def test_merge_plan_rejects_bad_widths_before_any_device_work():
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    addr = [1 << 20, 1 << 21, 1 << 22, 1 << 23, 1 << 24, 1 << 25]

    def call(vocab, text_cols):
        rc = lib.tvbf_merge_plan(addr[0], addr[1], 10, vocab, text_cols, addr[2], addr[3], addr[4], addr[5], 1 << 30,
                                 None)
        return rc, lib.tvbf_last_error().decode()

    for vocab, text_cols in ((100, 101), (100, 1), (100, 0)):
        rc, msg = call(vocab, text_cols)
        assert rc != 0 and "text_cols" in msg
    rc, msg = call(20_000_000, 4000)
    assert rc != 0 and "at most 4096" in msg


def test_merged_features_need_non_negative_text():
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    f = _lib.Features(n_shows=10, n_pad=256, k_pad=64, text_dtype=_lib.TEXT_FP16, vocab=100, operand=1 << 20,
                      text_indptr=1 << 21, text_indices=1 << 22, text_values=1 << 23, col_side=1 << 24,
                      meta_scale=1 << 25, genre_mode=_lib.GROUP_PACKED, genre_dim=20, meta_mode=_lib.GROUP_PACKED)
    p = _lib.Params(genre_weight=0.4, text_weight=0.5, metadata_weight=0.1, min_similarity=0.1, k=20,
                    exclude_self=1, row_begin=0, row_end=10)
    out = (C.c_int64 * 4)()
    f.text_cols, f.text_signed = 60, 1
    assert lib.tvbf_plan_tiles(C.byref(f), C.byref(p), 0, 1, 0, out) != 0
    assert "non-negative text" in lib.tvbf_last_error().decode()
    f.text_cols, f.text_signed = 101, 0
    assert lib.tvbf_plan_tiles(C.byref(f), C.byref(p), 0, 1, 0, out) != 0
    assert "text_cols" in lib.tvbf_last_error().decode()


# ---------------------------------------------------------------------------------------------- bound
@pytest.mark.parametrize("text_cols", [4024, 2000, 600])
def test_merged_dot_bounds_the_exact_text_cosine(text_cols):
    from sklearn.preprocessing import normalize

    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    x = normalize(make_catalogue(400, 5000, nnz=40, n_genres=20, seed=3).features()["text_features"].tocsr())
    col_map, _, _ = model_plan(x.indices, x.shape[1], text_cols)
    exact = (x @ x.T).toarray()
    xm = merged_dense(x, col_map, text_cols)
    upper = xm @ xm.T
    assert np.all(upper >= exact * (1 - 1e-12) - 1e-300)
    if text_cols >= 0.4 * x.shape[1]:     # from 0.4 V on, most pairs gain nothing from the merge
        assert np.mean(upper - exact <= 1e-12) > 0.5


def test_merged_dot_of_adversarial_rows_still_bounds():
    """rows whose terms all share one merged column: the bound is loose but holds"""
    import scipy.sparse as sp
    from sklearn.preprocessing import normalize

    vocab, text_cols = 1000, 100
    df_idx = np.r_[np.repeat(np.arange(50), 10), np.arange(50, vocab)]     # 50 frequent columns, then the rest
    col_map, slot_ptr, slot_cols = model_plan(df_idx, vocab, text_cols)
    group = slot_cols[slot_ptr[70]:slot_ptr[71]]
    rng = np.random.default_rng(0)
    rows = [np.sort(rng.choice(group, size=min(4, group.size), replace=False)) for _ in range(30)]
    x = sp.csr_matrix((rng.random(sum(r.size for r in rows)) + 0.1,
                       np.concatenate(rows), np.r_[0, np.cumsum([r.size for r in rows])]), shape=(30, vocab))
    x = normalize(x)
    exact = (x @ x.T).toarray()
    xm = merged_dense(x, col_map, text_cols)
    assert np.all(xm @ xm.T >= exact * (1 - 1e-12))
