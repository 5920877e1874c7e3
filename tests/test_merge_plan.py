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


def bf16_bits(x) -> np.ndarray:
    """float64 -> bfloat16 bits, rounded once to nearest with ties to even (``cvt.rn.bf16.f64``,
    which ``__double2bfloat16`` is on sm_100).  A float32 step would round twice."""
    x = np.asarray(x, dtype=np.float64)
    _, e = np.frexp(x)                                  # |x| in [2^(e-1), 2^e)
    q = np.ldexp(1.0, np.maximum(e - 8, -133))          # bf16 spacing there: 8 significant bits, subnormals 2^-133
    r = np.rint(x / q) * q                              # x / q is exact (q is a power of two); rint: ties to even
    with np.errstate(over="ignore"):
        return (r.astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)


def model_operand(indptr, indices, values, plan, k_pad: int, col_offset: int, scale: float,
                  dtype: str = "fp16") -> np.ndarray:
    """uint16 [n_rows, k_pad]: the bits tvbf_prep_csr_to_operand_mapped writes into a zeroed
    buffer.  Operand column s of a row is the float64 sum of the row's entries in the vocabulary
    columns of slot s, added one by one in ``slot_cols`` order (the kernel's order), times ``scale``,
    rounded once to fp16 / bf16; every other position stays zero.  ``plan``: (col_map, slot_ptr,
    slot_cols) as ``model_plan`` returns them."""
    col_map, slot_ptr, slot_cols = (np.asarray(a) for a in plan)
    indptr, indices = np.asarray(indptr, dtype=np.int64), np.asarray(indices, dtype=np.int64)
    values = np.asarray(values, dtype=np.float64)
    n = indptr.size - 1
    text_cols = slot_ptr.size - 1
    rank = np.empty(slot_cols.size, dtype=np.int64)
    rank[slot_cols] = np.arange(slot_cols.size)         # position of a vocabulary column in slot_cols
    row = np.repeat(np.arange(n), np.diff(indptr))
    order = np.lexsort((rank[indices], row))            # per row, in slot_cols order
    acc = np.zeros(n * text_cols)
    np.add.at(acc, row[order] * text_cols + col_map[indices[order]], values[order])   # sequential, in order
    touched = np.zeros(n * text_cols, dtype=bool)
    touched[row * text_cols + col_map[indices]] = True
    out = np.zeros((n, k_pad), dtype=np.uint16)
    scaled = acc.reshape(n, text_cols) * scale
    bits = scaled.astype(np.float16).view(np.uint16) if dtype == "fp16" else bf16_bits(scaled)
    out[:, col_offset:col_offset + text_cols] = np.where(touched.reshape(n, text_cols), bits, 0)
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
    rc, msg = call(4098, 2)                     # one tail slot of 4 097 columns; 4 097 / 2 is the largest accepted
    assert rc != 0 and "4097 vocabulary columns per operand column" in msg


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


# ---------------------------------------------------------------------------------------------- operand model
def test_bf16_rounder_rounds_once_to_nearest_even():
    cases = [(1.0, 0x3F80), (-1.5, 0xBFC0), (0.0, 0x0000),
             (1 + 2.0 ** -8, 0x3F80),                   # halfway, down to the even neighbour
             (1 + 3 * 2.0 ** -8, 0x3F82),               # halfway, up to the even neighbour
             (1 + 2.0 ** -8 + 2.0 ** -40, 0x3F81),      # just above halfway: a float32 step would make it a tie
             (1 + 2.0 ** -8 - 2.0 ** -40, 0x3F80),
             (2 - 2.0 ** -9, 0x4000),                   # carries into the exponent
             (256 * (1 + 2.0 ** -8), 0x4380), (-(1 + 3 * 2.0 ** -8), 0xBF82),
             (2.0 ** -133, 0x0001), (1.5 * 2.0 ** -133, 0x0002), (0.5 * 2.0 ** -133, 0x0000),   # subnormals
             (2.0 ** -126 * (1 - 2.0 ** -9), 0x0080),   # the largest subnormal rounds up to the smallest normal
             (2.0 ** 128 - 2.0 ** 119, 0x7F80), (2.0 ** 128 - 2.0 ** 119 - 2.0 ** 90, 0x7F7F)]   # overflow edge
    got = bf16_bits([x for x, _ in cases])
    for (x, want), g in zip(cases, got):
        assert int(g) == want, (x, hex(int(g)), hex(want))
    # the double rounding the model avoids
    x = np.float64(1 + 2.0 ** -8 + 2.0 ** -40)
    assert int(np.float32(x).view(np.uint32) >> 16) == 0x3F80
    # float32 inputs round once either way: compare with torch's float32 -> bfloat16
    import torch

    rng = np.random.default_rng(1)
    f32 = (rng.standard_normal(200_000) * np.exp2(rng.integers(-130, 120, 200_000))).astype(np.float32)
    f32 = np.r_[f32, (np.arange(1 << 16, dtype=np.uint32) << 16 | 0x8000).view(np.float32)]   # every tie
    f32 = f32[np.isfinite(f32)]
    ref = torch.from_numpy(f32).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    assert np.array_equal(bf16_bits(f32.astype(np.float64)), ref)


def _csr_rows(rows, values, vocab):
    import scipy.sparse as sp

    indptr = np.r_[0, np.cumsum([len(r) for r in rows])]
    return sp.csr_matrix((np.asarray(values, dtype=np.float64), np.concatenate(rows).astype(np.int64), indptr),
                         shape=(len(rows), vocab))


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_operand_model_is_the_rounded_merged_rows(dtype):
    """On ordinary rows the model is merged_dense times the scale, rounded once, at the layout's
    offset, zero elsewhere"""
    import torch
    from sklearn.preprocessing import normalize

    from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue

    x = normalize(make_catalogue(300, 10_000, nnz=60, n_genres=20, seed=4).features()["text_features"].tocsr())
    x.sort_indices()
    plan = model_plan(x.indices, 10_000, 4024)
    got = model_operand(x.indptr, x.indices, x.data, plan, 4160, 64, 256.0, dtype)
    m = merged_dense(x, plan[0], 4024) * 256.0
    want = m.astype(np.float16).view(np.uint16) if dtype == "fp16" else bf16_bits(m)
    assert np.array_equal(got[:, 64:64 + 4024], want)
    assert not got[:, :64].any() and not got[:, 64 + 4024:].any()
    assert np.array_equal(got[:, 64:64 + 4024] != 0, m > 0)
    if dtype == "bf16":      # merged sums are not float32 numbers in general; where they are, torch agrees
        sub = m.astype(np.float32).astype(np.float64) == m
        ref = torch.from_numpy(m.astype(np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
        assert np.array_equal(want[sub], ref[sub])


def test_operand_model_adds_in_slot_order():
    """Entries of one slot are added in slot_cols order, not in column order: a value on an fp16 tie
    and two tiny ones, whose float64 sum lands on either side of the tie depending on the order."""
    vocab, text_cols = 6, 2                     # head: rank 0; the tail slot takes the five others
    plan = model_plan(np.r_[np.repeat(5, 4), np.repeat(1, 3), np.repeat(3, 2), 0, 2, 4], vocab, text_cols)
    assert list(plan[2]) == [5, 1, 3, 0, 2, 4]
    a, b = 1 + 2.0 ** -11, 2.0 ** -53           # a: halfway between the fp16 numbers 1 and 1 + 2^-10
    x = _csr_rows([[1, 3, 4]], [a, b, b], vocab)
    got = model_operand(x.indptr, x.indices, x.data, plan, 2, 0, 1.0, "fp16")
    assert (a + b) + b == a and got[0, 1] == 0x3C00              # column 1 first: the tiny ones vanish
    plan2 = (plan[0], plan[1], np.array([5, 3, 4, 1, 0, 2]))     # columns 3 and 4 first: they add up to 2^-52
    got2 = model_operand(x.indptr, x.indices, x.data, plan2, 2, 0, 1.0, "fp16")
    assert (b + b) + a > a and got2[0, 1] == 0x3C01


def test_merged_slack_grows_the_subnormal_term_only():
    """tvbf_debug_slack (host only): a merged operand entry sums at most V - text_cols + 1 entries of
    a unit row, so the fp16 subnormal allowance eps_term grows by sqrt(V - text_cols + 1); the
    relative terms stay as they are"""
    from tvbingefriend_recommendation_service_b200 import _lib

    lib = _lib.load()
    for vocab, text_cols in ((10_000, 4024), (50_000, 20_000), (4097, 2), (6000, 4024)):
        f = _lib.Features(n_shows=10, n_pad=256, k_pad=(text_cols + 63) // 64 * 64, text_dtype=_lib.TEXT_FP16,
                          text_scale_log2=8, vocab=vocab, operand=1 << 20, text_indptr=1 << 21,
                          text_indices=1 << 22, text_values=1 << 23, col_side=1 << 24, meta_scale=1 << 25,
                          genre_mode=_lib.GROUP_PACKED, genre_dim=40, meta_mode=_lib.GROUP_PACKED)
        p = _lib.Params(genre_weight=0.4, text_weight=0.5, metadata_weight=0.1, min_similarity=0.1, k=60,
                        exclude_self=1, row_begin=0, row_end=10)
        out = {}
        for cols in (0, text_cols):
            f.text_cols = cols
            o = (C.c_float * 5)()
            assert lib.tvbf_debug_slack(C.byref(f), C.byref(p), o) == 0
            out[cols] = list(o)
        plain, merged = out[0], out[text_cols]
        assert merged[:4] == plain[:4], (vocab, text_cols)
        assert plain[4] > 0.0
        assert merged[4] / plain[4] == pytest.approx(np.sqrt(vocab - text_cols + 1), rel=2 ** -22), (vocab, text_cols)
        f.text_dtype = _lib.TEXT_BF16                 # bf16 has no subnormal range that matters here
        f.text_cols = text_cols
        o = (C.c_float * 5)()
        assert lib.tvbf_debug_slack(C.byref(f), C.byref(p), o) == 0 and o[4] == 0.0
