"""Host side of the B200 hybrid-similarity -> top-K path.

PyTorch is plumbing here: it owns device memory, streams and (for several GPUs)
``torch.distributed``; all arithmetic is in ``libtvbf.so`` (hand-written sm_100a CUDA) reached
through the C ABI of ``include/tvbf.h``.  There is no CPU fallback.

Pipeline for one catalogue (reference: scripts/populate_database.py:125-218):

    stage()   host: classify the five feature matrices, convert to the transfer layout, pin
    upload()  H2D + K0 prep kernels: fp64 row normalisation, fp16 operand, genre bitmasks, ids
    top_k()   K1 tcgen05 candidate pass -> K5 fp64 rescore + certificate -> K6 exact repair
    to_host() D2H of the [rows, k] table
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import os

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib
from ._lib import Features, Params, TopKOut, check

TEXT_SCALE_LOG2 = 8          # operand text columns hold x * 2^8 (keeps tiny tf-idf values normal in fp16)
_DTYPES = {"fp16": (_lib.TEXT_FP16, torch.float16), "bf16": (_lib.TEXT_BF16, torch.bfloat16)}


def _is_binary(a: np.ndarray) -> bool:
    if a.dtype == np.bool_:
        return True
    return bool(np.all((a == 0) | (a == 1)))


def _is_one_hot(a: np.ndarray) -> bool:
    """values in {0,1}, at most one 1 per row."""
    if a.ndim != 2 or a.shape[1] == 0:
        return False
    if not _is_binary(a):
        return False
    return bool((np.count_nonzero(a, axis=1) <= 1).all())


def _pin(t: torch.Tensor, pin: bool) -> torch.Tensor:
    return t.pin_memory() if pin and torch.cuda.is_available() else t


@dataclass
class StagedCatalogue:
    """Host-side transfer buffers (pinned when a GPU is present) + how each group is scored."""

    n_shows: int
    vocab: int
    metadata_mode: str                      # "mean3" | "hstack"
    text_indptr: torch.Tensor               # int64 [N+1]
    text_indices: torch.Tensor              # int32 [nnz]
    text_values: torch.Tensor               # float64 [nnz]
    genre_packed: bool
    genre: torch.Tensor                     # uint8 [N,G] (packed) or float64 [N,G] (folded)
    meta_packed: bool
    meta: list                              # 3 x uint8 one-hot (packed) or float64 groups (folded)
    text_signed: bool = False               # any negative text value (embeddings / SVD instead of TF-IDF)

    def h2d_bytes(self) -> int:
        ts = [self.text_indptr, self.text_indices, self.text_values, self.genre, *self.meta]
        return int(sum(t.numel() * t.element_size() for t in ts))


def stage(features: dict, metadata_mode: str = "mean3", pin: bool = True) -> StagedCatalogue:
    """Classify and convert the reference's feature dict (keys of compute_all_similarities,
    ml/similarity_computer.py:132-155) into transfer buffers.  Pure host code."""
    if metadata_mode not in ("mean3", "hstack"):
        raise ValueError(f"metadata_mode must be 'mean3' or 'hstack', got {metadata_mode!r}")
    genre = np.asarray(features["genre_features"])
    text = features["text_features"]
    plat = np.asarray(features["platform_features"])
    typ = np.asarray(features["type_features"])
    lang = np.asarray(features["language_features"])
    n = int(genre.shape[0])
    text = sp.csr_matrix(text, dtype=np.float64) if not sp.issparse(text) or text.format != "csr" \
        or text.dtype != np.float64 else text
    if not text.has_canonical_format:
        text = text.copy()
        text.sum_duplicates()
        text.sort_indices()
    for name, a in (("text", text), ("platform", plat), ("type", typ), ("language", lang)):
        if a.shape[0] != n:
            raise ValueError(f"{name}_features has {a.shape[0]} rows, genre_features has {n}")
    genre_packed = genre.ndim == 2 and 1 <= genre.shape[1] <= 128 and _is_binary(genre)   # two 64-bit words
    # the three one-hot groups are packed into one 32-bit mask per show (reference defaults:
    # 21 platforms + 5 types + 6 languages = 32 columns, feature_extractor.py:122-193)
    meta_packed = (plat.shape[1] + typ.shape[1] + lang.shape[1] <= 32) and \
        all(_is_one_hot(a) for a in (plat, typ, lang))
    if genre_packed:
        g_t = torch.from_numpy(np.ascontiguousarray(genre != 0).astype(np.uint8))
    else:
        g_t = torch.from_numpy(np.ascontiguousarray(genre, dtype=np.float64))
    if meta_packed:
        meta = [torch.from_numpy(np.ascontiguousarray(a != 0).astype(np.uint8)) for a in (plat, typ, lang)]
    elif metadata_mode == "mean3":
        meta = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)) for a in (plat, typ, lang)]
    else:  # similarity_computer.py:84 -- one cosine over the concatenation
        meta = [torch.from_numpy(np.ascontiguousarray(np.hstack([plat, typ, lang]), dtype=np.float64))]
    return StagedCatalogue(
        n_shows=n, vocab=int(text.shape[1]), metadata_mode=metadata_mode,
        text_indptr=_pin(torch.from_numpy(text.indptr.astype(np.int64)), pin),
        text_indices=_pin(torch.from_numpy(text.indices.astype(np.int32)), pin),
        text_values=_pin(torch.from_numpy(np.ascontiguousarray(text.data, dtype=np.float64)), pin),
        genre_packed=genre_packed, genre=_pin(g_t, pin),
        meta_packed=meta_packed, meta=[_pin(m, pin) for m in meta],
        text_signed=bool(text.nnz and text.data.min() < 0.0))


def merge_text_cols(vocab: int, genre_dim: int, fold_max_k: int = 4096, ratio: float = 0.4) -> int:
    """Text columns of the candidate pass' second operand for a vocabulary of ``vocab`` columns and
    ``genre_dim`` packed genre columns (``HybridTopKEngine.fold_max_k`` / ``merge_ratio``).  ``vocab``
    -- no merge -- while the text and the packed groups fit the fold limit (``vocab + genre_dim + 32
    <= fold_max_k``), when ``ratio`` or ``fold_max_k`` is 0, or when merging would not narrow the
    64-column padded operand; else ``max(fold_max_k - genre_dim - 32, ceil(ratio * vocab))``, so that
    the merged text and the packed groups still fit the fold limit.  Depends on shapes only, so the
    host never waits for the device to choose it."""
    v, lim = int(vocab), int(fold_max_k)
    if ratio <= 0.0 or lim <= 0 or v + genre_dim + 32 <= lim:
        return v
    kt = max(lim - genre_dim - 32, int(np.ceil(ratio * v)), 2)
    head = kt // 2
    # tvbf_merge_plan takes at most 4096 vocabulary columns per operand column
    if (kt + 63) // 64 >= (v + 63) // 64 or -(-(v - head) // (kt - head)) > 4096:
        return v
    return kt


@dataclass
class DeviceCatalogue:
    """Prepared, device-resident features (``tvbf_features``) and the tensors that back it."""

    c: Features
    n_shows: int
    folded: bool
    weights_baked: tuple | None            # folded groups bake sqrt(w/w_text) into the operand
    keep: list = field(default_factory=list)
    operand: torch.Tensor | None = None    # [n_pad, k_pad] fp16 / bf16
    text_indptr: torch.Tensor | None = None
    text_indices: torch.Tensor | None = None
    fold: dict | None = None               # second operand of the candidate pass: merged text and / or the packed groups (engine._folded)
    buffers: dict = field(default_factory=dict)   # named per-catalogue device buffers a later catalogue can take over
    h2d_set: tuple | None = None           # (h2d buffer set, its write stamp) when the CSR lives in an h2d(reuse=True) set
    parts: dict = field(default_factory=dict)     # the tensors behind ``c`` by name and the text nnz (``extend``)


@dataclass
class TopK:
    """Columnar top-K table of source rows [row_begin, row_begin + R) -- the record stream of
    scripts/populate_database.py:211-217."""

    indices: np.ndarray      # int32 [R, k], -1 padded (column = position in show_ids)
    counts: np.ndarray       # int32 [R]
    hybrid: np.ndarray       # float64 [R, k] similarity_score
    genre: np.ndarray        # float64 [R, k]
    text: np.ndarray         # float64 [R, k]
    metadata: np.ndarray     # float64 [R, k]
    row_begin: int = 0
    flagged_rows: int = 0    # rows the certificate sent to the exact kernel
    rescored_pairs: int = 0
    changed_rows: np.ndarray | None = None   # extend_top_k / update_top_k: sorted int32 rows that changed

    @property
    def k(self) -> int:
        return int(self.indices.shape[1])

    def slice(self, begin: int, end: int) -> "TopK":
        """Rows [begin, end) of this table (positions within the table) as a view."""
        return TopK(self.indices[begin:end], self.counts[begin:end], self.hybrid[begin:end], self.genre[begin:end],
                    self.text[begin:end], self.metadata[begin:end], row_begin=self.row_begin + begin)

    @staticmethod
    def _ids(show_ids) -> np.ndarray:
        return show_ids if isinstance(show_ids, np.ndarray) else np.asarray(list(show_ids))

    def to_dict(self, show_ids, id_key: str = "similar_show_id") -> dict:
        """``all_similarities`` exactly as the hot loop builds it (populate_database.py:208-221):
        shows without a qualifying neighbour are omitted."""
        ids = self._ids(show_ids)
        # bulk conversion to Python scalars first: 2 M records of C3 take 2.2 s this way, 3.0 s with
        # per-element float()/int() calls (the dicts themselves are the rest)
        sim = ids[np.where(self.indices >= 0, self.indices, 0)].tolist()
        hyb, gen, txt, met = self.hybrid.tolist(), self.genre.tolist(), self.text.tolist(), self.metadata.tolist()
        cnt = self.counts.tolist()
        own = ids[self.row_begin:self.row_begin + len(cnt)].tolist()
        out = {}
        for r, c in enumerate(cnt):
            if c == 0:
                continue
            sr, hr, gr, tr, mr = sim[r], hyb[r], gen[r], txt[r], met[r]
            out[own[r]] = [{id_key: sr[e], "similarity_score": hr[e], "genre_score": gr[e], "text_score": tr[e],
                            "metadata_score": mr[e]} for e in range(c)]
        return out

    def records(self, show_ids) -> dict:
        """Flat columnar records (one per kept pair, in table order) for a bulk sink
        (repos/similarity_repository.py:72-108 row shape) without building N*k dicts."""
        ids = self._ids(show_ids)
        n, k = self.indices.shape
        if n and int(self.counts.min()) == k:      # every show has k neighbours: plain reshapes, no masks
            return {"show_id": np.repeat(ids[self.row_begin:self.row_begin + n], k),
                    "similar_show_id": ids[self.indices.reshape(-1)],
                    "similarity_score": self.hybrid.reshape(-1), "genre_score": self.genre.reshape(-1),
                    "text_score": self.text.reshape(-1), "metadata_score": self.metadata.reshape(-1)}
        mask = np.arange(k)[None, :] < self.counts[:, None]
        rows = np.nonzero(mask)[0]
        return {"show_id": ids[self.row_begin + rows],
                "similar_show_id": ids[self.indices[mask]],
                "similarity_score": self.hybrid[mask], "genre_score": self.genre[mask],
                "text_score": self.text[mask], "metadata_score": self.metadata[mask]}


@dataclass
class NeighbourTable:
    """Every neighbour at or above ``min_similarity`` of source rows [row_begin, row_begin + R): row r is
    entries ``row_ptr[r] .. row_ptr[r + 1]``, ordered by (score descending, column ascending) -- the
    record stream of scripts/populate_database.py:211-217 cut by the threshold alone (or also by
    ``max_per_row``)."""

    row_ptr: np.ndarray      # int64 [R + 1], row_ptr[0] == 0
    indices: np.ndarray      # int32 [row_ptr[R]] (column = position in show_ids)
    hybrid: np.ndarray       # float64 [row_ptr[R]] similarity_score
    genre: np.ndarray
    text: np.ndarray
    metadata: np.ndarray
    candidate_pairs: int = 0   # pairs i < j the tensor-core sweep passed to the float64 finish
    row_begin: int = 0
    flagged_rows: int = 0      # always 0: the threshold job has no certificate to fail

    @property
    def counts(self) -> np.ndarray:
        return np.diff(self.row_ptr).astype(np.int32)

    def slice(self, begin: int, end: int) -> "NeighbourTable":
        """Rows [begin, end) of this table (positions within the table); the arrays are views."""
        b, e = int(self.row_ptr[begin]), int(self.row_ptr[end])
        return NeighbourTable(self.row_ptr[begin:end + 1] - b, self.indices[b:e], self.hybrid[b:e], self.genre[b:e],
                              self.text[b:e], self.metadata[b:e], candidate_pairs=self.candidate_pairs,
                              row_begin=self.row_begin + begin)

    def to_dict(self, show_ids, id_key: str = "similar_show_id") -> dict:
        """``all_similarities`` as the hot loop builds it, in the shape of ``TopK.to_dict``: shows
        without a qualifying neighbour are omitted."""
        ids = TopK._ids(show_ids)
        sim = ids[self.indices].tolist()
        hyb, gen, txt, met = self.hybrid.tolist(), self.genre.tolist(), self.text.tolist(), self.metadata.tolist()
        ptr = self.row_ptr.tolist()
        own = ids[self.row_begin:self.row_begin + len(ptr) - 1].tolist()
        out = {}
        for r in range(len(ptr) - 1):
            b, e = ptr[r], ptr[r + 1]
            if b == e:
                continue
            out[own[r]] = [{id_key: sim[q], "similarity_score": hyb[q], "genre_score": gen[q], "text_score": txt[q],
                            "metadata_score": met[q]} for q in range(b, e)]
        return out

    def records(self, show_ids) -> dict:
        """Flat columnar records (one per pair, in table order), as ``TopK.records``."""
        ids = TopK._ids(show_ids)
        rows = np.repeat(np.arange(len(self.row_ptr) - 1), np.diff(self.row_ptr))
        return {"show_id": ids[self.row_begin + rows], "similar_show_id": ids[self.indices],
                "similarity_score": self.hybrid, "genre_score": self.genre, "text_score": self.text,
                "metadata_score": self.metadata}


class HybridTopKEngine:
    """One engine per process / GPU.  It caches a device workspace and pinned host buffers, so it
    must not be shared between threads that run jobs concurrently (the reference's callers are
    single-threaded, SURVEY.md section 8b); create one engine per thread instead.  All work is
    issued on the current torch CUDA stream of ``device``."""

    def __init__(self, device: int | str | torch.device | None = None, text_dtype: str = "fp16"):
        self.lib = _lib.load()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() \
                else torch.device("cuda", 0)
        self.device = torch.device(device) if not isinstance(device, int) else torch.device("cuda", device)
        with torch.cuda.device(self.device) if torch.cuda.is_available() else _NullCtx():
            self.sm_count, self.cc_major, self.cc_minor = _lib.require_device()
        if text_dtype not in _DTYPES:
            raise ValueError(f"text_dtype must be one of {list(_DTYPES)}")
        self.text_dtype = text_dtype
        self._launch_base = int(self.lib.tvbf_kernel_launches())
        self._ws: torch.Tensor | None = None
        self._pinned: dict = {}
        # Small vocabularies: the candidate pass is bound by its epilogue, not by the MMAs, so the
        # packed genre / metadata groups are ALSO written into a second operand as K columns and the
        # epilogue drops its popcounts (tvbf_features.bits_folded).  Used while the widened operand
        # has at most fold_max_k columns (0 disables; TVBF_FOLD_MAX_K overrides).  Measured at
        # N = 80 000 (tools/time_fold_crossover.py), K1 ms popcount / folded: V = 500 8.9 / 6.3,
        # 1 000 7.9 / 6.0, 1 900 9.4 / 7.9, 3 000 12.2 / 11.5, 4 500 17.2 / 16.9 -- the gain fades as the
        # MMAs take over; the folded bound is slightly looser (3-5 % more rows go to the exact kernel).
        self.fold_max_k = int(os.environ.get("TVBF_FOLD_MAX_K", "4096"))
        # Large vocabularies: the candidate pass is bound by its MMAs over an operand that is 99.5 %
        # zeros.  For non-negative text it only needs an upper bound of the text cosine, and summing
        # vocabulary columns gives one (x_i . x_j <= merged x_i . merged x_j), so the second operand
        # carries the text merged into merge_text_cols(V, G, ...) columns (DESIGN.md section 14).  0 disables
        # (TVBF_MERGE_RATIO overrides); fold_max_k = 0 disables it too.
        self.merge_ratio = float(os.environ.get("TVBF_MERGE_RATIO", "0.4"))
        self._fold_buf: torch.Tensor | None = None
        self._fold_owner: dict | None = None      # the catalogue fold whose content the buffer holds
        self._theta: torch.Tensor | None = None    # seeded thresholds of the tile-sharded job (valid until the next job)
        self._h2d_stamp = 0                         # writes into the h2d(reuse=True) sets so far

    @property
    def kernel_launches(self) -> int:
        """CUDA kernels libtvbf has launched since this engine was created (counted inside the
        library at every launch)."""
        return int(self.lib.tvbf_kernel_launches()) - self._launch_base

    # ------------------------------------------------------------------------------------ utils
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def release(self) -> None:
        """Drop the cached device workspace and pinned host buffers (they are re-created on demand);
        useful between jobs of very different size, e.g. after a 200 k x 50 k catalogue."""
        self._ws = None
        self._pinned.clear()
        self._fold_buf = None
        self._fold_owner = None
        self._theta = None
        if torch.cuda.is_available():
            with torch.cuda.device(self.device):
                torch.cuda.empty_cache()

    def _workspace(self, nbytes: int) -> torch.Tensor:
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
        return self._ws

    # ------------------------------------------------------------------------------------ upload
    def h2d(self, st: StagedCatalogue, reuse: bool = False) -> dict:
        """Host -> device copies of the staged buffers on the current stream (no kernels).
        ``reuse``: copy into cached device buffers (two sets used in turn, so a stream of jobs allocates
        nothing and the previous job's arrays -- which ``prepare(recycle=...)`` still reads to un-scatter
        the operand -- stay intact); the tensors of the call before the previous one are overwritten.
        Each write stamps its set, so ``prepare`` can tell when a recycled catalogue's CSR arrays have
        been overwritten since (it then zeroes the whole operand instead of un-scattering it); a
        catalogue whose set has been overwritten must not run jobs any more."""
        dev = self.device
        cache = None
        if reuse:
            gen = self._pinned.setdefault(("h2d_gen",), [0])
            gen[0] ^= 1
            cache = self._pinned.setdefault(("h2d", gen[0]), {})
            self._h2d_stamp += 1
            cache["stamp"] = self._h2d_stamp

        def up(name: str, h: torch.Tensor) -> torch.Tensor:
            if cache is None:
                return h.to(dev, non_blocking=True)
            d = cache.get(name)
            if d is None or d.shape != h.shape or d.dtype != h.dtype:
                d = cache[name] = torch.empty(h.shape, dtype=h.dtype, device=dev)
            d.copy_(h, non_blocking=True)
            return d

        with torch.cuda.device(dev):
            return {"st": st, "indptr": up("indptr", st.text_indptr), "indices": up("indices", st.text_indices),
                    "values": up("values", st.text_values), "genre": up("genre", st.genre),
                    "meta": [up(f"meta{i}", m) for i, m in enumerate(st.meta)],
                    "h2d_set": None if cache is None else (cache, cache["stamp"])}

    def upload(self, st: StagedCatalogue, weights: tuple[float, float, float] = (0.4, 0.5, 0.1),
               recycle: DeviceCatalogue | None = None) -> DeviceCatalogue:
        """H2D copies + K0 prep kernels."""
        return self.prepare(self.h2d(st), weights, recycle)

    def _zero(self, t: torch.Tensor) -> None:
        check(self.lib.tvbf_device_zero(t.data_ptr(), t.numel() * t.element_size(), self._stream()),
              "tvbf_device_zero")

    def prepare(self, raw: dict, weights: tuple[float, float, float] = (0.4, 0.5, 0.1),
                recycle: DeviceCatalogue | None = None) -> DeviceCatalogue:
        """K0 prep kernels on device-resident raw features.  ``weights`` matter only when a group
        is folded into the tensor-core operand (general float features).

        ``recycle``: a catalogue this engine prepared earlier and the caller no longer needs.  Its
        operand buffer is taken over -- the positions its CSR had set are zeroed (one store per old
        non-zero) instead of clearing a fresh N x V array -- and the old catalogue becomes unusable.
        When that CSR came from an ``h2d(reuse=True)`` set that a later ``h2d`` has overwritten (the
        call before the previous one, e.g. ``raw`` itself), its positions are no longer known and the
        whole operand is zeroed instead."""
        lib, dev, stream = self.lib, self.device, None
        st: StagedCatalogue = raw["st"]
        gw, tw, mw = (float(w) for w in weights)
        with torch.cuda.device(dev):
            stream = self._stream()
            n, v = st.n_shows, st.vocab
            n_pad = (n + 255) // 256 * 256
            folded_dims = (0 if st.genre_packed else st.genre.shape[1]) + \
                (0 if st.meta_packed else sum(m.shape[1] for m in st.meta))
            k_pad = max(64, (v + folded_dims + 63) // 64 * 64)
            code, tdt = _DTYPES[self.text_dtype]
            keep = []
            indptr, indices, rawv = raw["indptr"], raw["indices"], raw["values"]
            if rawv.numel() == 0:
                # a catalogue without any text: the C ABI wants non-NULL arrays, which are never read
                indices = torch.zeros((1,), dtype=torch.int32, device=dev)
                rawv = torch.zeros((1,), dtype=torch.float64, device=dev)
            # a recycled catalogue hands over all its same-shaped buffers: a steady stream of jobs then
            # allocates nothing (torch's caching allocator otherwise falls back to cudaMalloc -- a device
            # synchronisation of tens of milliseconds -- whenever the lifetimes of a step's tensors shift)
            spare = dict(recycle.buffers) if recycle is not None else {}

            def take(name, shape, dtype):
                t = spare.pop(name, None)
                if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != dev:
                    t = torch.empty(shape, dtype=dtype, device=dev)
                return t

            values, operand = self._text_operand(indptr, indices, rawv, n, n_pad, k_pad, recycle,
                                                 folded=folded_dims > 0, values=take("values", rawv.shape, rawv.dtype))
            col_side = take("col_side", (n_pad, 2), torch.int64)   # 16-byte records
            meta_scale = take("meta_scale", (n_pad,), torch.float32)
            self._zero(col_side)
            self._zero(meta_scale)
            keep += [indptr, indices, values, operand, col_side, meta_scale]
            scale = float(2 ** TEXT_SCALE_LOG2)

            f = Features()
            f.n_shows, f.n_pad, f.k_pad, f.text_dtype = n, n_pad, k_pad, code
            f.text_scale_log2, f.vocab = TEXT_SCALE_LOG2, v
            f.operand = operand.data_ptr()
            f.text_indptr, f.text_indices, f.text_values = indptr.data_ptr(), indices.data_ptr(), values.data_ptr()
            f.text_nnz = int(raw["values"].numel())
            f.col_side, f.meta_scale = col_side.data_ptr(), meta_scale.data_ptr()
            f.text_signed = int(st.text_signed)
            f.meta_kind = _lib.META_MEAN3 if st.metadata_mode == "mean3" else _lib.META_HSTACK
            col = v
            folded = False
            dense = {}

            def fold(g_raw: torch.Tensor, weight: float, what: str) -> int:
                nonlocal col, folded
                if tw <= 0.0 or weight < 0.0:
                    raise _lib.TvbfError(
                        f"{what} features are not binary/one-hot and must be folded into the tensor-core "
                        "operand, which needs text_weight > 0 and non-negative weights; "
                        "use force_exact=True for this weight combination")
                ratio = weight / tw
                if ratio > 6.0e4:
                    raise _lib.TvbfError(f"{what}: weight ratio {ratio} overflows the fp16 operand")
                g_norm = torch.empty_like(g_raw)
                check(lib.tvbf_prep_dense_normalize(g_raw.data_ptr(), n, g_raw.shape[1], g_norm.data_ptr(), stream),
                      "tvbf_prep_dense_normalize")
                check(lib.tvbf_prep_dense_to_operand(g_norm.data_ptr(), n, g_norm.shape[1], operand.data_ptr(),
                                                     k_pad, col, scale * float(np.sqrt(ratio)), code, stream),
                      "tvbf_prep_dense_to_operand")
                keep.append(g_norm)
                dense.setdefault(what, []).append(g_norm)
                col += g_norm.shape[1]
                folded = True
                return g_norm.data_ptr()

            if st.genre_packed:
                g8 = raw["genre"]
                genre_hi = None
                if g8.shape[1] > 64:      # second mask word for genre columns 64..127
                    genre_hi = take("genre_hi", (n_pad,), torch.int64)
                    self._zero(genre_hi)
                    keep.append(genre_hi)
                    f.genre_hi = genre_hi.data_ptr()
                check(lib.tvbf_prep_genre_bits(g8.data_ptr(), n, g8.shape[1], col_side.data_ptr(),
                                               None if genre_hi is None else genre_hi.data_ptr(), stream),
                      "tvbf_prep_genre_bits")
                f.genre_mode, f.genre_dim = _lib.GROUP_PACKED, int(g8.shape[1])
            else:
                f.genre_mode, f.genre_dim = _lib.GROUP_FOLDED, int(st.genre.shape[1])
                f.genre_dense = fold(raw["genre"], gw, "genre")
            if st.meta_packed:
                m8 = raw["meta"]
                check(lib.tvbf_prep_meta_ids(m8[0].data_ptr(), m8[0].shape[1], m8[1].data_ptr(), m8[1].shape[1],
                                             m8[2].data_ptr(), m8[2].shape[1], n, n_pad, f.meta_kind,
                                             col_side.data_ptr(), meta_scale.data_ptr(), stream),
                      "tvbf_prep_meta_ids")
                f.meta_mode = _lib.GROUP_PACKED
            else:
                f.meta_mode = _lib.GROUP_FOLDED
                f.meta_groups = len(st.meta)
                per_group_w = mw / 3.0 if st.metadata_mode == "mean3" else mw
                for gi, m in enumerate(raw["meta"]):
                    f.meta_dims[gi] = int(m.shape[1])
                    f.meta_dense[gi] = fold(m, per_group_w, "metadata")
            keep.append(raw)
        bufs = {"values": values, "col_side": col_side, "meta_scale": meta_scale}
        if f.genre_hi:
            bufs["genre_hi"] = genre_hi
        if recycle is not None:
            recycle.buffers = {}
        parts = {"values": values, "col_side": col_side, "meta_scale": meta_scale,
                 "genre_hi": genre_hi if f.genre_hi else None, "nnz": int(raw["values"].numel()),
                 "genre_dense": dense.get("genre", [None])[0], "meta_dense": dense.get("metadata", []),
                 "meta_widths": tuple(int(m.shape[1]) for m in st.meta)}
        return DeviceCatalogue(c=f, n_shows=n, folded=folded,
                               weights_baked=(gw, tw, mw) if folded else None, keep=keep,
                               operand=operand, text_indptr=indptr, text_indices=indices, buffers=bufs,
                               h2d_set=raw.get("h2d_set"), parts=parts)

    # ------------------------------------------------------------------------------------ device-side ingest
    _RAW_DTYPES = {np.dtype(np.bool_): 0, np.dtype(np.uint8): 0, np.dtype(np.int32): 1, np.dtype(np.int64): 2,
                   np.dtype(np.float32): 3, np.dtype(np.float64): 4}

    def _stage_bytes(self, name: str, arr: np.ndarray) -> torch.Tensor:
        """Copy ``arr``'s bytes into a cached pinned buffer and start the H2D copy; returns the device
        bytes (uint8).  The pinned buffers are reused from call to call (no page-locking per job)."""
        import warnings

        a = np.ascontiguousarray(arr)
        nbytes = a.nbytes
        buf = self._pinned.get(("raw", name))
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty((max(nbytes, 1),), dtype=torch.uint8, pin_memory=True)
            self._pinned[("raw", name)] = buf
        dev = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=self.device)
        if nbytes:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")          # read-only arrays (np.load with mmap_mode) are fine here
                src = torch.from_numpy(a.reshape(-1).view(np.uint8))
            buf[:nbytes].copy_(src)
            dev[:nbytes].copy_(buf[:nbytes], non_blocking=True)
        return dev

    def ingest(self, features: dict, metadata_mode: str = "mean3",
               weights: tuple[float, float, float] = (0.4, 0.5, 0.1),
               recycle: DeviceCatalogue | None = None) -> DeviceCatalogue:
        """features dict (as ``np.load`` / ``load_npz`` hand it over) -> device catalogue with the
        classification and narrowing done ON THE GPU (SURVEY.md section 8f-3): the host only copies
        the raw bytes -- int64 multi-hot genres, float64 / bool one-hots, the CSR arrays in whatever
        index width scipy chose -- through cached pinned buffers; kernels check {0,1}-valuedness /
        one-hotness / sortedness / sign while they pack, and one int32 of flags comes back.  Inputs
        the packed path cannot take (general float groups, more than 64 genre or 32 metadata
        columns, exotic dtypes) go through the host ``stage()`` as before."""
        if metadata_mode not in ("mean3", "hstack"):
            raise ValueError(f"metadata_mode must be 'mean3' or 'hstack', got {metadata_mode!r}")
        genre = np.asarray(features["genre_features"])
        text = features["text_features"]
        groups = [np.asarray(features[k_]) for k_ in ("platform_features", "type_features", "language_features")]

        def slow():
            return self.upload(stage(features, metadata_mode), weights, recycle)

        if not (sp.issparse(text) and text.format == "csr"):
            return slow()
        ok = genre.ndim == 2 and 1 <= genre.shape[1] <= 128 and genre.dtype in self._RAW_DTYPES
        ok = ok and all(a.ndim == 2 and a.dtype in self._RAW_DTYPES for a in groups)
        ok = ok and sum(a.shape[1] for a in groups) <= 32 and all(a.shape[1] >= 1 for a in groups)
        ok = ok and text.data.dtype in (np.float32, np.float64) and text.indptr.dtype in (np.int32, np.int64) \
            and text.indices.dtype in (np.int32, np.int64)
        if not ok:
            return slow()
        n = int(genre.shape[0])
        for name, a in (("text", text), ("platform", groups[0]), ("type", groups[1]), ("language", groups[2])):
            if a.shape[0] != n:
                raise ValueError(f"{name}_features has {a.shape[0]} rows, genre_features has {n}")
        lib, dev = self.lib, self.device
        v = int(text.shape[1])
        nnz = int(text.indptr[-1])
        n_pad = (n + 255) // 256 * 256
        kind = _lib.META_MEAN3 if metadata_mode == "mean3" else _lib.META_HSTACK
        with torch.cuda.device(dev):
            stream = self._stream()
            d_indptr = self._stage_bytes("indptr", text.indptr)
            d_indices = self._stage_bytes("indices", text.indices[:nnz])
            d_values = self._stage_bytes("values", text.data[:nnz])
            d_genre = self._stage_bytes("genre", genre)
            d_groups = [self._stage_bytes(f"meta{g}", a) for g, a in enumerate(groups)]
            flags = torch.empty((1,), dtype=torch.int32, device=dev)
            self._zero(flags)
            indptr = torch.empty((n + 1,), dtype=torch.int64, device=dev)
            indices = torch.empty((max(nnz, 1),), dtype=torch.int32, device=dev)
            rawv = torch.empty((max(nnz, 1),), dtype=torch.float64, device=dev)
            col_side = torch.empty((n_pad, 2), dtype=torch.int64, device=dev)
            meta_scale = torch.empty((n_pad,), dtype=torch.float32, device=dev)
            check(lib.tvbf_ingest_csr(d_indptr.data_ptr(), int(text.indptr.dtype == np.int64), d_indices.data_ptr(),
                                      int(text.indices.dtype == np.int64), d_values.data_ptr(),
                                      int(text.data.dtype == np.float64), n, indptr.data_ptr(), indices.data_ptr(),
                                      rawv.data_ptr(), flags.data_ptr(), stream), "tvbf_ingest_csr")
            genre_hi = torch.empty((n_pad,), dtype=torch.int64, device=dev) if genre.shape[1] > 64 else None
            check(lib.tvbf_ingest_genre(d_genre.data_ptr(), self._RAW_DTYPES[genre.dtype], n, n_pad, int(genre.shape[1]),
                                        col_side.data_ptr(), None if genre_hi is None else genre_hi.data_ptr(),
                                        flags.data_ptr(), stream), "tvbf_ingest_genre")
            g0, g1, g2 = groups
            check(lib.tvbf_ingest_meta(d_groups[0].data_ptr(), self._RAW_DTYPES[g0.dtype], int(g0.shape[1]),
                                       d_groups[1].data_ptr(), self._RAW_DTYPES[g1.dtype], int(g1.shape[1]),
                                       d_groups[2].data_ptr(), self._RAW_DTYPES[g2.dtype], int(g2.shape[1]), n, n_pad,
                                       kind, col_side.data_ptr(), meta_scale.data_ptr(), flags.data_ptr(), stream),
                  "tvbf_ingest_meta")
            bits = int(flags.item())           # the one synchronisation of the ingest
            if bits & 7:
                # not binary / not one-hot -> general float path; unsorted or duplicated CSR entries ->
                # scipy canonicalises on the host (both rare: compute_features.py writes neither)
                return slow()
            code, tdt = _DTYPES[self.text_dtype]
            k_pad = max(64, (v + 63) // 64 * 64)
            values, operand = self._text_operand(indptr, indices, rawv, n, n_pad, k_pad, recycle)
            f = Features()
            f.n_shows, f.n_pad, f.k_pad, f.text_dtype = n, n_pad, k_pad, code
            f.text_scale_log2, f.vocab = TEXT_SCALE_LOG2, v
            f.operand = operand.data_ptr()
            f.text_indptr, f.text_indices, f.text_values = indptr.data_ptr(), indices.data_ptr(), values.data_ptr()
            f.text_nnz = nnz
            f.col_side, f.meta_scale = col_side.data_ptr(), meta_scale.data_ptr()
            f.meta_kind = kind
            f.genre_mode, f.genre_dim = _lib.GROUP_PACKED, int(genre.shape[1])
            f.genre_hi = None if genre_hi is None else genre_hi.data_ptr()
            f.meta_mode = _lib.GROUP_PACKED
            f.text_signed = int(bool(bits & 8))
        return DeviceCatalogue(c=f, n_shows=n, folded=False, weights_baked=None,
                               keep=[indptr, indices, values, operand, col_side, meta_scale, genre_hi],
                               operand=operand, text_indptr=indptr, text_indices=indices,
                               parts={"values": values, "col_side": col_side, "meta_scale": meta_scale,
                                      "genre_hi": genre_hi, "nnz": nnz, "genre_dense": None, "meta_dense": [],
                                      "meta_widths": tuple(int(a.shape[1]) for a in groups)})

    def _text_operand(self, indptr, indices, rawv, n: int, n_pad: int, k_pad: int,
                      recycle: DeviceCatalogue | None, folded: bool = False, values: torch.Tensor | None = None):
        """fp64 row normalisation of the CSR values + the fp16 / bf16 tensor-core operand (fresh and
        zeroed, or ``recycle``'s with its old positions cleared)."""
        lib, dev, stream = self.lib, self.device, self._stream()
        code, tdt = _DTYPES[self.text_dtype]
        if values is None:
            values = torch.empty_like(rawv)
        operand = None
        if (recycle is not None and recycle.operand is not None and not recycle.folded and not folded
                and tuple(recycle.operand.shape) == (n_pad, k_pad) and recycle.operand.dtype == tdt
                and recycle.operand.device == dev):
            operand = recycle.operand
            src = recycle.h2d_set
            if src is None or src[0]["stamp"] == src[1]:
                check(lib.tvbf_prep_clear_csr_positions(recycle.text_indptr.data_ptr(),
                                                        recycle.text_indices.data_ptr(), recycle.n_shows,
                                                        operand.data_ptr(), k_pad, 0, code, stream),
                      "tvbf_prep_clear_csr_positions")
            else:           # the h2d set holding its CSR has been overwritten since
                self._zero(operand)
            recycle.operand = None          # ownership moved: the old catalogue must not be used again
            recycle.c.operand = None
            recycle.keep.clear()
        if operand is None:
            operand = torch.empty((n_pad, k_pad), dtype=tdt, device=dev)
            self._zero(operand)
        check(lib.tvbf_prep_csr_normalize(indptr.data_ptr(), rawv.data_ptr(), n, values.data_ptr(), stream),
              "tvbf_prep_csr_normalize")
        check(lib.tvbf_prep_csr_to_operand(indptr.data_ptr(), indices.data_ptr(), values.data_ptr(), n,
                                           operand.data_ptr(), k_pad, 0, float(2 ** TEXT_SCALE_LOG2), code, stream),
              "tvbf_prep_csr_to_operand")
        return values, operand

    def _second_layout(self, cat: DeviceCatalogue, gw: float, tw: float, mw: float, k: int, tuning: int = 0,
                       candidates: int = 0) -> tuple[int, bool] | None:
        """(text columns, packed groups folded) of the operand the candidate pass of this job runs on
        instead of the catalogue's, or None for the catalogue's own operand (host only)."""
        c = cat.c
        if cat.folded or c.text_signed or self.text_dtype != "fp16" or cat.operand is None:
            return None
        g_dim = int(c.genre_dim)
        kt = merge_text_cols(int(c.vocab), g_dim, self.fold_max_k, self.merge_ratio)
        # the folded kernels exist for CTA pairs and up to 64 candidates per list
        bits = ((kt + g_dim + 32 + 63) // 64 * 64 <= self.fold_max_k and k <= 48
                and (tuning & 0xF) != 1 and candidates <= 64
                and c.genre_mode == _lib.GROUP_PACKED and c.meta_mode == _lib.GROUP_PACKED
                and tw > 0.0 and gw >= 0.0 and mw >= 0.0
                and all(w == 0.0 or 1e-8 <= w / tw <= 1e4 for w in (gw, mw)))   # columns stay normal fp16 numbers
        if bits:
            return kt, True
        if kt < int(c.vocab) and tw >= 0.0:
            return kt, False
        return None

    def _merge_plan(self, cat: DeviceCatalogue, text_cols: int) -> dict:
        """``tvbf_merge_plan`` of ``cat``'s text CSR onto ``text_cols`` columns (device tensors)."""
        lib, dev, c = self.lib, self.device, cat.c
        v = int(c.vocab)
        plan = {"col_map": torch.empty((v,), dtype=torch.int32, device=dev),
                "slot_ptr": torch.empty((text_cols + 1,), dtype=torch.int32, device=dev),
                "slot_cols": torch.empty((v,), dtype=torch.int32, device=dev)}
        ws = torch.empty((int(lib.tvbf_merge_plan_workspace_bytes(v)),), dtype=torch.uint8, device=dev)
        check(lib.tvbf_merge_plan(c.text_indptr, c.text_indices, cat.n_shows, v, text_cols,
                                  plan["col_map"].data_ptr(), plan["slot_ptr"].data_ptr(), plan["slot_cols"].data_ptr(),
                                  ws.data_ptr(), ws.numel(), self._stream()), "tvbf_merge_plan")
        return plan

    def _second_rows(self, fc: dict, indptr: int, indices: int, values: int, n_rows: int, dst: int,
                     col_side: int, genre_hi: int | None, meta_scale: int) -> None:
        """Write ``n_rows`` shows into the zeroed rows at ``dst`` of the second operand ``fc``: their
        text (through the merge plan when it has one) and, once the weights are set, their packed
        groups."""
        lib, stream = self.lib, self._stream()
        f = fc["c"]
        code, _ = _DTYPES[self.text_dtype]
        k2, scale = int(f.k_pad), float(2 ** TEXT_SCALE_LOG2)
        plan = fc["plan"]
        if plan is None:
            check(lib.tvbf_prep_csr_to_operand(indptr, indices, values, n_rows, dst, k2, 0, scale, code, stream),
                  "tvbf_prep_csr_to_operand")
        else:
            check(lib.tvbf_prep_csr_to_operand_mapped(indptr, indices, values, n_rows, plan["col_map"].data_ptr(),
                                                      plan["slot_ptr"].data_ptr(), plan["slot_cols"].data_ptr(), dst,
                                                      k2, 0, scale, code, stream), "tvbf_prep_csr_to_operand_mapped")
        if fc["weights"] is not None:
            gw, tw, mw = fc["weights"]
            check(lib.tvbf_prep_fold_bits(col_side, genre_hi, meta_scale, n_rows, int(f.genre_dim), dst, k2,
                                          int(f.fold_col0), scale * float(np.sqrt(gw / tw)),
                                          scale * float(np.sqrt(mw / tw)), code, stream), "tvbf_prep_fold_bits")

    def _folded(self, cat: DeviceCatalogue, gw: float, tw: float, mw: float, k: int, tuning: int = 0,
                candidates: int = 0) -> Features | None:
        """``tvbf_features`` of ``cat`` over the engine's second operand, or None when the job runs on
        the catalogue's own operand.  The second operand carries the text -- merged into fewer
        columns for large vocabularies (``merge_text_cols``) -- and, when the job qualifies, the
        packed genre / metadata groups as K columns for these weights (``_second_layout``)."""
        layout = self._second_layout(cat, gw, tw, mw, k, tuning, candidates)
        if layout is None:
            return None
        text_cols, bits = layout
        c = cat.c
        fc = cat.fold
        if fc is not None and (self._fold_owner is not fc or fc["layout"] != layout):
            fc = cat.fold = None                # the engine's buffer went to another catalogue or layout since
        if fc is None:
            n_pad = int(c.n_pad)
            k2 = (text_cols + (int(c.genre_dim) + 32 if bits else 0) + 63) // 64 * 64
            _, tdt = _DTYPES[self.text_dtype]
            buf = self._fold_buf
            if buf is None or tuple(buf.shape) != (n_pad, k2) or buf.dtype != tdt:
                self._fold_buf = None
                buf = torch.empty((n_pad, k2), dtype=tdt, device=self.device)
                self._fold_buf = buf            # one buffer per engine, reused by the next catalogue of this shape
            self._zero(buf)
            merged = text_cols < int(c.vocab)
            f = Features.from_buffer_copy(c)
            f.operand, f.k_pad = buf.data_ptr(), k2
            f.text_cols = text_cols if merged else 0
            f.bits_folded, f.fold_col0 = int(bits), text_cols if bits else 0
            fc = cat.fold = {"c": f, "operand": buf, "weights": None, "layout": layout,
                             "plan": self._merge_plan(cat, text_cols) if merged else None}
            self._fold_owner = fc
            self._second_rows(fc, c.text_indptr, c.text_indices, c.text_values, cat.n_shows, buf.data_ptr(),
                              c.col_side, c.genre_hi, c.meta_scale)
        if bits and fc["weights"] != (gw, tw, mw):
            f = fc["c"]
            fc["weights"] = (gw, tw, mw)
            f.fold_weights[0], f.fold_weights[1], f.fold_weights[2] = gw, tw, mw
            code, _ = _DTYPES[self.text_dtype]
            scale = float(2 ** TEXT_SCALE_LOG2)
            check(self.lib.tvbf_prep_fold_bits(c.col_side, c.genre_hi, c.meta_scale, cat.n_shows, int(c.genre_dim),
                                               f.operand, int(f.k_pad), int(f.fold_col0),
                                               scale * float(np.sqrt(gw / tw)), scale * float(np.sqrt(mw / tw)),
                                               code, self._stream()), "tvbf_prep_fold_bits")
        return fc["c"]

    # ------------------------------------------------------------------------------------ top-k
    _TABLE_FIELDS = ("indices", "counts", "hybrid", "genre", "text", "metadata", "stats")

    def _alloc_tables(self, rows: int, k: int, row_begin: int | None = None) -> dict:
        """Device result table: indices int32[rows, k] (-1 padded), counts int32[rows], four
        float64[rows, k] score arrays, stats int32[8]."""
        dev = self.device
        t = {"indices": torch.empty((rows, k), dtype=torch.int32, device=dev),
             "counts": torch.empty((rows,), dtype=torch.int32, device=dev)}
        for name in ("hybrid", "genre", "text", "metadata"):
            t[name] = torch.empty((rows, k), dtype=torch.float64, device=dev)
        t["stats"] = torch.empty((8,), dtype=torch.int32, device=dev)     # zeroed by the library calls
        if row_begin is not None:
            t["row_begin"] = row_begin
        return t

    def _c_tables(self, t: dict) -> TopKOut:
        return TopKOut(**{name: t[name].data_ptr() for name in self._TABLE_FIELDS})

    def top_k_device(self, cat: DeviceCatalogue, weights=(0.4, 0.5, 0.1), k: int = 20,
                     min_similarity: float = 0.1, exclude_self: bool = True, row_begin: int = 0,
                     row_end: int | None = None, splits: int = 0, candidates: int = 0,
                     force_exact: bool = False, skip_fallback: bool = False, phases: int = 0,
                     out: dict | None = None, tuning: int = 0) -> dict:
        """Launch the K1 -> K5 -> K6 sequence on the current stream; returns device tensors.
        ``phases`` (bitmask 1|2|4) launches a subset so that a caller can bracket each kernel with
        its own CUDA events; pass the dict returned by the first call as ``out`` to the others."""
        gw, tw, mw = (float(w) for w in weights)
        if cat.folded and cat.weights_baked != (gw, tw, mw) and not force_exact:
            raise _lib.TvbfError("this catalogue was uploaded with folded (non-binary) groups for weights "
                                 f"{cat.weights_baked}; upload again for weights {(gw, tw, mw)}")
        row_end = cat.n_shows if row_end is None else int(row_end)
        rows = row_end - row_begin
        p = Params(genre_weight=gw, text_weight=tw, metadata_weight=mw, min_similarity=float(min_similarity),
                   k=int(k), exclude_self=int(bool(exclude_self)), row_begin=int(row_begin), row_end=row_end,
                   splits=int(splits), candidates=int(candidates), force_exact=int(bool(force_exact)),
                   skip_fallback=int(bool(skip_fallback)), text_rel_err=0.0, phases=int(phases), tuning=int(tuning))
        with torch.cuda.device(self.device):
            feats = None if force_exact else self._folded(cat, gw, tw, mw, int(k), int(tuning), int(candidates))
            if feats is None:
                feats = cat.c
            nbytes = self.lib.tvbf_topk_workspace_bytes(C.byref(feats), C.byref(p))
            if nbytes == 0:
                check(-1, "tvbf_topk_workspace_bytes")
            ws = self._workspace(nbytes)
            t = out if out is not None else self._alloc_tables(rows, k)
            cout = self._c_tables(t)
            check(self.lib.tvbf_hybrid_topk(C.byref(feats), C.byref(p), C.byref(cout), ws.data_ptr(),
                                            ws.numel(), self._stream()), "tvbf_hybrid_topk")
        t["row_begin"] = row_begin
        return t

    # ------------------------------------------------------------------------------------ appends
    def _ingest_like(self, cat: DeviceCatalogue, features: dict, caller: str) -> DeviceCatalogue:
        """``features`` ingested as rows of ``cat``: same metadata mode and baked weights.  Raises
        ``ValueError`` when ``cat`` was consumed, or when the rows differ from it in vocabulary size,
        genre or metadata width, group encoding (binary / float) or operand width."""
        c = cat.c
        if cat.operand is None or not cat.parts:
            raise ValueError(f"{caller}: the catalogue was recycled or does not come from ingest / prepare")
        mode = "mean3" if c.meta_kind == _lib.META_MEAN3 else "hstack"
        new = self.ingest(features, mode, cat.weights_baked or (0.4, 0.5, 0.1))
        nc = new.c
        for what, a, b in (("vocabulary size", c.vocab, nc.vocab), ("genre encoding", c.genre_mode, nc.genre_mode),
                           ("genre columns", c.genre_dim, nc.genre_dim),
                           ("metadata encoding", c.meta_mode, nc.meta_mode),
                           ("metadata groups", c.meta_groups, nc.meta_groups),
                           ("metadata widths", cat.parts["meta_widths"], new.parts["meta_widths"]),
                           ("operand width", c.k_pad, nc.k_pad), ("text dtype", c.text_dtype, nc.text_dtype)):
            if a != b:
                raise ValueError(f"{caller}: the new shows' {what} ({b}) differs from the catalogue's ({a})")
        if cat.folded and (not new.folded or new.weights_baked != cat.weights_baked):
            raise ValueError(f"{caller}: the new shows' float groups do not match the catalogue's")
        return new

    def extend(self, cat: DeviceCatalogue, new_features: dict) -> DeviceCatalogue:
        """``cat`` grown by the shows of ``new_features`` (rows N .. N+Q-1 after its N shows).  Only
        the new rows are prepared (ingest, normalisation, operand rows, CSR, column-side records);
        the old rows are kept -- in place when the spare rows up to ``n_pad`` suffice, else copied
        into buffers grown with headroom.  ``cat`` is consumed, as with ``prepare(recycle=...)``.

        Precondition: the old shows' features are unchanged and the new shows are encoded in the
        same vocabulary and widths (transformed by the already fitted extractor).  A different
        vocabulary size, genre or metadata width, group encoding (binary / float) or metadata mode
        raises ``ValueError``; a refitted extractor changes every row and needs a whole job."""
        c = cat.c
        new = self._ingest_like(cat, new_features, "extend")
        nc = new.c
        n_old, q = cat.n_shows, new.n_shows
        n = n_old + q
        dev = self.device
        p_old, p_new = cat.parts, new.parts
        with torch.cuda.device(dev):
            n_pad = int(c.n_pad)
            grow = n > n_pad
            if grow:
                n_pad = (n + n // 8 + 255) // 256 * 256     # headroom for the next appends

            def rows(old: torch.Tensor | None, fresh: torch.Tensor | None) -> torch.Tensor | None:
                """[n_pad, ...] buffer: old rows (in place or copied), then the new rows."""
                if old is None:
                    return None
                if grow:
                    t = torch.zeros((n_pad, *old.shape[1:]), dtype=old.dtype, device=dev)
                    t[:n_old].copy_(old[:n_old])
                else:
                    t = old
                t[n_old:n].copy_(fresh[:q])
                return t

            operand = rows(cat.operand, new.operand)
            col_side = rows(p_old["col_side"], p_new["col_side"])
            meta_scale = rows(p_old["meta_scale"], p_new["meta_scale"])
            genre_hi = rows(p_old["genre_hi"], p_new["genre_hi"])
            nnz_old, nnz_new = p_old["nnz"], p_new["nnz"]
            indptr = torch.cat([cat.text_indptr[:n_old + 1], new.text_indptr[1:] + cat.text_indptr[n_old]])
            indices = torch.cat([cat.text_indices[:nnz_old], new.text_indices[:nnz_new]])
            values = torch.cat([p_old["values"][:nnz_old], p_new["values"][:nnz_new]])
            if nnz_old + nnz_new == 0:     # the C ABI wants non-NULL arrays, which are never read
                indices = torch.zeros((1,), dtype=torch.int32, device=dev)
                values = torch.zeros((1,), dtype=torch.float64, device=dev)
            genre_dense = None if p_old["genre_dense"] is None else \
                torch.cat([p_old["genre_dense"][:n_old], p_new["genre_dense"][:q]])
            meta_dense = [torch.cat([a[:n_old], b[:q]]) for a, b in zip(p_old["meta_dense"], p_new["meta_dense"])]
            f = Features.from_buffer_copy(c)
            f.n_shows, f.n_pad = n, n_pad
            f.operand = operand.data_ptr()
            f.text_indptr, f.text_indices, f.text_values = indptr.data_ptr(), indices.data_ptr(), values.data_ptr()
            f.text_nnz = nnz_old + nnz_new
            f.col_side, f.meta_scale = col_side.data_ptr(), meta_scale.data_ptr()
            f.genre_hi = None if genre_hi is None else genre_hi.data_ptr()
            f.text_signed = int(bool(c.text_signed) or bool(nc.text_signed))
            if genre_dense is not None:
                f.genre_dense = genre_dense.data_ptr()
            for gi, m in enumerate(meta_dense):
                f.meta_dense[gi] = m.data_ptr()
            grown = DeviceCatalogue(
                c=f, n_shows=n, folded=cat.folded, weights_baked=cat.weights_baked,
                keep=[indptr, indices, values, operand, col_side, meta_scale, genre_hi, genre_dense, *meta_dense],
                operand=operand, text_indptr=indptr, text_indices=indices,
                parts={"values": values, "col_side": col_side, "meta_scale": meta_scale, "genre_hi": genre_hi,
                       "nnz": nnz_old + nnz_new, "genre_dense": genre_dense, "meta_dense": meta_dense,
                       "meta_widths": p_old["meta_widths"]})
            fc = cat.fold
            if fc is not None and self._fold_owner is fc and not grow and not f.text_signed:
                # the second operand: write the new rows' text (through the catalogue's merge plan)
                # and group columns
                ff = Features.from_buffer_copy(fc["c"])
                buf = fc["operand"]
                self._second_rows(fc, new.text_indptr.data_ptr(), new.text_indices.data_ptr(),
                                  p_new["values"].data_ptr(), q, buf[n_old:].data_ptr(), col_side[n_old:].data_ptr(),
                                  None if genre_hi is None else genre_hi[n_old:].data_ptr(),
                                  meta_scale[n_old:].data_ptr())
                for name in ("n_shows", "text_indptr", "text_indices", "text_values", "text_nnz", "col_side",
                             "meta_scale", "genre_hi"):
                    setattr(ff, name, getattr(f, name))
                grown.fold = self._fold_owner = {**fc, "c": ff}
            grown.keep.append(new)          # the new rows' tensors stay alive while the grown catalogue uses them
        cat.operand = None                  # consumed: its buffers now belong to the grown catalogue
        cat.c.operand = None
        cat.keep.clear()
        cat.parts = {}
        cat.fold = None
        cat.buffers = {}                    # prepare(recycle=cat) must not take the grown catalogue's buffers
        cat.h2d_set = None
        return grown

    def top_k_append_device(self, cat: DeviceCatalogue, n_old: int, previous: dict, weights=(0.4, 0.5, 0.1),
                            k: int = 20, min_similarity: float = 0.1, out: dict | None = None) -> dict:
        """Table of the grown catalogue ``cat`` (from ``extend``) from ``previous``, the device table
        (``top_k_device``) of its first ``n_old`` shows for the same weights, ``k`` and
        ``min_similarity`` (``exclude_self=True``).  Bit-identical to ``top_k_device(cat, ...)``
        (indices, counts and the four scores); ``changed_rows`` of the result holds the sorted int32
        old rows whose indices or counts differ from ``previous`` (every other old row is
        byte-identical to its previous row).

        The incremental path (``tvbf_append_topk``) computes only the 256 x 256 tiles that hold a new
        show and copies the previous row of every old show that received no new candidate.  Jobs the
        symmetric sweep does not take (float-valued groups, negative weights, k > 100, ...) and
        catalogues with signed text run the whole job and compare.  ``incremental`` of the result
        says which of the two ran."""
        n_old, k = int(n_old), int(k)
        if previous["indices"].dim() != 2 or tuple(previous["indices"].shape) != (n_old, k) \
                or tuple(previous["counts"].shape) != (n_old,):
            raise ValueError(f"previous table has shape {tuple(previous['indices'].shape)}, expected ({n_old}, {k})")
        if not 0 <= n_old <= cat.n_shows:
            raise ValueError(f"n_old {n_old} outside [0, {cat.n_shows}]")
        gw, tw, mw = (float(w) for w in weights)
        if n_old == cat.n_shows:
            return {**previous, "changed_rows": torch.zeros((0,), dtype=torch.int32, device=self.device),
                    "incremental": True}
        p = self._params(cat, weights, k, min_similarity)
        with torch.cuda.device(self.device):
            feats = self._append_features(cat, n_old, weights, k, min_similarity)
            if feats is None:
                # whole job on the grown catalogue, changed rows by comparison (for old rows, a score
                # changes only with the indices: the score of two old shows is the same)
                t = self.top_k_device(cat, weights, k, min_similarity, out=out)
                t["changed_rows"] = self._changed_rows(t, previous)
                t["incremental"] = False
                return t
            nbytes = self.lib.tvbf_append_workspace_bytes(C.byref(feats), C.byref(p), n_old)
            if nbytes == 0:
                check(-1, "tvbf_append_workspace_bytes")
            ws = self._workspace(nbytes)
            t = out if out is not None else self._alloc_tables(cat.n_shows, k)
            changed = torch.empty((n_old,), dtype=torch.int32, device=self.device)
            prev = self._c_tables({**previous, "stats": t["stats"]})
            check(self.lib.tvbf_append_topk(C.byref(feats), C.byref(p), n_old, C.byref(prev), C.byref(self._c_tables(t)),
                                            changed.data_ptr(), ws.data_ptr(), ws.numel(), self._stream()),
                  "tvbf_append_topk")
            t["changed_rows"] = torch.nonzero(changed).flatten().to(torch.int32)
            t["incremental"] = True
        t["row_begin"] = 0
        return t

    @staticmethod
    def _changed_rows(t: dict, previous: dict, row_map: torch.Tensor | None = None) -> torch.Tensor:
        """Sorted int32 rows of ``previous`` that differ from the same rows of ``t`` in any of the six
        fields (the scores bit for bit).  With ``row_map`` (a removal: previous row o is row
        ``row_map[o]`` of ``t``, -1 when it was removed) the rows of ``t`` are compared with their
        previous rows, whose indices are renumbered by ``row_map`` (a removed show becomes -1)."""
        if row_map is not None:
            keep = torch.nonzero(row_map >= 0).flatten()
            previous = {name: previous[name].index_select(0, keep)
                        for name in ("indices", "counts", "hybrid", "genre", "text", "metadata")}
            idx = previous["indices"]
            previous["indices"] = torch.where(idx >= 0, row_map[idx.clamp(min=0).long()].to(idx.dtype), idx)
        n = previous["counts"].shape[0]
        diff = (t["counts"][:n] != previous["counts"]) | (t["indices"][:n] != previous["indices"]).any(dim=1)
        for name in ("hybrid", "genre", "text", "metadata"):
            diff |= (t[name][:n].view(torch.int64) != previous[name].view(torch.int64)).any(dim=1)
        return torch.nonzero(diff).flatten().to(torch.int32)

    def _append_features(self, cat: DeviceCatalogue, n_old: int, weights, k: int, min_similarity: float):
        """``tvbf_features`` the incremental append runs on (the folded second operand when the job
        qualifies), or None when the job needs the whole job: signed text, or not eligible for the
        symmetric sweep."""
        return None if n_old <= 0 else self._incremental_features(cat, weights, k, min_similarity)

    def _incremental_features(self, cat: DeviceCatalogue, weights, k: int, min_similarity: float):
        """``tvbf_features`` an incremental append or update of ``cat`` runs on (the folded second
        operand when the job qualifies), or None when it needs the whole job: signed text, or not
        eligible for the symmetric sweep."""
        gw, tw, mw = (float(w) for w in weights)
        if cat.c.text_signed:
            return None
        p = self._params(cat, weights, k, min_similarity)
        if not self.lib.tvbf_sym_eligible(C.byref(cat.c), C.byref(p)):
            return None
        feats = self._folded(cat, gw, tw, mw, int(k))
        return cat.c if feats is None else feats

    def append_tiles(self, cat: DeviceCatalogue, n_old: int, weights=(0.4, 0.5, 0.1), k: int = 20,
                     min_similarity: float = 0.1) -> dict | None:
        """Tensor-core tiles (256 x 256 x k_pad) the incremental append of ``top_k_append_device``
        executes on ``cat`` (host only): its threshold seed pass over the super blocks that hold new
        shows and the append sweep.  None when the job runs the whole job instead."""
        with torch.cuda.device(self.device):
            feats = self._append_features(cat, int(n_old), weights, int(k), float(min_similarity))
            if feats is None or int(n_old) >= cat.n_shows:
                return None
            out = (C.c_int64 * 2)()
            check(self.lib.tvbf_append_plan_tiles(C.byref(feats), C.byref(self._params(cat, weights, k, min_similarity)),
                                                  int(n_old), out), "tvbf_append_plan_tiles")
        return {"seed_tiles": int(out[0]), "sweep_tiles": int(out[1])}

    # ------------------------------------------------------------------------------------ updates
    @staticmethod
    def _update_rows(rows, n: int) -> np.ndarray:
        """``rows`` as a sorted int64 array; ``ValueError`` unless they are distinct integers in [0, n)."""
        r = np.asarray(rows)
        if r.ndim != 1 or (r.size and not np.issubdtype(r.dtype, np.integer)):
            raise ValueError(f"rows must be a 1-D array of integers, got shape {r.shape} and dtype {r.dtype}")
        r = np.sort(r.astype(np.int64))
        if r.size and (r[0] < 0 or r[-1] >= n):
            raise ValueError(f"rows must lie in [0, {n}), got [{r[0]}, {r[-1]}]")
        if r.size > 1 and (r[1:] == r[:-1]).any():
            raise ValueError("rows must be distinct")
        return r

    def update(self, cat: DeviceCatalogue, rows, new_features: dict) -> DeviceCatalogue:
        """``cat`` with the shows ``rows`` (distinct, any order) given the features of
        ``new_features`` (row e of it for the e-th smallest of ``rows``).  Only the Q new rows are
        prepared; they are written over the old ones in place (operand rows, column-side records,
        metadata scales, second genre words, dense float groups, the rows of the engine's second
        operand when this catalogue owns it) and the text CSR is spliced on the device.  The result
        equals a fresh ``ingest`` of the updated features.  ``cat`` is consumed, as with ``extend``.

        Precondition: the new features are encoded in the catalogue's vocabulary and widths (the
        already fitted extractor); a different vocabulary size, genre or metadata width, group
        encoding (binary / float) or metadata mode raises ``ValueError``."""
        r = self._update_rows(rows, cat.n_shows)
        q = int(r.size)
        n_feat = int(np.asarray(new_features["genre_features"]).shape[0])
        if n_feat != q:
            raise ValueError(f"update: {q} rows but new features for {n_feat} shows")
        if q == 0:
            if cat.operand is None or not cat.parts:
                raise ValueError("update: the catalogue was recycled or does not come from ingest / prepare")
            return cat
        c = cat.c
        new = self._ingest_like(cat, new_features, "update")
        nc = new.c
        n = cat.n_shows
        dev = self.device
        p_old, p_new = cat.parts, new.parts
        with torch.cuda.device(dev):
            idx = torch.from_numpy(r).to(dev)
            operand = cat.operand
            operand.index_copy_(0, idx, new.operand[:q])
            col_side, meta_scale, genre_hi = p_old["col_side"], p_old["meta_scale"], p_old["genre_hi"]
            col_side.index_copy_(0, idx, p_new["col_side"][:q])
            meta_scale.index_copy_(0, idx, p_new["meta_scale"][:q])
            if genre_hi is not None:
                genre_hi.index_copy_(0, idx, p_new["genre_hi"][:q])
            genre_dense = p_old["genre_dense"]
            if genre_dense is not None:
                genre_dense.index_copy_(0, idx, p_new["genre_dense"][:q])
            meta_dense = p_old["meta_dense"]
            for a, b in zip(meta_dense, p_new["meta_dense"]):
                a.index_copy_(0, idx, b[:q])
            # CSR splice: row lengths -> indptr, then every output entry gathered from [old nnz | new nnz]
            nnz_old, nnz_new = p_old["nnz"], p_new["nnz"]
            ip_old = cat.text_indptr[:n + 1].to(torch.int64)
            ip_new = new.text_indptr[:q + 1].to(torch.int64)
            lens = ip_old[1:] - ip_old[:-1]
            lens[idx] = ip_new[1:] - ip_new[:-1]
            indptr = torch.zeros((n + 1,), dtype=torch.int64, device=dev)
            indptr[1:] = torch.cumsum(lens, 0)
            start = ip_old[:-1].clone()
            start[idx] = ip_new[:-1] + nnz_old
            nnz = int(indptr[-1].item())
            if nnz == 0:               # the C ABI wants non-NULL arrays, which are never read
                indices = torch.zeros((1,), dtype=torch.int32, device=dev)
                values = torch.zeros((1,), dtype=torch.float64, device=dev)
            else:
                row_of = torch.repeat_interleave(torch.arange(n, device=dev), lens, output_size=nnz)
                pos = torch.arange(nnz, device=dev) - indptr[row_of] + start[row_of]
                indices = torch.cat([cat.text_indices[:nnz_old], new.text_indices[:nnz_new]])[pos]
                values = torch.cat([p_old["values"][:nnz_old], p_new["values"][:nnz_new]])[pos]
            f = Features.from_buffer_copy(c)
            f.text_indptr, f.text_indices, f.text_values = indptr.data_ptr(), indices.data_ptr(), values.data_ptr()
            f.text_nnz = nnz
            signed = bool(c.text_signed) or bool(nc.text_signed)
            f.text_signed = int(signed and nnz > 0 and bool((values < 0).any()))
            parts = {**p_old, "values": values, "nnz": nnz}
            buffers = {**cat.buffers, "values": values} if "values" in cat.buffers else dict(cat.buffers)
            upd = DeviceCatalogue(c=f, n_shows=n, folded=cat.folded, weights_baked=cat.weights_baked,
                                  keep=[indptr, indices, values, operand, col_side, meta_scale, genre_hi, genre_dense,
                                        *meta_dense], operand=operand,
                                  text_indptr=indptr, text_indices=indices, buffers=buffers, parts=parts)
            fc = cat.fold
            if fc is not None and self._fold_owner is fc and not f.text_signed:
                # the second operand: rebuild the updated rows (through the catalogue's merge plan) and
                # write them over
                ff = Features.from_buffer_copy(fc["c"])
                buf = fc["operand"]
                rows_fold = torch.zeros((q, int(ff.k_pad)), dtype=buf.dtype, device=dev)
                self._second_rows(fc, new.text_indptr.data_ptr(), new.text_indices.data_ptr(),
                                  p_new["values"].data_ptr(), q, rows_fold.data_ptr(), p_new["col_side"].data_ptr(),
                                  None if p_new["genre_hi"] is None else p_new["genre_hi"].data_ptr(),
                                  p_new["meta_scale"].data_ptr())
                buf.index_copy_(0, idx, rows_fold)
                for name in ("text_indptr", "text_indices", "text_values", "text_nnz"):
                    setattr(ff, name, getattr(f, name))
                upd.fold = self._fold_owner = {**fc, "c": ff}
        cat.operand = None                  # consumed: its buffers now belong to the updated catalogue
        cat.c.operand = None
        cat.keep.clear()
        cat.parts = {}
        cat.fold = None
        cat.buffers = {}
        cat.h2d_set = None
        return upd

    def top_k_update_device(self, cat: DeviceCatalogue, rows, previous: dict, weights=(0.4, 0.5, 0.1),
                            k: int = 20, min_similarity: float = 0.1, out: dict | None = None) -> dict:
        """Table of ``cat`` after the shows ``rows`` got new features (``update``) from
        ``previous``, the device table (``top_k_device``) of the catalogue before the update for the
        same weights, ``k`` and ``min_similarity`` (``exclude_self=True``).  Bit-identical to
        ``top_k_device(cat, ...)`` (indices, counts and the four scores); ``changed_rows`` of the
        result holds the sorted int32 rows, updated or not, that differ from ``previous`` in any
        field (every other row is byte-identical to its previous row).

        The incremental path (``tvbf_update_topk``) sweeps only the updated shows' rows against all
        columns and copies the previous row of every show that names no updated show and received
        no candidate from one.  Jobs the symmetric sweep does not take (float-valued groups,
        negative weights, k > 100, ...) and catalogues with signed text run the whole job and
        compare.  ``incremental`` of the result says which of the two ran."""
        n, k = cat.n_shows, int(k)
        r = self._update_rows(rows, n)
        if previous["indices"].dim() != 2 or tuple(previous["indices"].shape) != (n, k) \
                or tuple(previous["counts"].shape) != (n,):
            raise ValueError(f"previous table has shape {tuple(previous['indices'].shape)}, expected ({n}, {k})")
        if r.size == 0:
            return {**previous, "changed_rows": torch.zeros((0,), dtype=torch.int32, device=self.device),
                    "incremental": True}
        p = self._params(cat, weights, k, min_similarity)
        with torch.cuda.device(self.device):
            feats = self._incremental_features(cat, weights, k, min_similarity)
            if feats is None:
                # whole job on the updated catalogue, changed rows by comparison
                t = self.top_k_device(cat, weights, k, min_similarity, out=out)
                t["changed_rows"] = self._changed_rows(t, previous)
                t["incremental"] = False
                return t
            nbytes = self.lib.tvbf_update_workspace_bytes(C.byref(feats), C.byref(p), int(r.size))
            if nbytes == 0:
                check(-1, "tvbf_update_workspace_bytes")
            ws = self._workspace(nbytes)
            t = out if out is not None else self._alloc_tables(n, k)
            rows_d = torch.from_numpy(r.astype(np.int32)).to(self.device)
            changed = torch.empty((n,), dtype=torch.int32, device=self.device)
            prev = self._c_tables({**previous, "stats": t["stats"]})
            check(self.lib.tvbf_update_topk(C.byref(feats), C.byref(p), rows_d.data_ptr(), int(r.size), C.byref(prev),
                                            C.byref(self._c_tables(t)), changed.data_ptr(), ws.data_ptr(), ws.numel(),
                                            self._stream()), "tvbf_update_topk")
            t["changed_rows"] = torch.nonzero(changed).flatten().to(torch.int32)
            t["incremental"] = True
        t["row_begin"] = 0
        return t

    def update_tiles(self, cat: DeviceCatalogue, n_rows: int, weights=(0.4, 0.5, 0.1), k: int = 20,
                     min_similarity: float = 0.1) -> dict | None:
        """Tensor-core tiles (256 x 256 x k_pad) the incremental update of ``top_k_update_device``
        executes on ``cat`` with ``n_rows`` updated shows (host only): its threshold seed pass over
        the gathered rows and the update sweep.  None when the job runs the whole job instead."""
        with torch.cuda.device(self.device):
            feats = self._incremental_features(cat, weights, int(k), float(min_similarity))
            if feats is None or not 1 <= int(n_rows) <= cat.n_shows:
                return None
            out = (C.c_int64 * 2)()
            check(self.lib.tvbf_update_plan_tiles(C.byref(feats), C.byref(self._params(cat, weights, k, min_similarity)),
                                                  int(n_rows), out), "tvbf_update_plan_tiles")
        return {"seed_tiles": int(out[0]), "sweep_tiles": int(out[1])}

    # ------------------------------------------------------------------------------------ removals
    def remove(self, cat: DeviceCatalogue, rows) -> DeviceCatalogue:
        """``cat`` without the shows ``rows`` (distinct, any order): the remaining shows keep their
        order and become rows 0 .. N - Q - 1.  Compacted on the device (operand rows, column-side
        records, metadata scales, second genre words, dense float groups, the text CSR and the rows of
        the engine's second operand when this catalogue owns it); the freed rows are zeroed and
        ``n_pad`` shrinks to that of N - Q shows.  The result equals a fresh ``ingest`` of the
        remaining features.  ``cat`` is consumed, as with ``extend``.  Removing every show raises
        ``ValueError``."""
        n = cat.n_shows
        r = self._update_rows(rows, n)
        if cat.operand is None or not cat.parts:
            raise ValueError("remove: the catalogue was recycled or does not come from ingest / prepare")
        q = int(r.size)
        if q == 0:
            return cat
        if q == n:
            raise ValueError("remove: removing every show leaves no catalogue")
        m = n - q
        c = cat.c
        dev = self.device
        p_old = cat.parts
        keep_np = np.delete(np.arange(n, dtype=np.int64), r)
        with torch.cuda.device(dev):
            keep = torch.from_numpy(keep_np).to(dev)
            n_pad = (m + 255) // 256 * 256

            def compact(t: torch.Tensor | None) -> torch.Tensor | None:
                """rows ``keep`` of a padded buffer moved to the front, the freed rows zeroed; the first
                ``n_pad`` rows (a view)"""
                if t is None:
                    return None
                t[:m].copy_(t.index_select(0, keep))
                t[m:n].zero_()
                return t[:n_pad]

            operand = compact(cat.operand)
            col_side = compact(p_old["col_side"])
            meta_scale = compact(p_old["meta_scale"])
            genre_hi = compact(p_old["genre_hi"])
            genre_dense = None if p_old["genre_dense"] is None else p_old["genre_dense"].index_select(0, keep)
            meta_dense = [a.index_select(0, keep) for a in p_old["meta_dense"]]
            # CSR: the kept rows' lengths -> indptr, every output entry gathered from its old position
            ip_old = cat.text_indptr[:n + 1].to(torch.int64)
            lens = (ip_old[1:] - ip_old[:-1]).index_select(0, keep)
            indptr = torch.zeros((m + 1,), dtype=torch.int64, device=dev)
            indptr[1:] = torch.cumsum(lens, 0)
            nnz = int(indptr[-1].item())
            if nnz == 0:               # the C ABI wants non-NULL arrays, which are never read
                indices = torch.zeros((1,), dtype=torch.int32, device=dev)
                values = torch.zeros((1,), dtype=torch.float64, device=dev)
            else:
                row_of = torch.repeat_interleave(torch.arange(m, device=dev), lens, output_size=nnz)
                pos = torch.arange(nnz, device=dev) - indptr[row_of] + ip_old[:-1].index_select(0, keep)[row_of]
                indices = cat.text_indices[pos]
                values = p_old["values"][pos]
            f = Features.from_buffer_copy(c)
            f.n_shows, f.n_pad = m, n_pad
            f.operand = operand.data_ptr()
            f.text_indptr, f.text_indices, f.text_values = indptr.data_ptr(), indices.data_ptr(), values.data_ptr()
            f.text_nnz = nnz
            f.text_signed = int(bool(c.text_signed) and nnz > 0 and bool((values < 0).any()))
            if genre_dense is not None:
                f.genre_dense = genre_dense.data_ptr()
            for gi, a in enumerate(meta_dense):
                f.meta_dense[gi] = a.data_ptr()
            parts = {**p_old, "values": values, "nnz": nnz, "col_side": col_side, "meta_scale": meta_scale,
                     "genre_hi": genre_hi, "genre_dense": genre_dense, "meta_dense": meta_dense}
            buffers = {"values": values, "col_side": col_side, "meta_scale": meta_scale}
            if genre_hi is not None:
                buffers["genre_hi"] = genre_hi
            rem = DeviceCatalogue(c=f, n_shows=m, folded=cat.folded, weights_baked=cat.weights_baked,
                                  keep=[indptr, indices, values, operand, col_side, meta_scale, genre_hi, genre_dense,
                                        *meta_dense], operand=operand,
                                  text_indptr=indptr, text_indices=indices,
                                  buffers=buffers if cat.buffers else {}, parts=parts)
            fc = cat.fold
            if fc is not None and self._fold_owner is fc and not f.text_signed:
                # the second operand: its rows move with the shows
                buf = compact(fc["operand"])
                ff = Features.from_buffer_copy(fc["c"])
                ff.n_shows, ff.n_pad, ff.operand = m, n_pad, buf.data_ptr()
                for name in ("text_indptr", "text_indices", "text_values", "text_nnz", "col_side", "meta_scale", "genre_hi"):
                    setattr(ff, name, getattr(f, name))
                rem.fold = self._fold_owner = {**fc, "c": ff, "operand": buf}
        cat.operand = None                  # consumed: its buffers now belong to the compacted catalogue
        cat.c.operand = None
        cat.keep.clear()
        cat.parts = {}
        cat.fold = None
        cat.buffers = {}
        cat.h2d_set = None
        return rem

    def top_k_remove_device(self, cat: DeviceCatalogue, rows, previous: dict, weights=(0.4, 0.5, 0.1),
                            k: int = 20, min_similarity: float = 0.1, out: dict | None = None) -> dict:
        """Table of ``cat`` after the shows ``rows`` (old numbering) were removed (``remove``) from
        ``previous``, the device table (``top_k_device``) of the catalogue before the removal for the
        same weights, ``k`` and ``min_similarity`` (``exclude_self=True``).  Row r of the result is
        the r-th remaining show, with indices in the new numbering.  Bit-identical to
        ``top_k_device(cat, ...)`` (indices, counts and the four scores); ``changed_rows`` of the
        result holds the sorted int32 new rows that differ in any field from their previous row with
        its indices renumbered (every other row is byte-identical to it).  These are exactly the rows
        whose previous row names a removed show.

        The incremental path (``tvbf_remove_topk``) copies every other row and sweeps only those rows
        against all columns.  Jobs the symmetric sweep does not take (float-valued groups, negative
        weights, k > 100, ...) and catalogues with signed text run the whole job and compare.
        ``incremental`` of the result says which of the two ran."""
        m, k = cat.n_shows, int(k)
        n = int(previous["counts"].shape[0])
        r = self._update_rows(rows, n)
        q = int(r.size)
        if previous["indices"].dim() != 2 or tuple(previous["indices"].shape) != (m + q, k) \
                or tuple(previous["counts"].shape) != (m + q,):
            raise ValueError(f"previous table has shape {tuple(previous['indices'].shape)}, expected ({m + q}, {k})")
        if q == 0:
            return {**previous, "changed_rows": torch.zeros((0,), dtype=torch.int32, device=self.device),
                    "incremental": True}
        p = self._params(cat, weights, k, min_similarity)
        with torch.cuda.device(self.device):
            feats = self._incremental_features(cat, weights, k, min_similarity)
            if feats is None:
                # whole job on the remaining catalogue, changed rows by comparison with the renumbered rows
                t = self.top_k_device(cat, weights, k, min_similarity, out=out)
                row_map = torch.full((n,), -1, dtype=torch.int64)
                row_map[np.delete(np.arange(n), r)] = torch.arange(m)
                t["changed_rows"] = self._changed_rows(t, previous, row_map.to(self.device))
                t["incremental"] = False
                return t
            nbytes = self.lib.tvbf_remove_workspace_bytes(C.byref(feats), C.byref(p), q)
            if nbytes == 0:
                check(-1, "tvbf_remove_workspace_bytes")
            ws = self._workspace(nbytes)
            t = out if out is not None else self._alloc_tables(m, k)
            rows_d = torch.from_numpy(r.astype(np.int32)).to(self.device)
            changed = torch.empty((m,), dtype=torch.int32, device=self.device)
            prev = self._c_tables({**previous, "stats": t["stats"]})
            check(self.lib.tvbf_remove_topk(C.byref(feats), C.byref(p), rows_d.data_ptr(), q, C.byref(prev),
                                            C.byref(self._c_tables(t)), changed.data_ptr(), ws.data_ptr(), ws.numel(),
                                            self._stream()), "tvbf_remove_topk")
            t["changed_rows"] = torch.nonzero(changed).flatten().to(torch.int32)
            t["incremental"] = True
        t["row_begin"] = 0
        return t

    def remove_tiles(self, cat: DeviceCatalogue, n_rows: int, weights=(0.4, 0.5, 0.1), k: int = 20,
                     min_similarity: float = 0.1) -> dict | None:
        """Tensor-core tiles (256 x 256 x k_pad) the incremental removal of ``top_k_remove_device``
        executes on the remaining catalogue ``cat`` when ``n_rows`` of its rows named a removed show
        (the length of ``changed_rows``; host only): its threshold seed pass over their gathered rows
        and the repair sweep.  {0, 0} for no such row; None when the job runs the whole job instead."""
        with torch.cuda.device(self.device):
            feats = self._incremental_features(cat, weights, int(k), float(min_similarity))
            if feats is None or not 0 <= int(n_rows) <= cat.n_shows:
                return None
            if int(n_rows) == 0:
                return {"seed_tiles": 0, "sweep_tiles": 0}
            out = (C.c_int64 * 2)()
            check(self.lib.tvbf_remove_plan_tiles(C.byref(feats), C.byref(self._params(cat, weights, k, min_similarity)),
                                                  int(n_rows), out), "tvbf_remove_plan_tiles")
        return {"seed_tiles": int(out[0]), "sweep_tiles": int(out[1])}

    # ------------------------------------------------------------------------------------ refreshes
    def top_k_refresh_device(self, cat: DeviceCatalogue, previous: dict, removed=(), updated=(), n_appended: int = 0,
                             weights=(0.4, 0.5, 0.1), k: int = 20, min_similarity: float = 0.1,
                             exclude_self: bool = True, out: dict | None = None) -> dict:
        """Table of ``cat`` after a refresh that removed the shows ``removed``, gave the shows
        ``updated`` new features (both rows of ``previous``, distinct and disjoint, any order) and
        appended ``n_appended`` shows, from ``previous``, the device table (``top_k_device``) of the
        catalogue before it for the same weights, ``k``, ``min_similarity`` and ``exclude_self``.
        ``cat`` holds the remaining shows in their old order, the updated ones with their new
        features, then the appended shows: the chain ``update(cat, updated, new_features)``,
        ``remove(cat, removed)``, ``extend(cat, appended_features)`` builds it (no other catalogue
        operation is needed), and so does a fresh ``ingest`` of the features after the refresh.

        Row r of the result is row r of ``cat``, with indices in that numbering.  Bit-identical to
        ``top_k_device(cat, ...)`` (indices, counts and the four scores); ``changed_rows`` of the
        result holds the sorted int32 rows to rewrite: every appended row, and every remaining row
        that differs in any field from its previous row with the indices renumbered (every other row
        is byte-identical to that).  Unlike ``top_k_append_device``, whose ``changed_rows`` holds old
        rows only, the appended rows are listed too.

        The incremental path (``tvbf_refresh_topk``) sweeps the updated and appended shows, and the
        remaining shows whose previous row names a removed show, against all columns; it copies
        every row no changed score can reach, and sweeps the rows whose lost neighbours it cannot
        refill a second time on the tensor cores (``stats[5]`` counts them; ``stats[0]`` counts the
        rows left to the exact kernel).  Jobs the symmetric sweep does not take (float-valued
        groups, negative weights, k > 100, ...), catalogues with signed text and
        ``exclude_self=False`` run the whole job and compare.  ``incremental`` of the result says
        which of the two ran.  Rows out of range, duplicates, ``removed`` and ``updated``
        overlapping, a ``previous`` of the wrong shape, an ``n_appended`` that does not match
        ``cat.n_shows`` and removing every old show raise ``ValueError``."""
        k, qa = int(k), int(n_appended)
        if previous["indices"].dim() != 2 or previous["indices"].shape[1] != k \
                or tuple(previous["counts"].shape) != (previous["indices"].shape[0],):
            raise ValueError(f"previous table has shape {tuple(previous['indices'].shape)}, expected (N, {k})")
        n_old, n = int(previous["counts"].shape[0]), cat.n_shows
        rem = self._update_rows(removed, n_old)
        upd = self._update_rows(updated, n_old)
        if np.intersect1d(rem, upd).size:
            raise ValueError("removed and updated rows overlap")
        if rem.size == n_old:
            raise ValueError("refresh: removing every old show leaves no catalogue to refresh")
        if qa < 0 or n_old - rem.size + qa != n:
            raise ValueError(f"n_appended {qa}: {n_old} previous rows - {rem.size} removed + {qa} appended "
                             f"!= {n} shows in the catalogue")
        if rem.size == 0 and upd.size == 0 and qa == 0:
            return {**previous, "changed_rows": torch.zeros((0,), dtype=torch.int32, device=self.device),
                    "incremental": True}
        p = self._params(cat, weights, k, min_similarity)
        with torch.cuda.device(self.device):
            feats = self._incremental_features(cat, weights, k, min_similarity) if exclude_self else None
            if feats is None:
                # whole job, changed rows by comparison with the renumbered rows, plus the appended ones
                t = self.top_k_device(cat, weights, k, min_similarity, exclude_self=exclude_self, out=out)
                row_map = torch.full((n_old,), -1, dtype=torch.int64)
                row_map[np.delete(np.arange(n_old), rem)] = torch.arange(n_old - rem.size)
                ch = self._changed_rows(t, previous, row_map.to(self.device))
                t["changed_rows"] = torch.cat([ch, torch.arange(n - qa, n, dtype=torch.int32, device=self.device)])
                t["incremental"] = False
                return t
            nbytes = self.lib.tvbf_refresh_workspace_bytes(C.byref(feats), C.byref(p), int(rem.size), int(upd.size), qa)
            if nbytes == 0:
                check(-1, "tvbf_refresh_workspace_bytes")
            ws = self._workspace(nbytes)
            t = out if out is not None else self._alloc_tables(n, k)
            rem_d = torch.from_numpy(rem.astype(np.int32)).to(self.device)
            upd_d = torch.from_numpy(upd.astype(np.int32)).to(self.device)
            changed = torch.empty((n,), dtype=torch.int32, device=self.device)
            prev = self._c_tables({**previous, "stats": t["stats"]})
            check(self.lib.tvbf_refresh_topk(C.byref(feats), C.byref(p), rem_d.data_ptr() if rem.size else None,
                                             int(rem.size), upd_d.data_ptr() if upd.size else None, int(upd.size), qa,
                                             C.byref(prev), C.byref(self._c_tables(t)), changed.data_ptr(),
                                             ws.data_ptr(), ws.numel(), self._stream()), "tvbf_refresh_topk")
            t["changed_rows"] = torch.nonzero(changed).flatten().to(torch.int32)
            t["incremental"] = True
        t["row_begin"] = 0
        return t

    def refresh_tiles(self, cat: DeviceCatalogue, n_gathered: int, n_repaired: int = 0, weights=(0.4, 0.5, 0.1),
                      k: int = 20, min_similarity: float = 0.1) -> dict | None:
        """Tensor-core tiles (256 x 256 x k_pad) the incremental refresh of ``top_k_refresh_device``
        executes on the catalogue after the refresh ``cat`` (host only) when ``n_gathered`` rows are
        updated, appended or named a removed show, and ``n_repaired`` rows go to the second sweep
        (``stats[5]`` of the result): the threshold seed pass and the sweep of each stage, 0 for a
        stage without rows.  None when the job runs the whole job instead."""
        with torch.cuda.device(self.device):
            feats = self._incremental_features(cat, weights, int(k), float(min_similarity))
            if feats is None or not 0 <= int(n_repaired) <= cat.n_shows or not 0 <= int(n_gathered) <= cat.n_shows:
                return None
            if int(n_gathered) == 0:
                return {"seed_tiles": 0, "sweep_tiles": 0, "repair_seed_tiles": 0, "repair_sweep_tiles": 0}
            out = (C.c_int64 * 4)()
            check(self.lib.tvbf_refresh_plan_tiles(C.byref(feats), C.byref(self._params(cat, weights, k, min_similarity)),
                                                   int(n_gathered), int(n_repaired), out), "tvbf_refresh_plan_tiles")
        return {"seed_tiles": int(out[0]), "sweep_tiles": int(out[1]), "repair_seed_tiles": int(out[2]),
                "repair_sweep_tiles": int(out[3])}

    def top_k_sweep_device(self, cat: DeviceCatalogue, weight_list, k: int = 20, min_similarity: float = 0.1,
                           exclude_self: bool = True, shared: bool | None = None, tuning: int = 0,
                           out: list | None = None, **kw) -> list[dict]:
        """Weight sweep (BASELINE config C5; notebooks/03 cell 6 of the reference): one table per
        weight triple over ONE device-resident catalogue.  H2D, normalisation, the fp16 operand and
        the packed genre / metadata words never depend on the weights.  ``shared`` (default: when
        every triple is eligible for the symmetric sweep and the catalogue has >= 40 000 shows)
        also shares the tensor-core sweep between up to 5 triples per launch
        (``tvbf_hybrid_topk_sweep``: one candidate list per (triple, show)); otherwise the candidate
        sweep runs once per triple.  Either way the tables equal those of separate jobs.
        ``out``: the list an earlier call of the same shape returned, to be overwritten (no allocation)."""
        if cat.folded:
            raise _lib.TvbfError("a catalogue with folded (non-binary) groups bakes the weights into the "
                                 "operand; use compute_top_k_sweep, which uploads once per triple")
        triples = [tuple(float(x) for x in w) for w in weight_list]
        if shared is None:
            shared = (exclude_self and cat.n_shows >= 40_000 and len(triples) > 1 and not kw
                      and not cat.c.genre_hi        # the shared sweep keeps one-word genre masks
                      and all(self.sym_eligible(cat, w, k, min_similarity) for w in triples))
        if not shared:
            return [self.top_k_device(cat, w, k, min_similarity, exclude_self, tuning=tuning, **kw) for w in triples]
        k, rows, dev, spare, out = int(k), cat.n_shows, self.device, list(out or []), []
        with torch.cuda.device(dev):
            for g0 in range(0, len(triples), 5):
                part = triples[g0:g0 + 5]
                n = len(part)
                ps = (Params * n)()
                for w, (gw, tw, mw) in enumerate(part):
                    ps[w] = Params(genre_weight=gw, text_weight=tw, metadata_weight=mw,
                                   min_similarity=float(min_similarity), k=k, exclude_self=int(bool(exclude_self)),
                                   row_begin=0, row_end=rows, splits=0, candidates=0, force_exact=0,
                                   skip_fallback=0, text_rel_err=0.0, phases=0, tuning=int(tuning))
                nbytes = self.lib.tvbf_topk_sweep_workspace_bytes(C.byref(cat.c), ps, n)
                if nbytes == 0:
                    check(-1, "tvbf_topk_sweep_workspace_bytes")
                ws = self._workspace(nbytes)
                tabs = [spare.pop(0) if spare and tuple(spare[0]["indices"].shape) == (rows, k)
                        else self._alloc_tables(rows, k, 0) for _ in range(n)]
                couts = (TopKOut * n)()
                for w, t in enumerate(tabs):
                    couts[w] = self._c_tables(t)
                check(self.lib.tvbf_hybrid_topk_sweep(C.byref(cat.c), ps, n, couts, ws.data_ptr(), ws.numel(),
                                                      self._stream()), "tvbf_hybrid_topk_sweep")
                out += tabs
        return out

    def compute_top_k_sweep(self, features: dict, weight_list, k: int = 20, min_similarity: float = 0.1,
                            metadata_mode: str = "mean3", exclude_self: bool = True, **kw) -> list[TopK]:
        """features dict -> one host TopK per weight triple (staging and upload shared when the
        features are binary / one-hot)."""
        triples = [tuple(float(x) for x in w) for w in weight_list]
        if not triples:
            return []
        cat = self.ingest(features, metadata_mode, triples[0])
        if cat.folded:   # weights are baked into the operand: one upload per triple
            st = stage(features, metadata_mode)
            return [self.to_host(self.top_k_device(self.upload(st, w), w, k, min_similarity, exclude_self, **kw))
                    for w in triples]
        return [self.to_host(t) for t in self.top_k_sweep_device(cat, triples, k, min_similarity, exclude_self, **kw)]

    def to_host(self, t: dict, copy: bool = True) -> TopK:
        """D2H of a result table into cached pinned buffers (synchronises).  With ``copy=False`` the
        returned arrays alias the pinned buffers and are valid until the next ``to_host`` of the
        same shape on this engine."""
        names = ("indices", "counts", "hybrid", "genre", "text", "metadata", "stats")
        host = {}
        with torch.cuda.device(self.device):
            for n in names:
                src = t[n]
                key = (n, tuple(src.shape), src.dtype)
                buf = self._pinned.get(key)
                if buf is None:
                    if len(self._pinned) > 64:
                        self._pinned.clear()
                    buf = torch.empty(src.shape, dtype=src.dtype, pin_memory=True)
                    self._pinned[key] = buf
                buf.copy_(src, non_blocking=True)
                host[n] = buf
            torch.cuda.current_stream(self.device).synchronize()
        host = {n: (v.numpy().copy() if copy else v.numpy()) for n, v in host.items()}
        if host["stats"].ndim == 2:            # gathered [world, 8]: per-rank counters
            host["stats"] = host["stats"].sum(axis=0)
        return TopK(indices=host["indices"], counts=host["counts"], hybrid=host["hybrid"], genre=host["genre"],
                    text=host["text"], metadata=host["metadata"], row_begin=int(t.get("row_begin", 0)),
                    flagged_rows=int(host["stats"][0]), rescored_pairs=int(host["stats"][1]))

    def compute_top_k(self, features: dict, weights=(0.4, 0.5, 0.1), k: int = 20, min_similarity: float = 0.1,
                      metadata_mode: str = "mean3", exclude_self: bool = True, **kw) -> TopK:
        """features dict -> TopK for all rows on this GPU (raw bytes up, classified and packed on the
        device: ``ingest``)."""
        cat = self.ingest(features, metadata_mode, weights)
        return self.to_host(self.top_k_device(cat, weights, k, min_similarity, exclude_self, **kw))

    # ------------------------------------------------------------------------------------ threshold
    def neighbours_device(self, cat: DeviceCatalogue, weights=(0.4, 0.5, 0.1), min_similarity: float = 0.1,
                          exclude_self: bool = True, max_per_row: int = 0, capacity: int | None = None,
                          max_pairs: int | None = None) -> dict:
        """Every pair with hybrid >= ``min_similarity``, one row per show (``tvbf_neighbours_*``):
        the tensor-core sweep emits the candidate pairs (a superset, by the upper bound), the finish
        rescores them in float64 and orders each row.  The sweep writes into ``capacity`` pair slots
        (default 64 N: 8 bytes per pair, 51 MB at 100 000 shows); when it finds more candidates it runs
        once more with room for all of them (one synchronisation per sweep reads the count).
        ``max_pairs`` bounds the output: a ValueError is raised before anything larger than
        ``max_pairs`` entries (2 candidates + N) is allocated.  It also bounds the default pair buffer
        to the (max_pairs - N) / 2 candidates such an output can take; an explicit ``capacity`` is
        used as given.
        ``max_per_row`` > 0 keeps the first entries of every row.  Returns device tensors ``row_ptr``
        (int64 [N + 1]), ``indices``, ``hybrid``, ``genre``, ``text``, ``metadata`` and the count
        ``candidate_pairs``."""
        gw, tw, mw = (float(w) for w in weights)
        n = cat.n_shows
        p = self._params(cat, weights, 1, min_similarity, exclude_self)
        lib, dev = self.lib, self.device
        cap = 64 * n if capacity is None else int(capacity)
        if capacity is None and max_pairs is not None:
            cap = min(cap, max(0, (int(max_pairs) - n) // 2))   # more candidates raise anyway
        if cap < 0:
            raise ValueError(f"capacity must be >= 0, got {cap}")
        with torch.cuda.device(dev):
            if lib.tvbf_neighbours_workspace_bytes(C.byref(cat.c), C.byref(p), 0) == 0:
                check(-1, "tvbf_neighbours_workspace_bytes")
            feats = self._folded(cat, gw, tw, mw, 1)
            if feats is None:
                feats = cat.c
            count = torch.zeros((1,), dtype=torch.int64, device=dev)

            def workspace(n_pairs: int) -> torch.Tensor:
                # the sweep itself needs the workspace of 0 pairs; the finish that of the pairs it takes
                nbytes = lib.tvbf_neighbours_workspace_bytes(C.byref(feats), C.byref(p), n_pairs)
                if nbytes == 0:
                    check(-1, "tvbf_neighbours_workspace_bytes")
                return self._workspace(nbytes)

            def sweep(cap: int):
                ws = workspace(0)
                pairs = torch.empty((max(cap, 1), 2), dtype=torch.int32, device=dev)
                check(lib.tvbf_neighbours_sweep(C.byref(feats), C.byref(p), pairs.data_ptr(), cap, count.data_ptr(),
                                                ws.data_ptr(), ws.numel(), self._stream()), "tvbf_neighbours_sweep")
                return pairs, int(count.item())

            def guard(n_cand: int) -> None:
                if max_pairs is not None and 2 * n_cand + n > int(max_pairs):
                    raise ValueError(f"the sweep found {n_cand} candidate pairs: the output needs room for "
                                     f"{2 * n_cand + n} entries, more than max_pairs={int(max_pairs)}")

            pairs, n_cand = sweep(cap)
            while n_cand > cap:
                guard(n_cand)
                cap = n_cand
                pairs = None
                pairs, n_cand = sweep(cap)
            guard(n_cand)
            ws = workspace(n_cand)
            m = 2 * n_cand + n
            out = {"row_ptr": torch.empty((n + 1,), dtype=torch.int64, device=dev),
                   "indices": torch.empty((m,), dtype=torch.int32, device=dev)}
            for name in ("hybrid", "genre", "text", "metadata"):
                out[name] = torch.empty((m,), dtype=torch.float64, device=dev)
            check(lib.tvbf_neighbours_finish(C.byref(feats), C.byref(p), pairs.data_ptr(), n_cand, int(max_per_row),
                                             *(out[k].data_ptr() for k in ("row_ptr", "indices", "hybrid", "genre",
                                                                             "text", "metadata")),
                                             ws.data_ptr(), ws.numel(), self._stream()), "tvbf_neighbours_finish")
            nnz = int(out["row_ptr"][-1].item())
        for name in ("indices", "hybrid", "genre", "text", "metadata"):
            out[name] = out[name][:nnz]
        out["candidate_pairs"] = n_cand
        return out

    @staticmethod
    def neighbours_to_host(t: dict) -> NeighbourTable:
        """D2H of a ``neighbours_device`` result (synchronises)."""
        host = {k: t[k].cpu().numpy() for k in ("row_ptr", "indices", "hybrid", "genre", "text", "metadata")}
        return NeighbourTable(**host, candidate_pairs=int(t["candidate_pairs"]))

    def compute_neighbours(self, features: dict, weights=(0.4, 0.5, 0.1), min_similarity: float = 0.1,
                           metadata_mode: str = "mean3", exclude_self: bool = True, max_per_row: int = 0,
                           **kw) -> NeighbourTable:
        """features dict -> every neighbour at or above ``min_similarity`` of every show, on this GPU."""
        cat = self.ingest(features, metadata_mode, weights)
        return self.neighbours_to_host(self.neighbours_device(cat, weights, min_similarity, exclude_self,
                                                              max_per_row, **kw))

    # ------------------------------------------------------------------------------------ several GPUs
    def _params(self, cat: DeviceCatalogue, weights, k, min_similarity, exclude_self=True, row_begin=0,
                row_end=None, splits=0, tuning=0) -> Params:
        gw, tw, mw = (float(w) for w in weights)
        return Params(genre_weight=gw, text_weight=tw, metadata_weight=mw, min_similarity=float(min_similarity),
                      k=int(k), exclude_self=int(bool(exclude_self)), row_begin=int(row_begin),
                      row_end=int(cat.n_shows if row_end is None else row_end), splits=int(splits), candidates=0,
                      force_exact=0, skip_fallback=0, text_rel_err=0.0, phases=0, tuning=int(tuning))

    def sym_eligible(self, cat: DeviceCatalogue, weights, k, min_similarity) -> bool:
        """Can this job use the symmetric (tile-sharded) sweep?  (packed groups, non-negative
        weights, positive threshold, k <= 100)"""
        if cat.folded:
            return False
        p = self._params(cat, weights, k, min_similarity)
        with torch.cuda.device(self.device):
            return bool(self.lib.tvbf_sym_eligible(C.byref(cat.c), C.byref(p)))

    def sym_seed(self, cat: DeviceCatalogue, weights, k, min_similarity, rank: int, world: int,
                 splits: int = 0, tuning: int = 0, reuse_theta: bool = False) -> torch.Tensor:
        """Phase 1 of the tile-sharded symmetric job: thresholds of this rank's shows seeded from a
        sampled sweep; returns theta int32[n_pad] (raw bits of positive floats), to be MAX-reduced
        over the ranks."""
        p = self._params(cat, weights, k, min_similarity, splits=splits, tuning=tuning)
        with torch.cuda.device(self.device):
            feats = self._k1_features(cat, weights, k, tuning)
            nbytes = self.lib.tvbf_sym_workspace_bytes(C.byref(feats), C.byref(p), world)
            if nbytes == 0:
                check(-1, "tvbf_sym_workspace_bytes")
            ws = self._workspace(nbytes)
            theta = self._theta if reuse_theta else None     # reuse: valid until this engine's next seeded job
            if theta is None or theta.numel() != int(cat.c.n_pad):
                theta = torch.empty((int(cat.c.n_pad),), dtype=torch.int32, device=self.device)
                if reuse_theta:
                    self._theta = theta
            check(self.lib.tvbf_sym_seed(C.byref(feats), C.byref(p), rank, world, theta.data_ptr(), ws.data_ptr(),
                                         ws.numel(), self._stream()), "tvbf_sym_seed")
        return theta

    def _k1_features(self, cat: DeviceCatalogue, weights, k, tuning: int = 0) -> Features:
        """The features the candidate pass runs on: the folded operand when the job qualifies."""
        gw, tw, mw = (float(w) for w in weights)
        return self._folded(cat, gw, tw, mw, int(k), int(tuning)) or cat.c

    def sym_sweep(self, cat: DeviceCatalogue, weights, k, min_similarity, rank: int, world: int,
                  theta: torch.Tensor, splits: int = 0, tuning: int = 0, packed_rows: int = 0,
                  peer_ptrs=None, peer_shard_rows: int = 0):
        """Phase 2: sweep this rank's tiles; returns partial candidate lists for ALL shows:
        (cand int32[N, L, 2], cnt int32[N], bound f32[N]), or -- with ``packed_rows`` >= N -- one
        int32[packed_rows, L + 1, 2] tensor whose entry L of each row holds {count, bound bits}
        (what ``sharding.exchange_packed`` moves in one all-to-all)."""
        p = self._params(cat, weights, k, min_similarity, splits=splits, tuning=tuning)
        dev, n = self.device, cat.n_shows
        with torch.cuda.device(dev):
            feats = self._k1_features(cat, weights, k, tuning)
            ws = self._workspace(self.lib.tvbf_sym_workspace_bytes(C.byref(feats), C.byref(p), world))
            L = int(self.lib.tvbf_sym_list_len(C.byref(feats), C.byref(p)))
            if peer_ptrs is not None:     # compaction fused with the exchange: rows go to their owners' buffers
                check(self.lib.tvbf_sym_sweep_peer(C.byref(feats), C.byref(p), rank, world, theta.data_ptr(), peer_ptrs,
                                                   int(peer_shard_rows), ws.data_ptr(), ws.numel(), self._stream()),
                      "tvbf_sym_sweep_peer")
                return None
            if packed_rows:
                assert packed_rows >= n
                packed = torch.empty((packed_rows, L + 1, 2), dtype=torch.int32, device=dev)
                check(self.lib.tvbf_sym_sweep(C.byref(feats), C.byref(p), rank, world, theta.data_ptr(),
                                              packed.data_ptr(), None, None, ws.data_ptr(), ws.numel(), self._stream()),
                      "tvbf_sym_sweep")
                return packed
            cand = torch.empty((n, L, 2), dtype=torch.int32, device=dev)
            cnt = torch.empty((n,), dtype=torch.int32, device=dev)
            bound = torch.empty((n,), dtype=torch.float32, device=dev)
            check(self.lib.tvbf_sym_sweep(C.byref(feats), C.byref(p), rank, world, theta.data_ptr(), cand.data_ptr(),
                                          cnt.data_ptr(), bound.data_ptr(), ws.data_ptr(), ws.numel(), self._stream()),
                  "tvbf_sym_sweep")
        return cand, cnt, bound

    def sym_rescore(self, cat: DeviceCatalogue, weights, k, min_similarity, cand_all: torch.Tensor,
                    cnt_all: torch.Tensor | None, bound_all: torch.Tensor | None, row_begin: int, row_end: int,
                    splits: int = 0, tuning: int = 0, table_row0: int = 0, out: dict | None = None) -> dict:
        """Phase 3: fp64 rescoring + certificate + exact repair of rows [row_begin, row_end) from the
        exchanged candidate tables ([world, R, L, 2] / [world, R], or packed [world, R, L + 1, 2] with
        ``cnt_all = bound_all = None``) that cover the shows [table_row0, table_row0 + R): R = N after
        an all-gather, R = this rank's (padded) shard after an all-to-all.  ``out``: tables to write
        (e.g. ``sharding.shard_views`` of the gather buffer); allocated when omitted."""
        dev, rows, world = self.device, row_end - row_begin, int(cand_all.shape[0])
        table_rows = int(cand_all.shape[1])
        with torch.cuda.device(dev):
            t = out if out is not None else self._alloc_tables(rows, k, row_begin)
            t["row_begin"] = row_begin
            if rows > 0:
                p = self._params(cat, weights, k, min_similarity, row_begin=row_begin, row_end=row_end,
                                 splits=splits, tuning=tuning)
                ws = self._workspace(self.lib.tvbf_sym_workspace_bytes(C.byref(cat.c), C.byref(p), world))
                cout = self._c_tables(t)
                check(self.lib.tvbf_rescore_lists(C.byref(cat.c), C.byref(p), cand_all.data_ptr(),
                                                  None if cnt_all is None else cnt_all.data_ptr(),
                                                  None if bound_all is None else bound_all.data_ptr(), world,
                                                  int(table_row0), table_rows,
                                                  C.byref(cout), ws.data_ptr(),
                                                  ws.numel(), self._stream()), "tvbf_rescore_lists")
            else:
                self._zero(t["stats"])
        return t

    def top_k_device_sym_sharded(self, cat: DeviceCatalogue, weights, k, min_similarity, rank: int, world: int,
                                 all_reduce_max, exchange, row_range, splits: int = 0, tuning: int = 0,
                                 events: dict | None = None, out: dict | None = None,
                                 padded_rows: int | None = None, peer=None) -> dict:
        """This GPU's part of the tile-sharded symmetric job: the three phases with the two
        collectives between them passed in as callables: ``all_reduce_max(int32 tensor)`` in place,
        and ``exchange(packed [world * shard_rows, L + 1, 2]) -> [world, shard_rows, L + 1, 2]``
        holding every rank's lists for THIS rank's rows ``row_range`` (one all-to-all over the row
        shards).  ``events``: dict that receives CUDA events around every phase (bench.py)."""
        def mark(name):
            if events is not None:
                ev = torch.cuda.Event(enable_timing=True)
                with torch.cuda.device(self.device):
                    ev.record()
                events.setdefault(name, []).append(ev)

        b, e = row_range
        padded_rows = padded_rows or cat.n_shows
        mark("seed0")
        theta = self.sym_seed(cat, weights, k, min_similarity, rank, world, splits, tuning, reuse_theta=True)
        mark("seed1")
        all_reduce_max(theta)            # raw bits of positive floats order like integers
        mark("reduce1")
        if peer is not None:
            # fused: K4s stores every finished candidate row into its owner's receive buffer (NVLink);
            # a device-side barrier makes the rows visible -- no all-to-all
            ptrs, packed_all, barrier = peer.next()
            self.sym_sweep(cat, weights, k, min_similarity, rank, world, theta, splits, tuning,
                           peer_ptrs=ptrs, peer_shard_rows=peer.rows)
            mark("sweep1")
            barrier()
        else:
            packed = self.sym_sweep(cat, weights, k, min_similarity, rank, world, theta, splits, tuning,
                                    packed_rows=padded_rows)
            mark("sweep1")
            packed_all = exchange(packed)
        mark("exchange1")
        t = self.sym_rescore(cat, weights, k, min_similarity, packed_all, None, None, b, e, splits, tuning,
                             table_row0=b, out=out)
        mark("rescore1")
        return t

    # ------------------------------------------------------------------------------------ exact
    def exact_rows(self, cat: DeviceCatalogue, rows, weights=(0.4, 0.5, 0.1), k: int = 10,
                   min_similarity: float = 0.0, exclude_self: bool = True) -> TopK:
        """Exact fp64 top-k of explicit source rows (the single-show query of
        services/content_based_service.py:161-236, any n up to 1024)."""
        rows_np = np.ascontiguousarray(np.asarray(rows, dtype=np.int32))
        if rows_np.size == 0:
            z = np.zeros((0, k))
            return TopK(np.zeros((0, k), np.int32), np.zeros(0, np.int32), z, z.copy(), z.copy(), z.copy())
        gw, tw, mw = (float(w) for w in weights)
        p = Params(genre_weight=gw, text_weight=tw, metadata_weight=mw, min_similarity=float(min_similarity),
                   k=int(k), exclude_self=int(bool(exclude_self)), row_begin=0, row_end=cat.n_shows)
        with torch.cuda.device(self.device):
            dev = self.device
            r = rows_np.shape[0]
            rows_d = torch.from_numpy(rows_np).to(dev)
            t = self._alloc_tables(r, k)
            out = self._c_tables(t)
            nbytes = self.lib.tvbf_exact_workspace_bytes(C.byref(cat.c), r)
            ws = self._workspace(nbytes)
            check(self.lib.tvbf_exact_rows(C.byref(cat.c), C.byref(p), rows_d.data_ptr(), r, C.byref(out),
                                           ws.data_ptr(), ws.numel(), self._stream()), "tvbf_exact_rows")
        return self.to_host(t)

    def matrix_rows_topk(self, hybrid: torch.Tensor, genre: torch.Tensor, text: torch.Tensor,
                         metadata: torch.Tensor, rows, k: int = 10, min_similarity: float = 0.0) -> TopK:
        """Top-k over rows of precomputed N x N device matrices (variant C,
        content_based_service.py:206-234)."""
        rows_np = np.ascontiguousarray(np.asarray(rows, dtype=np.int32))
        n = int(hybrid.shape[0])
        r = rows_np.shape[0]
        p = Params(genre_weight=0.0, text_weight=0.0, metadata_weight=0.0, min_similarity=float(min_similarity),
                   k=int(k), exclude_self=1, row_begin=0, row_end=n)
        with torch.cuda.device(self.device):
            dev = self.device
            rows_d = torch.from_numpy(rows_np).to(dev)
            t = self._alloc_tables(r, k)
            out = self._c_tables(t)
            nbytes = min(2 * self.sm_count, r) * n * 8 + 256
            ws = self._workspace(nbytes)
            check(self.lib.tvbf_matrix_rows_topk(hybrid.data_ptr(), genre.data_ptr(), text.data_ptr(),
                                                 metadata.data_ptr(), n, C.byref(p), rows_d.data_ptr(), r,
                                                 C.byref(out), ws.data_ptr(), ws.numel(), self._stream()),
                  "tvbf_matrix_rows_topk")
        return self.to_host(t)

    # ------------------------------------------------------------------------------------ matrices
    def cosine_matrix(self, x) -> torch.Tensor:
        """cosine_similarity(X) as an N x N float64 device tensor (similarity_computer.py:41,58,86);
        ``x`` is a dense array or a scipy sparse matrix."""
        with torch.cuda.device(self.device):
            dev, stream = self.device, self._stream()
            if sp.issparse(x):
                m = sp.csr_matrix(x, dtype=np.float64)
                if not m.has_canonical_format:
                    m = m.copy()
                    m.sum_duplicates()
                    m.sort_indices()
                n, d = m.shape
                if m.nnz == 0:       # every row is zero: so is every cosine (and there is nothing to upload)
                    return torch.zeros((n, n), dtype=torch.float64, device=dev)
                indptr = torch.from_numpy(m.indptr.astype(np.int64)).to(dev)
                indices = torch.from_numpy(m.indices.astype(np.int32)).to(dev)
                raw = torch.from_numpy(np.ascontiguousarray(m.data, dtype=np.float64)).to(dev)
                vals = torch.empty_like(raw)
                check(self.lib.tvbf_prep_csr_normalize(indptr.data_ptr(), raw.data_ptr(), n, vals.data_ptr(), stream),
                      "tvbf_prep_csr_normalize")
                xn = torch.zeros((n, d), dtype=torch.float64, device=dev)
                check(self.lib.tvbf_csr_to_dense_f64(indptr.data_ptr(), indices.data_ptr(), vals.data_ptr(), n, d,
                                                     xn.data_ptr(), stream), "tvbf_csr_to_dense_f64")
            else:
                a = np.ascontiguousarray(np.asarray(x), dtype=np.float64)
                if a.ndim != 2:
                    raise ValueError("feature matrix must be 2-D")
                n, d = a.shape
                raw = torch.from_numpy(a).to(dev)
                xn = torch.empty_like(raw)
                check(self.lib.tvbf_prep_dense_normalize(raw.data_ptr(), n, d, xn.data_ptr(), stream),
                      "tvbf_prep_dense_normalize")
            out = torch.empty((n, n), dtype=torch.float64, device=dev)
            check(self.lib.tvbf_cosine_matrix_f64(xn.data_ptr(), n, d, out.data_ptr(), stream),
                  "tvbf_cosine_matrix_f64")
        return out

    def hybrid_combine(self, g: torch.Tensor, t: torch.Tensor, m: torch.Tensor, wg: float, wt: float,
                       wm: float) -> torch.Tensor:
        """wg*g + wt*t + wm*m elementwise on the device (similarity_computer.py:122-124)."""
        with torch.cuda.device(self.device):
            out = torch.empty_like(g)
            check(self.lib.tvbf_hybrid_combine_f64(g.data_ptr(), t.data_ptr(), m.data_ptr(), float(wg), float(wt),
                                                   float(wm), g.numel(), out.data_ptr(), self._stream()),
                  "tvbf_hybrid_combine_f64")
        return out

    def matrix_stats(self, mat: torch.Tensor) -> dict:
        """Upper-triangle statistics (similarity_computer.py:171-190)."""
        n = int(mat.shape[0])
        with torch.cuda.device(self.device):
            ws = self._workspace(self.lib.tvbf_matrix_stats_workspace_bytes())
            out5 = (C.c_double * 5)()
            check(self.lib.tvbf_matrix_stats_f64(mat.data_ptr(), n, out5, ws.data_ptr(), ws.numel(), self._stream()),
                  "tvbf_matrix_stats_f64")
        return {"mean": float(out5[0]), "std": float(out5[1]), "min": float(out5[2]),
                "max": float(out5[3]), "median": float(out5[4])}

    # ------------------------------------------------------------------------------------ streaming statistics
    _STATS_DTYPE = np.dtype([("sum", "<f8", 4), ("sumsq", "<f8", 4), ("zeros", "<u8", 4),
                             ("hist", "<u8", (4, 1024)), ("min_bits", "<u4", 4), ("max_bits", "<u4", 4),
                             ("hi", "<f4", 4), ("n_cand", "<i4"), ("cand_ij", "<i4", (2, 2048, 2)),
                             ("cand_val", "<f4", (2, 2048)), ("sum_gm", "<f8")], align=True)

    def similarity_stats(self, cat: DeviceCatalogue, weights, exact_moments: bool = True,
                         gram_bytes_limit: int | None = None) -> dict:
        """Upper-triangle statistics of the genre / text / metadata / hybrid similarity matrices
        (ml/similarity_computer.py:171-190) WITHOUT materialising them: one symmetric tensor-core
        sweep accumulates sums, extrema, zero counts and 1024-bin histograms on the device; the
        largest text and hybrid elements are rescored exactly in float64.

        The fp16 text operand alone would limit mean / std of text and hybrid to ~1e-5 (its rounding
        is correlated per vocabulary column).  With ``exact_moments`` every text-dependent sum --
        sum t, sum t^2, sum g*t, sum m*t -- is computed exactly in float64 from small Gram-type
        matrices (``tvbf_text_moments``: column sums, [64, V], [32, V] and, memory permitting, the
        [V, V] vocabulary Gram matrix) and the hybrid's moments are assembled from them, so mean and
        std agree with the reference's float64 to ~1e-9 (genre / metadata elements are fp32 values
        summed in float64: ~1e-8); std has an absolute floor of ~2^-26 sqrt(rms^2 + 2 / (N - 1)), where
        the one-pass variance cancels (nearly equal elements, tiny N).  min: an exact 0.0 when some element is zero, otherwise the fp32
        element value.  median to one histogram bin (``median_resolution``).

        The text and hybrid max are the float64 maxima, bit-identical to ``tvbf_score_pairs`` of the
        pair that attains them.  The sweep keeps the pair with the largest fp16 / fp32 element value
        of every epilogue warp; many pairs can share that value, so the true maximum need not be among
        them.  Their best exact score tau is a score some pair attains, hence a lower bound of the
        maximum.  An exact top-1 job at ``min_similarity = tau`` (``top_k_device``: certified, its
        scores those of ``tvbf_score_pairs``) then finds every row's best neighbour scoring >= tau;
        the largest of those is the maximum over all pairs, in O(N) memory however many pairs tie.
        Text runs with weights (0, 1, 0), the hybrid with ``weights``; tau <= 0 means the maximum is
        0 and needs no job.  genre / metadata max: the fp32 element value.

        Needs N >= 2 (ValueError: the upper triangle is empty) and non-negative text: signed text
        (embeddings) raises ``TvbfError``; the N x N path (``matrix_stats``) takes it."""
        gw, tw, mw = (float(w) for w in weights)
        n = cat.n_shows
        if n < 2:
            raise ValueError(f"similarity statistics need at least 2 shows: the upper triangle of {n} x {n} "
                             "is empty")
        p = self._params(cat, (gw, tw, mw), 20, 0.5)
        lib, dev = self.lib, self.device
        with torch.cuda.device(dev):
            nbytes = int(lib.tvbf_stats_accum_bytes())
            assert nbytes == self._STATS_DTYPE.itemsize, (nbytes, self._STATS_DTYPE.itemsize)
            accum = torch.zeros((nbytes,), dtype=torch.uint8, device=dev)
            p1 = self._params(cat, (gw, tw, mw), 20, 0.5, tuning=1 << 20)
            ws = self._workspace(max(int(lib.tvbf_topk_workspace_bytes(C.byref(cat.c), C.byref(p1))), 1 << 20))
            check(lib.tvbf_similarity_stats(C.byref(cat.c), C.byref(p), accum.data_ptr(), ws.data_ptr(), ws.numel(),
                                            self._stream()), "tvbf_similarity_stats")
            raw = np.frombuffer(accum.cpu().numpy().tobytes(), dtype=self._STATS_DTYPE)[0]
            # exact float64 value of the largest text / hybrid elements
            pairs = raw["cand_ij"].reshape(-1, 2)
            keep = pairs[:, 0] >= 0
            exact_max = {}
            if keep.any():
                pk = np.ascontiguousarray(pairs[keep].astype(np.int32))
                pd = torch.from_numpy(pk).to(dev)
                out4 = torch.empty((pk.shape[0], 4), dtype=torch.float64, device=dev)
                check(lib.tvbf_score_pairs(C.byref(cat.c), C.byref(p), pd.data_ptr(), pk.shape[0], out4.data_ptr(),
                                           self._stream()), "tvbf_score_pairs")
                o = out4.cpu().numpy()
                for name, w, col in (("text_similarity", (0.0, 1.0, 0.0), 2), ("hybrid_similarity", (gw, tw, mw), 0)):
                    tau = float(o[:, col].max())
                    if tau > 0.0:
                        top = self.to_host(self.top_k_device(cat, w, 1, tau))
                        best = getattr(top, "text" if col == 2 else "hybrid")[top.counts > 0, 0]
                        tau = float(best.max(initial=tau))
                    exact_max[name] = tau
            moments = None
            if exact_moments:
                v = int(cat.c.vocab)
                free, _tot = torch.cuda.mem_get_info()
                limit = int(free * 0.5) if gram_bytes_limit is None else int(gram_bytes_limit)
                with_gram = 1 if 8 * v * v <= limit else 0
                mb = int(lib.tvbf_text_moments_workspace_bytes(C.byref(cat.c), with_gram))
                mws = torch.empty((mb,), dtype=torch.uint8, device=dev)
                out8 = torch.empty((24,), dtype=torch.float64, device=dev)
                check(lib.tvbf_text_moments(C.byref(cat.c), with_gram, out8.data_ptr(), mws.data_ptr(), mb,
                                            self._stream()), "tvbf_text_moments")
                moments = out8.cpu().numpy()
                del mws
        count = n * (n - 1) // 2
        names = ("genre_similarity", "text_similarity", "metadata_similarity", "hybrid_similarity")
        s1 = [float(x) for x in raw["sum"]]
        s2 = [float(x) for x in raw["sumsq"]]
        exact = {"text_mean": False, "text_std": False}
        if moments is not None:
            # strict upper triangle = (all pairs - diagonal) / 2
            st_, st2, sgt, smt = ((moments[a] - moments[a + 4]) / 2 for a in range(4))
            sg_, sg2, sm_, sm2, sgm = ((moments[8 + a] - moments[13 + a]) / 2 for a in range(5))
            s1[0], s2[0], s1[2], s2[2] = sg_, sg2, sm_, sm2       # genre / metadata: exact as well
            s1[1] = st_
            s1[3] = gw * sg_ + tw * st_ + mw * sm_
            exact["text_mean"] = True
            if with_gram:
                s2[1] = st2
                s2[3] = (gw * gw * sg2 + tw * tw * st2 + mw * mw * sm2 + 2 * gw * tw * sgt
                         + 2 * gw * mw * sgm + 2 * tw * mw * smt)
                exact["text_std"] = True
        out = {}
        for q, name in enumerate(names):
            mean = s1[q] / count
            var = max(0.0, s2[q] / count - mean * mean)
            zeros = int(raw["zeros"][q])
            hist = raw["hist"][q].astype(np.int64)
            width = float(raw["hi"][q]) / 1024.0

            def value_at(rank: int) -> float:
                if rank < zeros:
                    return 0.0
                cum = zeros + np.cumsum(hist)
                b = int(np.searchsorted(cum, rank, side="right"))
                before = zeros + int(hist[:b].sum())
                return (b + (rank - before + 0.5) / max(int(hist[b]), 1)) * width

            vmin = 0.0 if zeros else float(np.frombuffer(np.uint32(raw["min_bits"][q]).tobytes(), np.float32)[0])
            vmax = float(np.frombuffer(np.uint32(raw["max_bits"][q]).tobytes(), np.float32)[0])
            out[name] = {"mean": mean, "std": float(np.sqrt(var)), "min": vmin,
                         "max": exact_max.get(name, vmax),
                         "median": 0.5 * (value_at((count - 1) // 2) + value_at(count // 2)),
                         "median_resolution": width,
                         "exact_moments": dict(exact) if q in (1, 3) else {"text_mean": True, "text_std": True}}
        return out

    def plan_tiles(self, cat: DeviceCatalogue, weights, k, min_similarity, rank: int = 0, world: int = 1,
                   tile_sharded: bool = False, row_begin: int = 0, row_end: int | None = None, splits: int = 0,
                   tuning: int = 0) -> dict:
        """Tensor-core tiles the candidate pass of this job executes (``tvbf_plan_tiles``, host only).
        A job that runs over the second operand (``_folded``) is planned over it (k_pad)."""
        p = self._params(cat, weights, k, min_similarity, row_begin=row_begin, row_end=row_end, splits=splits,
                         tuning=tuning)
        out = (C.c_int64 * 4)()
        feats = cat.c
        w = tuple(float(x) for x in weights)
        layout = self._second_layout(cat, *w, int(k), int(tuning))
        fc = cat.fold
        if layout is not None and fc is not None and self._fold_owner is fc and fc["layout"] == layout \
                and (not layout[1] or fc["weights"] == w):
            feats = fc["c"]
        with torch.cuda.device(self.device):
            check(self.lib.tvbf_plan_tiles(C.byref(feats), C.byref(p), int(rank), int(world), int(bool(tile_sharded)),
                                           out), "tvbf_plan_tiles")
        seed, sweep, rows, sym = (int(x) for x in out)
        return {"seed_tiles": seed, "sweep_tiles": sweep, "tile_rows": rows, "symmetric": bool(sym),
                "k_pad": int(feats.k_pad), "folded_bits": bool(feats.bits_folded), "text_cols": int(feats.text_cols),
                "flops": 2.0 * (seed + sweep) * rows * 256 * int(feats.k_pad)}

    def debug_slack(self, cat: DeviceCatalogue, weights, feats: Features | None = None) -> dict:
        """Constants of the candidate pass' upper bound (``tvbf_debug_slack``; tests only).  ``feats``:
        the ``_folded`` variant of ``cat``'s features."""
        p = self._params(cat, weights, 20, 0.1)
        out = (C.c_float * 5)()
        check(self.lib.tvbf_debug_slack(C.byref(cat.c if feats is None else feats), C.byref(p), out), "tvbf_debug_slack")
        return dict(zip(("w_text", "w_text_err", "w_text_acc", "eps", "eps_term"), (float(x) for x in out)))

    def debug_gemm_tile(self, cat: DeviceCatalogue, row0: int, col0: int, pair: bool = False,
                        feats: Features | None = None) -> torch.Tensor:
        """Raw fp32 accumulators of one tensor-core tile (diagnostics / tests): 128 x 256 through
        cta_group::1, or 256 x 256 through a cta_group::2 CTA pair."""
        with torch.cuda.device(self.device):
            out = torch.zeros((256 if pair else 128, 256), dtype=torch.float32, device=self.device)
            fn = self.lib.tvbf_debug_gemm_tile_pair if pair else self.lib.tvbf_debug_gemm_tile
            check(fn(C.byref(cat.c if feats is None else feats), int(row0), int(col0), out.data_ptr(), self._stream()),
                  "tvbf_debug_gemm_tile")
        return out


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


_default_engine: HybridTopKEngine | None = None


def default_engine() -> HybridTopKEngine:
    """Process-wide engine on the current CUDA device (raises without a B200)."""
    global _default_engine
    if _default_engine is None:
        _default_engine = HybridTopKEngine()
    return _default_engine
