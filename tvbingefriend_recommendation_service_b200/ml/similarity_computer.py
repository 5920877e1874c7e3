"""Drop-in ``SimilarityComputer`` (reference: ml/similarity_computer.py:12-190) on B200.

Same constructor, methods, defaults and return types as the reference class; every method runs
CUDA kernels of ``libtvbf.so`` and raises if the library or an sm_100 GPU is missing.  The
additive ``compute_top_k`` is the production path: features -> hybrid score -> per-show top-K
without materialising any N x N matrix.
"""

from __future__ import annotations

import logging

import numpy as np
import torch

from ..engine import HybridTopKEngine, TopK, default_engine

logger = logging.getLogger(__name__)


def _split_rows(features: dict, n: int) -> tuple[dict, dict]:
    """(rows [0, n), rows [n, ...)) of the five feature matrices of a features dict."""
    keys = ("genre_features", "text_features", "platform_features", "type_features", "language_features")
    old, new = dict(features), dict(features)
    for key in keys:
        a = features[key]
        old[key], new[key] = a[:n], a[n:]
    return old, new


def _changed_rows(top: TopK, previous: TopK, row_map: np.ndarray | None = None) -> np.ndarray:
    """Sorted int32 rows of ``previous`` that differ from the same rows of ``top`` in any of the six
    fields (the scores bit for bit).  With ``row_map`` (a removal: previous row o is row
    ``row_map[o]`` of ``top``, -1 when it was removed) the rows of ``top`` are compared with their
    previous rows, whose indices are renumbered by ``row_map`` (a removed show becomes -1)."""
    prev = {name: getattr(previous, name) for name in ("indices", "counts", "hybrid", "genre", "text", "metadata")}
    if row_map is not None:
        keep = np.nonzero(row_map >= 0)[0]
        prev = {name: a[keep] for name, a in prev.items()}
        idx = prev["indices"]
        prev["indices"] = np.where(idx >= 0, row_map[np.maximum(idx, 0)], idx).astype(idx.dtype)
    n = prev["counts"].shape[0]
    diff = (top.counts[:n] != prev["counts"]) | (top.indices[:n] != prev["indices"]).any(axis=1)
    for name in ("hybrid", "genre", "text", "metadata"):
        diff |= (getattr(top, name)[:n].view(np.int64) != prev[name].view(np.int64)).any(axis=1)
    return np.nonzero(diff)[0].astype(np.int32)


# noinspection PyMethodMayBeStatic
class SimilarityComputer:
    """Compute similarity matrices (and top-K tables) from feature arrays."""

    def __init__(self, genre_weight: float = 0.4, text_weight: float = 0.5,
                 metadata_weight: float = 0.1, engine: HybridTopKEngine | None = None):
        # reference :15-28
        self.genre_weight = genre_weight
        self.text_weight = text_weight
        self.metadata_weight = metadata_weight
        self._engine = engine

    @property
    def engine(self) -> HybridTopKEngine:
        if self._engine is None:
            self._engine = default_engine()
        return self._engine

    # ---- N x N variant (reference :30-130) ------------------------------------------------------
    def _cosine(self, x, label: str) -> torch.Tensor:
        logger.info(f"Computing {label} similarity...")
        sim = self.engine.cosine_matrix(x)
        logger.info(f" {label.capitalize()} similarity: {tuple(sim.shape)}")
        return sim

    @staticmethod
    def _out_dtype(*arrays):
        """sklearn's dtype rule (check_pairwise_arrays / _return_float_dtype, SURVEY.md section 3.6):
        the result is float32 only when EVERY input is float32, else float64.  The arithmetic here is
        float64 either way (more precise than the reference's float32 run, within 1e-6 of it)."""
        return np.float32 if all(getattr(a, "dtype", None) == np.float32 for a in arrays) else np.float64

    def compute_genre_similarity(self, genre_features: np.ndarray) -> np.ndarray:
        """cosine_similarity(genre_features) -> (n_shows, n_shows) float64 (reference :30-45)."""
        return self._cosine(genre_features, "genre").cpu().numpy().astype(self._out_dtype(genre_features), copy=False)

    def compute_text_similarity(self, text_features) -> np.ndarray:
        """cosine_similarity on TF-IDF vectors, dense or scipy sparse (reference :47-62)."""
        return self._cosine(text_features, "text").cpu().numpy().astype(self._out_dtype(text_features), copy=False)

    def compute_metadata_similarity(self, platform_features: np.ndarray, type_features: np.ndarray,
                                    language_features: np.ndarray) -> np.ndarray:
        """cosine of the hstack of platform/type/language (reference :64-90)."""
        metadata_features = np.hstack([platform_features, type_features, language_features])
        return self._cosine(metadata_features, "metadata").cpu().numpy().astype(
            self._out_dtype(metadata_features), copy=False)

    def _normalized_weights(self) -> tuple[float, float, float]:
        total_weight = self.genre_weight + self.text_weight + self.metadata_weight  # reference :112-115
        return (self.genre_weight / total_weight, self.text_weight / total_weight,
                self.metadata_weight / total_weight)

    def compute_hybrid_similarity(self, genre_similarity: np.ndarray, text_similarity: np.ndarray,
                                  metadata_similarity: np.ndarray) -> np.ndarray:
        """Weighted combination with weights normalised by their sum (reference :92-130)."""
        logger.info("Computing hybrid similarity...")
        gw, tw, mw = self._normalized_weights()
        logger.info(f"  Weights - Genre: {gw:.2f}, Text: {tw:.2f}, Metadata: {mw:.2f}")
        dev = self.engine.device
        g, t, m = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
                   for a in (genre_similarity, text_similarity, metadata_similarity))
        return self.engine.hybrid_combine(g, t, m, gw, tw, mw).cpu().numpy()

    def compute_all_similarities(self, features: dict[str, np.ndarray]) -> dict[str, np.ndarray]:
        """All four matrices (reference :132-169); intermediates stay on the GPU."""
        logger.info("=" * 60)
        logger.info("COMPUTING ALL SIMILARITIES")
        logger.info("=" * 60)
        g = self._cosine(features["genre_features"], "genre")
        t = self._cosine(features["text_features"], "text")
        m = self._cosine(np.hstack([features["platform_features"], features["type_features"],
                                    features["language_features"]]), "metadata")
        gw, tw, mw = self._normalized_weights()
        h = self.engine.hybrid_combine(g, t, m, gw, tw, mw)
        logger.info("=" * 60)
        logger.info("SIMILARITY COMPUTATION COMPLETE")
        logger.info("=" * 60)
        return {"genre_similarity": g.cpu().numpy(), "text_similarity": t.cpu().numpy(),
                "metadata_similarity": m.cpu().numpy(), "hybrid_similarity": h.cpu().numpy()}

    def get_similarity_statistics(self, similarity_matrix: np.ndarray) -> dict[str, float]:
        """mean/std/min/max/median of the strict upper triangle (reference :171-190)."""
        mat = torch.from_numpy(np.ascontiguousarray(similarity_matrix, dtype=np.float64)).to(self.engine.device)
        return self.engine.matrix_stats(mat)

    def compute_similarity_statistics(self, features: dict, metadata_mode: str = "hstack",
                                      normalize_weights: bool = True) -> dict[str, dict[str, float]]:
        """The four ``get_similarity_statistics`` results of scripts/compute_similarities.py:119-131
        for catalogues whose N x N matrices cannot exist: one streaming tensor-core sweep (defaults =
        this class' conventions: hstack metadata, normalised weights).  mean / std / min / max as
        the reference's, median to ``median_resolution``.  Needs binary genre and one-hot metadata
        features."""
        weights = self._normalized_weights() if normalize_weights else \
            (self.genre_weight, self.text_weight, self.metadata_weight)
        cat = self.engine.ingest(features, metadata_mode, weights)
        return self.engine.similarity_stats(cat, weights)

    # ---- production variant: no N x N ------------------------------------------------------------
    def compute_top_k(self, features: dict, k: int = 20, min_similarity: float = 0.1,
                      exclude_self: bool = True, metadata_mode: str = "mean3",
                      normalize_weights: bool = False, device_ids=None, **kw) -> TopK:
        """features -> per-show top-K table.

        Defaults reproduce the production loop (scripts/populate_database.py:170-218): mean of the
        three metadata cosines and RAW weights.  ``metadata_mode="hstack", normalize_weights=True``
        reproduces what this class + the service produce (reference :84-86, :112-115).
        Ties are broken by (score descending, column index ascending)."""
        weights = self._normalized_weights() if normalize_weights else \
            (self.genre_weight, self.text_weight, self.metadata_weight)
        if device_ids is not None and len(device_ids) > 1:
            from ..multi_gpu import compute_top_k_multi_gpu
            return compute_top_k_multi_gpu(features, weights, k, min_similarity, metadata_mode,
                                           exclude_self, list(device_ids), **kw)
        eng = self.engine if device_ids is None else HybridTopKEngine(device_ids[0])
        return eng.compute_top_k(features, weights, k, min_similarity, metadata_mode, exclude_self, **kw)

    def extend_top_k(self, features: dict, previous: TopK, k: int = 20, min_similarity: float = 0.1,
                     exclude_self: bool = True, metadata_mode: str = "mean3",
                     normalize_weights: bool = False) -> TopK:
        """Top-K table after appending shows to a catalogue whose table exists.

        ``features`` covers all N + Q shows: the N shows of ``previous`` (the ``compute_top_k``
        table of the first N rows with the same arguments) followed by the Q new ones.  The result
        equals ``compute_top_k(features, ...)`` bit for bit; its ``changed_rows`` lists the old rows
        (sorted int32) whose neighbours or their count changed -- every other old row is identical
        to its row in ``previous``, so a caller only has to store the listed rows and the new ones.
        Only the pairs with a new show are scored on the tensor cores.

        Precondition: the first N shows' features are those ``previous`` was computed from, and the
        new shows are encoded in the same vocabulary and widths (the already fitted extractor); a
        refitted extractor changes every row and needs ``compute_top_k``.  Jobs the incremental path
        does not take (signed text, float-valued groups, k > 100, ``exclude_self=False``, ...) run the
        whole job and compare."""
        weights = self._normalized_weights() if normalize_weights else \
            (self.genre_weight, self.text_weight, self.metadata_weight)
        n_all = int(np.asarray(features["genre_features"]).shape[0])
        n_old = int(previous.counts.shape[0])
        if previous.indices.ndim != 2 or previous.indices.shape != (n_old, k) or previous.row_begin != 0:
            raise ValueError(f"previous table has shape {previous.indices.shape}, expected ({n_old}, {k}) from row 0")
        if n_old > n_all:
            raise ValueError(f"previous table has {n_old} rows, features only {n_all}")
        eng = self.engine

        def full() -> TopK:
            top = eng.compute_top_k(features, weights, k, min_similarity, metadata_mode, exclude_self)
            top.changed_rows = _changed_rows(top, previous)
            return top

        if n_old == n_all:
            return TopK(previous.indices, previous.counts, previous.hybrid, previous.genre, previous.text,
                        previous.metadata, changed_rows=np.zeros(0, dtype=np.int32))
        if not exclude_self or n_old == 0:
            return full()
        old, new = _split_rows(features, n_old)
        try:
            cat = eng.extend(eng.ingest(old, metadata_mode, weights), new)
        except ValueError:
            # the two parts classify differently (e.g. binary genres before, fractional ones among the
            # new shows): one catalogue encoding for all rows needs the whole job
            return full()
        with torch.cuda.device(eng.device):
            dev = eng.device
            prev = {name: torch.from_numpy(np.ascontiguousarray(getattr(previous, name))).to(dev)
                    for name in ("indices", "counts", "hybrid", "genre", "text", "metadata")}
            t = eng.top_k_append_device(cat, n_old, prev, weights, k, min_similarity)
            changed = t["changed_rows"].cpu().numpy()
        top = eng.to_host(t)
        top.changed_rows = changed
        return top

    def update_top_k(self, features: dict, previous: TopK, rows, k: int = 20, min_similarity: float = 0.1,
                     exclude_self: bool = True, metadata_mode: str = "mean3",
                     normalize_weights: bool = False) -> TopK:
        """Top-K table after the shows ``rows`` of a catalogue whose table exists got new features.

        ``features`` is the whole catalogue after the update; ``previous`` is the ``compute_top_k``
        table of the catalogue before it, with the same arguments.  The result equals
        ``compute_top_k(features, ...)`` bit for bit; its ``changed_rows`` lists the rows (sorted
        int32, updated or not) that differ from ``previous`` in any field -- every other row is
        identical to its row in ``previous``, so a caller only has to store the listed rows.  Only
        the updated shows' rows are scored against the catalogue on the tensor cores.

        Precondition, which the library cannot check: every row not in ``rows`` has the features
        ``previous`` was computed from, and all rows are encoded in the same vocabulary and widths
        (the already fitted extractor); a refitted extractor changes every row and needs
        ``compute_top_k``.  Jobs the incremental path does not take (signed text, float-valued
        groups, k > 100, ``exclude_self=False``, ...) run the whole job and compare."""
        weights = self._normalized_weights() if normalize_weights else \
            (self.genre_weight, self.text_weight, self.metadata_weight)
        n_all = int(np.asarray(features["genre_features"]).shape[0])
        if previous.indices.ndim != 2 or previous.indices.shape != (n_all, k) or previous.counts.shape != (n_all,) \
                or previous.row_begin != 0:
            raise ValueError(f"previous table has shape {previous.indices.shape}, expected ({n_all}, {k}) from row 0")
        eng = self.engine
        r = eng._update_rows(rows, n_all)
        fields = ("indices", "counts", "hybrid", "genre", "text", "metadata")

        if r.size == 0:
            return TopK(*(getattr(previous, name) for name in fields), changed_rows=np.zeros(0, dtype=np.int32))
        if not exclude_self:
            top = eng.compute_top_k(features, weights, k, min_similarity, metadata_mode, exclude_self)
            top.changed_rows = _changed_rows(top, previous)
            return top
        # one catalogue encoding for all rows: when the updated rows make a group float-valued (or the
        # others are), the whole catalogue is ingested that way and the whole job runs
        cat = eng.ingest(features, metadata_mode, weights)
        with torch.cuda.device(eng.device):
            prev = {name: torch.from_numpy(np.ascontiguousarray(getattr(previous, name))).to(eng.device)
                    for name in fields}
            t = eng.top_k_update_device(cat, r, prev, weights, k, min_similarity)
            changed = t["changed_rows"].cpu().numpy()
        top = eng.to_host(t)
        top.changed_rows = changed
        return top

    def remove_top_k(self, features: dict, previous: TopK, rows, k: int = 20, min_similarity: float = 0.1,
                     exclude_self: bool = True, metadata_mode: str = "mean3",
                     normalize_weights: bool = False) -> TopK:
        """Top-K table after the shows ``rows`` left a catalogue whose table exists.

        ``features`` is the catalogue after the removal (the remaining shows in their old order);
        ``previous`` is the ``compute_top_k`` table of the catalogue before it, with the same
        arguments, and ``rows`` are the removed shows' rows in it.  Row r of the result is the r-th
        remaining show, and its indices are rows of ``features``.  The result equals
        ``compute_top_k(features, ...)`` bit for bit; its ``changed_rows`` lists the rows (sorted
        int32) that differ in any field from their previous row with its indices renumbered -- every
        other row is identical to that, so a caller only has to store the listed rows.  Only the
        shows whose previous row names a removed show are scored against the catalogue on the
        tensor cores.  Removing every show raises ``ValueError``.

        Precondition, which the library cannot check: the remaining shows have the features
        ``previous`` was computed from.  Jobs the incremental path does not take (signed text,
        float-valued groups, k > 100, ``exclude_self=False``, ...) run the whole job and compare."""
        weights = self._normalized_weights() if normalize_weights else \
            (self.genre_weight, self.text_weight, self.metadata_weight)
        n_all = int(np.asarray(features["genre_features"]).shape[0])
        n_old = int(previous.counts.shape[0])
        eng = self.engine
        r = eng._update_rows(rows, n_old)
        if previous.indices.ndim != 2 or previous.indices.shape != (n_all + r.size, k) \
                or previous.counts.shape != (n_all + r.size,) or previous.row_begin != 0:
            raise ValueError(f"previous table has shape {previous.indices.shape}, expected "
                             f"({n_all + r.size}, {k}) from row 0")
        if n_all == 0:
            raise ValueError("remove_top_k: removing every show leaves no catalogue")
        fields = ("indices", "counts", "hybrid", "genre", "text", "metadata")

        if r.size == 0:
            return TopK(*(getattr(previous, name) for name in fields), changed_rows=np.zeros(0, dtype=np.int32))
        if not exclude_self:
            row_map = np.full(n_old, -1, dtype=np.int64)
            row_map[np.delete(np.arange(n_old), r)] = np.arange(n_all)
            top = eng.compute_top_k(features, weights, k, min_similarity, metadata_mode, exclude_self)
            top.changed_rows = _changed_rows(top, previous, row_map)
            return top
        cat = eng.ingest(features, metadata_mode, weights)
        with torch.cuda.device(eng.device):
            prev = {name: torch.from_numpy(np.ascontiguousarray(getattr(previous, name))).to(eng.device)
                    for name in fields}
            t = eng.top_k_remove_device(cat, r, prev, weights, k, min_similarity)
            changed = t["changed_rows"].cpu().numpy()
        top = eng.to_host(t)
        top.changed_rows = changed
        return top

    def refresh_top_k(self, features: dict, previous: TopK, removed=(), updated=(), k: int = 20,
                      min_similarity: float = 0.1, exclude_self: bool = True, metadata_mode: str = "mean3",
                      normalize_weights: bool = False) -> TopK:
        """Top-K table after a refresh of a catalogue whose table exists: the shows ``removed`` left,
        the shows ``updated`` got new features and new shows were appended, all at once.

        ``features`` is the catalogue after the refresh: the remaining shows in their old order (the
        updated ones with their new features), then the appended shows.  ``previous`` is the
        ``compute_top_k`` table of the catalogue before it, with the same arguments; ``removed`` and
        ``updated`` are rows of it (distinct, disjoint).  The number of appended shows follows from
        the shapes.  Row r of the result is row r of ``features``.  The result equals
        ``compute_top_k(features, ...)`` bit for bit; its ``changed_rows`` lists the rows to store
        (sorted int32): every appended row, and every remaining row that differs in any field from
        its previous row with the indices renumbered -- every other row is identical to that.
        Unlike ``extend_top_k``, whose ``changed_rows`` holds old rows only, the appended rows are
        listed too.  Only the updated and appended shows, the shows whose previous row names a
        removed show, and rows that lost a neighbour they cannot refill otherwise are scored against
        the catalogue on the tensor cores.  Removing every old show raises ``ValueError``.

        Precondition, which the library cannot check: every remaining show not in ``updated`` has
        the features ``previous`` was computed from, and all rows are encoded in the same vocabulary
        and widths (the already fitted extractor).  Jobs the incremental path does not take (signed
        text, float-valued groups, k > 100, ``exclude_self=False``, ...) run the whole job and
        compare."""
        weights = self._normalized_weights() if normalize_weights else \
            (self.genre_weight, self.text_weight, self.metadata_weight)
        n_all = int(np.asarray(features["genre_features"]).shape[0])
        n_old = int(previous.counts.shape[0])
        if previous.indices.ndim != 2 or previous.indices.shape != (n_old, k) or previous.row_begin != 0:
            raise ValueError(f"previous table has shape {previous.indices.shape}, expected ({n_old}, {k}) from row 0")
        eng = self.engine
        rem = eng._update_rows(removed, n_old)
        upd = eng._update_rows(updated, n_old)
        if np.intersect1d(rem, upd).size:
            raise ValueError("removed and updated rows overlap")
        if rem.size == n_old:
            raise ValueError("refresh_top_k: removing every old show leaves no catalogue to refresh")
        n_app = n_all - (n_old - int(rem.size))
        if n_app < 0:
            raise ValueError(f"features hold {n_all} shows, fewer than the {n_old - rem.size} remaining ones")
        fields = ("indices", "counts", "hybrid", "genre", "text", "metadata")

        if rem.size == 0 and upd.size == 0 and n_app == 0:
            return TopK(*(getattr(previous, name) for name in fields), changed_rows=np.zeros(0, dtype=np.int32))
        if not exclude_self:
            row_map = np.full(n_old, -1, dtype=np.int64)
            row_map[np.delete(np.arange(n_old), rem)] = np.arange(n_old - rem.size)
            top = eng.compute_top_k(features, weights, k, min_similarity, metadata_mode, exclude_self)
            top.changed_rows = np.concatenate([_changed_rows(top, previous, row_map),
                                               np.arange(n_all - n_app, n_all, dtype=np.int32)])
            return top
        cat = eng.ingest(features, metadata_mode, weights)
        with torch.cuda.device(eng.device):
            prev = {name: torch.from_numpy(np.ascontiguousarray(getattr(previous, name))).to(eng.device)
                    for name in fields}
            t = eng.top_k_refresh_device(cat, prev, rem, upd, n_app, weights, k, min_similarity)
            changed = t["changed_rows"].cpu().numpy()
        top = eng.to_host(t)
        top.changed_rows = changed
        return top

    def compute_top_k_sweep(self, features: dict, weight_list, k: int = 20, min_similarity: float = 0.1,
                            exclude_self: bool = True, metadata_mode: str = "mean3",
                            normalize_weights: bool = False, **kw) -> list[TopK]:
        """One top-K table per (genre, text, metadata) weight triple -- the comparison of weighting
        schemes the reference does by re-running everything per scheme (notebooks/03 cell 6) -- with
        staging, upload and feature prep shared by all triples and, on large catalogues of binary /
        one-hot features, ONE tensor-core sweep for up to five triples.  Each table is identical to
        what ``SimilarityComputer(*triple).compute_top_k(...)`` returns."""
        triples = []
        for gw, tw, mw in weight_list:
            tot = float(gw) + float(tw) + float(mw)
            triples.append((gw / tot, tw / tot, mw / tot) if normalize_weights else (float(gw), float(tw), float(mw)))
        return self.engine.compute_top_k_sweep(features, triples, k, min_similarity, metadata_mode, exclude_self, **kw)
