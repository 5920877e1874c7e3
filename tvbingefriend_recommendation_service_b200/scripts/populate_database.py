"""Drop-in for the hot function of scripts/populate_database.py:
``compute_and_store_similarities`` (reference :85-259).

Same arguments and defaults, same record stream (``similar_show_id, similarity_score, genre_score,
text_score, metadata_score``; shows without a qualifying neighbour omitted; flushed to the sink
every 5000 shows with ``clear_existing=False``), same returned statistics keys -- but the N
iterations of five cosine_similarity calls + argsort become one GPU pass."""

from __future__ import annotations

import argparse
import logging
import sys
from pathlib import Path

import numpy as np

from ..ml.similarity_computer import SimilarityComputer
from ..services.content_based_service import load_feature_files, load_show_ids
from ..sinks import InMemorySimilaritySink

logger = logging.getLogger(__name__)

BATCH_SIZE = 5000  # reference :166


def compute_and_store_similarities(input_dir: Path, genre_weight: float = 0.4, text_weight: float = 0.5,
                                   metadata_weight: float = 0.1, top_n_per_show: int | None = 20,
                                   min_similarity: float = 0.1, sink=None, device_ids=None) -> dict:
    """``top_n_per_show=None`` stores every neighbour at or above ``min_similarity`` (no top-n cut): the
    threshold job of ``SimilarityComputer.compute_neighbours``, single GPU."""
    input_dir = Path(input_dir)
    logger.info("COMPUTING AND STORING SIMILARITIES")
    logger.info(f"Genre weight: {genre_weight}  Text weight: {text_weight}  Metadata weight: {metadata_weight}")
    logger.info(f"Top N per show: {top_n_per_show}  Min similarity: {min_similarity}")
    features = load_feature_files(input_dir)
    show_ids = load_show_ids(input_dir)
    logger.info(f"✓ Loaded features for {len(show_ids)} shows")
    computer = SimilarityComputer(genre_weight=genre_weight, text_weight=text_weight,
                                  metadata_weight=metadata_weight)
    # production conventions (reference :184-192): mean of three metadata cosines, raw weights
    if top_n_per_show is None:
        if device_ids is not None and len(device_ids) > 1:
            raise ValueError("every neighbour above the threshold (top_n_per_show=None) runs on one GPU")
        top = computer.compute_neighbours(features, min_similarity=min_similarity, metadata_mode="mean3",
                                          normalize_weights=False)
    else:
        top = computer.compute_top_k(features, k=top_n_per_show, min_similarity=min_similarity,
                                     exclude_self=True, metadata_mode="mean3", normalize_weights=False,
                                     device_ids=device_ids)
    sink = sink if sink is not None else InMemorySimilaritySink()
    total_records_stored = store_similarity_batches(top, show_ids, sink)
    return finish_stats(sink, total_records_stored, top.flagged_rows, top_n_per_show, min_similarity)


def store_similarity_batches(top, show_ids, sink) -> int:
    """The storage half of the reference loop: delete-all up front (reference :156-162), then one
    ``bulk_store_all_similarities(batch, clear_existing=False)`` per 5000 shows (:223-234).  A sink
    with ``bulk_store_records`` gets the columnar batch instead of 5000 x k dicts.  ``top`` is a
    ``TopK`` or a ``NeighbourTable`` (both slice into the same record shape)."""
    ids = np.asarray(list(show_ids))
    n = len(ids)
    columnar = getattr(sink, "bulk_store_records", None)
    if columnar is not None:
        columnar({c: ids[:0] for c in ("show_id", "similar_show_id", "similarity_score", "genre_score",
                                       "text_score", "metadata_score")}, clear_existing=True)
    else:
        sink.bulk_store_all_similarities({}, clear_existing=True)
    total_records_stored = 0
    for b in range(0, n, BATCH_SIZE):
        e = min(b + BATCH_SIZE, n)
        part = top.slice(b, e)
        if columnar is not None:
            total_records_stored += columnar(part.records(ids), clear_existing=False)
        else:
            batch = part.to_dict(ids)
            if batch:
                total_records_stored += sink.bulk_store_all_similarities(batch, clear_existing=False)
        logger.info(f"  Processed {e}/{n} shows... (stored {total_records_stored} similarity records)")
    logger.info(f"✓ Stored {total_records_stored} total similarity records")
    return total_records_stored


def finish_stats(sink, total_records_stored: int, flagged_rows: int, top_n_per_show, min_similarity) -> dict:
    """reference :243-255"""
    stats = dict(sink.get_similarity_stats())
    stats["total_records"] = total_records_stored
    stats["top_n_per_show"] = top_n_per_show
    stats["min_similarity"] = min_similarity
    stats["flagged_rows"] = flagged_rows
    return stats


def load_and_sync_metadata(service, input_dir: Path) -> int:
    """reference :46-82 -- persistence of show metadata is storage (out of scope); the drop-in
    forwards the CSV records to the service's sink when that offers ``bulk_store_shows``."""
    import pandas as pd

    metadata_path = Path(input_dir) / "shows_metadata.csv"
    if not metadata_path.exists():
        raise FileNotFoundError(f"Metadata file not found: {metadata_path}\n" "Run fetch_and_prepare_data.py first.")
    shows_df = pd.read_csv(metadata_path)
    shows_df = shows_df.astype(object).where(pd.notnull(shows_df), None)
    count = service.sync_metadata_to_db(shows_df.to_dict("records"))
    logger.info(f"✓ Synced {count} shows to database")
    return count


def verify_recommendations(service, metadata_path: Path, num_tests: int = 3) -> None:
    """reference :262-295"""
    import pandas as pd

    shows_df = pd.read_csv(metadata_path)
    for show_id in shows_df["id"].head(num_tests).tolist():
        recommendations = service.get_recommendations_from_db(show_id=show_id, n=5)
        logger.info(f"\nRecommendations for show {show_id}:")
        if recommendations:
            for i, rec in enumerate(recommendations, 1):
                logger.info(f"  {i}. {rec.get('name', rec.get('similar_show_id'))} "
                            f"(score: {rec['similarity_score']:.3f})")
        else:
            logger.warning("  No recommendations found")


def main(argv=None, sink=None):
    """reference :298-401: same flags, same order of steps, ``sys.exit(1)`` on any exception."""
    parser = argparse.ArgumentParser(description="Populate database with show metadata and similarities")
    parser.add_argument("--input-dir", type=str, default="data/processed")
    parser.add_argument("--top-n", type=int, default=20)
    parser.add_argument("--min-similarity", type=float, default=0.1)
    parser.add_argument("--all-above-threshold", action="store_true",
                        help="Store every neighbour with score >= --min-similarity (no --top-n cut)")
    parser.add_argument("--skip-metadata", action="store_true", help="Skip metadata sync (only compute similarities)")
    parser.add_argument("--skip-test", action="store_true", help="Skip recommendation testing")
    parser.add_argument("--genre-weight", type=float, default=0.4)
    parser.add_argument("--text-weight", type=float, default=0.5)
    parser.add_argument("--metadata-weight", type=float, default=0.1)
    args = parser.parse_args(argv)
    input_dir = Path(args.input_dir)
    try:
        from ..services.content_based_service import ContentBasedRecommendationService

        sink = sink if sink is not None else InMemorySimilaritySink()
        service = ContentBasedRecommendationService(processed_data_dir=input_dir, use_blob=False, sink=sink)
        metadata_count = 0
        if not args.skip_metadata:
            if hasattr(sink, "bulk_store_shows"):
                metadata_count = load_and_sync_metadata(service, input_dir)
            else:   # metadata persistence is storage: nothing to do without a sink that stores shows
                logger.info("\n⊘ No metadata store configured (sink has no bulk_store_shows): skipping metadata sync")
        else:
            logger.info("\n⊘ Skipping metadata sync")
        stats = compute_and_store_similarities(input_dir, args.genre_weight, args.text_weight, args.metadata_weight,
                                               None if args.all_above_threshold else args.top_n,
                                               args.min_similarity, sink=sink)
        if not args.skip_test:
            verify_recommendations(service, input_dir / "shows_metadata.csv", num_tests=3)
        else:
            logger.info("\n⊘ Skipping recommendation testing")
        if not args.skip_metadata:
            logger.info(f"Shows synced: {metadata_count}")
        logger.info(f"Similarity records: {stats['total_records']}")
        logger.info(f"Unique shows with recommendations: {stats['unique_shows']}")
        logger.info(f"Average similarities per show: {stats['avg_similarities_per_show']:.1f}")
        return stats
    except Exception as e:  # reference :399-401
        logger.error(f"Error during database population: {str(e)}", exc_info=True)
        sys.exit(1)


if __name__ == "__main__":
    logging.basicConfig(level=logging.INFO)
    main()
