"""Drop-in for scripts/compute_similarities.py (reference :29-262): load the feature files,
compute the four similarity matrices and their statistics on the GPU, optionally save them."""

from __future__ import annotations

import argparse
import logging
import sys
from pathlib import Path

import numpy as np

from .._lib import TvbfError
from ..ml.similarity_computer import SimilarityComputer

logger = logging.getLogger(__name__)

REQUIRED_FILES = ["genre_features.npy", "text_features.npz", "platform_features.npy",
                  "type_features.npy", "language_features.npy"]


def load_features(input_dir: Path) -> dict:
    """reference :29-81 (same required files, same error text)."""
    from scipy.sparse import load_npz

    input_dir = Path(input_dir)
    for filename in REQUIRED_FILES:
        filepath = input_dir / filename
        if not filepath.exists():
            raise FileNotFoundError(f"Feature file not found: {filepath}\n" "Run compute_features.py first.")
    features = {}
    for filename in REQUIRED_FILES:
        key = filename.split(".")[0]
        features[key] = load_npz(input_dir / filename) if filename.endswith(".npz") else np.load(input_dir / filename)
        logger.info(f"✓ Loaded {key}: {features[key].shape}")
    return features


STAT_KEYS = ("mean", "std", "min", "max", "median")
SIM_NAMES = ("genre_similarity", "text_similarity", "metadata_similarity", "hybrid_similarity")


def matrices_fit(n_shows: int, max_matrix_bytes: int | None = None) -> bool:
    """Can the four N x N float64 matrices (32 * N^2 bytes, reference :152-157: "~205 GB for 80 k
    shows") be materialised?  They live on the GPU and are copied to the host, so both must hold them."""
    need = 32 * n_shows * n_shows
    if max_matrix_bytes is not None:
        return need <= max_matrix_bytes
    import torch

    budget = 64 << 30
    if torch.cuda.is_available():
        free, _total = torch.cuda.mem_get_info()
        budget = min(budget, int(free * 0.6))
    try:
        import psutil

        budget = min(budget, int(psutil.virtual_memory().available * 0.6))
    except Exception:
        pass
    return need <= budget


def compute_similarities(features: dict, genre_weight: float = 0.4, text_weight: float = 0.5,
                         metadata_weight: float = 0.1, max_matrix_bytes: int | None = None) -> dict:
    """reference :84-133.  Small catalogues: the four N x N matrices, as the reference returns them.
    Catalogues whose matrices do not fit (the reference dies of memory there): the same four
    statistics from ONE streaming tensor-core sweep that never materialises N x N; the returned dict
    then maps each name to ``None`` and carries the statistics under ``"statistics"``."""
    computer = SimilarityComputer(genre_weight=genre_weight, text_weight=text_weight,
                                  metadata_weight=metadata_weight)
    n_shows = int(features["genre_features"].shape[0])
    if matrices_fit(n_shows, max_matrix_bytes):
        similarities = computer.compute_all_similarities(features)
        all_stats = {name: computer.get_similarity_statistics(similarities[name]) for name in SIM_NAMES}
    else:
        logger.info(f"⊘ {n_shows} shows: 4 N x N float64 matrices = {32 * n_shows * n_shows / 1e9:.1f} GB do not fit; "
                    "computing their statistics with the streaming sweep")
        try:
            all_stats = computer.compute_similarity_statistics(features)
        except TvbfError as e:
            if "signed text" not in str(e):
                raise
            raise ValueError(f"the streaming statistics do not take text features with negative values ({e}); "
                             "the N x N matrices do: raise --max-matrix-bytes (32 * N^2 bytes are needed, "
                             f"{32 * n_shows * n_shows} here)") from e
        similarities = {name: None for name in SIM_NAMES}
        similarities["statistics"] = all_stats
    for sim_name in SIM_NAMES:
        stats = all_stats[sim_name]
        logger.info(f"\n{sim_name}:")
        for key in STAT_KEYS:
            logger.info(f"  {key.capitalize()}: {stats[key]:.4f}")
    return similarities


def save_similarities(similarities: dict, output_dir: Path, save_to_disk: bool = False):
    """reference :136-177 -- skipped unless asked (N x N matrices are large)."""
    if not save_to_disk:
        logger.info("⊘ Skipping similarity matrix storage (storage optimization)")
        return
    output_dir = Path(output_dir)
    output_dir.mkdir(parents=True, exist_ok=True)
    for name, matrix in similarities.items():
        if name == "statistics":
            continue
        if matrix is None:
            logger.warning(f"⊘ {name} was not materialised (catalogue too large): nothing to save")
            continue
        np.save(output_dir / f"{name}.npy", matrix)
        logger.info(f"✓ Saved {name}.npy")


def main(argv=None):
    """reference :180-262"""
    parser = argparse.ArgumentParser(description="Compute similarity matrices from feature matrices")
    parser.add_argument("--input-dir", type=str, default="data/processed")
    parser.add_argument("--output-dir", type=str, default="data/processed")
    parser.add_argument("--genre-weight", type=float, default=0.4)
    parser.add_argument("--text-weight", type=float, default=0.5)
    parser.add_argument("--metadata-weight", type=float, default=0.1)
    parser.add_argument("--save-similarities", action="store_true")
    parser.add_argument("--max-matrix-bytes", type=int, default=None,
                        help="materialise the N x N matrices only if 32*N*N <= this (default: what memory allows)")
    args = parser.parse_args(argv)
    total_weight = args.genre_weight + args.text_weight + args.metadata_weight
    if total_weight <= 0:
        logger.error("Error: Sum of weights must be greater than 0")
        sys.exit(1)
    try:
        features = load_features(Path(args.input_dir))
        similarities = compute_similarities(features, args.genre_weight, args.text_weight, args.metadata_weight,
                                            max_matrix_bytes=args.max_matrix_bytes)
        save_similarities(similarities, Path(args.output_dir), save_to_disk=args.save_similarities)
        return similarities
    except Exception as e:  # same contract as the reference: log and exit 1
        logger.error(f"Error during similarity computation: {str(e)}", exc_info=True)
        sys.exit(1)


if __name__ == "__main__":
    logging.basicConfig(level=logging.INFO)
    main()
