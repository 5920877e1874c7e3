"""Streaming similarity statistics (``SimilarityComputer.compute_similarity_statistics``):
    python tools/time_statistics.py [REPS] [--root CHECKOUT]

Times the whole call -- ingest, the statistics sweep, the exact moments and the exact text / hybrid
maxima -- from the host clock around a device synchronise, at N = 3 000 (``make_catalogue(3000,
2048)``) and at C3 (100 000 shows x 10 000 terms), after one warm-up call per shape.  Prints the
median and minimum of REPS calls, the reported maxima and the card with its power limit.
``--root`` imports the package from another checkout (built in place), so that two versions can
be timed one after the other on the same card; run them alternately to see the spread."""
import json
import subprocess
import sys
import time
from pathlib import Path

args = sys.argv[1:]
root = Path(__file__).resolve().parent.parent
if "--root" in args:
    i = args.index("--root")
    root = Path(args[i + 1]).resolve()
    del args[i:i + 2]
reps = int(args[0]) if args else 5
sys.path.insert(0, str(root))
import numpy as np
import torch

from tvbingefriend_recommendation_service_b200 import engine as engine_module
from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine
from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer
from tvbingefriend_recommendation_service_b200.synthetic import make_catalogue, make_config


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


print(f"# {card()}; package from {Path(engine_module.__file__).resolve().parent}", flush=True)
comp = SimilarityComputer(engine=HybridTopKEngine(0))
for name, cat in (("N3000", make_catalogue(3000, 2048, nnz=30, seed=17)), ("C3", make_config("C3"))):
    f = cat.features()
    comp.compute_similarity_statistics(f)
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = comp.compute_similarity_statistics(f)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    print(json.dumps({"shape": name, "n": cat.n_shows, "median_ms": round(float(np.median(ts)), 2),
                      "min_ms": round(min(ts), 2), "text_max": out["text_similarity"]["max"],
                      "hybrid_max": out["hybrid_similarity"]["max"]}), flush=True)
    comp.engine.release()
