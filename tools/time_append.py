"""Append Q shows to a computed catalogue (``extend`` + ``top_k_append_device``) against the whole job
on the grown catalogue, alternating in one process:  python tools/time_append.py [REPS]

Shapes: C3 (100 000 shows x 10 000 terms) + Q = 256 / 1 000 / 5 000 and P80k (80 000 x 500, the
reference's production vocabulary) + Q = 1 000.  The append's time covers growing the device
catalogue (ingest and prep of the new rows) and the update; the old catalogue and its table are
resident, as they are for a service that keeps them.  The whole job's time covers the job on the
resident grown catalogue.  Both end in a device synchronise and are read from the host clock.
Prints the card, its power limit, the tiles each computes and whether the tables are identical."""
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import scipy.sparse as sp
import torch

from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine
from tvbingefriend_recommendation_service_b200.synthetic import make_config

KEYS = ("genre_features", "text_features", "platform_features", "type_features", "language_features")
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def rows(feats, sel):
    return {**feats, **{k: (feats[k][sel].tocsr() if sp.issparse(feats[k]) else feats[k][sel]) for k in KEYS}}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


print(f"# {card()}")
eng = HybridTopKEngine(0)
W, K, MS = (0.4, 0.5, 0.1), 20, 0.1
for cfg, n_old, q in (("C3", 100_000, 256), ("C3", 100_000, 1000), ("C3", 100_000, 5000), ("P80k", 80_000, 1000)):
    feats = make_config(cfg, n_old + q).features()
    old, new = rows(feats, slice(0, n_old)), rows(feats, slice(n_old, None))
    grown_full = eng.ingest(feats, "mean3", W)
    t_app, t_full, same = [], [], True
    for r in range(reps + 1):                      # first round: warm-up
        cat = eng.ingest(old, "mean3", W)
        prev = eng.top_k_device(cat, W, K, MS)
        torch.cuda.synchronize()
        res, ta = wall(lambda: eng.top_k_append_device(eng.extend(cat, new), n_old, prev, W, K, MS))
        eng.top_k_device(grown_full, W, K, MS)     # untimed: the engine's one second operand (P80k) back to it
        ref, tf = wall(lambda: eng.top_k_device(grown_full, W, K, MS))
        if r:
            t_app.append(ta)
            t_full.append(tf)
        same = same and all(torch.equal(res[n].nan_to_num(), ref[n].nan_to_num())
                            for n in ("indices", "counts", "hybrid", "genre", "text", "metadata"))
        changed = int(res["changed_rows"].numel())
        incremental = bool(res["incremental"])
        grown = eng.extend(eng.ingest(old, "mean3", W), new)     # untimed: for the tile plan below
        del res, ref, prev, cat
    plan = eng.plan_tiles(grown_full, W, K, MS)
    tiles = eng.append_tiles(grown, n_old, W, K, MS)
    del grown
    app, full = float(np.median(t_app)), float(np.median(t_full))
    print(f"{cfg} N={n_old} Q={q}: append {app:.2f} ms (min {min(t_app):.2f}), whole job {full:.2f} ms "
          f"(min {min(t_full):.2f}), ratio {app / full:.3f}; tiles (seed pass + sweep): append "
          f"{tiles['seed_tiles']} + {tiles['sweep_tiles']}, whole job {plan['seed_tiles']} + {plan['sweep_tiles']}; "
          f"incremental {incremental}; changed old rows {changed}; tables identical {same}")
