"""Update the features of Q shows of a computed catalogue (``update`` + ``top_k_update_device``) against
the whole job on the updated catalogue, alternating in one process:  python tools/time_update.py [REPS]

Shapes: C3 (100 000 shows x 10 000 terms) with Q = 1 / 100 / 1 000 / 5 000 random rows and P80k
(80 000 x 500, the reference's production vocabulary) with Q = 1 000.  The new features are the same
rows of a second catalogue of the same config with another seed: every updated show changes
completely, the worst case for neighbours lost below the previous k-th entry.  The update's time
covers writing the new rows into the resident catalogue (ingest and prep of the Q rows, CSR splice)
and the incremental table; the whole job's time covers the job on the resident updated catalogue.
Both end in a device synchronise and are read from the host clock; median and minimum of REPS rounds.
Prints the card, its power limit, the tiles each computes, the rows K5 sent to K6 (stats[0]), the
rescored pairs, the changed rows and whether the tables are identical."""
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
from tvbingefriend_recommendation_service_b200.synthetic import CONFIGS, make_catalogue

KEYS = ("genre_features", "text_features", "platform_features", "type_features", "language_features")
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def rows(feats, sel):
    return {**feats, **{k: (feats[k][sel].tocsr() if sp.issparse(feats[k]) else feats[k][sel]) for k in KEYS}}


def replace(feats, sel, new):
    n = feats["genre_features"].shape[0]
    perm = np.arange(n)
    perm[sel] = n + np.arange(len(sel))
    return {**feats, **{k: (sp.vstack([feats[k], new[k]]).tocsr()[perm] if sp.issparse(feats[k])
                            else np.concatenate([feats[k], new[k]])[perm]) for k in KEYS}}


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
for cfg, n, q in (("C3", 100_000, 1), ("C3", 100_000, 100), ("C3", 100_000, 1000), ("C3", 100_000, 5000),
                  ("P80k", 80_000, 1000)):
    conf = {**CONFIGS[cfg], "n_shows": n}
    before = make_catalogue(**conf).features()
    other = make_catalogue(**{**conf, "seed": conf.get("seed", 0) + 1}).features()
    sel = np.sort(np.random.default_rng(q).choice(n, size=q, replace=False))
    new = rows(other, sel)
    after_full = eng.ingest(replace(before, sel, new), "mean3", W)
    t_upd, t_full, same = [], [], True
    for r in range(reps + 1):                      # first round: warm-up
        cat = eng.ingest(before, "mean3", W)
        prev = eng.top_k_device(cat, W, K, MS)
        torch.cuda.synchronize()
        res, tu = wall(lambda: eng.top_k_update_device(eng.update(cat, sel, new), sel, prev, W, K, MS))
        eng.top_k_device(after_full, W, K, MS)     # untimed: the engine's one second operand (P80k) back to it
        ref, tf = wall(lambda: eng.top_k_device(after_full, W, K, MS))
        if r:
            t_upd.append(tu)
            t_full.append(tf)
        same = same and all(torch.equal(res[f].nan_to_num(), ref[f].nan_to_num())
                            for f in ("indices", "counts", "hybrid", "genre", "text", "metadata"))
        stats = res["stats"].cpu().numpy()
        changed = int(res["changed_rows"].numel())
        incremental = bool(res["incremental"])
        del res, ref, prev, cat
    plan = eng.plan_tiles(after_full, W, K, MS)
    tiles = eng.update_tiles(after_full, q, W, K, MS)
    upd, full = float(np.median(t_upd)), float(np.median(t_full))
    print(f"{cfg} N={n} Q={q}: update {upd:.2f} ms (min {min(t_upd):.2f}), whole job {full:.2f} ms "
          f"(min {min(t_full):.2f}), ratio {upd / full:.3f}; tiles (seed pass + sweep): update "
          f"{tiles['seed_tiles']} + {tiles['sweep_tiles']}, whole job {plan['seed_tiles']} + {plan['sweep_tiles']}; "
          f"K6 rows {int(stats[0])}; rescored pairs {int(stats[1])}; changed rows {changed}; "
          f"incremental {incremental}; tables identical {same}", flush=True)
