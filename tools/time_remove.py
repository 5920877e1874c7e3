"""Remove Q shows from a computed catalogue (``remove`` + ``top_k_remove_device``) against the same
removal on the update path and against the whole job on the remaining catalogue, alternating in one
process:  python tools/time_remove.py [REPS]

Shapes: C3 (100 000 shows x 10 000 terms) with Q = 1 / 100 / 1 000 / 5 000 random rows and P80k
(80 000 x 500, the reference's production vocabulary) with Q = 1 000.  The update path is the
baseline of DESIGN.md §12: compact the catalogue, renumber the previous table and give its rows that
name a removed show (A) count 0, then ``top_k_update_device`` of the rows A.  Both removal times
cover compacting the resident catalogue and the table; the whole job's time covers the job on the
resident remaining catalogue.  Each ends in a device synchronise and is read from the host clock;
median and minimum of REPS rounds.  Prints the card, its power limit, |A|, the tiles of both paths,
the rows K5 sent to K6 (stats[0]), the rescored pairs and whether the tables are identical."""
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
FIELDS = ("indices", "counts", "hybrid", "genre", "text", "metadata")
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


def via_update(eng, cat, sel, prev, n):
    """the removal on the update path: the rows A are 'updated' to the features they have"""
    rem = eng.remove(cat, sel)
    dev = prev["counts"].device
    keep = torch.from_numpy(np.delete(np.arange(n), sel)).to(dev)
    row_map = torch.full((n,), -1, dtype=torch.int64, device=dev)
    row_map[keep] = torch.arange(keep.numel(), device=dev)
    t = {f: prev[f].index_select(0, keep) for f in FIELDS}
    idx = t["indices"]
    t["indices"] = torch.where(idx >= 0, row_map[idx.clamp(min=0).long()].to(idx.dtype), idx)
    in_row = torch.arange(idx.shape[1], device=dev)[None, :] < t["counts"][:, None]
    a = torch.nonzero(((t["indices"] < 0) & in_row).any(dim=1)).flatten()
    t["counts"] = t["counts"].index_fill(0, a, 0)
    a_host = a.cpu().numpy()
    return eng.top_k_update_device(rem, a_host, t, W, K, MS), a_host.size


print(f"# {card()}")
eng = HybridTopKEngine(0)
W, K, MS = (0.4, 0.5, 0.1), 20, 0.1
for cfg, n, q in (("C3", 100_000, 1), ("C3", 100_000, 100), ("C3", 100_000, 1000), ("C3", 100_000, 5000),
                  ("P80k", 80_000, 1000)):
    conf = {**CONFIGS[cfg], "n_shows": n}
    before = make_catalogue(**conf).features()
    sel = np.sort(np.random.default_rng(q).choice(n, size=q, replace=False))
    after_full = eng.ingest(rows(before, np.delete(np.arange(n), sel)), "mean3", W)
    t_rem, t_upd, t_full, same = [], [], [], True
    for r in range(reps + 1):                      # first round: warm-up
        cat = eng.ingest(before, "mean3", W)
        prev = eng.top_k_device(cat, W, K, MS)
        res, tr = wall(lambda: eng.top_k_remove_device(eng.remove(cat, sel), sel, prev, W, K, MS))
        cat2 = eng.ingest(before, "mean3", W)
        (base, n_a_upd), tu = wall(lambda: via_update(eng, cat2, sel, prev, n))
        eng.top_k_device(after_full, W, K, MS)     # untimed: the engine's one second operand (P80k) back to it
        ref, tf = wall(lambda: eng.top_k_device(after_full, W, K, MS))
        if r:
            t_rem.append(tr)
            t_upd.append(tu)
            t_full.append(tf)
        same = same and all(torch.equal(x[f].nan_to_num(), ref[f].nan_to_num()) for x in (res, base) for f in FIELDS)
        stats = res["stats"].cpu().numpy()
        stats_u = base["stats"].cpu().numpy()
        n_a = int(res["changed_rows"].numel())
        incremental = bool(res["incremental"]) and bool(base["incremental"])
        del res, base, ref, prev, cat, cat2
    plan = eng.plan_tiles(after_full, W, K, MS)
    tiles = eng.remove_tiles(after_full, n_a, W, K, MS)
    tiles_u = eng.update_tiles(after_full, n_a_upd, W, K, MS)
    rem, upd, full = (float(np.median(t)) for t in (t_rem, t_upd, t_full))
    print(f"{cfg} N={n} Q={q}: |A| {n_a}; remove {rem:.2f} ms (min {min(t_rem):.2f}), via update {upd:.2f} ms "
          f"(min {min(t_upd):.2f}), whole job {full:.2f} ms (min {min(t_full):.2f}), remove / whole job "
          f"{rem / full:.3f}; tiles (seed pass + sweep): remove {tiles['seed_tiles']} + {tiles['sweep_tiles']}, "
          f"via update {tiles_u['seed_tiles']} + {tiles_u['sweep_tiles']}, whole job {plan['seed_tiles']} + "
          f"{plan['sweep_tiles']}; K6 rows remove {int(stats[0])} / via update {int(stats_u[0])}; rescored pairs "
          f"remove {int(stats[1])} / via update {int(stats_u[1])}; incremental {incremental}; "
          f"tables identical {same}", flush=True)
