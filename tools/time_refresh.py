"""Refresh a computed catalogue -- remove R shows, update U and append Qa at once (the catalogue chain
``update`` + ``remove`` + ``extend``, then ``top_k_refresh_device``) -- against the single-kind call or
the chain of the three single-kind calls, and against the whole job on the refreshed catalogue,
alternating in one process:  python tools/time_refresh.py [REPS]

Shapes: C3 (100 000 shows x 10 000 terms) with (R, U, Qa) = (0, 1, 0), (0, 100, 0), (0, 1 000, 0)
against ``top_k_update_device``, (1 000, 0, 0) against ``top_k_remove_device``, (0, 0, 1 000) against
``top_k_append_device``, and (100, 100, 100), (1 000, 1 000, 1 000), (5 000, 5 000, 5 000) against
update, then remove, then append; P80k (80 000 x 500, the reference's production vocabulary) with
(1 000, 1 000, 1 000).  Removed and updated rows are random; the new features of the updated and
appended shows are rows of a second catalogue of the same config with another seed, so every updated
show changes completely.  Each incremental time covers the catalogue operations and the table(s); the
whole job's time covers the job on the resident refreshed catalogue.  Each ends in a device
synchronise and is read from the host clock; median and minimum of REPS rounds after a warm-up round.
Prints the card and its power limit, the tiles of both stages, |G| (updated, appended and the shows
whose previous row names a removed show), the rows of the second sweep (stats[5]) and of the exact
kernel (stats[0]), the rescored pairs, the changed rows and whether the tables are identical."""
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


def after(before, rem, upd, new, app):
    n = before["genre_features"].shape[0]
    src = np.arange(n)
    src[upd] = n + np.arange(len(upd))
    sel = np.r_[np.delete(src, rem), n + len(upd) + np.arange(app["genre_features"].shape[0])]
    allf = {**before, **{k: (sp.vstack([before[k], new[k], app[k]]).tocsr() if sp.issparse(before[k])
                             else np.concatenate([before[k], new[k], app[k]])) for k in KEYS}}
    return rows(allf, sel)


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


def same(a, b):
    return all(torch.equal(a[f].nan_to_num(), b[f].nan_to_num()) for f in FIELDS)


print(f"# {card()}")
eng = HybridTopKEngine(0)
W, K, MS = (0.4, 0.5, 0.1), 20, 0.1
SHAPES = [("C3", 0, 1, 0, "update"), ("C3", 0, 100, 0, "update"), ("C3", 0, 1000, 0, "update"),
          ("C3", 1000, 0, 0, "remove"), ("C3", 0, 0, 1000, "append"),
          ("C3", 100, 100, 100, "chain"), ("C3", 1000, 1000, 1000, "chain"), ("C3", 5000, 5000, 5000, "chain"),
          ("P80k", 1000, 1000, 1000, None)]
for cfg, nr, nu, na, other_path in SHAPES:
    conf = CONFIGS[cfg]
    n = conf["n_shows"]
    before = make_catalogue(**conf).features()
    second = make_catalogue(**{**conf, "seed": conf.get("seed", 0) + 1}).features()
    rng = np.random.default_rng(nr * 7 + nu * 3 + na)
    pick = rng.permutation(n)
    rem, upd = np.sort(pick[:nr]), np.sort(pick[nr:nr + nu])
    new, app = rows(second, np.arange(nu)), rows(second, nu + np.arange(na))
    full_cat = eng.ingest(after(before, rem, upd, new, app), "mean3", W)

    def chain(cat):
        if nu:
            cat = eng.update(cat, upd, new)
        if nr:
            cat = eng.remove(cat, rem)
        if na:
            cat = eng.extend(cat, app)
        return cat

    def single(cat, prev):
        if other_path == "update":
            return eng.top_k_update_device(eng.update(cat, upd, new), upd, prev, W, K, MS)
        if other_path == "remove":
            return eng.top_k_remove_device(eng.remove(cat, rem), rem, prev, W, K, MS)
        if other_path == "append":
            return eng.top_k_append_device(eng.extend(cat, app), n, prev, W, K, MS)
        cat = eng.update(cat, upd, new)
        t = eng.top_k_update_device(cat, upd, prev, W, K, MS)
        cat = eng.remove(cat, rem)
        t = eng.top_k_remove_device(cat, rem, t, W, K, MS)
        cat = eng.extend(cat, app)
        return eng.top_k_append_device(cat, n - nr, t, W, K, MS)

    t_ref, t_one, t_full, ident = [], [], [], True
    for r in range(reps + 1):                      # first round: warm-up
        cat = eng.ingest(before, "mean3", W)
        prev = eng.top_k_device(cat, W, K, MS)
        res, tr = wall(lambda: eng.top_k_refresh_device(chain(cat), prev, rem, upd, na, W, K, MS))
        stats = res["stats"].cpu().numpy()
        changed, incremental = int(res["changed_rows"].numel()), bool(res["incremental"])
        if other_path is not None:
            cat = eng.ingest(before, "mean3", W)
            prev = eng.top_k_device(cat, W, K, MS)
            one, to = wall(lambda: single(cat, prev))
        eng.top_k_device(full_cat, W, K, MS)       # untimed: the engine's one second operand (P80k) back to it
        ref, tf = wall(lambda: eng.top_k_device(full_cat, W, K, MS))
        ident = ident and same(res, ref) and (other_path is None or same(one, ref))
        if r:
            t_ref.append(tr)
            t_full.append(tf)
            if other_path is not None:
                t_one.append(to)
        if r == 0:
            # |G|: the updated and appended shows, and the other remaining ones whose previous row names a
            # removed show
            p_idx, p_cnt = prev["indices"].cpu().numpy(), prev["counts"].cpu().numpy()
            gone = np.zeros(n, dtype=bool)
            gone[rem] = True
            named = (gone[np.maximum(p_idx, 0)] & (np.arange(K)[None, :] < p_cnt[:, None])).any(axis=1)
            named[upd] = True
            n_g = int(named[~gone].sum()) + na
        del res, ref, prev, cat
    tiles = eng.refresh_tiles(full_cat, n_g, int(stats[5]), W, K, MS)
    plan = eng.plan_tiles(full_cat, W, K, MS)
    ref_ms, full_ms = float(np.median(t_ref)), float(np.median(t_full))
    line = (f"{cfg} (R, U, Qa) = ({nr}, {nu}, {na}): refresh {ref_ms:.2f} ms (min {min(t_ref):.2f})")
    if other_path is not None:
        line += f", {other_path} {float(np.median(t_one)):.2f} ms (min {min(t_one):.2f})"
    line += (f", whole job {full_ms:.2f} ms (min {min(t_full):.2f}), refresh / whole job {ref_ms / full_ms:.3f}; "
             f"tiles (seed pass + sweep): stage 1 {tiles['seed_tiles']} + {tiles['sweep_tiles']}, stage 2 "
             f"{tiles['repair_seed_tiles']} + {tiles['repair_sweep_tiles']}, whole job {plan['seed_tiles']} + "
             f"{plan['sweep_tiles']}; |G| {n_g}; stage-2 rows {int(stats[5])}; K6 rows {int(stats[0])}; "
             f"rescored pairs {int(stats[1])}; changed rows {changed}; incremental {incremental}; "
             f"tables identical {ident}")
    print(line, flush=True)
    del full_cat
