"""Every neighbour at or above a threshold (``neighbours_device``) against the top-20 job on the same
catalogue:  python tools/time_neighbours.py [REPS]

Shapes: C3 (100 000 shows x 10 000 terms) and P80k (80 000 x 500, the reference's production
vocabulary), thresholds 0.9 / 0.7 / 0.5.  Per threshold: the candidate pairs the tensor-core sweep
emits and the exact pairs (i < j) the float64 finish keeps; the sweep (``tvbf_neighbours_sweep``) and
the finish (``tvbf_neighbours_finish``) each from CUDA events around that call alone, with a capacity
that holds every candidate; the whole ``neighbours_device`` call (both, the count read-back and the
output allocation) from the host clock around a device synchronise.  For comparison the top-20 job
(``top_k_device``): its candidate pass alone (phases=1: seed pass + symmetric sweep) and the whole
job, from CUDA events.  Median and minimum of REPS rounds after one warm-up round.  Prints the card
and its power limit first."""
import ctypes as C
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np
import torch

from tvbingefriend_recommendation_service_b200._lib import check
from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine
from tvbingefriend_recommendation_service_b200.synthetic import make_config

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
W = (0.4, 0.5, 0.1)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def events(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    b.synchronize()
    return out, a.elapsed_time(b)


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def med(ts):
    return f"{float(np.median(ts)):.2f} ms (min {min(ts):.2f})"


print(f"# {card()}", flush=True)
eng = HybridTopKEngine(0)
lib, dev = eng.lib, eng.device
for cfg in ("C3", "P80k"):
    cat = eng.ingest(make_config(cfg).features(), "mean3", W)
    n = cat.n_shows
    t_topk, t_k1 = [], []
    for r in range(reps + 1):
        _, tk = events(lambda: eng.top_k_device(cat, W, 20, 0.1))
        _, t1 = events(lambda: eng.top_k_device(cat, W, 20, 0.1, phases=1))
        if r:
            t_topk.append(tk)
            t_k1.append(t1)
    print(f"{cfg} N={n}: top_k_device k=20 whole job {med(t_topk)}, its candidate pass (seed + sweep) "
          f"{med(t_k1)}", flush=True)
    for tau in (0.9, 0.7, 0.5):
        res = eng.neighbours_device(cat, W, tau)
        n_cand, n_exact = int(res["candidate_pairs"]), int(res["row_ptr"][-1].item()) // 2
        del res
        feats = eng._folded(cat, *W, 1) or cat.c
        p = eng._params(cat, W, 1, tau)
        cap = max(n_cand, 1)
        nbytes = lib.tvbf_neighbours_workspace_bytes(C.byref(feats), C.byref(p), cap)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        pairs = torch.empty((cap, 2), dtype=torch.int32, device=dev)
        count = torch.zeros((1,), dtype=torch.int64, device=dev)
        m = 2 * n_cand + n
        out = [torch.empty((n + 1,), dtype=torch.int64, device=dev), torch.empty((m,), dtype=torch.int32, device=dev)]
        out += [torch.empty((m,), dtype=torch.float64, device=dev) for _ in range(4)]
        st = torch.cuda.current_stream(dev).cuda_stream
        t_sw, t_fi, t_all = [], [], []
        for r in range(reps + 1):
            _, ts = events(lambda: check(lib.tvbf_neighbours_sweep(C.byref(feats), C.byref(p), pairs.data_ptr(), cap,
                                                                   count.data_ptr(), ws.data_ptr(), nbytes, st),
                                         "tvbf_neighbours_sweep"))
            assert int(count.item()) == n_cand
            _, tf = events(lambda: check(lib.tvbf_neighbours_finish(C.byref(feats), C.byref(p), pairs.data_ptr(),
                                                                    n_cand, 0, *(o.data_ptr() for o in out),
                                                                    ws.data_ptr(), nbytes, st),
                                         "tvbf_neighbours_finish"))
            _, tw = wall(lambda: eng.neighbours_device(cat, W, tau))
            if r:
                t_sw.append(ts)
                t_fi.append(tf)
                t_all.append(tw)
        del ws, pairs, out
        print(f"{cfg} N={n} tau={tau}: candidate pairs {n_cand}, exact pairs {n_exact} "
              f"({n_cand / max(n_exact, 1):.2f}x); sweep {med(t_sw)}, finish {med(t_fi)}, "
              f"neighbours_device {med(t_all)}", flush=True)
    del cat
    eng.release()
