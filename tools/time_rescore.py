"""Kernel breakdown of the stage after the candidate pass (K4s + K5 + K6) on the bench's flagship job:
    python tools/time_rescore.py [CONFIG] [STEPS]

Builds CONFIG (default C3) with bench.py's inputs (weights 0.4 / 0.5 / 0.1, min_similarity 0.1,
exclude self, mean3 metadata) and times it twice in one process: with the engine's merge ratio
(TVBF_MERGE_RATIO, default 0.4) and with merging off.  For each it prints
  - the stage's time per step from CUDA events around the K4s + K5 + K6 launches, profiler off;
  - the mean device time per step of every kernel in a torch.profiler run (CUDA activities) of
    its own, K1 included, so that the sum can be set against the step;
  - flagged rows with and without text (stats[2], stats[3]) and the candidate list entries that
    K4s compacts (stats[4], in units of 16: TVBF_DEBUG_COUNTS is set here).
The card's name and power limit are printed first."""
import os
import subprocess
import sys
from pathlib import Path

os.environ.setdefault("TVBF_DEBUG_COUNTS", "1")
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine, stage  # noqa: E402
from tvbingefriend_recommendation_service_b200.synthetic import CONFIGS, make_config  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "C3"
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
W, MS = (0.4, 0.5, 0.1), 0.1


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


print(f"# {card()}", flush=True)
cat = make_config(name)
k = CONFIGS[name]["k"]
eng = HybridTopKEngine(0)
raw = eng.h2d(stage(cat.features(), "mean3", pin=True))
ratios = (eng.merge_ratio, 0.0)
for ratio in ratios:
    eng.merge_ratio = ratio
    state = {"prev": None, "tables": None}

    def step(ev=None):
        dc = eng.prepare(raw, W, recycle=state["prev"])
        state["prev"] = dc
        t = eng.top_k_device(dc, W, k, MS, True, phases=1, out=state["tables"])
        state["tables"] = t
        if ev is not None:
            ev[0].record()
        eng.top_k_device(dc, W, k, MS, True, phases=6, out=t)
        if ev is not None:
            ev[1].record()
        return t

    for _ in range(3):
        t = step()
    torch.cuda.synchronize()
    st = t["stats"].cpu().numpy()
    stage_ms = []
    for _ in range(steps):
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        step(ev)
        torch.cuda.synchronize()
        stage_ms.append(ev[0].elapsed_time(ev[1]))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            key = e.name.split("(")[0].replace("void ", "")[:100]
            per[key] = per.get(key, 0.0) + (e.time_range.end - e.time_range.start) / 1e3 / steps
    print(f"\n{name}, merge ratio {ratio}: K4s + K5 + K6 {np.mean(stage_ms):.3f} ms per step "
          f"(min {np.min(stage_ms):.3f}, max {np.max(stage_ms):.3f}, CUDA events, profiler off); "
          f"flagged rows {int(st[0])}: text {int(st[2])}, no text {int(st[3])}; rescored pairs {int(st[1])}; "
          f"list entries ~{int(st[4]) * 16} (stats[4] x 16, one step)", flush=True)
    print(f"{'ms/step':>9s}  kernel (torch.profiler, {steps} steps)")
    for key, ms in sorted(per.items(), key=lambda kv: -kv[1]):
        print(f"{ms:9.3f}  {key}")
    print(f"{sum(per.values()):9.3f}  total device time", flush=True)
    del t, state
