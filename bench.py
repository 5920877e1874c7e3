#!/usr/bin/env python
"""Benchmark of the hybrid all-pairs similarity -> top-K path (BASELINE.json metric:
shows/sec to top-20, TFLOP/s vs peak, at 1/2/4/8 B200, beside the host-CPU reference).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C3] [--impl b200|reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole synthetic catalogue: K0 prep kernels ->
K1 tcgen05 candidate pass -> K5 fp64 rescore/certify -> K6 exact repair (with N GPUs > 1: candidate
lists exchanged by all-to-all before K5, [N, k] tables all-gathered after K6).  ``value`` is timed with the raw features already resident in HBM;
``e2e`` adds, inside the timed region, the H2D copy of the staged (pinned) feature buffers and the
D2H read of the result table through the public engine API.  Prints ONE JSON line on rank 0.

``--dump-outputs DIR`` writes the table the last timed step of ``value`` computed (indices, counts
and the four score columns, as float64 ``DIR/<name>.npy``, plus ``rows``: the source rows they
cover), so that two builds can be compared output for output.  The inputs are seeded: the same
arguments give the same inputs on every run.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "shows_per_sec_to_top_k"
UNIT = "shows/s"
DUMP_LIMIT_BYTES = 64_000_000


def output_sample(table, limit: int = DUMP_LIMIT_BYTES, seed: int = 0) -> dict:
    """A host result table as float64 arrays of at most ``limit`` bytes in all: every row when it
    fits, else a fixed seeded sample of source rows (ascending).  ``rows`` names the rows kept."""
    n, k = table.indices.shape
    row_bytes = 8 * (5 * k + 2)                        # five [k] columns, the count and the row number
    cap = (limit - 4096) // row_bytes                  # 4 KB for the seven .npy headers
    rows = np.arange(n) if n <= cap else np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))
    out = {"rows": rows + table.row_begin}
    out.update({f: getattr(table, f)[rows] for f in ("indices", "counts", "hybrid", "genre", "text", "metadata")})
    return {name: np.asarray(a, dtype=np.float64) for name, a in out.items()}


def _peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"bf16_tflops": float(d["bf16_tflops"]), "bf16_tflops_sustained": float(d["bf16_tflops_sustained"]),
                "hbm_gbs": float(d["hbm_gbs"]), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region: NVML every 10 ms from a thread
    (the timed region of a default run lasts ~0.3 s), ``nvidia-smi -lms 100`` if NVML is unavailable."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None
        self.nvml, self.handle, self.thread, self.stop_flag = None, None, None, threading.Event()
        self.sm, self.mx, self.reasons, self.source = [], [], set(), "nvidia-smi"

    def _nvml_handle(self):
        import pynvml
        import torch

        pynvml.nvmlInit()
        try:      # the CUDA ordinal need not be the NVML index (CUDA_VISIBLE_DEVICES): go by UUID
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)     # probe
        return pynvml, handle

    def _poll(self):
        nv, h = self.nvml, self.handle
        flags = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                for name, bit in flags.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.source = "nvml"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None,
                    "sm_max_mhz": max(self.mx) if self.mx else None, "samples": len(self.sm),
                    "reasons": sorted(self.reasons), "source": "nvml, 10 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


def cpu_baseline(cat, cfg, weights, budget_s: float = 20.0, use_sklearn: bool = True, min_rows: int = 256) -> dict:
    """The reference's production loop (scripts/populate_database.py:170-218) on a bounded,
    evenly spaced row sample of the same catalogue, on this box's host cores."""
    from oracle.reference_paths import production_loop

    cos = None
    label = "oracle numpy restatement of cosine_similarity"
    if use_sklearn:
        try:
            from sklearn.metrics.pairwise import cosine_similarity as cos  # the reference's own dependency
            label = "sklearn.metrics.pairwise.cosine_similarity (the reference's dependency)"
        except Exception:
            cos = None
    kw = {} if cos is None else {"cosine": cos}
    n = cat.n_shows
    ids = cat.show_ids.tolist()
    feats = cat.features()
    # all the host threads the BLAS under numpy can use (torchrun exports OMP_NUM_THREADS=1)
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        limiter = threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        threadpool_info, limiter = None, None
    t0 = time.perf_counter()
    production_loop(feats, ids, *weights, top_n_per_show=cfg["k"], min_similarity=0.1, rows=[0, n // 2], **kw)
    per_row = (time.perf_counter() - t0) / 2
    # SURVEY.md section 8d: at least 256 sampled rows (capped at 40 s of CPU work)
    rows = int(max(4, min(n, max(budget_s, min(40.0, min_rows * per_row)) / max(per_row, 1e-6))))
    sample = np.linspace(0, n - 1, rows).astype(np.int64).tolist()
    t0 = time.perf_counter()
    production_loop(feats, ids, *weights, top_n_per_show=cfg["k"], min_similarity=0.1, rows=sample, **kw)
    dt = time.perf_counter() - t0
    threads = os.cpu_count() or 1
    if threadpool_info is not None:
        threads = max([i.get("num_threads", 1) for i in threadpool_info()] or [1])
    if limiter is not None:
        limiter.restore_original_limits()
    # variant A (SimilarityComputer.compute_all_similarities, ml/similarity_computer.py:132-169) where the four
    # N x N float64 matrices fit comfortably: BASELINE.json configs[0] (C1) with the same sklearn cosine
    variant_a = None
    try:
        from oracle.reference_paths import SimilarityComputerOracle
        from tvbingefriend_recommendation_service_b200.synthetic import make_config

        c1 = make_config("C1")
        comp = SimilarityComputerOracle(*weights, **kw)
        t0 = time.perf_counter()
        sims = comp.compute_all_similarities(c1.features())
        variant_a = {"config": "C1 (1000 shows x 5000 vocab)", "seconds": time.perf_counter() - t0,
                     "what": "compute_all_similarities: 3 cosine_similarity calls + weighted sum, four N x N float64"}
        del sims
    except Exception as exc:
        variant_a = {"error": str(exc)}
    return {"value": rows / dt, "unit": UNIT, "cores": int(threads), "kind": "port", "variant_a": variant_a,
            "sample": f"{rows} evenly spaced source rows of {n} through the verbatim production loop "
                      f"(5 cosine_similarity calls + argsort per row; {label}); "
                      f"host has {os.cpu_count()} logical cpus; scipy CSR product and argsort are single-threaded",
            "seconds": dt}


def run_reference(args, cfg, cat, weights) -> dict:
    """--impl reference: the reference's CPU implementation of the path (oracle port: the
    reference is pure Python over sklearn, nothing to compile), bounded sample per step."""
    steps, warm = args.steps, args.warmup
    per_step_budget = max(2.0, min(20.0, 120.0 / max(1, steps + warm)))
    res = None
    vals = []
    for i in range(warm + steps):
        res = cpu_baseline(cat, cfg, weights, budget_s=per_step_budget, min_rows=0)
        if i >= warm:
            vals.append(res["value"])
    v = float(np.mean(vals))
    res["value"] = v
    return {"metric": METRIC, "value": v, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * cat.n_shows / v, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(args, cfg), "cpu_baseline": res,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def parity_check(eng, cat, cfg, weights, table, single=None, rows: int = 96) -> dict:
    """Correctness of the table this run produced, carried in the JSON line: an evenly spaced sample
    of source rows against the CPU oracle (float64 restatement of the production loop; the oracle is
    the checker here, nothing it computes is timed or reported as the product's), and -- when the
    job ran on several GPUs -- exact equality with the single-GPU table computed by rank 0."""
    from oracle.compare import compare_topk
    from oracle.reference_paths import ProductionRows

    n, k = cat.n_shows, cfg["k"]
    pr = ProductionRows(cat.features(), *weights)
    sample = np.unique(np.linspace(0, n - 1, rows).astype(np.int64))
    ridx, rcnt, rsc = pr.topk_arrays(sample, k, 0.1)
    rep = compare_topk(ridx, rcnt, rsc[0], table.indices[sample], table.counts[sample], table.hybrid[sample],
                       lambda r, js: pr.pair_scores(int(sample[r]), js), k, 0.1)
    out = {"rows": int(len(sample)), "identical": int(rep.rows_identical_ordered),
           "tie_permuted": int(rep.rows_tie_permuted), "failures": int(len(rep.failures)), "ok": bool(rep.ok),
           "max_rel_score_err": float(rep.max_rel_score_err),
           "checker": "oracle.reference_paths.ProductionRows + tie-aware comparator (eps 1e-9)"}
    if single is not None:
        m = single.indices >= 0
        same = (np.array_equal(single.indices, table.indices) and np.array_equal(single.counts, table.counts)
                and np.array_equal(single.hybrid[m], table.hybrid[m]))
        out["identical_to_single_gpu"] = bool(same)
        out["ok"] = bool(out["ok"] and same)
    return out


def dense_text_probe(eng, dc, weights, k, tuning, steps: int = 3) -> dict:
    """K1 on a dense-random operand of the same shape (SURVEY.md section 8d's pure-GEMM variant): the
    synthetic TF-IDF operand is 99.5 % zeros, which keeps the tensor pipe's switching power -- and so
    the power-capped clock -- far from what a dense GEMM sees.  Only the candidate kernel runs (the
    random operand has no CSR behind it, so nothing is rescored or reported from it)."""
    import torch

    operand = dc.keep[3]
    saved = operand.clone()
    g = torch.Generator(device=operand.device)
    g.manual_seed(1234)
    operand.copy_(torch.rand(operand.shape, device=operand.device, dtype=torch.float32, generator=g).to(operand.dtype))
    sampler = ClockSampler(operand.device.index or 0)
    times = []
    try:
        eng.top_k_device(dc, weights, k, 0.1, True, phases=1, tuning=tuning)     # warm-up
        torch.cuda.synchronize()
        sampler.start()
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.top_k_device(dc, weights, k, 0.1, True, phases=1, tuning=tuning)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
    finally:
        clocks = sampler.stop()
        operand.copy_(saved)
    return {"k1_ms": float(np.mean(times)), "clocks": clocks,
            "operand": "U(0,1) fp16 in every entry (dense), same [N_pad, K_pad] shape"}


def nxn_variant(eng, weights, names=("C1", "C2")) -> dict:
    """The reference's full-matrix variant (SimilarityComputer.compute_all_similarities,
    ml/similarity_computer.py:132-169: four N x N float64 matrices) on the GPU, beside the survey's
    CPU figures for the same shapes (SURVEY.md section 6: 0.08 s at N = 1 000, 30.6 s at N = 20 000)."""
    import torch

    from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer
    from tvbingefriend_recommendation_service_b200.synthetic import make_config

    comp = SimilarityComputer(*weights, engine=eng)
    out = {}
    for name in names:
        cat = make_config(name)
        f = cat.features()
        n = cat.n_shows
        free, _ = torch.cuda.mem_get_info()
        if 32 * n * n > 0.5 * free:
            out[name] = {"skipped": "4 N x N float64 matrices do not fit"}
            continue
        res = {}
        for it in range(2):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            g = eng.cosine_matrix(f["genre_features"])
            t = eng.cosine_matrix(f["text_features"])
            m = eng.cosine_matrix(np.hstack([f["platform_features"], f["type_features"], f["language_features"]]))
            gw, tw, mw = comp._normalized_weights()
            h = eng.hybrid_combine(g, t, m, gw, tw, mw)
            e1.record()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            res = {"n_shows": n, "device_ms": e0.elapsed_time(e1), "wall_ms_incl_upload": 1e3 * (t1 - t0),
                   "matrices_gb": 32 * n * n / 1e9}
            del g, t, m, h
        out[name] = res
        eng.release()
    out["survey_cpu_seconds"] = {"C1": 0.08, "C2": 30.6}
    return out


def weight_sweep(eng, config: str = "C3", reps: int = 3) -> dict:
    """The reference notebook's five weight schemes (notebooks/03_content_similarity cell 6; BASELINE
    config C5's sweep) on ``config`` through ONE shared symmetric tensor-core sweep (kMode 5): the text
    GEMM is executed once, the epilogue scores every triple."""
    import torch

    from tvbingefriend_recommendation_service_b200.engine import stage
    from tvbingefriend_recommendation_service_b200.synthetic import CONFIGS, WEIGHT_SWEEP, make_config

    cat = make_config(config)
    k = CONFIGS[config]["k"]
    dc = eng.upload(stage(cat.features()))
    ts, out = [], None
    for _ in range(1 + reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = eng.top_k_sweep_device(dc, WEIGHT_SWEEP, k, 0.1, shared=True, out=out)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    res = {"config": config, "triples": [list(w) for w in WEIGHT_SWEEP], "k": k, "ms_all_triples": float(np.mean(ts[1:])),
           "ms_all_triples_per_rep": [round(t, 2) for t in ts[1:]],
           "ms_per_triple": float(np.mean(ts[1:])) / len(WEIGHT_SWEEP),
           "flagged_rows": [int(t["stats"][0]) for t in out]}
    del dc, out, cat
    eng.release()
    return res


def run_extra(name: str, eng, args, world: int, rank: int, weights, peaks: dict, steps: int = 3,
              tuning: int = 0, config: str | None = None) -> dict:
    """One more BASELINE.json shape in the same run (same kernels, same drivers, device-resident
    inputs, ``steps`` timed steps after one warm-up): ms per catalogue, K1 ms and executed TFLOP/s."""
    import torch
    import torch.distributed as dist

    from tvbingefriend_recommendation_service_b200.engine import stage
    from tvbingefriend_recommendation_service_b200.multi_gpu import top_k_device_distributed
    from tvbingefriend_recommendation_service_b200.sharding import row_shard
    from tvbingefriend_recommendation_service_b200.synthetic import CONFIGS, make_config

    cfg = CONFIGS[config or name]
    cat = make_config(config or name)
    n, k = cat.n_shows, cfg["k"]
    st = stage(cat.features(), "mean3", pin=True)
    raw = eng.h2d(st)
    prev = [None]

    def step(events=None):
        def mark(key):
            if events is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                events.setdefault(key, []).append(ev)

        dc = eng.prepare(raw, weights, recycle=prev[0])
        prev[0] = dc
        if world > 1:
            return top_k_device_distributed(eng, dc, weights, k, 0.1, True, events=events, tuning=tuning,
                                            symmetric=False if (tuning >> 20) & 3 == 1 else None)
        mark("seed0")
        t = eng.top_k_device(dc, weights, k, 0.1, True, phases=1, tuning=tuning)
        mark("sweep1")
        eng.top_k_device(dc, weights, k, 0.1, True, phases=6, out=t, tuning=tuning)
        return t

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(2):       # warm-up (allocations, clocks)
        out = step()
    sync()
    events: dict = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step(events)
    e1.record()
    sync()
    if world > 1:
        k1 = float(np.mean([a.elapsed_time(b) + c.elapsed_time(d) for a, b, c, d in
                            zip(events["seed0"], events["seed1"], events["reduce1"], events["sweep1"])]))
    else:
        k1 = float(np.mean([a.elapsed_time(b) for a, b in zip(events["seed0"], events["sweep1"])]))
    t_ms = torch.tensor([e0.elapsed_time(e1) / steps, k1], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    dc = prev[0]
    if world > 1:
        sharded = n >= 40_000 and eng.sym_eligible(dc, weights, k, 0.1) and (tuning >> 20) & 3 != 1
        rb, re_ = row_shard(n, world, 0)
        plan = eng.plan_tiles(dc, weights, k, 0.1, rank=0, world=world, tile_sharded=True) if sharded else \
            eng.plan_tiles(dc, weights, k, 0.1, row_begin=rb, row_end=re_, tuning=1 << 20)
    else:
        plan = eng.plan_tiles(dc, weights, k, 0.1, tuning=tuning)
    stats = out["stats"].cpu().numpy().reshape(-1, 8).sum(axis=0)
    ms, k1 = t_ms[0].item(), t_ms[1].item()
    tf = plan["flops"] / (k1 * 1e-3) / 1e12 if k1 > 0 else 0.0
    res = {"workload": f"{n} shows x vocab {cfg['vocab']} (~{cfg['nnz']} nnz/row), top-{k}, metadata {cfg['meta']}",
           "ms_per_step": ms, "shows_per_s": n / (ms * 1e-3), "k1_ms": k1, "executed_tflops": tf,
           "frac": tf / peaks["bf16_tflops_sustained"], "symmetric_sweep": plan["symmetric"],
           "tiles": plan["seed_tiles"] + plan["sweep_tiles"], "tile": f"{plan['tile_rows']}x256x{plan['k_pad']}",
           "genre_metadata_in_operand": plan["folded_bits"], "flagged_rows": int(stats[0]), "steps": steps}
    del raw, st, cat, out, dc
    prev[0] = None
    eng.release()
    return res


def bench_config(args, cfg) -> dict:
    return {"workload": f"{args.config}: {cfg['n_shows']} synthetic shows, TF-IDF vocab {cfg['vocab']} "
                        f"(~{cfg['nnz']} nnz/row), {cfg['n_genres']} genres, metadata one-hot {cfg['meta']}, "
                        f"hybrid weights 0.4/0.5/0.1, top-{cfg['k']}, min_similarity 0.1",
            "n_shows": cfg["n_shows"], "vocab": cfg["vocab"], "k": cfg["k"],
            "parallelism": f"features replicated; x{args.gpus}: tile-sharded symmetric sweep, finished candidate "
                           f"rows stored into the owner GPU's buffer over NVLink (one all-to-all without "
                           f"symmetric memory), one coalesced all-gather of the tables (or row-sharded "
                           f"one-sided with --one-sided)",
            "l2_policy": "inputs larger than L2 (fp16 operand %.1f GB, streamed every step)"
                         % (cfg["n_shows"] * cfg["vocab"] * 2 / 1e9)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C3")
    ap.add_argument("--n-shows", type=int, default=None, help="override N (debug)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-dense-probe", action="store_true")
    ap.add_argument("--extra", default="P80k,C4,C5,one_sided,weight_sweep,nxn", help="comma-separated extra configs timed in the same run ('' = none)")
    ap.add_argument("--splits", type=int, default=0)
    ap.add_argument("--one-sided", action="store_true", help="disable the symmetric sweep at N > 1")
    ap.add_argument("--tuning", type=lambda x: int(x, 0), default=0, help="tvbf_params.tuning bitfield")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the table of the last timed step as DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the tables of --impl b200")

    from tvbingefriend_recommendation_service_b200.synthetic import CONFIGS, make_config

    cfg = dict(CONFIGS[args.config])
    if args.n_shows:
        cfg["n_shows"] = args.n_shows
    weights = (0.4, 0.5, 0.1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        cat = make_config(args.config, cfg["n_shows"])
        print(json.dumps(run_reference(args, cfg, cat, weights)), flush=True)
        return

    import torch
    import torch.distributed as dist

    from tvbingefriend_recommendation_service_b200.engine import HybridTopKEngine, stage
    from tvbingefriend_recommendation_service_b200.multi_gpu import top_k_device_distributed
    from tvbingefriend_recommendation_service_b200.sharding import row_shard

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.gpus != world and rank == 0 and world > 1:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}", file=sys.stderr)

    if args.one_sided and world == 1:
        args.tuning = (args.tuning & ~(3 << 20)) | (1 << 20)     # symmetric sweep off
    eng = HybridTopKEngine(local_rank)
    cat = make_config(args.config, cfg["n_shows"])
    n, k = cat.n_shows, cfg["k"]
    st = stage(cat.features(), "mean3", pin=True)
    raw = eng.h2d(st)                                 # inputs resident in HBM for `value`
    rb, re_ = row_shard(n, world, rank)
    peaks = _peaks()

    PHASES = ("prep", "seed", "reduce", "sweep", "exchange", "rescore", "gather")
    state = {"prev": None}

    def step_device(events: dict | None = None):
        """prep + top-k (+ threshold all-reduce, candidate all-to-all and table all-gather when N > 1);
        ``events`` receives CUDA events around every phase."""
        def mark(name):
            if events is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                events.setdefault(name, []).append(ev)

        mark("step0")
        h0 = time.perf_counter()
        dc = eng.prepare(raw, weights, recycle=state["prev"])     # the previous step's operand buffer is recycled
        state["prev"] = dc
        if world > 1:
            h1 = time.perf_counter()
            res = top_k_device_distributed(eng, dc, weights, k, 0.1, True, splits=args.splits, tuning=args.tuning,
                                           symmetric=None if not args.one_sided else False, events=events,
                                           tables=state.get("tables"))
            state["tables"] = res["_full"]      # the gather buffers are reused from step to step
            if os.environ.get("BENCH_DEBUG") and rank == 0 and events:
                print(f"host: prepare {1e3 * (h1 - h0):.2f} ms, distributed job {1e3 * (time.perf_counter() - h1):.2f} ms",
                      file=sys.stderr)
            return res
        if events is None:
            state["tables"] = eng.top_k_device(dc, weights, k, 0.1, True, splits=args.splits, tuning=args.tuning,
                                               out=state.get("tables"))
            return state["tables"]
        mark("seed0")
        t = eng.top_k_device(dc, weights, k, 0.1, True, splits=args.splits, phases=1, tuning=args.tuning,
                             out=state.get("tables"))
        state["tables"] = t
        for name in ("seed1", "reduce1", "sweep1", "exchange1"):   # one launch sequence: seed + sweep = "sweep"
            mark(name)
        eng.top_k_device(dc, weights, k, 0.1, True, splits=args.splits, phases=6, out=t, tuning=args.tuning)
        mark("rescore1")
        mark("gather1")
        return t

    def phase_ms(events: dict) -> dict:
        order = ("step0", "seed0", "seed1", "reduce1", "sweep1", "exchange1", "rescore1", "gather1")
        out = {}
        for name, a, b in zip(PHASES, order, order[1:]):
            out[name] = float(np.mean([x.elapsed_time(y) for x, y in zip(events[a], events[b])]))
        if world == 1:      # seed pass and sweep are one call on a single GPU
            out["sweep"] += out.pop("seed")
            out["seed"] = 0.0
        return out

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        out = step_device({})        # same code path as the timed steps (events recorded, then dropped)
    sync()
    stats_host = out["stats"].cpu().numpy().reshape(-1, 8).sum(axis=0)
    flagged, pairs = int(stats_host[0]), int(stats_host[1])

    # ---- timed region 1: device-resident inputs -------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches
    events: dict = {}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    ev0.record()
    host_t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step_device(events)
    host_enqueue_ms = 1e3 * (time.perf_counter() - host_t0) / args.steps   # host time to ISSUE a step (no sync inside)
    ev1.record()
    sync()
    launches = eng.kernel_launches - launches0
    total_ms = ev0.elapsed_time(ev1)
    ph = phase_ms(events)
    if os.environ.get("BENCH_DEBUG") and rank == 0:     # per-step phase times (averages hide host-side gaps)
        order = ("step0", "seed0", "seed1", "reduce1", "sweep1", "exchange1", "rescore1", "gather1")
        for i in range(args.steps):
            print("step", i, [round(events[a][i].elapsed_time(events[b][i]), 2) for a, b in zip(order, order[1:])],
                  file=sys.stderr)
    clocks = sampler.stop() if rank == 0 else None
    dumped = None
    if args.dump_outputs and rank == 0:     # read back before the e2e steps overwrite these tables
        dumped = output_sample(eng.to_host(last))
    t_ms = torch.tensor([total_ms, ph["seed"] + ph["sweep"]] + [ph[name] for name in PHASES], device="cuda",
                        dtype=torch.float64)
    t_min = t_ms.clone()
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_min, op=dist.ReduceOp.MIN)
    ms_per_step = t_ms[0].item() / args.steps
    k1_ms_mean = t_ms[1].item()
    phases_max = {name: round(t_ms[2 + i].item(), 4) for i, name in enumerate(PHASES)}
    phases_min = {name: round(t_min[2 + i].item(), 4) for i, name in enumerate(PHASES)}

    # ---- timed region 2: end to end through the public engine API (H2D + compute + D2H) --------
    dtk = None
    if world > 1:
        from tvbingefriend_recommendation_service_b200.multi_gpu import DistributedTopK

        dtk = DistributedTopK(eng, n, k)

    def step_e2e():
        if world > 1:     # sliced upload + NVLink replication in, shared pinned host table out
            return dtk.run(st, weights, 0.1, True, symmetric=None if not args.one_sided else False,
                           splits=args.splits, tuning=args.tuning)
        dc = eng.prepare(eng.h2d(st, reuse=True), weights, recycle=state["prev"])
        state["prev"] = dc
        t = state["tables"] = eng.top_k_device(dc, weights, k, 0.1, True, splits=args.splits, tuning=args.tuning,
                                               out=state.get("tables"))
        return eng.to_host(t, copy=False)

    for _ in range(3):      # warm-up: both sets of cached buffers and the pinned host tables exist afterwards
        step_e2e()
    sync()
    ev0.record()
    for _ in range(args.steps):
        host_table = step_e2e()
    ev1.record()
    sync()
    e2e_ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_ms_per_step = e2e_ms.item() / args.steps
    d2h = sum(getattr(host_table, f).nbytes for f in ("indices", "counts", "hybrid", "genre", "text", "metadata"))

    extra = {}
    if args.extra and not args.n_shows:
        state["prev"] = None
        del raw
        if dtk is None:
            eng.release()
        for name in [x for x in args.extra.split(",") if x and x != args.config]:
            time.sleep(1.0)      # let the power-cap controller settle: the next shape starts from an idle-ish GPU
            try:
                if name == "one_sided":     # the sweep every job that is not eligible for the symmetric one gets
                    extra[f"{args.config}_one_sided"] = run_extra(name, eng, args, world, rank, weights, peaks,
                                                                  tuning=1 << 20, config=args.config)
                elif name == "nxn":
                    if world == 1:
                        extra["nxn_variant"] = nxn_variant(eng, weights)
                elif name == "weight_sweep":
                    if world == 1:
                        extra["weight_sweep"] = weight_sweep(eng, args.config)
                else:
                    extra[name] = run_extra(name, eng, args, world, rank, weights, peaks)
            except Exception as exc:   # an extra must never take the headline down with it
                extra[name] = {"error": f"{type(exc).__name__}: {exc}"}
        raw = eng.h2d(st)

    final_table = single_table = value_table = None
    if world > 1 and not args.no_parity_check:     # the device-gathered table of the `value` path as well
        value_table = eng.to_host(step_device())
    if dtk is not None:
        sync()
    if rank == 0 and not args.no_parity_check:
        from tvbingefriend_recommendation_service_b200.engine import TopK

        final_table = TopK(**{f: getattr(host_table, f).copy() for f in
                              ("indices", "counts", "hybrid", "genre", "text", "metadata")})
        if world > 1:     # the same job on this GPU alone, for exact comparison with the gathered table
            single_table = eng.to_host(eng.top_k_device(eng.prepare(raw, weights), weights, k, 0.1, True))
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # algorithmic work of this GPU's share of the text contraction, counted as the reference
    # computes it (all N x N pairs); the symmetric sweep executes about half of it
    flops = 2.0 * n * n * cfg["vocab"] / world
    dc_plan = eng.prepare(raw, weights)
    sym_forced_off = ((args.tuning >> 20) & 3) == 1 or args.one_sided
    if world > 1:
        sharded_sym = (not sym_forced_off) and n >= 40_000 and eng.sym_eligible(dc_plan, weights, k, 0.1)
        plan = eng.plan_tiles(dc_plan, weights, k, 0.1, rank=0, world=world, tile_sharded=True, splits=args.splits,
                              tuning=args.tuning) if sharded_sym else \
            eng.plan_tiles(dc_plan, weights, k, 0.1, row_begin=rb, row_end=re_, splits=args.splits,
                           tuning=args.tuning | (1 << 20))
    else:
        eng._folded(dc_plan, *[float(w) for w in weights], k)   # small vocabularies: plan over the operand the job ran on
        plan = eng.plan_tiles(dc_plan, weights, k, 0.1, splits=args.splits, tuning=args.tuning)
    used_sym = plan["symmetric"]
    exec_flops = plan["flops"]      # this GPU's tiles (seed pass + sweep) x tile rows x 256 x K_pad x 2
    traffic = None
    try:   # DRAM bytes per K1 launch from the committed ncu capture of this configuration
        tj = json.loads((ROOT / "profiles" / "k1_traffic.json").read_text())
        if world == 1 and not args.n_shows:
            traffic = tj[args.config]["symmetric" if used_sym else "one_sided"]["bytes"]
    except Exception:
        traffic = None
    traffic_src = None
    try:
        traffic_src = tj[args.config]["symmetric" if used_sym else "one_sided"].get("source")
    except Exception:
        pass
    secs = k1_ms_mean * 1e-3
    alg_tflops = flops / secs / 1e12 if secs > 0 else 0.0
    exec_tflops = exec_flops / secs / 1e12 if secs > 0 else 0.0
    peak = peaks["bf16_tflops_sustained"]
    roofline = {"bound": "tensor", "achieved": exec_tflops, "peak": peak, "unit": "TFLOP/s",
                "frac": exec_tflops / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "hybrid_topk_kernel (K1: threshold seed pass + sweep)", "kernel_ms": k1_ms_mean,
                "flops_per_launch": exec_flops, "peak_kind": f"bf16 sustained, {peaks['source']}",
                "peak_burst": peaks["bf16_tflops"], "frac_of_burst": exec_tflops / peaks["bf16_tflops"],
                "symmetric_sweep": bool(used_sym), "seed_tiles": plan["seed_tiles"], "sweep_tiles": plan["sweep_tiles"],
                "tile": f"{plan['tile_rows']}x256x{plan['k_pad']}", "genre_metadata_in_operand": plan["folded_bits"],
                "algorithmic_flops_per_launch": flops, "algorithmic_tflops": alg_tflops,
                "frac_algorithmic": alg_tflops / peak if peak else None,
                "note": "achieved / frac count the flops the tensor pipe EXECUTES (256x256xK_pad tiles "
                        "launched, seed pass included); algorithmic_* count the reference's full 2*N*N*V "
                        "all-pairs contraction, of which the symmetric sweep needs about half.  The sparse "
                        "synthetic operand keeps the SM clock above what a dense GEMM holds under the power "
                        "cap: see dense_text for the same kernel on a dense-random operand"}
    line = {
        "metric": METRIC, "value": n / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f16 x f16 -> f32 (tcgen05) candidate pass, f64 for every reported score",
        "data": "synthetic", "config": bench_config(args, cfg),
        "roofline": roofline,
        "e2e": {"value": n / (e2e_ms_per_step * 1e-3), "unit": UNIT, "h2d_bytes_per_step": st.h2d_bytes(),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms_per_step,
                "path": "stage()d pinned features -> H2D -> K0..K6 -> D2H of the [N, k] table" if world == 1 else
                        f"every rank uploads 1/{world} of the pinned feature bytes (h2d_bytes_per_step is the "
                        f"whole-job total) and NVLink all-gathers them; every rank copies its shard of the table "
                        f"into one pinned host table in shared memory (d2h_bytes_per_step is the whole table)"},
        "gpu_launches": int(launches),
        "host_enqueue_ms_per_step": round(host_enqueue_ms, 3),   # rank 0; below ms_per_step = the GPU is the bound
        "phases_ms": phases_max,                 # max over ranks: a collective's entry includes waiting for the slowest rank
        "phases_ms_min_over_ranks": phases_min,  # ... the minimum is the collective itself
        "clocks": clocks,
        "flagged_rows": flagged, "rescored_pairs": pairs,
        "extra": extra,
    }
    if world == 1:
        # ---- API-level end to end: what a caller of the drop-in pays, wall clock.  features dict (numpy /
        # scipy objects as np.load and load_npz return them) -> SimilarityComputer.compute_top_k (raw
        # bytes staged through cached pinned buffers, classified and packed on the GPU, K0..K6, D2H)
        # -> TopK.records (the columnar record stream the sink stores)
        from tvbingefriend_recommendation_service_b200.ml.similarity_computer import SimilarityComputer

        comp = SimilarityComputer(*weights, engine=eng)
        feats, ids = cat.features(), cat.show_ids
        api_ms, rec_ms, n_rec = [], [], 0
        for i in range(1 + min(args.steps, 3)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            top = comp.compute_top_k(feats, k=k, min_similarity=0.1)
            t1 = time.perf_counter()
            rec = top.records(ids)
            t2 = time.perf_counter()
            if i:
                api_ms.append(1e3 * (t2 - t0))
                rec_ms.append(1e3 * (t2 - t1))
            n_rec = int(len(rec["show_id"]))
        line["api_e2e"] = {"ms": float(np.mean(api_ms)), "value": n / (float(np.mean(api_ms)) * 1e-3), "unit": UNIT,
                           "records_ms": float(np.mean(rec_ms)), "records": n_rec,
                           "path": "features dict -> SimilarityComputer.compute_top_k (device-side ingest) -> "
                                   "TopK.records; host wall clock, first call excluded (pinned staging buffers "
                                   "and workspace are allocated once per engine)"}
    if not args.no_dense_probe and world == 1:
        dc = eng.prepare(raw, weights)
        probe = dense_text_probe(eng, dc, weights, k, args.tuning)
        psecs = probe["k1_ms"] * 1e-3
        probe["executed_tflops"] = exec_flops / psecs / 1e12
        probe["frac"] = probe["executed_tflops"] / peak
        line["dense_text"] = probe
    if not args.no_parity_check:
        line["parity_check"] = parity_check(eng, cat, cfg, weights, final_table, single_table)
        if value_table is not None:
            m = single_table.indices >= 0
            line["parity_check"]["device_gathered_table_identical_to_single_gpu"] = bool(
                np.array_equal(single_table.indices, value_table.indices)
                and np.array_equal(single_table.counts, value_table.counts)
                and np.array_equal(single_table.hybrid[m], value_table.hybrid[m]))
            line["parity_check"]["ok"] = bool(line["parity_check"]["ok"] and
                                              line["parity_check"]["device_gathered_table_identical_to_single_gpu"])
    if not args.no_cpu_baseline and world == 1:      # rank 0 at N=1 only
        line["cpu_baseline"] = cpu_baseline(cat, cfg, weights, budget_s=20.0)
    if dumped is not None:
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for name, arr in dumped.items():
            np.save(out_dir / f"{name}.npy", arr)
        line["dump_outputs"] = {"dir": str(out_dir), "rows": int(len(dumped["rows"])), "of_rows": n,
                                "arrays": sorted(dumped)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
