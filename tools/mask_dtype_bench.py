"""float32 against uint8 semantic masks (Engine(mask_dtype=...)) on the bench workloads, in one process.

For each workload (c2: 4096 envs, c3: 8192, f4: size 256 with 4096) both engines run side by side on the same pool,
seed and actions with device auto-reset, at the same ring length: first L = 16, then the default ring-slot rule of
Engine (35 % of the free memory before either engine exists, up to 64 slots; the uint8 frame is a quarter of the
float32 one, so the rule grants it up to 4x the slots).  Timed blocks of K steps between CUDA events alternate between
the two dtypes; the median of 5 is reported, then one profiled block per dtype gives k_move / k_render / k_judge.

    python tools/mask_dtype_bench.py [--steps K] [--warmup W] [--workloads c2,c3,f4] [--out FILE]

Prints one JSON object per row and, with --out, writes them all plus the card's name, power limit and maximum SM clock
(nvidia-smi, read in the same process)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

DTYPES = ("float32", "uint8")
BLOCKS = 5
BOUND_HBM = 0.6  # stores at the measured peak take at least this share of k_render: the row is bound by HBM stores


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def make_engines(name, scenes, ring_slots, ring_budget):
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import ACTION_PROFILES
    from carlabev_env_b200.pool import pack_pool
    from carlabev_env_b200.vector_env import load_town01_map

    W = bench.WORKLOADS[name]
    discrete = W["actions"] == "discrete"
    size = W.get("size", 128)
    N = W["envs"]
    engs = {}
    for dt in DTYPES:
        e = E.Engine(N, mask_mode="6-class", frame_stack=4, ring_slots=ring_slots, ring_budget_bytes=ring_budget,
                     action_mode=E.ACTION_DISCRETE if discrete else E.ACTION_CONTINUOUS,
                     discrete_table=ACTION_PROFILES["discrete9_v1"]["discrete_actions"] if discrete else None,
                     autoreset=E.AUTORESET_NEXT_STEP, anchor=W["anchor"], seed=0, size=size,
                     max_actors=max(len(s["act_kind"]) for s in scenes), mask_dtype=dt)
        e.upload_map(load_town01_map(size))
        e.upload_pool(pack_pool(scenes))
        e.reset(torch.arange(N, dtype=torch.int32) % len(scenes))
        engs[dt] = e
    g = torch.Generator(device="cpu").manual_seed(0)
    if discrete:
        acts = [torch.randint(0, 9, (N,), generator=g, dtype=torch.int64).cuda() for _ in range(16)]
    else:
        lo, hi = torch.tensor([0.0, -1.0, 0.0]), torch.tensor([1.0, 1.0, 1.0])
        acts = [(lo + (hi - lo) * torch.rand(N, 3, generator=g)).float().cuda() for _ in range(16)]
    return engs, acts


def timed_block(eng, acts, K):
    import torch

    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        eng.step(acts[i % len(acts)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def run(name, ring_rule, K, warmup, scenes, peak_gbs):
    import torch

    N = bench.WORKLOADS[name]["envs"]
    if ring_rule == "L16":
        engs, acts = make_engines(name, scenes, 16, None)
    else:
        free, _ = torch.cuda.mem_get_info()
        engs, acts = make_engines(name, scenes, None, int(free * 0.35))
    for dt in DTYPES:
        for i in range(warmup):
            engs[dt].step(acts[i % len(acts)])
    blocks = {dt: [] for dt in DTYPES}
    for _ in range(BLOCKS):
        for dt in DTYPES:  # alternating: drift of clocks or neighbours hits both dtypes alike
            blocks[dt].append(timed_block(engs[dt], acts, K))
    rows = []
    for dt in DTYPES:
        eng = engs[dt]
        eng.profile(True)
        timed_block(eng, acts, K)
        move_ms, render_ms, judge_ms, n = eng.profile_read()
        eng.profile(False)
        n = max(n, 1)
        ms = statistics.median(blocks[dt]) / K
        store_bytes = N * eng.channels * eng.obs_hw[0] * eng.obs_hw[1] * (1 if dt == "uint8" else 4)
        render = render_ms / n
        floor_ms = store_bytes / (peak_gbs * 1e9) * 1e3
        share = floor_ms / render if render > 0 else None
        bound = ("HBM stores" if share is not None and share >= BOUND_HBM else
                 "on-chip phases (TMA, draw list, rotate, resize) and the launch's fill / drain")
        rows.append({"workload": name, "envs": N, "size": bench.WORKLOADS[name].get("size", 128), "mask_dtype": dt,
                     "ring_rule": ring_rule, "ring_slots": eng.L, "ring_bytes": N * eng.L * eng.frame_bytes,
                     "ms_per_step": ms, "env_steps_per_s": N / (ms * 1e-3), "blocks_ms": blocks[dt],
                     "k_move_ms": move_ms / n, "k_render_ms": render, "k_judge_ms": judge_ms / n,
                     "store_bytes_per_step": store_bytes, "store_ms_at_peak": floor_ms,
                     "store_share_of_k_render": share, "k_render_gbs": store_bytes / (render * 1e-3) / 1e9,
                     "bound": bound})
    for e in engs.values():
        e.close()
    del engs
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workloads", default="c2,c3,f4")
    ap.add_argument("--out", default=None, help="also write the JSON document (every row, the card, the HBM peak used) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("mask_dtype_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    peak, peak_src = bench.measured_peak_gbs()
    doc = {"gpu": info, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "steps": args.steps,
           "warmup": args.warmup, "blocks": BLOCKS, "rows": []}
    print(json.dumps({"gpu": info, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src}), flush=True)
    for name in args.workloads.split(","):
        scenes = bench.workload_pool(name, types.SimpleNamespace(pool=bench.POOL_SCENES))
        for rule in ("L16", "default"):
            for row in run(name, rule, args.steps, args.warmup, scenes, peak):
                print(json.dumps(row), flush=True)
                doc["rows"].append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
