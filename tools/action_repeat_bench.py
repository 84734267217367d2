"""Action repeat (Engine.set_action_repeat): one fused call of K simulator steps against K single steps.

Workloads (the engines of tools/lookahead_obs_bench.py: 6-class 96 x 96 masks, F = 4, a ring of 16 slots, device
auto-reset, trajectory tables):
  c2    4096 envs, lead_brake levels 1-3 (1024 scenes generated on the device), continuous actions, float32 masks
  c2u8  the same with uint8 masks
  c3    8192 envs, rdm rt_hard_v1 (25 vehicles; --c3-pool host-generated scenes), discrete actions, float32 masks

For each workload and K, in one process, blocks alternating, median of 5 blocks between CUDA events:
  repeat    one step call at action repeat K (k_step_repeat + the raster kernel; at K = 1 the three-launch step)
  singles   K consecutive step calls at repeat 1: a timing reference only (its auto-resets fall at other times)
Reported per call and per simulated step (call / K).  Then the fused path at K = 1 (debug flag 1024) against the
three-launch step, alternating the same way, and in a separate pass under torch.profiler the per-call device time of
k_step_repeat and of the raster kernel at each K.

    python tools/action_repeat_bench.py [--workloads c2,c2u8,c3] [--repeats 1,2,4,8] [--reps 40] [--out FILE]

Prints one JSON object per row and, with --out, writes them all plus the card's name, power limit and maximum SM clock
(nvidia-smi, read in the same process)."""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from lookahead_bench import actions  # noqa: E402
from lookahead_obs_bench import alternating, make_engine  # noqa: E402
from snapshot_bench import BLOCKS, gpu_info  # noqa: E402

FLAG_FUSED = 1024


def kernel_split(fn, calls):
    """Device time per call of k_step_repeat / k_move / k_judge / the raster kernel (torch.profiler, CUDA
    activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        name = ev.key
        for short in ("k_step_repeat", "k_move", "k_judge", "k_render_any", "k_render"):
            if short + "<" in name or short + "(" in name:
                us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                out[short] = out.get(short, 0.0) + us / 1e3 / calls
                break
    return out


def run(workload, repeats, reps, c3_pool):
    import torch

    eng = make_engine(workload, c3_pool)
    n = eng.N
    g = torch.Generator(device="cpu").manual_seed(0)
    acts = [actions(eng, g, (n,)) for _ in range(16)]
    it = [0]

    def step():
        eng.step(acts[it[0] % 16])
        it[0] += 1

    for _ in range(20):
        step()
    rows = []

    def row(op, k, ms, blocks, note, **extra):
        r = {"workload": workload, "op": op, "envs": n, "repeat": k, "ms_per_call": ms, "blocks_ms": blocks,
             "ms_per_sim_step": ms / k, "note": note, **extra}
        rows.append(r)
        print(json.dumps(r), flush=True)

    def at(k, calls=1):
        def fn():
            eng.set_action_repeat(k)
            for _ in range(calls):
                step()
        return fn

    for k in repeats:
        ops = [("repeat", at(k), reps), ("singles", at(1, k), max(1, reps // k))]
        at(k)()  # warm both shapes
        at(1, k)()
        res = alternating(ops, reps)
        ms, b = res["repeat"]
        ms_s, b_s = res["singles"]
        row("repeat", k, ms, b, f"one call at action repeat {k}")
        row("singles", k, ms_s, b_s, f"{k} calls at repeat 1 (timing reference)",
            repeat_speedup_per_sim_step=ms_s / ms)
    # the fused path at K = 1 against the three-launch step
    def fused():
        eng.set_action_repeat(1)
        eng.set_debug_flags(FLAG_FUSED)
        step()

    def three():
        eng.set_action_repeat(1)
        eng.set_debug_flags(0)
        step()

    res = alternating([("fused_k1", fused, reps), ("three_launch_k1", three, reps)], reps)
    for name, note in (("fused_k1", "k_step_repeat + raster at K = 1 (debug flag 1024)"),
                       ("three_launch_k1", "k_move + k_judge (side stream) + raster at K = 1")):
        row(name, 1, res[name][0], res[name][1], note)
    eng.set_debug_flags(0)
    # per-kernel split, profiler on (a separate pass: tracing slows the host)
    for k in repeats:
        split = kernel_split(at(k), 20)
        row("kernel_split", k, sum(split.values()), [], f"summed device time per call at repeat {k} (torch.profiler)",
            kernels_ms=split)
    split = kernel_split(fused, 20)
    eng.set_debug_flags(0)
    row("kernel_split_fused_k1", 1, sum(split.values()), [], "debug flag 1024 at K = 1 (torch.profiler)",
        kernels_ms=split)
    eng.close()
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="c2,c2u8,c3")
    ap.add_argument("--repeats", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--c3-pool", type=int, default=128)
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("action_repeat_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    repeats = [int(k) for k in args.repeats.split(",")]
    doc = {"gpu": info, "reps": args.reps, "blocks": BLOCKS, "repeats": repeats, "c3_pool": args.c3_pool, "rows": []}
    print(json.dumps({"gpu": info}), flush=True)
    for w in args.workloads.split(","):
        doc["rows"] += run(w, repeats, args.reps, args.c3_pool)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
