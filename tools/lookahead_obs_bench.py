"""Lookahead with rendered leaf observations (Engine.lookahead(obs=True)) against lookahead without them and against
the snapshot / restore / step recipe that gives a planner the same leaf observations by stepping.

Workloads (B branches = N envs, one branch per env, identity roots), F = 4, a ring of 16 slots, device auto-reset:
  c2      4096 envs, lead_brake levels 1-3 (1024 scenes generated on the device), continuous, 6-class float32 masks
  c2u8    the same with mask_dtype="uint8"
  c3      8192 envs, rdm rt_hard_v1 (25 vehicles, stepped by the 32-lane groups past the trajectory tables; a pool of
          --c3-pool host-generated scenes), discrete, 6-class float32 masks

For each workload and horizon H, in one process, blocks alternating between the three operations, each row the
median of 5 blocks between CUDA events:
  lookahead      cbev_lookahead, rewards only
  lookahead_obs  cbev_lookahead_obs: the branches with their draw records, the raster kernel over the B * F leaf
                 positions, the copy of the root frames
  plan           the recipe of tools/snapshot_bench.py: clone env 0 into every env, H rendered steps, whole-batch
                 restore (it also counts the planning episodes in the statistics, which lookahead does not)
Then, in a separate pass under torch.profiler, the per-kernel split of lookahead_obs (k_lookahead_obs, k_render /
k_render_any, k_leaf_window) and the k_lookahead time of the plain call, summed over the profiled calls.

    python tools/lookahead_obs_bench.py [--workloads c2,c2u8,c3] [--horizons 8,32] [--c3-horizons 8] [--out FILE]

Prints one JSON object per row and, with --out, writes them all plus the card's name, power limit and maximum SM clock
(nvidia-smi, read in the same process)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from lookahead_bench import actions  # noqa: E402
from snapshot_bench import BLOCKS, gpu_info  # noqa: E402


def make_engine(workload, c3_pool):
    import numpy as np
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    if workload in ("c2", "c2u8"):
        n, k = 4096, 1024
        eng = E.Engine(n, ring_slots=16, action_mode=E.ACTION_CONTINUOUS, autoreset=E.AUTORESET_NEXT_STEP,
                       max_actors=4, seed=0, mask_dtype="uint8" if workload == "c2u8" else "float32")
        eng.upload_map(load_town01_map(128))
        eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    else:
        from carlabev_env_b200.config import get_action_profile_spec
        from carlabev_env_b200.pool import pack_pool
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options
        from carlabev_env_b200.scenes import build_pool

        n, k = 8192, c3_pool
        scenes = build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                             for i in range(k)], pad=182, workers=min(32, os.cpu_count() or 1))
        table = np.asarray(get_action_profile_spec("discrete9_v1")["discrete_actions"], dtype=np.float32)
        eng = E.Engine(n, ring_slots=16, action_mode=E.ACTION_DISCRETE, discrete_table=table,
                       autoreset=E.AUTORESET_NEXT_STEP, max_actors=25, seed=0)
        eng.upload_map(load_town01_map(128))
        eng.upload_pool(pack_pool(scenes))
    eng.reset(torch.arange(n, dtype=torch.int32) % k)
    return eng


def alternating(ops, reps):
    """{name: (median ms per call, [ms per call of each block])}: BLOCKS rounds, each timing every op's block of
    `reps` calls in turn between CUDA events (synchronised)."""
    import torch

    blocks = {name: [] for name, _, _ in ops}
    for _ in range(BLOCKS):
        for name, fn, r in ops:
            r = r or reps
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(r):
                fn()
            e1.record()
            torch.cuda.synchronize()
            blocks[name].append(e0.elapsed_time(e1) / r)
    return {name: (statistics.median(b), b) for name, b in blocks.items()}


def kernel_split(fn, calls):
    """Device time per call of each kernel launched by fn, by kernel name (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        name = ev.key  # kernel names: "void (anonymous namespace)::k_render<0, 6, false>(...)"
        for short in ("k_lookahead_obs", "k_lookahead", "k_render_any", "k_render", "k_leaf_window", "k_fuse"):
            if short + "<" in name or short + "(" in name:
                us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                out[short] = out.get(short, 0.0) + us / 1e3 / calls
                break
    return out


def run(workload, horizons, reps, c3_pool):
    import torch

    eng = make_engine(workload, c3_pool)
    n = eng.N
    g = torch.Generator(device="cpu").manual_seed(0)
    step_acts = [actions(eng, g, (n,)) for _ in range(16)]
    for i in range(20):
        eng.step(step_acts[i % 16])
    snap = eng.snapshot()
    one = eng.snapshot(env_ids=[0])
    zeros = torch.zeros(n, dtype=torch.int32, device=eng.device)
    win_mb = n * eng.F * eng.frame_bytes / 2 ** 20
    rows = []
    for h in horizons:
        la_acts = actions(eng, g, (h, n))
        res = eng.lookahead(la_acts)
        res_obs = eng.lookahead(la_acts, obs=True)

        def plan():
            eng.restore(one, rows=zeros)
            for i in range(h):
                eng.step(step_acts[i % 16])
            eng.restore(snap)

        t = alternating([("lookahead", lambda: eng.lookahead(la_acts, out=res), None),
                         ("lookahead_obs", lambda: eng.lookahead(la_acts, obs=True, out=res_obs), None),
                         ("plan", plan, max(1, reps // 4))], reps)
        split = kernel_split(lambda: eng.lookahead(la_acts, obs=True, out=res_obs), reps)
        plain = kernel_split(lambda: eng.lookahead(la_acts, out=res), reps)
        s = res_obs.steps
        r = {"workload": workload, "branches": n, "horizon": h, "frame_stack": eng.F,
             "mask_dtype": eng.mask_dtype, "leaf_window_mb": win_mb,
             "mean_steps_taken": s.float().mean().item(),
             "leaf_frames_rendered": int(torch.clamp(s, max=eng.F).sum().item()),
             "lookahead_ms": t["lookahead"][0], "lookahead_obs_ms": t["lookahead_obs"][0], "plan_ms": t["plan"][0],
             "blocks_ms": {k: v[1] for k, v in t.items()},
             "kernels_ms": split, "k_lookahead_ms": plain.get("k_lookahead"),
             "obs_over_plain": t["lookahead_obs"][0] / t["lookahead"][0],
             "plan_over_obs": t["plan"][0] / t["lookahead_obs"][0]}
        rows.append(r)
        print(json.dumps(r), flush=True)
    eng.close()
    del snap, one
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="c2,c2u8,c3")
    ap.add_argument("--horizons", default="8,32")
    ap.add_argument("--c3-horizons", default="8")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--c3-pool", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("lookahead_obs_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    doc = {"gpu": info, "reps": args.reps, "blocks": BLOCKS, "rows": []}
    print(json.dumps({"gpu": info}), flush=True)
    for w in args.workloads.split(","):
        hs = args.c3_horizons if w == "c3" else args.horizons
        doc["rows"] += run(w, [int(h) for h in hs.split(",")], args.reps, args.c3_pool)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
