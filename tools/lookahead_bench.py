"""Observation-free lookahead (Engine.lookahead) against the two ways of getting the same numbers by stepping.

Workloads (B branches = N envs, one branch per env, identity roots):
  c2  4096 envs, lead_brake levels 1-3 (a pool of 1024 scenes generated on the device), continuous actions
  c3  8192 envs, rdm rt_hard_v1 (25 vehicles; a pool of --c3-pool host-generated scenes, scene_seed = i), discrete
Both with 6-class 96 x 96 float32 masks, F = 4, a ring of 16 slots, device auto-reset, trajectory tables.

For each workload and horizon H, in one process:
  lookahead   one cbev_lookahead call: B branches x H steps, rewards only
  plan        the snapshot/restore planning iteration of tools/snapshot_bench.py: clone env 0 into every env, H steps,
              whole-batch restore
  move+judge  k_move + k_judge per step, from the per-kernel events of cbev_profile_read_ex with debug flag 2 (k_judge
              serial on the step stream, so its events bracket it alone), over --profile-steps steps

Each timed row is the median of 5 blocks between CUDA events.  The per-branch-step time of the lookahead is its call
time over H; the bar is the move+judge time per step, the speed-up over `plan` is reported.

    python tools/lookahead_bench.py [--workloads c2,c3] [--horizons 8,32] [--reps 10] [--out FILE]

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

from snapshot_bench import BLOCKS, gpu_info, timed  # noqa: E402


def make_engine(workload, c3_pool):
    import numpy as np
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    if workload == "c2":
        n, k = 4096, 1024
        eng = E.Engine(n, ring_slots=16, action_mode=E.ACTION_CONTINUOUS, autoreset=E.AUTORESET_NEXT_STEP,
                       max_actors=4, seed=0)
        eng.upload_map(load_town01_map(128))
        eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    else:
        from carlabev_env_b200.pool import pack_pool
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options
        from carlabev_env_b200.scenes import build_pool

        n, k = 8192, c3_pool
        scenes = build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                             for i in range(k)], pad=182, workers=min(32, os.cpu_count() or 1))
        from carlabev_env_b200.config import get_action_profile_spec

        table = np.asarray(get_action_profile_spec("discrete9_v1")["discrete_actions"], dtype=np.float32)
        eng = E.Engine(n, ring_slots=16, action_mode=E.ACTION_DISCRETE, discrete_table=table,
                       autoreset=E.AUTORESET_NEXT_STEP, max_actors=25, seed=0)
        eng.upload_map(load_town01_map(128))
        eng.upload_pool(pack_pool(scenes))
    eng.reset(torch.arange(n, dtype=torch.int32) % k)
    return eng


def actions(eng, g, shape):
    import torch

    from carlabev_env_b200 import engine as E

    if eng.action_mode == E.ACTION_DISCRETE:
        return torch.randint(0, eng.cfg.n_discrete, shape, generator=g).cuda()
    lo, hi = torch.tensor([0.0, -1.0, 0.0]), torch.tensor([1.0, 1.0, 1.0])
    return (lo + (hi - lo) * torch.rand(*shape, 3, generator=g)).float().cuda()


def run(workload, horizons, reps, profile_steps, c3_pool):
    import torch

    eng = make_engine(workload, c3_pool)
    n = eng.N
    g = torch.Generator(device="cpu").manual_seed(0)
    step_acts = [actions(eng, g, (n,)) for _ in range(16)]
    for i in range(20):
        eng.step(step_acts[i % 16])
    rows = []

    def row(op, h, ms, blocks, note, **extra):
        r = {"workload": workload, "op": op, "branches": n, "horizon": h, "ms": ms, "blocks_ms": blocks,
             "us_per_step": ms * 1e3 / h if h else None, "note": note, **extra}
        rows.append(r)
        print(json.dumps(r), flush=True)

    # (b) k_move + k_judge per step, k_judge serial on the step stream
    eng.set_debug_flags(2)
    eng.profile(True)
    eng.profile_read()
    for i in range(profile_steps):
        eng.step(step_acts[i % 16])
    move_ms, render_ms, judge_ms, k = eng.profile_read()
    eng.profile(False)
    eng.set_debug_flags(0)
    sim_us = (move_ms + judge_ms) * 1e3 / k
    row("move_judge", 1, sim_us / 1e3, [], f"k_move + k_judge per step over {k} profiled steps (debug flag 2)",
        move_us=move_ms * 1e3 / k, judge_us=judge_ms * 1e3 / k, render_us=render_ms * 1e3 / k)

    snap = eng.snapshot()
    one = eng.snapshot(env_ids=[0])
    zeros = torch.zeros(n, dtype=torch.int32, device=eng.device)
    for h in horizons:
        la_acts = actions(eng, g, (h, n))
        res = eng.lookahead(la_acts)
        ms, b = timed(lambda: eng.lookahead(la_acts, out=res), reps)
        steps = res.steps.float().mean().item()
        row("lookahead", h, ms, b, f"one call, {n} branches x {h} steps, no rewards buffer",
            mean_steps_taken=steps, us_per_branch_step_taken=ms * 1e3 / steps if steps else None,
            vs_move_judge=(ms * 1e3 / h) / sim_us)

        def plan():
            eng.restore(one, rows=zeros)
            for i in range(h):
                eng.step(step_acts[i % 16])
            eng.restore(snap)

        ms_p, b_p = timed(plan, max(1, reps // 2))
        row("plan_clone_step_restore", h, ms_p, b_p, f"clone + {h} steps + whole-batch restore",
            lookahead_speedup=ms_p / ms)
    eng.close()
    del snap, one
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--horizons", default="8,32")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--profile-steps", type=int, default=200)
    ap.add_argument("--c3-pool", type=int, default=512)
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("lookahead_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    horizons = [int(h) for h in args.horizons.split(",")]
    doc = {"gpu": info, "reps": args.reps, "blocks": BLOCKS, "horizons": horizons, "rows": []}
    print(json.dumps({"gpu": info}), flush=True)
    for w in args.workloads.split(","):
        doc["rows"] += run(w, horizons, args.reps, args.profile_steps, args.c3_pool)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
