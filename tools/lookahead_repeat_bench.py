"""Lookahead in agent steps of action repeat K (Engine.lookahead(repeat=K)) against the two other ways of getting
the same work done.

Workloads as in tools/lookahead_rows_bench.py (B branches = N envs, identity roots, F = 4, a ring of 16 slots):
  c2      4096 envs, lead_brake levels 1-3, continuous, 6-class float32 masks
  c2u8    the same with mask_dtype="uint8"
  c3      8192 envs, rdm rt_hard_v1 (25 live-stepped vehicles, --c3-pool host-generated scenes), discrete, float32

For each horizon H (agent steps) and repeat K, in one process, blocks alternating between these arms, each the median
of 5 blocks between CUDA events after a warm-up call of every shape:
  repeat       lookahead(acts [H, B], repeat=K), no observations
  tiled        lookahead(acts tiled K times along the horizon, [H*K, B]), no observations: the same simulator steps,
               so repeat / tiled near 1 means the sub-step loop costs nothing extra (the outputs differ: tiled gives
               simulator-step rewards and discounting)
  repeat_obs   lookahead(repeat=K, obs=True): the leaf windows of agent-step frames
  repeat_leaf  lookahead(repeat=K, obs=True, leaf=True): the windows and the leaf rows
  clone        restore the roots into the live envs, set_action_repeat(K), step H times, copy out the windows, restore
               the live state and set the repeat back: the only other way to get agent-step leaf windows
`same_full_horizon_obs` checks that repeat_obs and clone give the same windows for the branches that ran all H agent
steps (the live envs auto-reset after a terminal step, a branch does not).

    python tools/lookahead_repeat_bench.py [--workloads c2,c2u8,c3] [--horizons 8,32] [--repeats 2,4] [--out FILE]

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
from lookahead_obs_bench import alternating  # noqa: E402
from lookahead_rows_bench import dumps, warm_engine  # noqa: E402
from snapshot_bench import BLOCKS, gpu_info  # noqa: E402


def run(workload, horizons, repeats, reps, c3_pool):
    import torch

    eng, g = warm_engine(workload, c3_pool)
    n = eng.N
    snap = eng.snapshot()
    win = torch.empty_like(eng.obs())
    rows = []
    for h in horizons:
        for k in repeats:
            acts = actions(eng, g, (h, n))
            tiled = acts.repeat_interleave(k, dim=0).contiguous()
            res = {"repeat": eng.lookahead(acts, repeat=k), "tiled": eng.lookahead(tiled),
                   "repeat_obs": eng.lookahead(acts, repeat=k, obs=True),
                   "repeat_leaf": eng.lookahead(acts, repeat=k, obs=True, leaf=True)}

            def clone():
                eng.restore(snap)
                eng.set_action_repeat(k)
                for t in range(h):
                    eng.step(acts[t])
                win.copy_(eng.obs())
                eng.set_action_repeat(1)
                eng.restore(snap)

            clone()
            full = res["repeat_obs"].steps == h
            same = bool(torch.equal(res["repeat_obs"].obs[full], win[full]))
            same_steps = bool(torch.equal(res["repeat"].steps, (res["tiled"].steps + k - 1) // k))
            t = alternating([("repeat", lambda: eng.lookahead(acts, repeat=k, out=res["repeat"]), None),
                             ("tiled", lambda: eng.lookahead(tiled, out=res["tiled"]), None),
                             ("repeat_obs", lambda: eng.lookahead(acts, repeat=k, obs=True, out=res["repeat_obs"]),
                              None),
                             ("repeat_leaf", lambda: eng.lookahead(acts, repeat=k, obs=True, leaf=True,
                                                                   out=res["repeat_leaf"]), None),
                             ("clone", clone, max(1, reps // 4))], reps)
            r = {"workload": workload, "branches": n, "horizon": h, "repeat": k, "frame_stack": eng.F,
                 "mask_dtype": eng.mask_dtype, "row_bytes": eng.snapshot_row_bytes,
                 "mean_agent_steps": res["repeat"].steps.float().mean().item(),
                 "full_horizon_branches": int(full.sum().item()), "same_full_horizon_obs": same,
                 "same_steps_as_tiled": same_steps, **{a + "_ms": v[0] for a, v in t.items()},
                 "blocks_ms": {a: v[1] for a, v in t.items()},
                 "repeat_over_tiled": t["repeat"][0] / t["tiled"][0],
                 "clone_over_repeat_obs": t["clone"][0] / t["repeat_obs"][0],
                 "clone_over_repeat_leaf": t["clone"][0] / t["repeat_leaf"][0]}
            rows.append(r)
            print(json.dumps(r), flush=True)
            del res
    eng.close()
    del snap, win
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="c2,c2u8,c3")
    ap.add_argument("--horizons", default="8,32")
    ap.add_argument("--repeats", default="2,4")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--c3-pool", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("lookahead_repeat_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    doc = {"gpu": info, "reps": args.reps, "blocks": BLOCKS, "rows": []}
    print(json.dumps({"gpu": info}), flush=True)
    hs = [int(h) for h in args.horizons.split(",")]
    ks = [int(k) for k in args.repeats.split(",")]
    for w in filter(None, args.workloads.split(",")):
        doc["rows"] += run(w, hs, ks, args.reps, args.c3_pool)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(dumps(doc))


if __name__ == "__main__":
    main()
