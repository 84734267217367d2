"""Lookahead from snapshot rows with leaf rows (Engine.lookahead(source=, leaf=True)): tree expansion through leaf rows
against replaying the action prefix from the live root, and the per-kernel split of a call.

Workloads as in tools/lookahead_obs_bench.py (B branches = N envs, identity roots, F = 4, a ring of 16 slots):
  c2      4096 envs, lead_brake levels 1-3, continuous, 6-class float32 masks
  c2u8    the same with mask_dtype="uint8"
  c3      8192 envs, rdm rt_hard_v1 (25 live-stepped vehicles, --c3-pool host-generated scenes), discrete, float32

Expansion (--expand-workloads, depth d = 1..--depth): a tree of B nodes per level, each expanded by one step.  In one
process, blocks alternating between the two ways of getting the depth-d leaf observations, each the median of 5 blocks
between CUDA events:
  rows    one step from the depth d - 1 leaf rows: lookahead(source=rows_{d-1}, obs=True, leaf=True), which also
          returns the depth-d rows the next level starts from
  replay  the whole prefix from the live root: lookahead(H = d, obs=True), no rows
The depth-d rows come from the depth d - 1 rows (two buffers used in turn), so branches that ended on the way give
done rows (steps = 0) as they would in a tree.  `crossover_depth` is the first depth at which rows is faster.

Split (--workloads, horizons --horizons, --c3-horizons for c3): in one process, blocks alternating between
lookahead_obs from the live envs and the same branches from their snapshot rows with leaf rows; then, in a separate
pass under torch.profiler, the device time per call of each kernel of the rows call (k_lookahead_ex, k_render /
k_render_any, k_leaf_window_rows, k_leaf_rows), with obs=True and with leaf rows only (windows in engine scratch).

    python tools/lookahead_rows_bench.py [--expand-workloads c2,c2u8] [--depth 32] [--workloads c2,c2u8,c3]
                                         [--horizons 8,32] [--c3-horizons 8] [--out FILE]

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

KERNELS = ("k_lookahead_ex", "k_lookahead_obs", "k_lookahead", "k_render_any", "k_render", "k_leaf_window_rows",
           "k_leaf_window", "k_leaf_rows")


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
        for short in KERNELS:
            if short + "<" in ev.key or short + "(" in ev.key:
                us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                out[short] = out.get(short, 0.0) + us / 1e3 / calls
                break
    return out


def warm_engine(workload, c3_pool):
    import torch

    eng = make_engine(workload, c3_pool)
    g = torch.Generator(device="cpu").manual_seed(0)
    step_acts = [actions(eng, g, (eng.N,)) for _ in range(16)]
    for i in range(20):
        eng.step(step_acts[i % 16])
    return eng, g


def expand(workload, depth, reps, c3_pool):
    import torch

    eng, g = warm_engine(workload, c3_pool)
    n = eng.N
    acts = actions(eng, g, (depth, n))
    root = eng.snapshot()
    # two leaf buffers used in turn: level d is expanded from one into the other
    bufs = [eng.lookahead(acts[:1].contiguous(), obs=True, leaf=True) for _ in range(2)]
    replay = {}
    prev = root
    rows = []
    for d in range(1, depth + 1):
        step = acts[d - 1:d].contiguous()
        prefix = acts[:d].contiguous()
        cur = bufs[d % 2]
        replay[d] = eng.lookahead(prefix, obs=True)
        src = prev
        t = alternating([("rows", lambda: eng.lookahead(step, source=src, obs=True, leaf=True, out=cur), None),
                         ("replay", lambda: eng.lookahead(prefix, obs=True, out=replay[d]), None)], reps)
        eng.lookahead(step, source=src, obs=True, leaf=True, out=cur)
        same = bool(torch.equal(cur.obs, replay[d].obs))  # the two ways give the same depth-d leaf observations
        prev = cur.leaf
        del replay[d]
        r = {"kind": "expand", "workload": workload, "branches": n, "depth": d, "mask_dtype": eng.mask_dtype,
             "row_bytes": eng.snapshot_row_bytes, "rows_ms": t["rows"][0], "replay_ms": t["replay"][0],
             "blocks_ms": {k: v[1] for k, v in t.items()}, "same_leaf_obs": same,
             "live_branches": int((cur.steps > 0).sum().item())}
        rows.append(r)
        print(json.dumps(r), flush=True)
    cross = next((r["depth"] for r in rows if r["rows_ms"] < r["replay_ms"]), None)
    summary = {"kind": "expand_summary", "workload": workload, "crossover_depth": cross,
               "rows_total_ms": sum(r["rows_ms"] for r in rows), "replay_total_ms": sum(r["replay_ms"] for r in rows)}
    print(json.dumps(summary), flush=True)
    eng.close()
    del bufs, prev, root
    torch.cuda.empty_cache()
    return rows + [summary]


def split(workload, horizons, reps, c3_pool):
    import torch

    eng, g = warm_engine(workload, c3_pool)
    n = eng.N
    snap = eng.snapshot()
    rows = []
    for h in horizons:
        la_acts = actions(eng, g, (h, n))
        res_obs = eng.lookahead(la_acts, obs=True)
        res_rows = eng.lookahead(la_acts, source=snap, obs=True, leaf=True)
        res_leaf = eng.lookahead(la_acts, source=snap, leaf=True)
        t = alternating([("lookahead_obs", lambda: eng.lookahead(la_acts, obs=True, out=res_obs), None),
                         ("rows_obs_leaf", lambda: eng.lookahead(la_acts, source=snap, obs=True, leaf=True,
                                                                 out=res_rows), None),
                         ("rows_leaf", lambda: eng.lookahead(la_acts, source=snap, leaf=True, out=res_leaf), None)],
                        reps)
        k_obs_leaf = kernel_split(lambda: eng.lookahead(la_acts, source=snap, obs=True, leaf=True, out=res_rows), reps)
        k_leaf = kernel_split(lambda: eng.lookahead(la_acts, source=snap, leaf=True, out=res_leaf), reps)
        k_live = kernel_split(lambda: eng.lookahead(la_acts, obs=True, out=res_obs), reps)
        r = {"kind": "split", "workload": workload, "branches": n, "horizon": h, "frame_stack": eng.F,
             "mask_dtype": eng.mask_dtype, "row_bytes": eng.snapshot_row_bytes,
             "leaf_rows_mb": n * eng.snapshot_row_bytes / 2 ** 20,
             "mean_steps_taken": res_rows.steps.float().mean().item(),
             "same_as_live": bool(torch.equal(res_rows.obs, res_obs.obs) and torch.equal(res_rows.ret, res_obs.ret)),
             **{k + "_ms": v[0] for k, v in t.items()}, "blocks_ms": {k: v[1] for k, v in t.items()},
             "kernels_ms_rows_obs_leaf": k_obs_leaf, "kernels_ms_rows_leaf": k_leaf,
             "kernels_ms_live_obs": k_live}
        rows.append(r)
        print(json.dumps(r), flush=True)
    eng.close()
    del snap
    torch.cuda.empty_cache()
    return rows


def dumps(doc):
    """The JSON document with one row per line."""
    head = {k: v for k, v in doc.items() if k != "rows"}
    rows = ",\n  ".join(json.dumps(r) for r in doc["rows"])
    return json.dumps(head)[:-1] + ',\n "rows": [\n  ' + rows + "\n ]}\n"


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--expand-workloads", default="c2,c2u8")
    ap.add_argument("--depth", type=int, default=32)
    ap.add_argument("--workloads", default="c2,c2u8,c3")
    ap.add_argument("--horizons", default="8,32")
    ap.add_argument("--c3-horizons", default="8")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--c3-pool", type=int, default=256)
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("lookahead_rows_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    doc = {"gpu": info, "reps": args.reps, "blocks": BLOCKS, "rows": []}
    print(json.dumps({"gpu": info}), flush=True)
    for w in filter(None, args.expand_workloads.split(",")):
        doc["rows"] += expand(w, args.depth, args.reps, args.c3_pool)
    for w in filter(None, args.workloads.split(",")):
        hs = args.c3_horizons if w == "c3" else args.horizons
        doc["rows"] += split(w, [int(h) for h in hs.split(",")], args.reps, args.c3_pool)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(dumps(doc))


if __name__ == "__main__":
    main()
