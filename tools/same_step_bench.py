"""Same-step auto-reset (AUTORESET_SAME_STEP) against next_step: the per-call cost of the reset pass.

Workloads (the engines of tools/lookahead_obs_bench.py: 6-class 96 x 96 masks, F = 4, a ring of 16 slots, trajectory
tables):
  c2    4096 envs, lead_brake levels 1-3 (1024 scenes generated on the device), continuous actions, float32 masks
  c2u8  the same with uint8 masks
  c3    8192 envs, rdm rt_hard_v1 (25 vehicles; --c3-pool host-generated scenes), discrete actions, float32 masks

For each workload and action repeat, two engines of the same configuration and seed live in one process, one per mode.
Their step calls are timed in alternating blocks, median of 5 blocks between CUDA events; the difference is the tail
the pass adds (k_same_step_reset and the raster launch of the reset frames).  Useful transitions per second count every
same_step call and, for next_step, the calls that are not auto-reset calls: calls/s x (1 - share of auto-reset calls),
the share measured from the run's own flags.  Then, in a separate pass under torch.profiler, the per-call device time of
every kernel, the raster launch that follows k_same_step_reset reported apart as the reset raster launch.  A second
alternating run times the same_step engine with its final-observation buffer unbound (the pass then copies no
terminal window), which separates the copy from the reset and its rendering.

    python tools/same_step_bench.py [--workloads c2,c2u8,c3] [--repeats 1,4] [--reps 40] [--out FILE]

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

KERNELS = ("k_same_step_reset", "k_step_repeat", "k_move", "k_judge", "k_render_any", "k_render")


def kernel_split(fn, calls):
    """Device time per call of each kernel fn launches (torch.profiler, CUDA activities); a raster launch right after
    k_same_step_reset counts as "reset_raster"."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    kernels = []
    for ev in prof.events():
        short = next((k for k in KERNELS if k + "<" in ev.name or k + "(" in ev.name), None)
        if short is None or not str(ev.device_type).endswith("CUDA"):
            continue
        kernels.append((ev.time_range.start, short, ev.time_range.end - ev.time_range.start))
    kernels.sort()
    out, prev = {}, None
    for _, short, us in kernels:
        key = "reset_raster" if short.startswith("k_render") and prev == "k_same_step_reset" else short
        out[key] = out.get(key, 0.0) + us / 1e3 / calls
        prev = short
    return out


def run(workload, repeats, reps, c3_pool):
    import torch

    from carlabev_env_b200 import engine as E

    engs = {"next_step": make_engine(workload, c3_pool, E.AUTORESET_NEXT_STEP),
            "same_step": make_engine(workload, c3_pool, E.AUTORESET_SAME_STEP)}
    n = engs["next_step"].N
    g = torch.Generator(device="cpu").manual_seed(0)
    acts = [actions(engs["next_step"], g, (n,)) for _ in range(16)]
    it = {m: 0 for m in engs}

    def stepper(mode):
        eng = engs[mode]

        def fn():
            eng.step(acts[it[mode] % 16])
            it[mode] += 1
        return fn

    rows = []

    def row(op, k, **extra):
        r = {"workload": workload, "op": op, "envs": n, "repeat": k, **extra}
        rows.append(r)
        print(json.dumps(r), flush=True)

    for k in repeats:
        for eng in engs.values():
            eng.set_action_repeat(k)
        for m in engs:
            for _ in range(20):
                stepper(m)()
        # share of next_step calls that are auto-reset calls (each ended env spends its next call on the reset)
        eng = engs["next_step"]
        ended = torch.zeros((), dtype=torch.int64, device=eng.device)
        calls = 200
        for _ in range(calls):
            stepper("next_step")()
            ended += (eng.terminated | eng.truncated).sum()
        share = float(ended) / (n * calls)
        res = alternating([(m, stepper(m), reps) for m in engs], reps)
        ms_n, b_n = res["next_step"]
        ms_s, b_s = res["same_step"]
        row("next_step", k, ms_per_call=ms_n, blocks_ms=b_n, auto_reset_call_share=share,
            useful_transitions_per_s=n * 1e3 / ms_n * (1.0 - share))
        row("same_step", k, ms_per_call=ms_s, blocks_ms=b_s, useful_transitions_per_s=n * 1e3 / ms_s,
            tail_ms=ms_s - ms_n)
        # the same engine with no final-observation buffer bound: the pass resets and renders, but copies nothing
        same = engs["same_step"]
        E._check(same.lib, same.lib.cbev_bind_final_obs(same.handle, None, 0))
        res = alternating([(m, stepper(m), reps) for m in engs], reps)
        row("same_step_unbound", k, ms_per_call=res["same_step"][0], blocks_ms=res["same_step"][1],
            next_step_ms_per_call=res["next_step"][0], tail_ms=res["same_step"][0] - res["next_step"][0],
            note="same_step without a bound final_obs buffer (no terminal-window copy)")
        E._check(same.lib, same.lib.cbev_bind_final_obs(same.handle, same.final_obs.data_ptr(),
                                                         same.final_obs.numel() * same.final_obs.element_size()))
        for m in engs:
            split = kernel_split(stepper(m), 20)
            row(f"kernel_split_{m}", k, kernels_ms=split, note="device time per call (torch.profiler)")
    for eng in engs.values():
        eng.close()
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="c2,c2u8,c3")
    ap.add_argument("--repeats", default="1,4")
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--c3-pool", type=int, default=128)
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("same_step_bench.py measures on the GPU; no CUDA device found")
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
