"""Snapshot / restore throughput (Engine.snapshot / Engine.restore) on the c2 workload, float32 and uint8 masks.

c2: 4096 envs, lead_brake levels 1-3 (a pool of 1024 scenes generated on the device), continuous actions, 6-class
96 x 96 masks, F = 4, ring of 16 slots, device auto-reset.  For each mask dtype, in one process:

  snapshot   whole batch: every env -> its row
  restore    whole batch: row i -> env i
  clone      row 0 -> every env (the rows are read from L2 after the first env; the cost is the writes)
  plan       one planning iteration: clone, H steps, restore the whole batch

Each is timed over --reps calls between CUDA events, median of 5 blocks; every working set is far larger than the
126 MB L2.  Bytes moved are counted from the row layout: a snapshot reads the window frames and state of every env and
writes the rows; a restore reads the rows it uses (one for a clone) and writes the state, the frames and the mirror
copies of the frames that land in the mirror zone (L - F + 1 <= slot).  The copy peak is measured in the same process:
a device-to-device cudaMemcpyAsync (torch copy_) of a buffer as large as one snapshot, 2 bytes moved per byte copied.

    python tools/snapshot_bench.py [--envs 4096] [--reps 20] [--horizon 16] [--out FILE]

Prints one JSON object per row and, with --out, writes them all plus the card's name, power limit and maximum SM clock
(nvidia-smi, read in the same process)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BLOCKS = 5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def timed(fn, reps):
    """Median over BLOCKS blocks of `reps` calls, ms per call (CUDA events, synchronised)."""
    import torch

    out = []
    for _ in range(BLOCKS):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / reps)
    return statistics.median(out), out


def copy_peak_gbs(nbytes, reps):
    import torch

    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms, _ = timed(lambda: dst.copy_(src), reps)
    del src, dst
    torch.cuda.empty_cache()
    return 2 * nbytes / (ms * 1e-3) / 1e9


def make_engine(n, dtype, ring_slots):
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    k = 1024
    eng = E.Engine(n, mask_mode="6-class", frame_stack=4, ring_slots=ring_slots, action_mode=E.ACTION_CONTINUOUS,
                   autoreset=E.AUTORESET_NEXT_STEP, max_actors=4, seed=0, mask_dtype=dtype)
    eng.upload_map(load_town01_map(128))
    eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    eng.reset(torch.arange(n, dtype=torch.int32) % k)
    g = torch.Generator(device="cpu").manual_seed(0)
    lo, hi = torch.tensor([0.0, -1.0, 0.0]), torch.tensor([1.0, 1.0, 1.0])
    acts = [(lo + (hi - lo) * torch.rand(n, 3, generator=g)).float().cuda() for _ in range(16)]
    return eng, acts


def mirrored_frames(eng):
    """Window frames a restore at the current head also writes to a mirror slot."""
    if eng.F == 1:
        return 0
    return sum(1 for k in range(eng.F) if eng.head - eng.F + 1 + k >= eng.L - eng.F + 1)


def run(dtype, n, reps, horizon, ring_slots, peak):
    import torch

    eng, acts = make_engine(n, dtype, ring_slots)
    for i in range(20):
        eng.step(acts[i % len(acts)])
    rb = eng.snapshot_row_bytes
    frames = eng.F * eng.frame_bytes
    state = rb - frames
    snap = eng.snapshot()
    one = eng.snapshot(env_ids=[0])
    zeros = torch.zeros(n, dtype=torch.int32, device=eng.device)
    rows = []

    def row(op, ms, blocks, nbytes, note):
        r = {"op": op, "mask_dtype": dtype, "envs": n, "row_bytes": rb, "state_bytes_per_row": state,
             "frame_bytes": eng.frame_bytes, "F": eng.F,
             "ring_slots": eng.L, "ms": ms, "blocks_ms": blocks, "bytes_moved": nbytes,
             "gbs": nbytes / (ms * 1e-3) / 1e9 if nbytes else None,
             "share_of_copy_peak": nbytes / (ms * 1e-3) / 1e9 / peak if nbytes else None, "note": note}
        rows.append(r)
        print(json.dumps(r), flush=True)

    ms, b = timed(lambda: eng.snapshot(out=snap), reps)
    row("snapshot", ms, b, 2 * n * rb, "reads window + state, writes rows")
    m = mirrored_frames(eng)
    writes = n * (rb + m * eng.frame_bytes)
    ms, b = timed(lambda: eng.restore(snap), reps)
    row("restore", ms, b, n * rb + writes, f"reads rows, writes state + window + {m} mirror frame(s) per env")
    ms, b = timed(lambda: eng.restore(one, rows=zeros), reps)
    row("clone_1_to_n", ms, b, rb + writes, "one row read (L2), every env written")

    def plan():
        eng.restore(one, rows=zeros)
        for i in range(horizon):
            eng.step(acts[i % len(acts)])
        eng.restore(snap)

    # H steps change the head: the mirror count of the last restore varies, bytes are not stated for this row
    ms, b = timed(plan, max(1, reps // 4))
    row(f"plan_clone_h{horizon}_restore", ms, b, 0, f"clone + {horizon} steps + whole-batch restore, ms per iteration")

    def steps_only():
        for i in range(horizon):
            eng.step(acts[i % len(acts)])

    ms, b = timed(steps_only, max(1, reps // 4))
    row(f"steps_h{horizon}", ms, b, 0, f"{horizon} steps alone, for comparison with the planning row")
    eng.close()
    del snap, one
    torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--horizon", type=int, default=16)
    ap.add_argument("--ring-slots", type=int, default=16)
    ap.add_argument("--dtypes", default="float32,uint8")
    ap.add_argument("--out", default=None, help="also write the JSON document (rows, card, copy peak) to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("snapshot_bench.py measures on the GPU; no CUDA device found")
    info = gpu_info()
    doc = {"gpu": info, "envs": args.envs, "reps": args.reps, "blocks": BLOCKS, "horizon": args.horizon, "copy_peak": {},
           "rows": []}
    print(json.dumps({"gpu": info}), flush=True)
    for dt in args.dtypes.split(","):
        # the copy peak at the size of this dtype's whole-batch snapshot
        frame = 6 * 96 * 96 * (1 if dt == "uint8" else 4)
        peak = copy_peak_gbs(args.envs * 4 * frame, args.reps)
        doc["copy_peak"][dt] = {"bytes_copied": args.envs * 4 * frame, "gbs": peak}
        print(json.dumps({"copy_peak_gbs": peak, "mask_dtype": dt}), flush=True)
        doc["rows"] += run(dt, args.envs, args.reps, args.horizon, args.ring_slots, peak)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
