#!/usr/bin/env python
"""bench.py -- env-steps/s of the CarlaBEV batched stepping hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # CUDA engine (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the outputs of the last timed step to DIR

Bench line workload (config.workload): BASELINE.json configs[1] -- 4096 envs per GPU, `lead_brake` scenes
(levels 1..3 round-robin, scene_seed = i), continuous actions U([0,1]x[-1,1]x[0,1]) from a seeded
generator, 6-class semantic-mask observations with a 4-frame stack, device auto-reset from the pool.
A "step" is one pass of the hot path over all envs of the rank: k_move -> (k_judge || k_render).
`extra_workloads` in the same JSON line carries configs[2], [3] and [4] at 8192 envs per GPU (under --gpus 8 the
first is the 65536-env configuration BASELINE.json names).
Multi-GPU (torchrun, one rank per GPU): envs shard independently, weak scaling, no data-path
collective; every timed block is bracketed by a barrier + synchronize and the max over ranks is taken.
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

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (obs+reward+done) at N envs, 1/2/4/8 B200; % HBM roofline"
UNIT = "env-steps/s"
POOL_SCENES = 4096
BLOCKS = 5  # timed blocks of exactly K steps each; the median block is reported (SURVEY.md section 8d)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------ scene pools
def _pool_cache_dir():
    import tempfile

    d = os.path.join(tempfile.gettempdir(), "cbev_bench_pools")
    os.makedirs(d, exist_ok=True)
    return d


def _log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')} rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def _host_workers():
    """Host cores one rank may use for scene generation: every rank generates its own share of a pool."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return max(1, min((os.cpu_count() or 1) // world, 32))


def _shared_pool(tag, requests, pad, size=128):
    """Scene pool `tag`, generated once per box by ALL ranks together: rank r builds requests[r::world] on its share
    of the host cores and publishes its part atomically; every rank then assembles the parts in order.  No collective
    is pending while the host works and nobody generates a scene twice.  Parts are cached under $TMPDIR."""
    from carlabev_env_b200.pool import load_pool, save_pool
    from carlabev_env_b200.scenes import build_pool as build

    n = len(requests)
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    base = os.path.join(_pool_cache_dir(), f"pool_{tag}_{n}")
    whole = f"{base}.npz"
    if os.path.exists(whole):
        try:
            return load_pool(whole)
        except Exception as ex:  # noqa: BLE001
            _log(f"cached pool {whole} unreadable ({ex}); rebuilding")
    part = f"{base}.w{world}.r{rank}.npz"
    if not os.path.exists(part):
        t0 = time.time()
        # other map scales: seeds the reference itself cannot reset ("hero_on_obstacle") are left out of the pool
        mine = [sc for sc in build(requests[rank::world], pad=pad, workers=_host_workers(), size=size,
                                   skip_invalid=size != 128) if sc is not None]
        tmp = f"{part}.{os.getpid()}.tmp.npz"
        save_pool(tmp, mine, compress=False)
        os.replace(tmp, whole if world == 1 else part)
        _log(f"pool {tag}: {len(mine)} of {n} scenes generated in {time.time() - t0:.1f} s on {_host_workers()} cores")
        if world == 1:
            return mine
    parts = []
    deadline = time.time() + 900.0
    for r in range(world):
        pr = f"{base}.w{world}.r{r}.npz"
        while not os.path.exists(pr):
            if time.time() > deadline:
                raise RuntimeError(f"rank {rank}: pool part {pr} did not appear within 900 s")
            time.sleep(0.2)
        parts.append(load_pool(pr))
    if size != 128:  # parts have unequal lengths (invalid seeds dropped): concatenate in rank order
        return [sc for part in parts for sc in part]
    scenes = [None] * n
    for r in range(world):
        scenes[r::world] = parts[r]
    return scenes


WORKLOADS = {
    # name: BASELINE.json config it restates (SURVEY.md section 8d); c2 is the bench line, the others are reported extras
    "c2": dict(desc="configs[1]: {N} envs/GPU lead_brake (levels 1-3, pool of {K} seeded scenes), continuous actions, "
                    "6-class semantic masks 96x96 float32, frame_stack 4, CaRL reward, device auto-reset (next-step) "
                    "from the pool", envs=4096, obs="semantic", actions="continuous", anchor=(0.5, 0.5), pool="lead_brake"),
    "c3": dict(desc="configs[2]: {N} envs/GPU rdm rt_hard_v1 (25 vehicles, pool of {K} host-generated scenes, scene_seed = i), "
                    "discrete9 actions, 6-class semantic F=4, auto-reset", envs=8192, obs="semantic",
               actions="discrete", anchor=(0.5, 0.5), pool="rdm_rt_hard_v1"),
    "c4": dict(desc="configs[3]: {N} envs/GPU 50/50 jaywalk (levels 1-4) / red_light_runner, continuous actions, "
                    "6-class semantic F=4, auto-reset from a pool of {K} scenes", envs=8192, obs="semantic",
               actions="continuous", anchor=(0.5, 0.5), pool="mixed_edge"),
    "c5": dict(desc="configs[4]: {N} envs/GPU raw RGB (128,128,3) uint8 obs, lookahead_75 camera, rdm with 50 vehicles "
                    "(pool of {K} host-generated scenes), continuous actions, auto-reset", envs=8192, obs="rgb",
               actions="continuous", anchor=(0.5, 0.75), pool="rdm_dense_50"),
    # SURVEY.md section 8 row f4 (not a BASELINE config): the other map scale the reference can run, EnvConfig.size = 256
    "f4": dict(desc="row f4: {N} envs/GPU at EnvConfig.size=256 (256x256 view of the Town01-256 map, 256 -> 96 area resize), "
                    "rdm with 12 vehicles (pool of {K} host-generated scenes the reference can reset at that scale), "
                    "discrete9 actions, 6-class semantic F=4, auto-reset", envs=4096, obs="semantic", actions="discrete",
               anchor=(0.5, 0.5), pool="rdm_size256", size=256),
}


def workload_pool(name, args):
    """Scene pools at the sizes SURVEY.md section 8(d) names: scene_seed = i, generated on the host cores by
    carlabev_env_b200.scenes (bit-identical to the reference's post-reset state for the same options)."""
    w = WORKLOADS[name]
    if w["pool"] == "lead_brake":         # configs[1]: level = 1 + i % 3, scene_seed = i
        return _shared_pool("lead_brake", [dict(scene="lead_brake", level=1 + i % 3, scene_seed=i)
                                           for i in range(args.pool)], 182)
    if w["pool"] == "rdm_rt_hard_v1":     # configs[2]: K = 4096 scenes, seeds 0..K-1
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options

        return _shared_pool("rdm_rt_hard_v1", [build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1",
                                                                                         scene_seed=i))
                                               for i in range(args.pool)], 182)
    if w["pool"] == "mixed_edge":         # configs[3]: K = 2048, jaywalk levels 1-4 round-robin / red_light_runner
        k = min(args.pool, 2048)
        return _shared_pool("mixed_edge", [dict(scene="jaywalk", level=1 + (i // 2) % 4, scene_seed=i) if i % 2 == 0
                                           else dict(scene="red_light_runner", scene_seed=i) for i in range(k)], 182)
    if w["pool"] == "rdm_size256":        # row f4: seeds 0..511 minus those the reference cannot reset at size 256
        k = min(args.pool, 512)
        return _shared_pool("rdm_size256", [dict(scene="rdm", num_vehicles=12, route_dist_range=(30, 100), scene_seed=i)
                                            for i in range(k)], 363, size=256)
    # configs[4]: rdm with num_vehicles = max_vehicles = 50, lookahead_75 camera (crop 230 px)
    k = min(args.pool, 1024)
    return _shared_pool("rdm_dense_50", [dict(scene="rdm", num_vehicles=50, route_dist_range=(30, 130), scene_seed=i)
                                         for i in range(k)], 230)


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({names[i] for r in self.rows for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(sm), "reasons": reasons}


# ------------------------------------------------------------------------------------ CPU baseline
def _ref_staged():
    return os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "CarlaBEV"))


def _cpu_worker_reference(args):
    """The UNMODIFIED reference (staged copy under oracle/_ref, oracle/make_ref.py) on the pygame / gymnasium shims:
    make_env(RunConfig(num_envs=1)) stepped through its own SyncVectorEnv, masked reset on termination."""
    wid, steps, seed = args[:3]
    workload = args[3] if len(args) > 3 else "c2"
    os.environ["CARLABEV_REFERENCE_ROOT"] = os.path.join(ROOT, "oracle", "_ref")
    from oracle.ref_loader import load_reference

    load_reference()
    from CarlaBEV.config import EnvConfig, RunConfig
    from CarlaBEV.envs import make_env

    f4 = workload == "f4"  # row f4: EnvConfig.size = 256, rdm with 12 vehicles, discrete9 actions
    envs = make_env(RunConfig(env=EnvConfig(render_mode="rgb_array", size=256) if f4 else
                              EnvConfig(render_mode="rgb_array", action_mode="continuous"), num_envs=1))
    rng = np.random.default_rng(seed + wid)
    mask = np.array([True])
    k = wid * 100003
    t_reset = t_step = 0.0

    def do_reset():
        nonlocal k
        while True:
            opts = (dict(scene="rdm", num_vehicles=12, route_dist_range=(30, 100), scene_seed=k) if f4 else
                    dict(scene="lead_brake", level=1 + k % 3, scene_seed=k))
            try:
                envs.reset(options=dict(opts, reset_mask=mask))
                return
            except RuntimeError:  # size 256: a seed the reference cannot reset ("hero_on_obstacle"): take the next one
                k += 1

    t0 = time.perf_counter()
    do_reset()
    t_reset += time.perf_counter() - t0
    n = n_reset = 0
    for _ in range(steps):
        a = (np.array([int(rng.integers(0, 9))]) if f4 else
             np.array([[rng.uniform(0, 1), rng.uniform(-1, 1), rng.uniform(0, 1)]], dtype=np.float32))
        t0 = time.perf_counter()
        _, _, term, trunc, _ = envs.step(a)
        t_step += time.perf_counter() - t0
        n += 1
        if term[0] or trunc[0]:
            k += 1
            n_reset += 1
            t0 = time.perf_counter()
            do_reset()
            t_reset += time.perf_counter() - t0
    return n, t_step, t_reset, n_reset


def _cpu_worker_port(args):
    """Fallback when the staged reference is absent: the oracle port (NumPy restatement of the reference step)."""
    wid, steps, seed = args[:3]
    from carlabev_env_b200.scenes import build_scripted_scene
    from carlabev_env_b200.vector_env import load_town01_map
    from oracle.env import OracleEnv

    cls = load_town01_map()
    rng = np.random.default_rng(seed + wid)
    scenes = [build_scripted_scene("lead_brake", wid * 64 + i, level=1 + i % 3, cls_map=cls) for i in range(8)]
    env = OracleEnv(cls, obs_mode="bev_semantic", semantic_mask_ch="6-class", frame_stack=4, action_mode="continuous")
    env.reset(scenes[0])
    t_reset = t_step = 0.0
    n = k = 0
    for _ in range(steps):
        a = np.array([rng.uniform(0, 1), rng.uniform(-1, 1), rng.uniform(0, 1)], dtype=np.float32)
        t0 = time.perf_counter()
        _, _, term, trunc, _ = env.step(a)
        t_step += time.perf_counter() - t0
        n += 1
        if term or trunc:
            k += 1
            t0 = time.perf_counter()
            env.reset(scenes[(k + wid) % len(scenes)])
            t_reset += time.perf_counter() - t0
    return n, t_step, t_reset, k


def cpu_baseline(steps_per_env=1500, max_workers=None, workload="c2"):
    """The reference's CPU path on all host cores: one single-env process per core (AsyncVectorEnv-style pool),
    step-only throughput = steps / slowest worker's time inside step(); reset time is reported separately."""
    import multiprocessing as mp

    cores = os.cpu_count() or 1
    workers = min(cores, max_workers or 64)
    staged = _ref_staged()
    if workload != "c2" and not staged:
        return None  # the oracle port is only wired for the bench line's workload
    fn = _cpu_worker_reference if staged else _cpu_worker_port
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(workers) as pool:
        res = pool.map(fn, [(w, steps_per_env, 1234, workload) for w in range(workers)])
    wall = time.perf_counter() - t0
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    resets = sum(r[3] for r in res)
    reset_s = sum(r[2] for r in res)
    what = ("the UNMODIFIED reference (byte-for-byte copy staged by oracle/make_ref.py) running on oracle/shims "
            "(pygame-lite / gymnasium-lite; neither library is installable in this image): make_env(num_envs=1) "
            "-> SyncVectorEnv.step" if staged else
            "oracle/ (NumPy port of the reference step incl. render/resize/masks/stack; no staged reference found)")
    return {"value": total / slowest, "unit": UNIT, "cores": workers, "kind": "reference-on-shims" if staged else "port",
            "reset_seconds_mean": reset_s / max(resets, 1), "resets": resets,
            "sample": f"{workers} worker processes x 1 env x {steps_per_env} steps of the " +
                      ("row-f4 workload (EnvConfig.size=256, rdm with 12 vehicles, discrete9, 6-class F=4)" if workload == "f4"
                       else "configs[1] workload (lead_brake, continuous actions, 6-class F=4)") +
                      f" through {what}; throughput = steps / slowest worker's time "
                      f"inside step() ({slowest:.1f} s; resets excluded and reported as reset_seconds_mean; wall incl. "
                      f"process spawn {wall:.1f} s); host has {cores} cores"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps_per_env = max(500, min(3000, args.steps * 3))  # bounded sample: roughly 5-25 s of stepping per core
    cb = cpu_baseline(steps_per_env=steps_per_env)
    n_env = cb["cores"]
    line = {
        "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * n_env / cb["value"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
        "config": {"workload": "configs[1] bounded sample: lead_brake, continuous actions, 6-class semantic F=4; "
                               f"{n_env} CPU envs (one per worker process)", "envs": n_env},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ the CUDA arm
class Ctx:
    """Process-wide plumbing: ranks, device, barrier."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def _timed_block(ctx, fn, steps):
    """EXACTLY `steps` calls of fn(i) between CUDA events on the launch stream, barrier + synchronize on both sides,
    max over ranks.  Returns milliseconds."""
    torch = ctx.torch
    stream = torch.cuda.current_stream(ctx.dev)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        fn(i)
    e1.record(stream)
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1))


DUMP_ENVS = 16384          # envs whose reward / flags / hero / episode rows are written (all of them up to this many)
DUMP_OBS_BYTES = 48 << 20  # observation windows are GBs: a sample of whole windows up to this size is written


def dump_outputs(out_dir, eng):
    """Write what a caller of Engine.step holds after the last step (observation window, reward, terminated,
    truncated, cause, hero and episode blocks) to out_dir/<name>.npy in float32 / float64, at most 64 MB in all.
    Envs are sampled by a fixed seed; obs_env_ids / env_ids name the sampled envs."""
    torch = eng.torch
    torch.cuda.synchronize(eng.device)
    obs = eng.obs()
    perm = np.random.default_rng(0).permutation(eng.N)
    env_ids = np.sort(perm[:DUMP_ENVS])
    obs_env_ids = np.sort(perm[:max(1, DUMP_OBS_BYTES // (obs[0].numel() * 4))])
    sel = torch.from_numpy(env_ids).to(eng.device)
    out = {"obs": obs[torch.from_numpy(obs_env_ids).to(eng.device)].float(),
           "obs_env_ids": obs_env_ids.astype(np.float64), "env_ids": env_ids.astype(np.float64),
           "reward": eng.reward[sel], "terminated": eng.terminated[sel].float(), "truncated": eng.truncated[sel].float(),
           "cause": eng.cause[sel].float(), "hero": eng.hero[sel], "episode": eng.episode[sel]}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.cpu().numpy() if torch.is_tensor(v) else v)
    _log(f"dumped {', '.join(out)} of the last timed step to {out_dir}")


def run_workload(ctx, name, args, with_cpu_baseline=False, dump_dir=None):
    torch = ctx.torch
    from carlabev_env_b200.config import EnvConfig, RunConfig
    from carlabev_env_b200.distributed import allreduce_stats, summarize_stats
    from carlabev_env_b200.vector_env import make_env

    world, rank, local, dev = ctx.world, ctx.rank, ctx.local, ctx.dev
    W = WORKLOADS[name]
    N = args.envs or W["envs"]
    K, Wm = args.steps, args.warmup
    scenes = workload_pool(name, args)
    _log(f"{name}: pool ready ({len(scenes)} scenes)")
    a_mean = float(np.mean([len(s["act_kind"]) for s in scenes]))
    discrete = W["actions"] == "discrete"
    semantic = W["obs"] == "semantic"
    ring_slots = args.ring_slots
    if ring_slots is None and semantic:
        # spend HBM on the observation ring: a longer ring wraps (and mirrors F-1 frames) less often;
        # up to 96 slots within half of the free memory (87 GB at 4096 envs)
        free, _ = torch.cuda.mem_get_info(local)
        ring_slots = int(max(8, min(96, (free // 2) // (N * 6 * 96 * 96 * 4))))
    # The product surface: the VectorEnv make_env returns (device auto-reset on); the device-resident legs drive its
    # engine through the C ABI directly, the e2e_vector_env leg goes through VectorEnv.step itself.
    cfg = RunConfig(env=EnvConfig(obs_mode="bev_semantic" if semantic else "bev_rgb",
                                  action_mode="discrete" if discrete else "continuous",
                                  ego_anchor_x_frac=W["anchor"][0], ego_anchor_y_frac=W["anchor"][1],
                                  size=W.get("size", 128)),
                    num_envs=N, seed=rank)
    envs = make_env(cfg, scenes=scenes, autoreset="next_step", device=local, ring_slots=ring_slots,
                    raw_rgb=not semantic, host_infos=True)
    eng = envs.engine
    if args.debug_flags:
        eng.set_debug_flags(args.debug_flags)
    frame_bytes = eng.frame_bytes
    ids = ((torch.arange(N, dtype=torch.int64) + rank * N) % len(scenes)).numpy()
    pool_note = "host generator (carlabev_env_b200/scenes.py), bit-identical to the reference's post-reset state"
    if args.device_pool and name == "c2":
        k = len(scenes)
        att = eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
        pool_note = (f"generated on the device (cbev_generate_scenes; {int((att > 1).sum())} of {k} scenes needed a retry): "
                     "draws bit-identical to the reference, smoothed routes within 1e-9 px")
    envs.reset(options={"scene_ids": ids})
    gen = torch.Generator(device="cpu").manual_seed(0 + rank)
    bank = 16
    if discrete:
        acts_host = [torch.randint(0, 9, (N,), generator=gen, dtype=torch.int64).pin_memory() for _ in range(bank)]
    else:
        lo = torch.tensor([0.0, -1.0, 0.0])
        hi = torch.tensor([1.0, 1.0, 1.0])
        acts_host = [(lo + (hi - lo) * torch.rand(N, 3, generator=gen)).float().pin_memory() for _ in range(bank)]
    if args.brake:  # diagnostic: full brake -> the ego stands still, no episode ends, no reset frames are written
        for a in acts_host:
            if not discrete:
                a[:, 0] = 0.0
                a[:, 1] = 0.0
                a[:, 2] = 1.0
            else:
                a[:] = 2
    acts_dev = [a.to(dev) for a in acts_host]
    acts_np = [a.numpy() for a in acts_host]
    stream = torch.cuda.current_stream(dev)

    def episodes_now():
        return float(eng.read_stats()[0].item())

    # ---- device-resident throughput ("value"): BLOCKS blocks of exactly K steps, median block ----
    for i in range(Wm):
        eng.step(acts_dev[i % bank])
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = eng.launches
    ep0 = episodes_now()
    blocks_ms = [_timed_block(ctx, lambda i: eng.step(acts_dev[i % bank]), K) for _ in range(BLOCKS)]
    launches = (eng.launches - l0) // BLOCKS
    resets_in_blocks = (episodes_now() - ep0) / BLOCKS   # every finished episode costs one auto-reset pass next step
    ms_med = statistics.median(blocks_ms)
    value = world * N * K / (ms_med * 1e-3)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, eng)
    # ---- one more block of K steps with CUDA events around every kernel (the roofline leg) ----
    eng.profile(True)
    prof_ms = _timed_block(ctx, lambda i: eng.step(acts_dev[i % bank]), K)
    move_ms, render_ms, judge_ms, prof_steps = eng.profile_read()
    eng.profile(False)
    n_prof = max(prof_steps, 1)
    move_avg, render_avg, judge_avg = move_ms / n_prof, render_ms / n_prof, judge_ms / n_prof

    # ---- e2e through the C ABI with HOST buffers (H2D actions, D2H reward/flags, stream synchronize every step) ----
    out_h = torch.zeros(N * 10, dtype=torch.uint8).pin_memory()   # reward f64[N] | terminated u8[N] | truncated u8[N]
    rew_h, term_h, trunc_h = out_h[: N * 8].view(torch.float64), out_h[N * 8: N * 9], out_h[N * 9:]
    chk = [0.0]

    def e2e_step(i):
        eng.step_host(acts_host[i % bank], rew_h, term_h, trunc_h)
        stream.synchronize()  # the host consumes reward / done before it can act again
        chk[0] += float(rew_h[0])

    for i in range(3):
        e2e_step(i)
    e2e_ms = statistics.median([_timed_block(ctx, e2e_step, K) for _ in range(3)])
    e2e_value = world * N * K / (e2e_ms * 1e-3)

    # ---- e2e through the reference-facing boundary: VectorEnv.step(host numpy actions) with host infos ----
    seen = [0]

    def venv_step(i):
        _, _, te, tr, infos = envs.step(acts_np[i % bank])
        stream.synchronize()
        if "episode" in infos:
            seen[0] += int(infos["_episode"].sum())

    for i in range(3):
        venv_step(i)
    venv_ms = statistics.median([_timed_block(ctx, venv_step, K) for _ in range(3)])
    venv_value = world * N * K / (venv_ms * 1e-3)

    def venv_step_pipelined(i):  # what step() itself waits for: the host copies, not the raster kernel
        _, _, te, tr, infos = envs.step(acts_np[i % bank])

    venv_pipe_ms = statistics.median([_timed_block(ctx, venv_step_pipelined, K) for _ in range(3)])
    venv_pipe_value = world * N * K / (venv_pipe_ms * 1e-3)

    clock_info = clocks.stop() if clocks else None   # sampled under load over every timed leg of this workload
    # ---- episode statistics: the only collective (all-reduce of a 21-double vector over NCCL) ----
    stats = summarize_stats(allreduce_stats(eng.read_stats().clone()))
    res = None
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        alg_bytes = N * frame_bytes
        achieved = alg_bytes / (render_avg * 1e-3) / 1e9 if render_avg > 0 else 0.0
        step_ms = ms_med / K
        traffic, traffic_source = None, None
        tp = os.path.join(ROOT, "profiles", "render_traffic.json")
        if os.path.exists(tp):
            try:
                with open(tp) as f:
                    tj = json.load(f)
                ent = tj.get(name) or {}
                traffic, traffic_source = ent.get("dram_bytes_per_launch"), ent.get("source")
            except Exception:  # noqa: BLE001
                pass
        Fs = 4
        resets_per_env_step = resets_in_blocks / (N * K)
        mirror_share = (Fs - 1) / max(eng.L - Fs + 1, 1) if semantic else 0.0
        written_est = alg_bytes * (1.0 + (Fs - 1) * resets_per_env_step + mirror_share) if semantic else alg_bytes
        res = {
            "value": value, "ms_per_step": step_ms, "blocks_ms": blocks_ms,
            "reset_steps_in_value": resets_in_blocks * world,
            "reset_steps_note": "env-steps of the median-sized block that were device auto-reset passes (NEXT_STEP "
                                "semantics: the step after a terminal one resets and renders the reset frame); they are "
                                "counted in `value` like any other step",
            "value_excluding_reset_steps": world * (N * K - resets_in_blocks) / (ms_med * 1e-3),
            "config": {"workload": W["desc"].format(N=N, K=len(scenes)), "envs_per_gpu": N, "envs_total": world * N,
                       "ring_slots": eng.L, "mean_actors_per_scene": a_mean, "pool": pool_note,
                       "l2": f"each step writes {alg_bytes / 1e6:.0f} MB of observations per GPU (> 126 MB L2), "
                             "no flush needed"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_source,
                         "kernel": "k_render" if W.get("size", 128) == 128 else "k_render_any", "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "written_bytes_per_launch_estimate": written_est,
                         "kernel_ms": render_avg, "sim_kernel_ms": move_avg, "judge_kernel_ms": judge_avg,
                         "judge_note": "k_judge runs on a side stream concurrently with k_render",
                         "profiled_steps": n_prof, "profiled_block_ms_per_step": prof_ms / K,
                         "launches_per_step": launches / K,
                         "step_frac": alg_bytes / (step_ms * 1e-3) / 1e9 / peak if peak else None,
                         "step_frac_note": "algorithmic bytes / whole-step time / peak (all three kernels and gaps)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": N * (8 if discrete else 12),
                    "d2h_bytes_per_step": N * 10,
                    "note": "cbev_step_host: pinned host actions in, reward/terminated/truncated out, stream synchronize "
                            "every step; observations stay device resident (ring view)"},
            "e2e_vector_env": {"value": venv_value, "unit": UNIT, "h2d_bytes_per_step": N * (8 if discrete else 12),
                               "d2h_bytes_per_step": N * 10 + N * 16 * 8, "ratio_to_e2e": venv_value / e2e_value,
                               "pipelined_value": venv_pipe_value, "terminal_infos_seen": seen[0],
                               "note": "make_env-style CarlaBEVVectorEnv(autoreset='next_step', host_infos=True).step("
                                       "host numpy actions): rewards / flags / episode block to the host, terminal infos "
                                       "built, stream synchronize every step; pipelined_value = without that extra "
                                       "synchronize (step() itself waits for the host copies only)"},
            "gpu_launches": int(launches),
            "clocks": clock_info,
            "episode_stats": stats,
        }
        if with_cpu_baseline:
            res["cpu_baseline"] = cpu_baseline(steps_per_env=args.cpu_steps)
        elif name == "f4" and world == 1 and not args.no_cpu_baseline:
            # the other map scale has no published number anywhere: time the reference's own path beside it (short sample)
            cb = cpu_baseline(steps_per_env=max(100, args.cpu_steps // 5), workload="f4")
            if cb is not None:
                res["cpu_baseline"] = cb
    envs.close()
    del envs, eng, acts_dev
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    ctx = Ctx()
    t_start = time.time()
    main = run_workload(ctx, args.workload, args, with_cpu_baseline=(ctx.world == 1 and not args.no_cpu_baseline),
                        dump_dir=args.dump_outputs)
    extras = []
    if args.workload == "c2" and not args.no_extras:
        for name in ("c3", "c4", "c5", "f4"):
            # every rank must take the same decision: the budget is checked on rank 0's clock
            flag = ctx.torch.tensor([1.0 if time.time() - t_start < args.extras_budget else 0.0], device=ctx.dev)
            if ctx.world > 1:
                ctx.dist.broadcast(flag, src=0)
            if flag.item() < 0.5:
                extras.append({"name": name, "skipped": f"time budget of {args.extras_budget:.0f} s spent"})
                continue
            try:
                r = run_workload(ctx, name, args)
            except Exception as ex:  # noqa: BLE001
                if ctx.world > 1:
                    raise
                r = {"error": repr(ex)[:300]}
            if ctx.rank == 0:
                extras.append({"name": name, **{k: r[k] for k in r if k != "clocks"}} if r else {"name": name})
    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "timing": f"median of {BLOCKS} blocks of exactly {args.steps} steps (CUDA events on the launch stream, barrier "
                      "+ synchronize on both sides of every block, max over ranks)",
        }
        line.update({k: v for k, v in main.items() if k not in ("value", "ms_per_step")})
        if extras:
            line["extra_workloads"] = extras
        print(json.dumps(line), flush=True)
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the workload's)")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS), help="BASELINE.json config; c2 is the bench line")
    ap.add_argument("--pool", type=int, default=POOL_SCENES)
    ap.add_argument("--ring-slots", type=int, default=None)
    ap.add_argument("--cpu-steps", type=int, default=1500,
                    help="reference steps per worker process for cpu_baseline (about 10-15 s of CPU work per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip extra_workloads (configs[2..4])")
    ap.add_argument("--extras-budget", type=float, default=240.0,
                    help="seconds after which no further extra workload is started")
    ap.add_argument("--brake", action="store_true", help="diagnostic: constant full-brake actions (no resets)")
    ap.add_argument("--device-pool", action="store_true",
                    help="c2 only: generate the lead_brake pool ON THE DEVICE (cbev_generate_scenes) instead of on the host")
    ap.add_argument("--debug-flags", type=int, default=0,
                    help="diagnostic (cbev_set_debug_flags): 2 = k_judge serial on the main stream, 32 = identity CTA order")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: after the timed steps of --workload (not of the extra workloads), write what its "
                         "last step computed to DIR/<name>.npy (rank 0's envs; a seeded sample of the observation windows)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA engine: it needs --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
