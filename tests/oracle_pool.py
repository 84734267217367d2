"""A pool of worker processes, each owning a slice of `OracleEnv`s, so that the scale-parity GPU tests step their
64-env oracle sample on all host cores instead of one (the oracle costs ~10 ms per env-step).  TEST INFRASTRUCTURE.

Protocol per call: the parent sends every worker a list of commands, one per env it owns --
("reset", scene_index), ("step", action), ("repeat", (action, K)) or None (leave the env alone) -- and gets back, per
env, a dict with the stacked observation, reward, flags, ego pose, actor poses, the hero block (`hero_vector`), the
cause and, on a terminal step, the episode row (`episode_vector`) after the command (None for a None command).

("repeat", (action, K)) is one agent step of action repeat K (Engine.set_action_repeat): up to K simulator steps with
the same action, stopping at the first terminated or truncated sub-step j.  Its dict holds the rewards summed in
order from r1 as Python floats, `j`, and everything else of sub-step j; only sub-step j is rendered.

Branch commands (the oracle side of Engine.lookahead; state never crosses processes, so branches from env r run on
r's worker):
  ("save", tag)       keep a deep copy of the env's current state (and scene index) under `tag`.
  ("branches", (tag, actions, K, keep))
                      one branch per action sequence actions[m] ([H, ...]), each from a deep copy of the env (tag None)
                      or of its copy under `tag`: up to H agent steps (`step` at K = 1, `_repeat`'s loop at K > 1),
                      stopping after the first terminated or truncated one.  Returns per branch a dict: per agent step
                      `reward` (the in-order sum at K > 1), `term`, `trunc`, `cause` and `j`; after the last step
                      taken `hero`, `episode` (when it terminated), `steps`, `header` (scene, episode count, ended), and with frames (see below) `obs` (the
                      observation in the env's form) and `frames` (np.stack of the raw frame stack); `retreat`, the
                      first agent step after which a pedestrian had started a retreat route (None if none did).
                      `keep` is None or one key per branch: the leaf copy is kept under that key, a valid `tag` of a
                      later call.  Only the last F agent steps of a branch are rendered, and only when `keep` is set
                      or `frames` (a fifth element, default False) asks for the observation.  Nothing the branches
                      copy from is changed.
  ("adopt", key)      replace the env by its kept copy `key`, scene index included."""
from __future__ import annotations

import copy
import multiprocessing as mp
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def hero_vector(env, scene_index):
    """The engine's hero block (engine.HERO_FIELDS order, csrc/sim.cu judge_body) from the oracle's state after a step."""
    s = env.sim
    e, last, ctl, cf = s.ego, s.last, s.control, s.comfort
    t = e.tidx
    return np.array([
        e.x, e.y, e.yaw, e.v,                      # x, y, yaw, v
        e.x_1, e.y_1, e.yaw_1, e.v_1,              # x_1, y_1, yaw_1, v_1
        last["dist2wp"],                           # dist2wp
        e.cx[t], e.cy[t], e.cyaw[t],               # set_point_x, set_point_y, set_point_yaw
        ctl["cmd_gas"], ctl["cmd_steer"], ctl["cmd_brake"],
        ctl["applied_delta"],
        cf["speed_mps"], cf["accel_long"], cf["accel_lat"], cf["jerk_long"], cf["jerk_lat"], cf["yaw_rate"],
        cf["yaw_acc"],
        s.acc,                                     # acc
        t,                                         # target_idx
        last["hit"], last["hit_id"], last["tile"], last["n_nearby"],
        s.dist2goal,                               # dist2goal
        s.t,                                       # t
        scene_index,                               # scene
    ], dtype=np.float64)


def reset_hero_vector(env, scene_index):
    """The hero block of a device auto-reset step (csrc/sim.cu auto_reset_env): zeros but the post-reset pose and scene."""
    h = np.zeros(32, dtype=np.float64)
    e = env.sim.ego
    h[:4] = e.x, e.y, e.yaw, e.v
    h[31] = scene_index
    return h


def episode_vector(info, scene_index):
    """info["episode_info"] of a terminal step as the engine's episode row (engine.EPISODE_FIELDS order)."""
    from oracle.sim import CAUSE_NAMES

    return np.array([info["return"], info["length"], CAUSE_NAMES.index(info["termination"]), info["mean_speed"],
                     info["mean_abs_accel_long"], info["mean_abs_accel_lat"], info["mean_abs_jerk_long"],
                     info["mean_abs_jerk_lat"], info["mean_abs_yaw_rate"], info["mean_abs_yaw_acc"],
                     info["comfort_violation_rate"], info["harsh_brake_rate"], scene_index, info["num_vehicles"],
                     info["len_ego_route"], info["episode"]], dtype=np.float64)


def active_terms(env):
    """Which reward terms of the step just taken were active, from the oracle's state (oracle/sim.py carl_reward /
    shaping_reward): name -> bool.  The reward-parameter tests count these to prove that each parameter was exercised."""
    from carlabev_env_b200.config import CARL_DEFAULTS, SHAPING_DEFAULTS
    from oracle.sim import (CAUSE_MAX_ACTIONS, CAUSE_NONE, CAUSE_OFFROAD, CLS_SIDEWALK, LANE_HALF_WIDTH_M, MPP,
                            SPEED_LIMIT)

    s = env.sim
    p = {**CARL_DEFAULTS, **SHAPING_DEFAULTS, **s.rp}
    cause, tile = s.last["cause"], s.last["tile"]
    h = s.hero_info()
    x, y, yaw, v = h["state"]
    lat = abs(s._lateral_error(x, y, *h["next_wps"]))
    body = cause == CAUSE_NONE  # the branch that evaluates the parameterised terms was reached
    if env.reward_mode == "carl":
        dist_m = lat * MPP
        over = v * MPP - SPEED_LIMIT / 3.6
        return dict(
            lane=body and dist_m > 0,
            lane_floor=body and dist_m > 0 and 1.0 - (dist_m / LANE_HALF_WIDTH_M) ** p["lane_center_exponent"]
            < p["lane_center_floor"],
            off_lane=body and (tile == CLS_SIDEWALK or dist_m > 1.5 * LANE_HALF_WIDTH_M),
            speeding=body and over > 0,
            speed_floor=body and over > 0 and np.exp(-over / p["speed_penalty_scale"]) < p["speed_penalty_floor"],
            ttc=body and s._ttc_raw(h["state"], s.last["nearby"], MPP) < p["ttc_threshold"])
    yaw_error = np.arctan2(np.sin(h["set_point"][2] - yaw), np.cos(h["set_point"][2] - yaw))
    sidewalk = tile == CLS_SIDEWALK
    return dict(
        sidewalk=cause in (CAUSE_NONE, CAUSE_OFFROAD) and sidewalk,
        offroad_term=cause == CAUSE_OFFROAD,
        route_dev=body and h["dist2wp"] > p["route_dev_start"],
        lat_clip=body and lat > p["lat_clip"],
        align=body and min(lat, p["lat_clip"]) < p["lat_small"] and abs(yaw_error) < p["yaw_small"],
        flow_cap=body and not sidewalk and v > p["max_speed_for_flow"],
        reverse=body and v < -0.1,
        truncation=cause == CAUSE_MAX_ACTIONS)


def _substeps(env, action, K):
    """Sub-steps 1..j of one agent step at action repeat K, none rendered: reward sum, terminated, truncated, info of
    sub-step j, and j."""
    total = 0.0
    for j in range(1, K + 1):
        _, r, te, tr, info = env.step(action, render=False)
        total += float(r)
        if te or tr:
            break
    return total, te, tr, info, j


def _repeat(env, action, K):
    """One agent step at action repeat K (see the module doc): obs, reward sum, terminated, truncated, info of sub-step
    j, and j."""
    total, te, tr, info, j = _substeps(env, action, K)
    return env.push_frame(), total, te, tr, info, j


def _copy(env):
    """Deep copy of an OracleEnv that shares the immutable map, FOV mask and scene arrays (a class map of scale 256 is
    5 MB; a branch needs none of its own)."""
    memo = {}
    for shared in (env.cls_map, env.fov_mask, env.geom, getattr(env.sim, "scene", None)):
        if shared is not None:
            memo[id(shared)] = shared
    return copy.deepcopy(env, memo)


def _retreating(env):
    return {k for k, a in enumerate(env.sim.actors) if getattr(a, "retreat_goal", None) is not None}


def _branch(env, scene_index, actions, K, render):
    """One branch on `env` (a copy: it is stepped in place), see ("branches", ...) in the module doc."""
    from oracle import raster

    before = _retreating(env)
    out = dict(reward=[], term=[], trunc=[], cause=[], j=[], retreat=None, episode=None)
    drawn = []  # (x, y, yaw, rects) of the agent steps whose frames the leaf window keeps
    for t, a in enumerate(actions):
        r, te, tr, info, j = _substeps(env, a, K)
        out["reward"].append(r)
        out["term"].append(bool(te))
        out["trunc"].append(bool(tr))
        out["cause"].append(int(env.sim.last["cause"]))
        out["j"].append(j)
        if render:
            e = env.sim.ego
            drawn = (drawn + [(e.x, e.y, e.yaw, raster.draw_list(env.sim))])[-env.frame_stack:]
        if out["retreat"] is None and _retreating(env) - before:
            out["retreat"] = t
        if te:
            out["episode"] = episode_vector(info["episode_info"], scene_index)
        if te or tr:
            break
    out["steps"] = len(out["reward"])
    for x, y, yaw, rects in drawn:  # what push_frame would have rendered after each of these agent steps
        env.frames.append(env._wrap_frame(raster.render_fov(env.cls_map, env.geom, x, y, yaw, rects, env.fov_mask)))
    out["hero"] = hero_vector(env, scene_index)
    out["header"] = (scene_index, env.episode, bool(out["term"] and (out["term"][-1] or out["trunc"][-1])))
    if render:
        out["obs"] = env._stacked()
        out["frames"] = np.stack(list(env.frames))
    return out


def _worker(conn, scenes, oracle_kw, n_envs, size):
    for p in (ROOT, os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    from golden_util import load_map
    from oracle.env import OracleEnv

    cls = load_map(size)
    envs = [OracleEnv(cls, size=size, **oracle_kw) for _ in range(n_envs)]
    scene_of = [-1] * n_envs
    kept = [{} for _ in range(n_envs)]  # per env: tag -> (copy, scene index), saved states and kept branch leaves
    while True:
        cmds = conn.recv()
        if cmds is None:
            break
        out = []
        for j, (env, cmd) in enumerate(zip(envs, cmds)):
            if cmd is None:
                out.append(None)
                continue
            op, arg = cmd
            if op == "save":
                kept[j][arg] = (_copy(env), scene_of[j])
                out.append(dict(scene=scene_of[j]))
                continue
            if op == "adopt":
                src, scene_of[j] = kept[j][arg]
                envs[j] = _copy(src)
                out.append(dict(scene=scene_of[j]))
                continue
            if op == "branches":
                tag, acts, K, keep = arg[:4]
                frames = len(arg) > 4 and bool(arg[4])
                root, scene = (env, scene_of[j]) if tag is None else kept[j][tag]
                res = []
                for m, a in enumerate(acts):
                    leaf = _copy(root)
                    res.append(_branch(leaf, scene, a, int(K), render=frames or keep is not None))
                    if keep is not None:
                        kept[j][keep[m]] = (leaf, scene)
                out.append(res)
                continue
            if op == "reset":
                scene_of[j] = int(arg)
                res = dict(obs=env.reset(scenes[int(arg)]), reward=0.0, term=False, trunc=False, cause=0,
                           hero=reset_hero_vector(env, scene_of[j]), episode=None)
            else:
                if op == "repeat":
                    o, r, te, tr, info, sub = _repeat(env, *arg)
                else:
                    o, r, te, tr, info = env.step(arg)
                res = dict(obs=o, reward=float(r), term=bool(te), trunc=bool(tr), cause=int(env.sim.last["cause"]),
                           hero=hero_vector(env, scene_of[j]),
                           episode=episode_vector(info["episode_info"], scene_of[j]) if te else None)
                if op == "repeat":
                    res["j"] = sub
                else:
                    res["terms"] = active_terms(env)
            e = env.sim.ego
            res["ego"] = np.array([e.x, e.y, e.yaw, e.v])
            res["actors"] = np.array([[b.x, b.y, b.yaw, b.v] for b in env.sim.actors]).reshape(-1, 4)
            out.append(res)
        conn.send(out)
    conn.close()


class OraclePool:
    def __init__(self, n_envs, scenes, oracle_kw, workers=None, timeout=300.0, size=128):
        """`size` is the map scale (EnvConfig.size) the workers load and their `OracleEnv`s run at."""
        self.timeout = timeout
        workers = max(1, min(workers or (os.cpu_count() or 2) - 1, 16, n_envs))
        ctx = mp.get_context("spawn")  # the parent holds a CUDA context: never fork it
        self.slices = np.array_split(np.arange(n_envs), workers)
        self.conns, self.procs = [], []
        for sl in self.slices:
            parent, child = ctx.Pipe()
            p = ctx.Process(target=_worker, args=(child, scenes, oracle_kw, len(sl), size), daemon=True)
            p.start()
            child.close()
            self.conns.append(parent)
            self.procs.append(p)

    def run(self, cmds):
        """cmds[j] = ("reset", scene_index) | ("step", action) | ("repeat", (action, K)) | ("save", tag) |
        ("branches", ...) | ("adopt", key) | None for oracle env j; returns the per-env results."""
        for conn, sl in zip(self.conns, self.slices):
            conn.send([cmds[j] for j in sl])
        out = [None] * len(cmds)
        for conn, sl, proc in zip(self.conns, self.slices, self.procs):
            waited = 0.0
            while not conn.poll(1.0):  # never block for ever on a dead worker (a hung test would hang the GPU box)
                waited += 1.0
                if not proc.is_alive() or waited > self.timeout:
                    raise RuntimeError(f"oracle worker {proc.pid} died or timed out (exit code {proc.exitcode})")
            for j, res in zip(sl, conn.recv()):
                out[j] = res
        return out

    def branches(self, roots, actions, K, tags=None, keep=None, frames=False, ids=None):
        """Branch b from oracle env roots[b] (or its copy under tags[b]) with actions[b] ([H, ...]); the branches of
        each root run on its worker, in order.  `keep` (a name) keeps leaf b under (keep, ids[b]) in env roots[b]'s
        store (ids: default 0..B-1, the branch's index in a larger call).  Returns the per-branch result dicts of
        ("branches", ...)."""
        ids = range(len(roots)) if ids is None else [int(i) for i in ids]
        n = len(self.slices) and int(self.slices[-1][-1]) + 1
        per_env = {}
        for b, r in enumerate(roots):
            per_env.setdefault((int(r), None if tags is None else tags[b]), []).append(b)
        out = [None] * len(roots)
        pending = list(per_env.items())
        while pending:  # one command per env and call: roots that need several tags take several calls
            cmds, taken, rest = [None] * n, [], []
            for (r, tag), bs in pending:
                if cmds[r] is not None:
                    rest.append(((r, tag), bs))
                    continue
                cmds[r] = ("branches", (tag, [actions[b] for b in bs], K,
                                        None if keep is None else [(keep, ids[b]) for b in bs], frames))
                taken.append((r, bs))
            res = self.run(cmds)
            for r, bs in taken:
                for b, x in zip(bs, res[r]):
                    out[b] = x
            pending = rest
        return out

    def close(self):
        for conn in self.conns:
            try:
                conn.send(None)
                conn.close()
            except Exception:  # noqa: BLE001
                pass
        for p in self.procs:
            p.join(timeout=10)
            if p.is_alive():
                p.kill()
