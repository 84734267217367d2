"""Lookahead rollouts against the oracle in every row of the pairwise table, action repeat included.

Each row of `ROWS` (test_pairwise_matrix's pairwise table over the auto-reset modes next_step and disabled) runs its
engine at the row's repeat K and N envs, with the oracle kept in step on every env as `run_row` does (observation, reward, flags, cause, hero block, actor poses, terminal episode rows and
at the end the statistics vector), and fires the probes of `PROBES` at chosen agent steps, all with
`lookahead(..., repeat=K)`:

  P1  live roots, repeated, rewards and hero blocks, gamma 0.97             B = 2N + 3   H = F + 3
  P2  live roots, identity, right after a step that ended some envs (before  B = N + 2    H = max(1, F - 1)
      the masked reset), plus the device roots -1 and N; obs=True, fused in
      the fusion rows; the same call again with leaf rows over a sentinel
  P3  rows of a snapshot taken 5 agent steps earlier, at the first episode   B = N        H = max(F + 2, 6)
      end from step 6 on; no frames
  P4  the same rows, repeated, plus the rows -1 and n_rows; obs=True        B = N + 5    H = max(F + 2, 6)
  P5  live roots, identity, leaf=True, obs=True                              B = N        H = F + 1
  P6  source = P5's leaf rows (chaining), leaf=True, obs=True                B = N        H = 3

so every row runs all six branch-kernel modes, and the rows reach every (group width, mode, K > 1) variant of
k_lookahead / _obs / _ex / _rep (`test_probes_reach_every_kernel_variant`).  Every branch is compared with an oracle
branch (`oracle_pool`'s "branches" command: deep copies of the root's oracle env stepped with the same actions):
steps exactly, per-step rewards within K * 1e-9 and exactly 0 after the last step, `ret` exactly the NumPy replay of
the rewards and within H * K * 1e-9 of the oracle's, flags and cause exactly, the hero block, and the leaf observation
(stacked, fused, uint8, gray or raw RGB) and raw leaf window byte for byte.  Terminal roots take 0 steps and keep the
root's window and row; invalid roots take 0 steps with a zero window and leave their leaf row unwritten.  Leaf rows
are checked by what they do: their header against the oracle branch, P6 continuing them against the kept oracle
copies continued, and after P6 the live envs restored from P5's rows and the oracle envs replaced by the kept copies,
so that the row's loop then compares the episodes those leaves finish (return, length in simulator steps, means) and
the statistics vector.

A branch in which a StopReturn pedestrian starts a retreat route is followed but not compared from that agent step on
(test_gpu_scale's RETREAT NOTE), and so is a root env that is already unpinned."""
import numpy as np
import pytest

from golden_util import load_map
from test_pairwise_matrix import AXES, OBS_SIZE, TRAJECTORY_STEPS, _scene_pool, engine_args, oracle_args

# The pairwise table of `test_pairwise_matrix` as its generator gave it with the auto-reset axis ("next_step",
# "disabled"), one tuple per row in COLUMNS order.  Branches do not depend on the live envs' auto-reset mode (a
# same-step engine's lookahead is compared with its next_step twin in test_gpu_same_step), so this matrix keeps the
# table whose every row it has passed, NO_MOVING_HISTORY below included.
COLUMNS = tuple(AXES) + ("n_envs", "steps", "max_actions")
ROWS = [
    (64, "block83", "f32", "binary", (0.5, 0.5), False, "stack", 3, "continuous", "carl", "tables", "next_step", 1, "device", 12, 80, None),
    (128, "block83", "u8", "2-class", (0.5, 0.75), False, "stack", 4, "discrete9", "shaping", "handover", "disabled", 3, "host", 16, 87, 45),
    (256, "block83", "gray", None, (0.0, 1.0), False, None, 5, "discrete13", "carl", "live", "disabled", 1, "host", 19, 94, None),
    (64, "area", "u8", "4-class", (0.95, 0.3), True, "vehicle_temporal", 5, "continuous", "shaping", "live", "next_step", 3, "device", 24, 101, None),
    (64, "half", "gray", None, (0.5, 0.75), True, None, 3, "discrete9", "carl", "handover", "next_step", 1, "device", 13, 108, None),
    (64, "copy", "f32", "5-class", (0.0, 1.0), True, "vehicle_weighted", 4, "discrete13", "shaping", "tables", "disabled", 3, "host", 20, 115, 45),
    (64, "enlarge", "f32", "6-class", (0.95, 0.3), False, "vehicle_temporal", 3, "discrete9", "carl", "tables", "disabled", 1, "host", 12, 81, None),
    (64, "nonsquare", "u8", "7-class", (0.5, 0.5), True, "vehicle_weighted", 5, "discrete9", "carl", "handover", "next_step", 4, "host", 16, 88, None),
    (64, "raw", "rgb", None, (0.5, 0.5), False, None, None, "discrete13", "shaping", "live", "next_step", 1, "device", 19, 95, None),
    (64, "area", "f32", "2-class", (0.5, 0.75), True, "stack", 5, "discrete13", "carl", "tables", "disabled", 1, "device", 24, 102, None),
    (128, "fast96", "gray", None, (0.95, 0.3), True, None, 4, "continuous", "carl", "handover", "next_step", 1, "device", 13, 109, None),
    (128, "area", "gray", None, (0.5, 0.5), False, None, 3, "discrete13", "shaping", "live", "disabled", 3, "host", 20, 116, 45),
    (128, "half", "f32", "4-class", (0.0, 1.0), False, "vehicle_weighted", 3, "continuous", "shaping", "tables", "disabled", 1, "host", 12, 82, None),
    (128, "copy", "u8", "binary", (0.5, 0.75), True, "stack", 5, "continuous", "shaping", "live", "next_step", 1, "device", 16, 89, 45),
    (128, "enlarge", "u8", "5-class", (0.0, 1.0), False, "vehicle_temporal", 4, "discrete13", "carl", "handover", "next_step", 3, "device", 19, 96, None),
    (128, "nonsquare", "gray", None, (0.95, 0.3), False, None, 4, "discrete13", "shaping", "tables", "disabled", 1, "device", 24, 103, None),
    (128, "raw", "rgb", None, (0.5, 0.75), True, None, None, "discrete9", "carl", "handover", "disabled", 3, "host", 13, 110, None),
    (128, "fast96", "u8", "6-class", (0.5, 0.5), True, "vehicle_temporal", 3, "discrete13", "shaping", "live", "next_step", 8, "host", 20, 117, 45),
    (128, "fast96", "f32", "7-class", (0.0, 1.0), False, "stack", 4, "discrete9", "shaping", "live", "disabled", 1, "device", 12, 83, None),
    (256, "area", "f32", "binary", (0.95, 0.3), True, "stack", 4, "discrete9", "shaping", "handover", "next_step", 3, "host", 16, 90, 45),
    (256, "half", "u8", "2-class", (0.5, 0.5), False, "stack", 3, "continuous", "carl", "tables", "next_step", 3, "device", 19, 97, None),
    (256, "copy", "gray", None, (0.5, 0.75), False, None, 3, "discrete9", "carl", "handover", "disabled", 3, "host", 24, 104, None),
    (256, "nonsquare", "f32", "4-class", (0.5, 0.75), True, "vehicle_temporal", 4, "continuous", "carl", "live", "next_step", 1, "device", 13, 111, None),
    (256, "raw", "rgb", None, (0.0, 1.0), True, None, None, "continuous", "shaping", "tables", "disabled", 4, "host", 20, 118, None),
    (256, "half", "u8", "5-class", (0.95, 0.3), False, "vehicle_weighted", 5, "continuous", "carl", "live", "next_step", 1, "device", 12, 84, None),
    (256, "copy", "f32", "6-class", (0.5, 0.5), True, "vehicle_weighted", 4, "continuous", "shaping", "handover", "disabled", 3, "device", 16, 91, 45),
    (256, "block83", "u8", "7-class", (0.95, 0.3), True, "vehicle_temporal", 3, "discrete13", "carl", "tables", "next_step", 1, "host", 19, 98, None),
    (128, "fast96", "f32", "binary", (0.0, 1.0), False, "stack", 5, "discrete13", "shaping", "tables", "disabled", 3, "host", 24, 105, None),
    (128, "fast96", "u8", "2-class", (0.5, 0.75), False, "stack", 5, "discrete9", "carl", "live", "next_step", 1, "device", 13, 112, None),
    (128, "fast96", "f32", "4-class", (0.5, 0.5), True, "vehicle_weighted", 5, "discrete9", "shaping", "handover", "disabled", 3, "host", 20, 119, 45),
    (128, "fast96", "u8", "5-class", (0.5, 0.5), False, "stack", 3, "discrete9", "carl", "tables", "next_step", 1, "device", 12, 85, None),
    (64, "area", "f32", "5-class", (0.0, 1.0), True, "vehicle_weighted", 4, "continuous", "shaping", "handover", "disabled", 8, "host", 16, 92, None),
    (64, "area", "u8", "6-class", (0.5, 0.75), False, "vehicle_weighted", 5, "discrete13", "carl", "live", "next_step", 1, "device", 19, 99, None),
    (256, "area", "f32", "7-class", (0.5, 0.75), True, "vehicle_temporal", 3, "continuous", "shaping", "tables", "disabled", 3, "host", 24, 106, 45),
    (64, "half", "u8", "binary", (0.95, 0.3), False, "stack", 4, "discrete13", "carl", "handover", "next_step", 1, "device", 13, 113, None),
    (256, "half", "f32", "6-class", (0.0, 1.0), True, "vehicle_temporal", 5, "discrete9", "shaping", "live", "disabled", 3, "host", 20, 120, None),
    (64, "half", "u8", "7-class", (0.95, 0.3), False, "vehicle_temporal", 3, "continuous", "carl", "tables", "next_step", 1, "device", 12, 86, None),
    (256, "copy", "f32", "2-class", (0.95, 0.3), True, "stack", 4, "discrete9", "shaping", "handover", "disabled", 3, "host", 16, 93, 45),
    (64, "copy", "u8", "4-class", (0.5, 0.5), False, "vehicle_temporal", 5, "discrete13", "carl", "live", "next_step", 1, "device", 19, 100, None),
    (256, "copy", "f32", "7-class", (0.0, 1.0), True, "vehicle_weighted", 3, "continuous", "shaping", "tables", "disabled", 4, "host", 24, 107, None),
    (64, "enlarge", "gray", None, (0.5, 0.5), True, None, 5, "continuous", "shaping", "live", "next_step", 1, "device", 13, 114, 45),
    (64, "enlarge", "u8", "binary", (0.5, 0.75), False, "stack", 4, "discrete9", "carl", "handover", "disabled", 3, "host", 20, 80, None),
    (128, "enlarge", "f32", "2-class", (0.0, 1.0), False, "stack", 3, "discrete13", "carl", "tables", "next_step", 1, "device", 12, 87, None),
    (64, "enlarge", "u8", "4-class", (0.95, 0.3), True, "vehicle_weighted", 4, "discrete9", "shaping", "handover", "disabled", 3, "host", 16, 94, None),
    (128, "enlarge", "f32", "7-class", (0.5, 0.5), False, "vehicle_temporal", 5, "discrete13", "carl", "live", "next_step", 1, "device", 19, 101, None),
    (256, "block83", "u8", "4-class", (0.5, 0.75), True, "vehicle_weighted", 3, "continuous", "shaping", "tables", "disabled", 3, "host", 24, 108, 45),
    (256, "block83", "f32", "5-class", (0.5, 0.75), False, "vehicle_temporal", 4, "discrete9", "carl", "handover", "next_step", 1, "device", 13, 115, None),
    (256, "block83", "u8", "6-class", (0.0, 1.0), True, "stack", 5, "discrete13", "shaping", "live", "disabled", 8, "host", 20, 81, None),
    (64, "nonsquare", "f32", "binary", (0.0, 1.0), False, "stack", 3, "continuous", "carl", "tables", "next_step", 1, "device", 12, 88, None),
    (128, "nonsquare", "u8", "2-class", (0.95, 0.3), True, "stack", 4, "discrete9", "shaping", "handover", "disabled", 3, "host", 16, 95, 45),
    (256, "nonsquare", "f32", "5-class", (0.5, 0.5), False, "vehicle_weighted", 5, "discrete13", "carl", "live", "next_step", 1, "device", 19, 102, None),
    (64, "nonsquare", "u8", "6-class", (0.95, 0.3), True, "vehicle_temporal", 3, "continuous", "shaping", "tables", "disabled", 3, "host", 24, 109, None),
    (128, "raw", "rgb", None, (0.95, 0.3), False, None, None, "discrete9", "carl", "handover", "next_step", 1, "device", 13, 116, None),
    (256, "area", "f32", "4-class", (0.5, 0.5), True, "stack", 4, "discrete13", "shaping", "live", "disabled", 3, "host", 20, 82, 45),
]


def _row(i):
    return dict(zip(COLUMNS, ROWS[i]))

SENTINEL = 0xA5
GAMMA = 0.97
# name: (roots, frames, rows, leaf); the kernel mode of a probe is (frames or leaf, rows, leaf)
PROBES = {
    "P1": ("live", False, False, False),
    "P2": ("live", True, False, False),
    "P3": ("rows", False, True, False),
    "P4": ("rows", True, True, False),
    "P5": ("live", True, False, True),
    "P6": ("leaf", True, True, True),
}
T_P3, T_P5, T_P1, T_P2_EARLIEST = 6, 34, 40, 8  # agent steps of the loop
SNAP_AGE = 5  # agent steps between P3 / P4's snapshot and the call


def group_width(row):
    """The engine's rule (sim.cu narrow_groups): 32-lane groups for pools with more than 8 actors stepped live.  Every
    row's scene pool has a scene with more than 8 actors (`_scene_pool`)."""
    return 8 if TRAJECTORY_STEPS[row["actors"]] > 0 else 32


def probe_variants(row):
    """(G, OBS, ROWS, LEAF, K > 1) of the branch kernel each probe of a row launches."""
    G, rep = group_width(row), row["repeat"] > 1
    out = set()
    for name, (_, frames, rows, leaf) in PROBES.items():
        out.add((G, frames or leaf, rows, leaf, rep))
    return out


def _frames_shape(row):
    return row["frame_stack"] or 1


def _branch_actions(hero, roots, H, rng, table):
    """Actions [H, B] of branches from `roots` (clipped into range) of envs whose hero blocks are `hero` [N, 32]: what
    `drive` gives the root env itself (so a branch goes on with the root's own driving and ends where its episode
    would), with a per-branch, per-step steering and throttle perturbation, and every fifth branch at full throttle
    with half lock, off the road."""
    import torch

    from test_gpu_reward_params import drive

    B = len(roots)
    base = drive(None, len(hero), 0, torch.from_numpy(np.ascontiguousarray(hero)))[roots]
    a = np.repeat(base[None], H, axis=0).astype(np.float64)
    a[..., 0] += rng.normal(0.0, 0.1, (H, B))
    a[..., 1] += rng.normal(0.0, 0.15, (H, B))
    wild = np.arange(B) % 5 == 4
    a[:, wild, 0], a[:, wild, 2] = 1.0, 0.0
    a[:, wild, 1] = np.where(np.arange(B)[wild] % 2 == 0, 0.5, -0.5)
    a[..., 0] = np.clip(a[..., 0], 0.0, 1.0)
    a[..., 1] = np.clip(a[..., 1], -1.0, 1.0)
    a[..., 2] = np.clip(a[..., 2], 0.0, 1.0)
    a = a.astype(np.float32)
    if table is None:
        return a
    return np.argmin(((table[None, None] - a[:, :, None]) ** 2).sum(-1), axis=2).astype(np.int64)


def _ret_numpy(rew, steps, gamma):
    """ret of every branch replayed in step order: ret + w * r, then w * gamma, unfused (Python floats)."""
    out = np.zeros(rew.shape[1])
    for b in range(rew.shape[1]):
        r, w = 0.0, 1.0
        for t in range(int(steps[b])):
            r = r + w * float(rew[t, b])
            w = w * gamma
        out[b] = r
    return out


def run_lookahead_row(row, seed=23):
    """The row's step loop with the probes of the module doc.  Returns the counters."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.config import ACTION_PROFILES
    from carlabev_env_b200.fovmask import corner_mask
    from carlabev_env_b200.pool import pack_pool
    from oracle import raster
    from oracle_pool import OraclePool
    from test_gpu_action_repeat import _stats_from_rows
    from test_gpu_reward_params import drive
    from test_gpu_scale import POSE_TOL, _check_episode, _check_hero, autoreset_scene
    from test_pairwise_matrix import ACTION_PROFILE

    size, n, K, steps = row["size"], row["n_envs"], row["repeat"], row["steps"]
    F = _frames_shape(row)
    scenes = _scene_pool(size, row["anchor"])
    S = len(scenes)
    amax = max(len(sc["act_kind"]) for sc in scenes)
    kw = engine_args(row)
    traj = kw["trajectory_steps"]
    eng = E.Engine(n, max_actors=amax, seed=seed, ring_budget_bytes=64 << 20, **kw)
    eng.upload_map(load_map(size))
    eng.upload_pool(pack_pool(scenes))
    if row["fov"]:
        eng.upload_fov_mask(corner_mask(size, 0.5))
    if K > 1:
        eng.set_action_repeat(K)
    eng.reset(torch.arange(n, dtype=torch.int32) % S)
    fuse = row["fusion"] if row["fusion"] not in (None, "stack") else None
    vch = raster.VEHICLE_CHANNEL.get(row["mask"]) if fuse else None
    next_step = row["autoreset"] == "next_step"
    host = row["path"] == "host"
    table = ACTION_PROFILES[ACTION_PROFILE[row["actions"]]].get("discrete_actions")
    table = None if table is None else np.asarray(table, dtype=np.float32)
    u8 = row["obs"] == "u8"
    rng = np.random.default_rng(1000 + seed)

    def observe():
        return (eng.fuse(fuse) if fuse else eng.obs()).cpu().numpy()

    def same_obs(got, ref):
        ref = ref[0] if row["obs"] == "rgb" else ref  # the raw frame has no frame stack
        if u8 and fuse != "vehicle_weighted":  # 0 / 1 bytes against the oracle's 0.0 / 1.0 floats
            assert np.isin(ref, (0.0, 1.0)).all()
        return got.shape == ref.shape and np.array_equal(got, ref)

    def same_window(got, frames):
        if u8:
            assert np.isin(frames, (0.0, 1.0)).all()
        return frames.size == got.size and np.array_equal(got, frames.reshape(got.shape))

    def actions(t):
        a = drive(None, n, t, eng.hero)
        if table is None:
            return a
        return np.argmin(((table[None] - a[:, None]) ** 2).sum(-1), axis=1).astype(np.int64)

    c = dict(compared=0, episodes=0, auto_resets=0, masked_resets=0, inside_repeat=0, unpinned=0,
             branches=0, branch_steps=0, followed_steps=0, ended_inside=0, ended_inside_repeat=0, terminal_roots=0,
             invalid_roots=0, retreat_branches=0, moving_history=0, leaf_rows=0, adopted=0, adopted_episodes=0)
    pool = OraclePool(n, scenes, oracle_args(row), size=size)

    def pose_tol(since):
        return POSE_TOL if traj == 0 or since * K > traj else 1e-9

    def check_branches(name, la, roots, valid, terminal, skip, refs, H, gamma, since, root_window=None,
                       root_rows=None):
        """Branch b of `la` against refs[b] (an oracle branch, or None for a root that was not run: invalid, terminal or
        skipped).  root_window(b) gives a steps-0 terminal root's window, root_rows(b) its leaf row."""
        frames = la.window is not None
        st = la.steps.cpu().numpy()
        ret = la.ret.cpu().numpy()
        term = la.terminated.cpu().numpy().astype(bool)
        trunc = la.truncated.cpu().numpy().astype(bool)
        cause = la.cause.cpu().numpy()
        rew = la.reward.cpu().numpy() if la.reward is not None else None
        hero = la.hero.cpu().numpy() if la.hero is not None else None
        win = la.window.cpu().numpy() if frames else None
        obs = la.obs.cpu().numpy() if frames else None
        hdr = la.leaf.header().cpu().numpy() if la.leaf is not None else None
        if rew is not None:
            assert np.array_equal(ret, _ret_numpy(rew, st, gamma)), (name, "ret != replay of la.reward")
            for b in range(len(st)):
                assert not rew[int(st[b]):, b].any(), (name, b, "reward after the last step")
        for b in range(len(st)):
            where = (name, b, int(roots[b]))
            c["branches"] += 1
            if not valid[b]:
                c["invalid_roots"] += 1
                assert st[b] == 0 and ret[b] == 0.0 and not term[b] and not trunc[b], where
                if frames:
                    assert not win[b].any(), (*where, "invalid root: window not zero")
                continue
            if terminal[b]:
                c["terminal_roots"] += 1
                assert st[b] == 0 and ret[b] == 0.0, (*where, "terminal root took steps", st[b])
                if frames and root_window is not None:
                    assert np.array_equal(win[b], root_window(b)), (*where, "terminal root: not the root's window")
                if hdr is not None and root_rows is not None:
                    assert np.array_equal(la.leaf.data[b].cpu().numpy(), root_rows(b)), (*where, "terminal leaf row")
                continue
            r = refs[b]
            if skip[b]:
                c["followed_steps"] += H
                continue
            if r["retreat"] is not None:  # followed from the agent step its retreat started on
                c["retreat_branches"] += 1
                c["branch_steps"] += r["retreat"]
                c["followed_steps"] += H - r["retreat"]
                assert st[b] > r["retreat"], (*where, "the engine ended before the oracle's retreat", st[b], r["retreat"])
                if rew is not None:
                    for t in range(r["retreat"]):
                        assert abs(rew[t, b] - r["reward"][t]) < K * 1e-9, (*where, t, "reward")
                continue
            c["branch_steps"] += H
            assert st[b] == r["steps"], (*where, "steps", st[b], r["steps"])
            s = int(st[b])
            if rew is not None:
                for t in range(s):
                    assert abs(rew[t, b] - r["reward"][t]) < K * 1e-9, (*where, t, "reward", rew[t, b], r["reward"][t])
            ref_ret = _ret_numpy(np.asarray(r["reward"], dtype=np.float64)[:, None], [s], gamma)[0]
            assert abs(ret[b] - ref_ret) <= H * K * 1e-9, (*where, "ret", ret[b], ref_ret)
            assert term[b] == r["term"][-1] and trunc[b] == r["trunc"][-1], (*where, "flags")
            assert cause[b] == r["cause"][-1], (*where, "cause", cause[b], r["cause"][-1])
            if hero is not None:
                _check_hero(hero[b], r["hero"], pose_tol(since[b] + s), where)
            if s < H and (term[b] or trunc[b]):
                c["ended_inside"] += 1
                if K > 1 and r["j"][-1] < K:
                    c["ended_inside_repeat"] += 1
            if frames:
                if la.obs is not la.window or not fuse:  # fused by the call, or the row's observation is the window
                    assert same_obs(obs[b], r["obs"]), (*where, "leaf observation", obs[b].shape, r["obs"].shape)
                assert same_window(win[b], r["frames"]), (*where, "leaf window")
                if fuse:
                    hist = r["frames"][-3:, vch]
                    c["moving_history"] += int(not (hist == hist[-1]).all())
            if hdr is not None:
                c["leaf_rows"] += 1
                got_hdr = (int(hdr[b, 0]), int(hdr[b, 1]), bool(hdr[b, 2] & 0xFF))
                assert got_hdr == tuple(r["header"]), (*where, "leaf row header", got_hdr, r["header"])

    def probe_live(name, roots, H, gamma, done, unpinned, since, **kw):
        """A call from live roots and its oracle branches."""
        valid = (roots >= 0) & (roots < n)
        rc = np.clip(roots, 0, n - 1)
        terminal = valid & done[rc]
        skip = valid & ~terminal & unpinned[rc]
        hero_live = eng.hero.cpu().numpy()
        acts = _branch_actions(hero_live, rc, H, rng, table)
        la = eng.lookahead(torch.from_numpy(acts).cuda(), env_ids=torch.from_numpy(roots.astype(np.int32)).cuda(),
                           gamma=gamma, repeat=K, **kw)
        run = np.flatnonzero(valid & ~terminal)
        got = pool.branches(rc[run], [acts[:, b] for b in run], K, keep="P5" if kw.get("leaf") else None,
                            frames=bool(kw.get("obs")), ids=run)
        refs = [None] * len(roots)
        for b, r in zip(run, got):
            refs[b] = r
        return la, acts, refs, valid, terminal, skip, rc

    def masked_reset(t, done, unpinned, adopted, since):
        ids = (np.arange(n) + 7 * (t + 1)) % S
        obs_r = eng.reset(torch.from_numpy(ids.astype(np.int32)), torch.from_numpy(done)).cpu().numpy()
        if fuse:
            obs_r = observe()
        ref = pool.run([("reset", int(ids[i])) if done[i] else None for i in range(n)])
        for i in np.flatnonzero(done):
            assert same_obs(obs_r[i], ref[i]["obs"]), (t, i, "masked reset observation")
        c["masked_resets"] += int(done.sum())
        unpinned[done] = adopted[done] = False
        since[done] = 0
        done[:] = False

    try:
        ref = pool.run([("reset", i % S) for i in range(n)])
        obs = observe()
        for i in range(n):
            assert same_obs(obs[i], ref[i]["obs"]), (i, "reset observation")
        done = np.zeros(n, bool)
        unpinned = np.zeros(n, bool)  # test_gpu_scale's RETREAT NOTE: followed, not compared, until the next reset
        adopted = np.zeros(n, bool)  # restored from a P5 leaf row, no episode compared since
        episodes = np.zeros(n, dtype=np.int64)
        since = np.zeros(n, dtype=np.int64)  # agent steps since the env's last reset
        term_total = 0
        rows = []
        fired = set()
        snaps = {}  # agent step -> (snapshot, the loop's bookkeeping then), for P3 / P4
        live_acts = {}  # agent step -> actions
        pin = None
        for t in range(steps):
            a = actions(t)
            live_acts[t] = a
            live_acts.pop(t - SNAP_AGE - 1, None)
            ended_now = []  # compared envs whose episode ended at this step (inside an agent step at K > 1)
            if host:
                if pin is None:
                    pin = torch.from_numpy(np.zeros_like(a)).pin_memory()
                pin.numpy()[...] = a
                eng.step_host_full(pin, episode=True)
            else:
                eng.step(torch.from_numpy(a).cuda())
            cmds = []
            for i in range(n):
                if done[i]:
                    cmds.append(("reset", int(autoreset_scene(seed, i, int(episodes[i]), S))))
                else:
                    cmds.append(("repeat", (a[i], K)) if K > 1 else ("step", a[i]))
            ref = pool.run(cmds)
            rew = eng.reward.cpu().numpy()
            term = eng.terminated.cpu().numpy().astype(bool)
            trunc = eng.truncated.cpu().numpy().astype(bool)
            cause = eng.cause.cpu().numpy()
            hero = eng.hero.cpu().numpy()
            episode = eng.episode.cpu().numpy()
            term_total += int(term.sum())
            obs = observe()
            act = eng.get_state(amax)[1]
            for i in range(n):
                r = ref[i]
                if done[i]:
                    assert np.array_equal(hero[i], r["hero"]), (t, i, "auto-reset hero block", hero[i], r["hero"])
                    assert rew[i] == 0.0 and not term[i] and not trunc[i], (t, i)
                    assert same_obs(obs[i], r["obs"]), (t, i, "auto-reset observation")
                    done[i] = unpinned[i] = adopted[i] = False
                    since[i] = 0
                    c["auto_resets"] += 1
                    continue
                since[i] += 1
                if unpinned[i]:
                    c["unpinned"] += 1
                    if term[i] or trunc[i]:
                        if term[i]:
                            rows.append(episode[i][None])
                        done[i] = True
                        episodes[i] += 1
                    continue
                c["compared"] += 1
                assert abs(r["reward"] - rew[i]) < K * 1e-9, (t, i, "reward", r["reward"], rew[i])
                assert r["term"] == term[i] and r["trunc"] == trunc[i], (t, i, "flags", r["term"], r["trunc"])
                assert r["cause"] == cause[i], (t, i, "cause", r["cause"], cause[i])
                _check_hero(hero[i], r["hero"], pose_tol(since[i]), (t, i))
                assert same_obs(obs[i], r["obs"]), (t, i, "observation", int((obs[i] != r["obs"]).sum()))
                na = len(r["actors"])
                if na:
                    assert np.allclose(act[i, :na, :4], r["actors"], rtol=POSE_TOL, atol=POSE_TOL), (t, i, "actors")
                    if np.any(act[i, :na, 7].astype(np.int64) & 32):
                        unpinned[i] = True
                if r["term"]:
                    _check_episode(episode[i], r["episode"], (t, i))
                    rows.append(r["episode"][None])
                    if adopted[i]:
                        c["adopted_episodes"] += 1
                if r["term"] or r["trunc"]:
                    done[i] = True
                    adopted[i] = False
                    episodes[i] += 1
                    c["episodes"] += 1
                    if K > 1 and r["j"] < K:
                        c["inside_repeat"] += 1
                    if K == 1 or r["j"] < K:
                        ended_now.append(i)

            # ---- P2: right after a step that ended envs, before the masked reset
            if "P2" not in fired and ((t >= T_P2_EARLIEST and done.any()) or t == steps - 1):
                fired.add("P2")
                H = max(1, F - 1)
                roots = np.concatenate([np.arange(n), [-1, n]])
                la, acts, refs, valid, terminal, skip, rc = probe_live("P2", roots, H, 1.0, done, unpinned, since,
                                                                       rewards=True, hero=True, obs=True, fuse=fuse)
                live_win = eng.obs().cpu().numpy()
                check_branches("P2", la, roots, valid, terminal, skip, refs, H, 1.0, since[rc],
                               root_window=lambda b: live_win[roots[b]])
                # the same call with leaf rows over a sentinel: same outputs, terminal roots' own rows, invalid
                # roots' rows untouched
                at = torch.from_numpy(acts).cuda()
                rt = torch.from_numpy(roots.astype(np.int32)).cuda()
                lf = eng.lookahead(at, env_ids=rt, obs=True, leaf=True, repeat=K)
                lf.leaf._buf.fill_(SENTINEL)
                lf = eng.lookahead(at, env_ids=rt, obs=True, leaf=True, repeat=K, out=lf)
                for k in ("steps", "ret", "terminated", "truncated", "cause", "window"):
                    assert torch.equal(getattr(lf, k), getattr(la, k)), ("P2 with leaf rows", k)
                leaf = lf.leaf.data.cpu().numpy()
                assert (leaf[~valid] == SENTINEL).all(), "P2: an invalid root's leaf row was written"
                live_rows = eng.snapshot().data.cpu().numpy()
                for b in np.flatnonzero(terminal):
                    assert np.array_equal(leaf[b], live_rows[roots[b]]), ("P2: terminal root's leaf row", b)
                c["p2_terminal_roots"] = int(terminal.sum())
            if not next_step and done.any():  # SyncVectorEnv-style masked reset of every env that ended
                masked_reset(t, done, unpinned, adopted, since)

            # ---- P1: live roots, repeated, rewards and hero blocks
            if t == T_P1:
                H = F + 3
                roots = rng.choice(np.flatnonzero(~unpinned), size=2 * n + 3)
                la, _, refs, valid, terminal, skip, rc = probe_live("P1", roots, H, GAMMA, done, unpinned, since,
                                                                    rewards=True, hero=True)
                check_branches("P1", la, roots, valid, terminal, skip, refs, H, GAMMA, since[rc])
            # ---- P3 / P4: roots from the rows of a snapshot taken SNAP_AGE agent steps earlier.  A snapshot is taken
            # every step (a ring of SNAP_AGE + 1); they fire at the first compared live episode end from T_P3 on (one
            # inside an agent step at K > 1), so that the branch of that env's row that replays the env's own actions
            # ends inside the horizon, or at the last step.
            if t >= T_P3 - SNAP_AGE and "P3" not in fired:
                old = snaps.get(t - SNAP_AGE)
                if old is not None and (t == steps - 1 or (t >= T_P3 and ended_now)):
                    fired.add("P3")
                    snap, snap_state = old
                    H = max(F + 2, SNAP_AGE + 1)  # F <= 3: the replayed branch ends before the horizon
                    replay = [i for i in ended_now if not snap_state["done"][i] and not snap_state["unpinned"][i]]
                    c["p3_step"], c["replays"] = t, len(replay)
                    for name in ("P3", "P4"):
                        if name == "P3":
                            roots = rng.permutation(n)
                        else:
                            roots = np.concatenate([rng.integers(0, n, size=n + 3), [-1, n]])
                            rng.shuffle(roots)
                        valid = (roots >= 0) & (roots < n)
                        rc = np.clip(roots, 0, n - 1)
                        terminal = valid & snap_state["done"][rc]
                        skip = valid & ~terminal & snap_state["unpinned"][rc]
                        acts = _branch_actions(snap_state["hero"], rc, H, rng, table)
                        for i in replay:  # the first branch of env i's row takes the env's own actions
                            at = np.flatnonzero(roots == i)
                            if len(at):
                                acts[:SNAP_AGE, at[0]] = np.stack([live_acts[t - SNAP_AGE + 1 + k][i]
                                                                   for k in range(SNAP_AGE)])
                        kwp = dict(obs=True, fuse=fuse) if name == "P4" else {}
                        la = eng.lookahead(torch.from_numpy(acts).cuda(), source=snap,
                                           rows=torch.from_numpy(roots.astype(np.int32)).cuda(), rewards=True,
                                           hero=True, repeat=K, **kwp)
                        run = np.flatnonzero(valid & ~terminal)
                        got = pool.branches(rc[run], [acts[:, b] for b in run], K,
                                            tags=[f"snap{(t - SNAP_AGE) % (SNAP_AGE + 1)}"] * len(run),
                                            frames=name == "P4")
                        refs = [None] * len(roots)
                        for b, r in zip(run, got):
                            refs[b] = r
                        check_branches(name, la, roots, valid, terminal, skip, refs, H, 1.0,
                                       snap_state["since"][rc], root_window=lambda b: snap_state["window"][roots[b]])
                snaps.pop(t - SNAP_AGE, None)
                if "P3" not in fired:
                    snaps[t] = (eng.snapshot(), dict(done=done.copy(), unpinned=unpinned.copy(), since=since.copy(),
                                                     hero=eng.hero.cpu().numpy(), window=eng.obs().cpu().numpy()))
                    pool.run([("save", f"snap{t % (SNAP_AGE + 1)}")] * n)
            # ---- P5 / P6: leaf rows, chained, then restored into the live envs
            if t == T_P5:
                H5 = F + 1
                roots = np.arange(n)
                la5, _, refs5, valid, terminal5, skip5, _ = probe_live("P5", roots, H5, 1.0, done, unpinned, since,
                                                                       rewards=True, hero=True, obs=True, leaf=True)
                live_rows = eng.snapshot().data.cpu().numpy()
                live_win = eng.obs().cpu().numpy()
                check_branches("P5", la5, roots, valid, terminal5, skip5, refs5, H5, 1.0, since,
                               root_window=lambda b: live_win[b], root_rows=lambda b: live_rows[b])
                st5 = la5.steps.cpu().numpy()
                end5 = (la5.terminated | la5.truncated).cpu().numpy().astype(bool)
                leaf5 = la5.leaf.data.cpu().numpy()
                # P6: continue the leaves; branches of ended leaves take 0 steps and keep the leaf's window and row
                H6 = 3
                terminal6 = terminal5 | end5
                skip6 = skip5 | np.array([r is not None and r["retreat"] is not None for r in refs5])
                hero5 = np.array([refs5[b]["hero"] if refs5[b] is not None else hero[b] for b in range(n)])
                acts6 = _branch_actions(hero5, roots, H6, rng, table)
                la6 = eng.lookahead(torch.from_numpy(acts6).cuda(), source=la5.leaf, rewards=True, hero=True,
                                    obs=True, leaf=True, repeat=K)
                run = np.flatnonzero(~terminal6)
                got = pool.branches(roots[run], [acts6[:, b] for b in run], K, tags=[("P5", b) for b in run],
                                    frames=True)
                refs6 = [None] * n
                for b, r in zip(run, got):
                    refs6[b] = r
                win5 = la5.window.cpu().numpy()
                check_branches("P6", la6, roots, valid, terminal6, skip6, refs6, H6, 1.0, since + st5,
                               root_window=lambda b: win5[b], root_rows=lambda b: leaf5[b])
                # restore P5's leaves into the live envs and the kept oracle copies into the oracle envs
                eng.restore(la5.leaf)
                pool.run([None if terminal5[i] else ("adopt", ("P5", i)) for i in range(n)])
                for i in np.flatnonzero(~terminal5):
                    since[i] += st5[i]
                    if skip6[i]:
                        unpinned[i] = True
                    if end5[i]:
                        done[i] = True
                        episodes[i] += 1
                    elif not unpinned[i]:
                        adopted[i] = True
                        c["adopted"] += 1
                if not next_step and done.any():
                    masked_reset(t, done, unpinned, adopted, since)
    finally:
        pool.close()
    stats = eng.read_stats().cpu().numpy()
    eng.close()
    assert stats[0] == term_total, "episode counter != number of terminal flags raised"
    assert stats[-1] == steps * n, "the step counter counts calls x N (branches do not step the live envs)"
    want = _stats_from_rows(np.concatenate(rows) if rows else np.zeros((0, len(E.EPISODE_FIELDS))))
    counts = [0, 2] + list(range(4, 12))
    assert np.array_equal(stats[counts], want[counts]), ("statistics counts", stats[counts], want[counts])
    sums = [k for k in range(len(stats) - 1) if k not in counts]
    assert np.allclose(stats[sums], want[sums], rtol=1e-7, atol=1e-7), ("statistics sums", stats[sums], want[sums])
    assert c["unpinned"] <= 0.25 * steps * n, c
    assert c["followed_steps"] <= 0.25 * (c["branch_steps"] + c["followed_steps"]), c
    return c


# Fusion rows in which no vehicle moves in any compared leaf window: no vehicle moves in view of these envs' cameras
# (the pairwise table's rows without moving vehicles in the live windows are 05, 22, 31 and 50).
NO_MOVING_HISTORY = (5, 22, 25, 31, 50)


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("i", range(len(ROWS)), ids=[f"row{i:02d}" for i in range(len(ROWS))])
def test_lookahead_row_against_the_oracle(i):
    row = _row(i)
    c = run_lookahead_row(row)
    print(f"row{i:02d} {row} {c}")
    assert c["episodes"] >= 1, c
    assert c["ended_inside"] >= 1, ("no branch ended inside the horizon", c)
    assert c["terminal_roots"] >= 1, ("no steps-0 terminal root", c)
    assert c["adopted_episodes"] >= 1, ("no restored leaf row reached a compared terminal episode", c)
    if row["repeat"] > 1:
        assert c["ended_inside_repeat"] >= 1, ("no branch ended inside an agent step", c)
    if row["fusion"] not in (None, "stack") and i not in NO_MOVING_HISTORY:
        assert c["moving_history"] >= 1, ("no fused leaf window with a moving vehicle", c)


# (OBS, ROWS, LEAF) of the six branch-kernel modes: k_lookahead, k_lookahead_obs and k_lookahead_ex's four
MODES = {(False, False, False), (True, False, False), (False, True, False), (True, True, False), (True, False, True),
         (True, True, True)}


def test_probes_reach_every_kernel_variant():
    """Over the rows, the probes launch every (G, mode, K > 1) branch kernel: k_lookahead<G>, k_lookahead_obs<G>,
    k_lookahead_ex<G, ...> (K = 1) and k_lookahead_rep<G, ...> (K > 1) for G = 8 and 32."""
    want = {(G, *m, rep) for G in (8, 32) for m in MODES for rep in (False, True)}
    assert len(want) == 24
    got = set()
    for i in range(len(ROWS)):
        got |= probe_variants(_row(i))
    assert got == want, sorted(want - got)
    assert {(f or lf, r, lf) for _, f, r, lf in PROBES.values()} == MODES


def test_probes_with_frames_reach_every_axis_value():
    """The probes that render leaf windows (P2, P4, P5, P6) run in every row, so they meet every resize branch, scale,
    observation form, mask mode, anchor, FOV mask and fusion mode."""
    framed = [k for k, (_, f, _, lf) in PROBES.items() if f or lf]
    assert {"P2", "P4", "P5", "P6"} <= set(framed)
    for ax in ("size", "resize", "obs", "mask", "anchor", "fov", "fusion"):
        seen = {_row(i)[ax] for i in range(len(ROWS))} - {None}
        assert seen == set(AXES[ax]), (ax, set(AXES[ax]) - seen)
    for ax, dom in OBS_SIZE.items():  # every (resize branch, scale) that exists
        for size in dom:
            assert any(_row(i)["resize"] == ax and _row(i)["size"] == size for i in range(len(ROWS))), (ax, size)


# ---- the oracle side: oracle_pool's branch commands against OracleEnv copies stepped by hand (no GPU)

ORACLE_KW = dict(obs_mode="bev_semantic", semantic_mask_ch="6-class", frame_stack=3, obs_size=(48, 48),
                 action_mode="continuous", action_profile="continuous_gsb_v1", temporal_fusion_mode="stack")


def _oracles(n=3, warm=6):
    """An OraclePool of n envs and n local OracleEnvs in the same states after `warm` steps."""
    from oracle.env import OracleEnv
    from oracle_pool import OraclePool
    from test_gpu_snapshot import _scripted

    scenes = _scripted(4, kinds=[("jaywalk", 3), ("lead_brake", 2), ("jaywalk", 4), ("lead_brake", 1)])
    pool = OraclePool(n, scenes, ORACLE_KW, workers=2)
    local = [OracleEnv(load_map(), **ORACLE_KW) for _ in range(n)]
    pool.run([("reset", i) for i in range(n)])
    for i in range(n):
        local[i].reset(scenes[i])
    for t in range(warm):
        a = [np.array([0.6, 0.1 * (i - 1), 0.0], dtype=np.float32) for i in range(n)]
        pool.run([("step", a[i]) for i in range(n)])
        for i in range(n):
            local[i].step(a[i])
    return pool, local


def _by_hand(env, scene, acts, K):
    """A copy of `env` stepped with `acts` as Engine.lookahead(repeat=K) does: per agent step the reward (sum) and
    flags, then the hero block, the observation and the frame stack after the last step."""
    import copy

    from oracle_pool import _repeat, hero_vector

    c = copy.deepcopy(env)
    rew, term, trunc = [], [], []
    for a in acts:
        if K == 1:
            _, r, te, tr, _ = c.step(a)
        else:
            _, r, te, tr, _, _ = _repeat(c, a, K)
        rew.append(float(r))
        term.append(bool(te))
        trunc.append(bool(tr))
        if te or tr:
            break
    return c, dict(reward=rew, term=term, trunc=trunc, hero=hero_vector(c, scene), obs=c._stacked(),
                   frames=np.stack(list(c.frames)))


def _actions(rng, H, B):
    a = np.stack([rng.uniform(0, 1, (B, H)), rng.uniform(-1, 1, (B, H)), rng.uniform(0, 0.3, (B, H))], axis=2)
    a[::3, :, 1] = 1.0  # full lock: some branches leave the road inside the horizon
    return a.astype(np.float32)


@pytest.mark.parametrize("K", [1, 3])
def test_branches_equal_copies_stepped_by_hand(K):
    """Branch outputs equal deep copies stepped with `step` (K = 1) or `_repeat` (K > 1) by hand, H below and above
    the frame stack."""
    pool, local = _oracles()
    try:
        rng = np.random.default_rng(K)
        roots = np.array([0, 1, 2, 0, 2, 1])
        for H in (2, 7):
            acts = _actions(rng, H, len(roots))
            got = pool.branches(roots, list(acts), K, frames=True)
            for b, r in enumerate(roots):
                _, want = _by_hand(local[r], r, acts[b], K)
                g = got[b]
                assert g["steps"] == len(want["reward"]) and g["reward"] == want["reward"], (K, H, b)
                assert g["term"] == want["term"] and g["trunc"] == want["trunc"], (K, H, b)
                assert np.array_equal(g["hero"], want["hero"]), (K, H, b)
                assert np.array_equal(g["obs"], want["obs"]) and np.array_equal(g["frames"], want["frames"]), (K, H, b)
                assert K == 1 or all(j == K for j in g["j"][:-1]), g["j"]
    finally:
        pool.close()


def test_branches_leave_the_env_unchanged():
    pool, local = _oracles()
    try:
        rng = np.random.default_rng(3)
        acts = _actions(rng, 5, 3)
        pool.branches(np.array([0, 1, 2]), list(acts), 1, keep="k", frames=True)
        pool.run([("save", "s")] * 3)
        a = np.array([0.5, 0.0, 0.0], dtype=np.float32)
        got = pool.run([("step", a)] * 3)
        for i in range(3):
            o, r, te, tr, _ = local[i].step(a)
            assert got[i]["reward"] == r and np.array_equal(got[i]["obs"], o), i
    finally:
        pool.close()


def test_save_and_adopt_round_trip():
    """("adopt", tag) of a saved state and of a kept branch leaf continues exactly as the copy it was taken from."""
    import copy

    from oracle_pool import hero_vector

    pool, local = _oracles()
    try:
        saved = [copy.deepcopy(e) for e in local]
        assert [r["scene"] for r in pool.run([("save", "s")] * 3)] == [0, 1, 2]
        a = np.array([0.8, -0.2, 0.0], dtype=np.float32)
        pool.run([("step", a)] * 3)
        assert [r["scene"] for r in pool.run([("adopt", "s")] * 3)] == [0, 1, 2]
        b = np.array([0.3, 0.4, 0.0], dtype=np.float32)
        got = pool.run([("step", b)] * 3)
        for i in range(3):
            o, r, _, _, _ = saved[i].step(b)
            assert got[i]["reward"] == r and np.array_equal(got[i]["obs"], o), i
            assert np.array_equal(got[i]["hero"], hero_vector(saved[i], i)), i
        # a kept leaf: adopted, it continues as the hand-stepped copy continues
        rng = np.random.default_rng(4)
        acts = _actions(rng, 4, 3)[:, :, :]
        acts[:, :, 1] = 0.0
        pool.branches(np.array([0, 1, 2]), list(acts), 3, keep="k", frames=True)
        pool.run([("adopt", ("k", i)) for i in range(3)])
        got = pool.run([("repeat", (b, 3))] * 3)
        from oracle_pool import _repeat

        for i in range(3):
            c, want = _by_hand(saved[i], i, acts[i], 3)
            if want["term"][-1] or want["trunc"][-1]:
                continue
            o, r, _, _, _, _ = _repeat(c, b, 3)
            assert got[i]["reward"] == r and np.array_equal(got[i]["obs"], o), i
    finally:
        pool.close()
