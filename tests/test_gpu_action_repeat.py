"""Action repeat (Engine.set_action_repeat / cbev_set_action_repeat, make_env(action_repeat=K)) on the GPU.

The reference is a twin engine B of the same configuration, seed and pool stepped at repeat 1.  Before each agent step
of engine A, B is restored from A's snapshot and stepped K times with the agent step's actions.  For every env, j is
its first terminal sub-step (1 for a pending NEXT_STEP auto-reset, else K), and A's outputs after its one call must be
B's after sub-step j: the reward is the in-order sum of B's rewards (bit for bit), flags, cause and hero are B's at j,
the episode row of a terminal env is B's, the state bytes of A's snapshot row are B's row at j, and A's newest frame is
B's newest frame at j.  Across agent steps A's window must hold those newest frames of the last F agent steps, and
A's statistics vector the sums of the terminal episode rows."""
import numpy as np
import pytest

from test_gpu_lookahead import _plan_actions
from test_gpu_lookahead_obs import TABLE
from test_gpu_snapshot import _engine, _rdm, _scripted

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]


def _frames(eng):
    """[N, F, frame elements] copy of the current observation windows (oldest first)."""
    return eng.obs().reshape(eng.N, eng.F, -1).clone()


def _stats_from_rows(rows):
    """The statistics vector (without the step counter) that the terminal episode rows `rows` [n, 16] add up to."""
    from carlabev_env_b200 import engine as E

    s = np.zeros(E.STATS_FIELDS, dtype=np.float64)
    if len(rows) == 0:
        return s
    f = {k: i for i, k in enumerate(E.EPISODE_FIELDS)}
    s[0], s[1], s[2], s[3] = len(rows), rows[:, f["return"]].sum(), rows[:, f["length"]].sum(), \
        rows[:, f["mean_speed"]].sum()
    for c in rows[:, f["cause"]].astype(int):
        s[4 + c] += 1
    s[12:18] = rows[:, f["mean_abs_accel_long"]:f["mean_abs_yaw_acc"] + 1].sum(0)
    s[18], s[19] = rows[:, f["comfort_violation_rate"]].sum(), rows[:, f["harsh_brake_rate"]].sum()
    return s


def _same_stats(got, ref, what):
    """Counts exact; sums to 1e-12 relative (the atomics add in another order; 1e-10 absolute near zero)."""
    counts = [0] + list(range(4, 12))
    assert np.array_equal(got[counts], ref[counts]), (what, got[counts], ref[counts])
    assert np.allclose(got, ref, rtol=1e-12, atol=1e-10), (what, got, ref)


class RepeatChecker:
    """Drives engine A at the repeat of each agent step and checks it against the twin B (see the module doc)."""

    def __init__(self, a, b):
        import torch

        self.a, self.b, self.t = a, b, torch
        N, F = a.N, a.F
        self.win = _frames(a)  # the expected window: newest frames of the last F agent steps
        self.rb = a.snapshot_row_bytes
        self.state_bytes = self.rb - F * a.frame_bytes
        self.terminal_rows = []
        self.calls = 0
        self.ends_inside = 0  # envs that ended before sub-step K of a repeat
        assert torch.equal(self.win, _frames(b))
        self.ar = torch.arange(N, device=a.device)
        # rows restore only into the engine that took them; B has A's layout, so A's rows go in under B's own info
        self.b_info = b.snapshot().info

    def agent_step(self, acts, K):
        from carlabev_env_b200 import engine as E

        t, a, b = self.t, self.a, self.b
        N = a.N
        snap = a.snapshot()
        b.restore(E.EnvSnapshot(snap._buf, self.b_info))
        pending = (snap.header()[:, 2] != 0).cpu().numpy() & (a.cfg.autoreset == E.AUTORESET_NEXT_STEP)
        rec = {k: [] for k in ("reward", "term", "trunc", "cause", "hero", "episode", "frame", "state")}
        for _ in range(K):
            b.step(acts)
            rec["reward"].append(b.reward.cpu().numpy().copy())
            rec["term"].append(b.terminated.cpu().numpy().astype(bool))
            rec["trunc"].append(b.truncated.cpu().numpy().astype(bool))
            rec["cause"].append(b.cause.clone())
            rec["hero"].append(b.hero.clone())
            rec["episode"].append(b.episode.clone())
            rec["frame"].append(_frames(b)[:, -1])
            rec["state"].append(b.snapshot().data[:, : self.state_bytes].clone())
        term, trunc = np.stack(rec["term"]), np.stack(rec["trunc"])  # [K, N]
        end = term | trunc
        j = np.where(end.any(0), end.argmax(0) + 1, K)
        j[pending] = 1
        self.ends_inside += int(((j < K) & ~pending).sum())
        rew = np.stack(rec["reward"])
        ref_reward = rew[0].copy()
        for k in range(1, K):  # in sub-step order from r1, as Python floats add
            more = k < j
            ref_reward[more] = ref_reward[more] + rew[k][more]
        a.set_action_repeat(K)
        a.step(acts)
        self.calls += 1
        jm = self.t.from_numpy(j - 1).to(a.device)
        at = lambda key: t.stack(rec[key])[jm, self.ar]  # noqa: E731
        got_r = a.reward.cpu().numpy()
        assert np.array_equal(got_r.view(np.int64), ref_reward.view(np.int64)), \
            ("reward", np.flatnonzero(got_r.view(np.int64) != ref_reward.view(np.int64))[:8])
        idx = (j - 1, np.arange(N))
        assert np.array_equal(a.terminated.cpu().numpy().astype(bool), term[idx]), "terminated"
        assert np.array_equal(a.truncated.cpu().numpy().astype(bool), trunc[idx]), "truncated"
        assert t.equal(a.cause, at("cause")), "cause"
        assert t.equal(a.hero, at("hero")), ("hero", t.nonzero((a.hero != at("hero")).any(1))[:8].flatten().tolist())
        done = term[idx]
        if done.any():
            sel = t.from_numpy(np.flatnonzero(done)).to(a.device)
            ref_ep = at("episode").index_select(0, sel)
            assert t.equal(a.episode.index_select(0, sel), ref_ep), "episode rows"
            self.terminal_rows.append(ref_ep.cpu().numpy())
        rows = a.snapshot().data
        ref_state = at("state")
        bad = t.nonzero((rows[:, : self.state_bytes] != ref_state).any(1)).flatten().tolist()
        assert not bad, ("state bytes", bad[:8], j[bad[:8]])
        newest = at("frame")
        got = _frames(a)
        assert t.equal(got[:, -1], newest), ("newest frame", t.nonzero((got[:, -1] != newest).any(1))[:8].flatten())
        # the window: the last F agent-step frames; an auto-reset fills every slot with the reset frame
        self.win = t.cat([self.win[:, 1:], newest[:, None]], dim=1)
        reset = t.from_numpy(pending).to(a.device)
        self.win[reset] = newest[reset][:, None]
        assert t.equal(got, self.win), ("window", t.nonzero((got != self.win).any(2).any(1)).flatten()[:8].tolist())
        return j

    def check_stats(self):
        rows = np.concatenate(self.terminal_rows) if self.terminal_rows else np.zeros((0, 16))
        got = self.a.read_stats().cpu().numpy().copy()
        ref = _stats_from_rows(rows)
        ref[-1] = self.calls * self.a.N  # CBEV_S_STEPS counts calls
        _same_stats(got, ref, "statistics")
        return len(rows)


def _pair(scenes, n, **kw):
    a, b = _engine(scenes, n, **kw), _engine(scenes, n, **kw)
    ids = np.arange(n, dtype=np.int32) % len(scenes)
    a.reset(ids)
    b.reset(ids)
    return a, b


def _run(a, b, rng, steps, K):
    chk = RepeatChecker(a, b)
    for s in range(steps):
        k = K[s % len(K)] if isinstance(K, (list, tuple)) else K
        chk.agent_step(_plan_actions(a, rng, 1, a.N)[0], k)
    return chk


CASES = {
    # name: (K, kwargs of _engine, scenes, envs, agent steps)
    "f32": (4, {}, None, 64, 40),
    "discrete": (3, dict(action_mode=0, discrete_table=TABLE), None, 64, 40),
    "u8_disabled": (2, dict(mask_dtype="uint8", autoreset=0), None, 64, 30),
    "gray": (4, dict(obs_mode=1), None, 32, 30),
    "rgb": (3, dict(obs_mode=2), None, 32, 30),
    "shaping_truncation": (4, dict(action_mode=0, discrete_table=TABLE, reward_mode=1,
                                   reward_params={"max_actions": 10}), None, 64, 30),
    "traj0": (8, dict(trajectory_steps=0), None, 32, 25),
    "traj8": (3, dict(trajectory_steps=8), None, 32, 25),
    "jaywalk_stop_return": (4, dict(trajectory_steps=0), "jaywalk", 32, 40),
    "red_light_runner": (4, {}, "red_light_runner", 32, 30),
    "size64": (2, dict(size=64, max_actors=16), "rdm64", 32, 30),
    "size256": (4, dict(size=256, max_actors=16), "rdm256", 32, 25),
    "c3_wide": (4, dict(max_actors=25, trajectory_steps=0, mask_dtype="uint8"), "c3", 64, 25),
}


def _scenes(name):
    from carlabev_env_b200.scenes import build_pool

    if name is None:
        return _scripted(16)
    if name == "jaywalk":
        return _scripted(16, kinds=[("jaywalk", 3 + i % 2) for i in range(16)])
    if name == "red_light_runner":
        return build_pool([dict(scene="red_light_runner", scene_seed=i) for i in range(8)], pad=182)
    if name.startswith("rdm"):
        return _rdm(int(name[3:]))
    from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options

    return build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                       for i in range(8)], pad=182)


@pytest.mark.parametrize("case", list(CASES))
def test_agent_step_equals_k_single_steps(case):
    K, kw, which, n, steps = CASES[case]
    scenes = _scenes(which)
    if which == "red_light_runner":
        kw = dict(kw, max_actors=max(len(s["act_kind"]) for s in scenes))
    a, b = _pair(scenes, n, **kw)
    chk = _run(a, b, np.random.default_rng(list(CASES).index(case)), steps, K)
    episodes = chk.check_stats()
    if case in ("f32", "discrete", "shaping_truncation"):
        assert episodes > 0 and chk.ends_inside > 0, "want episodes that end inside a repeat"
    a.close()
    b.close()


def test_switching_repeat_between_calls():
    from carlabev_env_b200 import engine as E

    a, b = _pair(_scripted(16), 48, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                 reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 14})
    chk = _run(a, b, np.random.default_rng(11), 36, [4, 1, 3])
    assert chk.check_stats() > 0 and a.action_repeat == 3
    a.close()
    b.close()


def test_flag_1024_at_repeat_1_equals_the_three_launch_step():
    """k_step_repeat at K = 1 against today's k_move + k_judge + raster step over 240 steps with auto-resets: every
    output buffer, the whole ring and the snapshot rows byte for byte, the statistics with exact counts."""
    import torch

    a, b = _pair(_scripted(16), 64)
    a.set_debug_flags(1024)
    rng = np.random.default_rng(2)
    step_launches = np.zeros(2, dtype=np.int64)  # launches of the step calls alone (snapshots launch too)
    resets = 0
    for s in range(240):
        acts = _plan_actions(a, rng, 1, a.N)[0]
        l0 = np.array([a.launches, b.launches])
        a.step(acts)
        b.step(acts)
        step_launches += np.array([a.launches, b.launches]) - l0
        for k in ("reward", "terminated", "truncated", "cause", "hero", "episode"):
            assert torch.equal(getattr(a, k), getattr(b, k)), (s, k)
        assert a.head == b.head and torch.equal(a.obs(), b.obs()), s
        if s >= 2 * a.L:  # by then every ring slot has been written (the rest of the ring starts uninitialised)
            assert torch.equal(a.ring, b.ring), s
        resets += int(a.terminated.sum())
        if s % 40 == 39:
            assert torch.equal(a.snapshot().data, b.snapshot().data), s
    assert resets > 0
    assert step_launches.tolist() == [2 * 240, 3 * 240]
    _same_stats(a.read_stats().cpu().numpy(), b.read_stats().cpu().numpy(), "statistics")
    a.close()
    b.close()


def test_profile_reports_the_fused_kernel_as_move():
    a, b = _pair(_scripted(8), 16)
    b.close()
    a.set_action_repeat(4)
    a.profile(True)
    rng = np.random.default_rng(4)
    for _ in range(5):
        a.step(_plan_actions(a, rng, 1, a.N)[0])
    move, render, judge, n = a.profile_read()
    assert n == 5 and move > 0 and render > 0 and judge == 0.0
    a.close()


@pytest.mark.parametrize("workload", ["c2", "c3"])
def test_scale(workload):
    """4096 envs on the c2 workload (lead_brake pool, continuous, float32 masks) and 8192 on a c3-style pool
    (25-vehicle rt_hard_v1 scenes stepped live: the 32-lane path, discrete, uint8 masks), a few agent steps at K = 4."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    def make(n, **kw):
        eng = E.Engine(n, ring_slots=7, autoreset=E.AUTORESET_NEXT_STEP, seed=0, **kw)
        eng.upload_map(load_town01_map(128))
        return eng

    if workload == "c2":
        n, k = 4096, 1024
        a, b = (make(n, action_mode=E.ACTION_CONTINUOUS, max_actors=4) for _ in range(2))
        for eng in (a, b):
            eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    else:
        from carlabev_env_b200.pool import pack_pool

        n, k = 8192, 32
        packed = pack_pool(_scenes("c3"))
        table = np.asarray([[0, 0, 0], [1, 0, 0], [0.5, -1, 0], [0.5, 1, 0], [0, 0, 1]], dtype=np.float32)
        a, b = (make(n, action_mode=E.ACTION_DISCRETE, discrete_table=table, max_actors=25, trajectory_steps=0,
                     mask_dtype="uint8") for _ in range(2))
        for eng in (a, b):
            eng.upload_pool(packed)
        k = 8
    ids = np.arange(n, dtype=np.int32) % k
    a.reset(ids)
    b.reset(ids)
    chk = _run(a, b, np.random.default_rng(1), 6, 4)
    chk.check_stats()
    a.close()
    b.close()


def test_make_env_action_repeat():
    """episode["l"] == ceil(length / 4), host rewards equal the device rewards, the masked-reset flow of autoreset
    "disabled", and ValueError for a repeat outside [1, 64]."""
    import torch

    from carlabev_env_b200.config import EnvConfig, RunConfig
    from carlabev_env_b200.vector_env import make_env

    scenes = _scripted(8)
    cfg = RunConfig(env=EnvConfig(action_mode="continuous"), num_envs=16)
    for bad in (0, 65, 2.5):
        with pytest.raises(ValueError, match="action_repeat"):
            make_env(cfg, scenes=scenes, action_repeat=bad, ring_budget_bytes=32 << 20)
    envs = make_env(cfg, scenes=scenes, action_repeat=4, ring_budget_bytes=32 << 20)
    assert envs.engine.action_repeat == 4
    obs, _ = envs.reset(options={"scene": "pool"})
    rng = np.random.default_rng(0)
    ended = 0
    for _ in range(60):
        a = np.stack([rng.uniform(0, 1, 16), rng.uniform(-1, 1, 16), rng.uniform(0, 1, 16)], 1).astype(np.float32)
        obs, rew, term, trunc, infos = envs.step(a)
        assert np.array_equal(envs.engine.host_reward.numpy(), rew.cpu().numpy())
        done = (term | trunc).cpu().numpy()
        if done.any():
            ep, info = infos["episode"], infos["episode_info"]
            i = np.flatnonzero(done)
            assert np.array_equal(ep["l"][i], -(-info["length"][i] // 4)), (ep["l"][i], info["length"][i])
            assert np.array_equal(ep["r"][i], info["return"][i])
            ended += len(i)
            with pytest.raises(AssertionError):
                envs.step(a)  # autoreset "disabled": terminated envs must be reset first
            obs, _ = envs.reset(options={"scene": "pool", "reset_mask": done})
            assert isinstance(obs, torch.Tensor)
    assert ended > 0
    envs.close()
