"""Lookahead in agent steps of action repeat K (Engine.lookahead(repeat=K) / cbev_lookahead_repeat) on the GPU.

The reference is a twin engine of the same configuration, seed and pool at set_action_repeat(K) with auto-reset
disabled.  The planner's snapshot rows are restored into the twin under the twin's own info (rows restore only into
the engine that took them, and the twin has the planner's layout), and the twin is stepped with each branch's action
rows, one agent step per call.  Rewards, ret, steps, flags, cause, hero, the leaf windows (raw and fused) and the leaf
rows must be the twin's bit for bit."""
import numpy as np
import pytest

from test_gpu_action_repeat import _frames
from test_gpu_lookahead import _live_state, _plan_actions, _ret_numpy, _same_state, _stepping_reference, _warm
from test_gpu_lookahead_obs import TABLE, _engine, _reference
from test_gpu_lookahead_rows import SENTINEL, EnvSnapshotCopy, _leaf_reference, _results, _same_results
from test_gpu_snapshot import _rdm, _scripted, _two_walkers

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]


class Twin:
    """Engine `b` at action repeat K standing in for the env the contract names: restore the root, step, read."""

    def __init__(self, a, b, K):
        from carlabev_env_b200 import engine as E

        self.E, self.a, self.b = E, a, b
        b.set_action_repeat(K)
        self.info = b.snapshot().info

    def rows(self, snap):
        """`snap` of the planner under the twin's info."""
        return self.E.EnvSnapshot(snap._buf, self.info)

    def check(self, la, snap, roots, acts, gamma, root_obs, fuse=None):
        """Every output of `la` (a call from the live roots `roots` of the planner when it had snapshot `snap`) against
        the twin.  Returns the agent steps taken."""
        import torch

        b = self.b
        roots = np.asarray(roots)
        B, H = len(roots), acts.shape[0]
        valid = (roots >= 0) & (roots < b.N)
        done = np.ones(B, bool)
        done[valid] = snap.header().cpu().numpy()[roots[valid], 2].astype(bool)
        steps = la.steps.cpu().numpy()
        sb = self.rows(snap)
        if valid.all():
            rew, term, trunc, cause, hero = _stepping_reference(b, sb, roots, acts)
            L = {k: getattr(la, k).cpu().numpy() for k in ("reward", "terminated", "truncated", "cause", "hero")}
            for i in range(B):
                s = int(steps[i])
                if done[i]:
                    assert s == 0 and not L["reward"][:, i].any() and not L["hero"][i].any(), i
                    continue
                ends = np.flatnonzero(term[:, i] | trunc[:, i])
                assert s == (int(ends[0]) + 1 if len(ends) else H), (i, s)
                assert np.array_equal(L["reward"][:s, i].view(np.int64), rew[:s, i].view(np.int64)), (i, "reward")
                assert not L["reward"][s:, i].any(), (i, "reward after the last step")
                assert (L["terminated"][i], L["truncated"][i], L["cause"][i]) == \
                       (term[s - 1, i], trunc[s - 1, i], cause[s - 1, i]), i
                assert np.array_equal(L["hero"][i], hero[s - 1, i]), (i, "hero")
            ret = _ret_numpy(L["reward"], steps, gamma)
            assert np.array_equal(la.ret.cpu().numpy().view(np.int64), ret.view(np.int64)), "ret"
        else:
            assert not steps[~valid].any() and not la.ret.cpu().numpy()[~valid].any()
        if la.obs is not None:
            ref = _reference(b, sb, roots, acts, steps, root_obs, fuse)
            bad = [i for i in range(B) if not torch.equal(la.obs[i], ref[i])]
            assert not bad, ("leaf window", len(bad), bad[:8], steps[bad[:8]])
        if la.leaf is not None:
            ref = _leaf_reference(b, sb, roots, acts, steps, valid)
            bad = [i for i in range(B) if not torch.equal(la.leaf.data[i], ref[i])]
            assert not bad, ("leaf row", len(bad), bad[:8], steps[bad[:8]])
        return steps


def _pair(scenes, n, **kw):
    a, b = _engine(scenes, n, **kw), _engine(scenes, n, **kw)
    ids = np.arange(n, dtype=np.int32) % len(scenes)
    a.reset(ids)
    b.reset(ids)
    return a, b


def _call(a, acts, K, roots, gamma=1.0, fuse=None, **kw):
    snap = a.snapshot()
    root_obs = (a.obs() if fuse is None else a.fuse(fuse)).clone()
    la = a.lookahead(acts, env_ids=roots, gamma=gamma, rewards=True, hero=True, obs=True, fuse=fuse, leaf=True,
                     repeat=K, **kw)
    return la, snap, root_obs


CASES = {
    # name: (K, kwargs of _engine, scenes, envs, warm-up steps, horizon)
    "f32": (4, {}, None, 32, 12, 16),
    "discrete": (3, dict(action_mode=0, discrete_table=TABLE), None, 32, 12, 16),
    "u8": (2, dict(mask_dtype="uint8"), None, 32, 10, 16),
    "gray": (4, dict(obs_mode=1), None, 32, 10, 12),
    "rgb": (3, dict(obs_mode=2), None, 24, 10, 12),
    "shaping_truncation": (4, dict(action_mode=0, discrete_table=TABLE, reward_mode=1,
                                   reward_params={"max_actions": 23}), None, 32, 2, 12),
    "traj8": (3, dict(trajectory_steps=8), None, 32, 1, 12),
    "jaywalk_stop_return": (8, dict(trajectory_steps=0), "jaywalk", 16, 8, 12),
    "red_light_runner": (4, {}, "red_light_runner", 16, 6, 12),
    "size64": (2, dict(size=64, max_actors=16), "rdm64", 24, 6, 12),
    "size256": (4, dict(size=256, max_actors=16), "rdm256", 16, 6, 10),
    "c3_wide": (4, dict(max_actors=25, trajectory_steps=0, mask_dtype="uint8"), "c3", 32, 6, 12),
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
def test_agent_steps_equal_the_twin_at_repeat_k(case):
    """Live roots, repeated (B > N), with per-step rewards, hero, leaf windows and leaf rows; gamma != 1."""
    K, kw, which, n, warm, H = CASES[case]
    scenes = _scenes(which)
    if which == "red_light_runner":
        kw = dict(kw, max_actors=max(len(s["act_kind"]) for s in scenes))
    a, b = _pair(scenes, n, **kw)
    rng = np.random.default_rng(list(CASES).index(case))
    _warm(a, rng, warm)
    twin = Twin(a, b, K)
    roots = rng.integers(0, n, size=3 * n // 2)
    acts = _plan_actions(a, rng, H, len(roots))
    before = _live_state(a)
    la, snap, root_obs = _call(a, acts, K, roots, gamma=0.97)
    _same_state(before, _live_state(a), "live engine")
    steps = twin.check(la, snap, roots, acts, 0.97, root_obs)
    if case in ("f32", "discrete", "shaping_truncation"):
        ended = (la.terminated | la.truncated).cpu().numpy()
        assert ended.any() and (steps < H).any(), "want branches that end inside the horizon"
    if case == "shaping_truncation":  # max_actions counts simulator steps: every branch ends inside the horizon
        assert (la.terminated | la.truncated).cpu().numpy().all() and la.truncated.any()
    a.close()
    b.close()


@pytest.mark.parametrize("fuse", ["vehicle_temporal", "vehicle_weighted"])
def test_fused_leaf_windows_equal_the_twin(fuse):
    a, b = _pair(_scripted(16), 24)
    rng = np.random.default_rng(7)
    _warm(a, rng, 9)
    twin = Twin(a, b, 3)
    roots = rng.integers(0, 24, size=30)
    acts = _plan_actions(a, rng, 9, 30)
    la, snap, root_obs = _call(a, acts, 3, roots, fuse=fuse)
    twin.check(la, snap, roots, acts, 1.0, root_obs, fuse=fuse)
    raw = a.lookahead(acts, env_ids=roots, obs=True, repeat=3)
    import torch

    assert torch.equal(raw.obs, la.window)
    a.close()
    b.close()


def test_terminations_inside_a_repeat_and_at_sub_step_k():
    """Roots one simulator step apart in episode length: shaping's max_actions truncation (and collisions) end the
    branches at every sub-step position of a repeat of 4, K - 1 of them inside it; the position is read from a
    repeat-1 call over the tiled actions (steps taken there are simulator steps)."""
    from carlabev_env_b200 import engine as E

    n, K, H = 32, 4, 12
    a, b = _pair(_scripted(16), n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                 reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 40})
    rng = np.random.default_rng(21)
    twin = Twin(a, b, K)
    positions = set()
    for _ in range(K):
        _warm(a, rng, 1)
        roots = np.arange(n)
        acts = _plan_actions(a, rng, H, n)
        la, snap, root_obs = _call(a, acts, K, roots)
        twin.check(la, snap, roots, acts, 1.0, root_obs)
        s1 = a.lookahead(acts.repeat_interleave(K, dim=0).contiguous(), env_ids=roots).steps.cpu().numpy()
        ended = (la.terminated | la.truncated).cpu().numpy() & (s1 > 0)
        positions |= set(((s1[ended] - 1) % K + 1).tolist())
    assert positions == set(range(1, K + 1)), positions
    a.close()
    b.close()


def test_rewards_equal_the_tiled_repeat_1_call():
    """Without the twin: reward[t] at repeat K is the in-order sum of a repeat-1 call's rewards over the action rows
    tiled K times, up to the first terminal sub-step; ret follows per agent step."""
    from carlabev_env_b200 import engine as E

    n, K, H = 32, 3, 10
    eng = _engine(_scripted(16), n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                  reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 30})
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(13)
    _warm(eng, rng, 5)
    roots = rng.integers(0, n, size=48)
    acts = _plan_actions(eng, rng, H, 48)
    la = eng.lookahead(acts, env_ids=roots, gamma=0.9, rewards=True, repeat=K)
    tiled = eng.lookahead(acts.repeat_interleave(K, dim=0).contiguous(), env_ids=roots, rewards=True)
    r1, s1 = tiled.reward.cpu().numpy(), tiled.steps.cpu().numpy()
    rk, sk = la.reward.cpu().numpy(), la.steps.cpu().numpy()
    assert np.array_equal(sk, -(-s1 // K))
    for i in range(48):
        for t in range(int(sk[i])):
            sub = r1[t * K:min((t + 1) * K, int(s1[i])), i]
            acc = sub[0]
            for x in sub[1:]:
                acc = acc + x
            assert rk[t, i] == acc, (i, t)
    assert np.array_equal(la.ret.cpu().numpy(), _ret_numpy(rk, sk, 0.9))
    for k in ("terminated", "truncated", "cause"):
        assert np.array_equal(getattr(la, k).cpu().numpy(), getattr(tiled, k).cpu().numpy()), k
    assert (la.truncated.cpu().numpy()).any()
    eng.close()


def test_terminal_roots_and_invalid_device_roots():
    import torch

    from carlabev_env_b200 import engine as E

    n, K = 16, 4
    a, b = _pair(_scripted(16), n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                 reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 48})
    rng = np.random.default_rng(3)
    _warm(a, rng, 5)
    twin = Twin(a, b, K)
    bad = torch.tensor([-1, n, 0, 10 ** 6, 3, 7], dtype=torch.int32, device=a.device)
    acts = _plan_actions(a, rng, 6, 6)
    la, snap, root_obs = _call(a, acts, K, bad)
    la.leaf._buf.fill_(SENTINEL)
    la = a.lookahead(acts, env_ids=bad, rewards=True, hero=True, obs=True, leaf=True, repeat=K, out=la)
    twin.check(la, snap, bad.cpu().numpy(), acts, 1.0, root_obs)
    assert la.steps.cpu().numpy()[[0, 1, 3]].tolist() == [0, 0, 0] and not la.obs[[0, 1, 3]].any()
    assert (la.leaf.data[[0, 1, 3]] == SENTINEL).all()
    # rows: done rows, out-of-range rows and header scenes outside the pool
    rows = snap.data.clone()
    hdr = rows[:, :12].view(torch.int32)
    hdr[1, 0], hdr[2, 0] = -1, 10 ** 6
    forged = E.EnvSnapshot(rows, snap.info)
    roots = torch.tensor([0, 1, 2, -5, n, 4], dtype=torch.int32, device=a.device)
    lr = a.lookahead(acts, source=forged, rows=roots, obs=True, leaf=True, repeat=K)
    lr.leaf._buf.fill_(SENTINEL)
    lr = a.lookahead(acts, source=forged, rows=roots, obs=True, leaf=True, repeat=K, out=lr)
    assert lr.steps.cpu().tolist()[1:5] == [0, 0, 0, 0]
    assert not lr.obs[1:5].any() and (lr.leaf.data[1:5] == SENTINEL).all()
    live = a.lookahead(acts[:, [0, 5]].contiguous(), env_ids=np.array([0, 4]), obs=True, leaf=True, repeat=K)
    assert torch.equal(lr.obs[[0, 5]], live.obs) and torch.equal(lr.leaf.data[[0, 5]], live.leaf.data)
    # every env truncated: terminal live roots and done rows give steps = 0, their own window and their own row
    _warm(a, rng, 44)
    snap = a.snapshot()
    assert snap.header()[:, 2].all()
    roots = rng.integers(0, n, size=24)
    acts = _plan_actions(a, rng, 5, 24)
    for kw in (dict(env_ids=roots), dict(source=snap, rows=roots)):
        lt = a.lookahead(acts, obs=True, leaf=True, rewards=True, repeat=K, **kw)
        assert not lt.steps.any() and not lt.reward.any() and not lt.ret.any()
        assert torch.equal(lt.leaf.data, snap.data[torch.from_numpy(roots).to(a.device)])
        assert torch.equal(lt.obs, a.obs()[torch.from_numpy(roots).to(a.device)])
    a.close()
    b.close()


def test_row_roots_equal_live_roots():
    """A call from snapshot rows, after the live batch moved on, reproduces the call from the live envs the rows were
    taken from, in every mode (no frames, windows, leaf rows)."""
    import torch

    n, K = 24, 3
    eng = _engine(_scripted(16), n)
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(8)
    _warm(eng, rng, 10)
    roots = rng.integers(0, n, size=36)
    acts = _plan_actions(eng, rng, 12, 36)
    snap = eng.snapshot()
    live = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True, leaf=True, repeat=K)
    res, leaf = _results(live), live.leaf.data.clone()
    _warm(eng, rng, 3)
    before = _live_state(eng)
    la = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, obs=True, leaf=True, repeat=K)
    _same_results(res, _results(la), "rows, leaf")
    assert torch.equal(la.leaf.data, leaf)
    lo = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, obs=True, repeat=K)
    _same_results(res, _results(lo), "rows, windows")
    ln = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, repeat=K)
    _same_results({k: v for k, v in res.items() if k != "obs"}, _results(ln), "rows, no frames")
    _same_state(before, _live_state(eng), "rows as roots")
    eng.close()


@pytest.mark.parametrize("R0", [0, 1])
def test_rows_taken_at_fewer_retreat_slots(R0):
    import torch

    from carlabev_env_b200.pool import pack_pool

    kinds = [("lead_brake", 1 + i % 3) for i in range(12)] if R0 == 0 else [("jaywalk", 3)] * 12
    scenes = _scripted(12, kinds=kinds)
    n = 24
    eng = _engine(scenes, n, trajectory_steps=0)
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(9)
    _warm(eng, rng, 9)
    snap = eng.snapshot()
    assert snap.info.retreat_slots == R0
    walkers = _scripted(4, seed0=900, kinds=[("jaywalk", 3)] * 4)
    eng.upload_pool(pack_pool(scenes + [_two_walkers(walkers[i], walkers[i + 1]) for i in range(0, 4, 2)]))
    assert eng.snapshot_row_bytes > snap.row_bytes
    roots = rng.integers(0, n, size=40)
    acts = _plan_actions(eng, rng, 10, 40)
    la = eng.lookahead(acts, source=snap, rows=roots, rewards=True, hero=True, obs=True, leaf=True, repeat=4)
    got, leaf = _results(la), la.leaf.data.clone()
    eng.restore(snap)
    ref = eng.lookahead(acts, env_ids=roots, rewards=True, hero=True, obs=True, leaf=True, repeat=4)
    _same_results(_results(ref), got, "grown pool")
    assert torch.equal(ref.leaf.data, leaf)
    eng.close()


def test_chaining_equals_one_call():
    import torch

    from carlabev_env_b200 import engine as E

    n, K = 32, 3
    eng = _engine(_scripted(16), n, action_mode=E.ACTION_DISCRETE, discrete_table=TABLE,
                  reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 50})
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(5)
    _warm(eng, rng, 6)
    for H1, H2 in ((1, 3), (3, 2), (5, 9)):  # H < F on both sides; truncation inside either part
        roots = rng.integers(0, n, size=48)
        acts = _plan_actions(eng, rng, H1 + H2, 48)
        kw = dict(rewards=True, hero=True, obs=True, leaf=True, repeat=K)
        full = eng.lookahead(acts, env_ids=roots, **kw)
        a = eng.lookahead(acts[:H1].contiguous(), env_ids=roots, **kw)
        b = eng.lookahead(acts[H1:].contiguous(), source=a.leaf, **kw)
        s1, s2 = a.steps.cpu().numpy(), b.steps.cpu().numpy()
        assert np.array_equal(full.steps.cpu().numpy(), s1 + s2)
        rew = torch.cat([a.reward, b.reward])
        assert torch.equal(full.reward, rew)
        assert np.array_equal(full.ret.cpu().numpy(), _ret_numpy(rew.cpu().numpy(), s1 + s2, 1.0))
        cont = torch.from_numpy(s2 > 0).to(eng.device)
        for k in ("terminated", "truncated", "cause"):
            assert torch.equal(getattr(full, k), torch.where(cont, getattr(b, k), getattr(a, k))), k
        assert torch.equal(full.hero, torch.where(cont[:, None], b.hero, a.hero))
        assert torch.equal(full.obs, b.obs)
        assert torch.equal(full.leaf.data, b.leaf.data)
    eng.close()


def test_leaf_row_restored_at_repeat_k_continues_like_the_twin():
    import torch

    n, H, K, M = 24, 6, 4, 5
    a, b = _pair(_scripted(16), n)
    rng = np.random.default_rng(6)
    _warm(a, rng, 7)
    twin = Twin(a, b, K)
    acts = _plan_actions(a, rng, H + M, n)
    live = a.snapshot()
    la = a.lookahead(acts[:H].contiguous(), leaf=True, repeat=K)
    leaf = EnvSnapshotCopy(la.leaf)
    b.restore(twin.rows(live))
    ref = []
    for t in range(H + M):
        b.step(acts[t].contiguous())
        if t >= H:
            ref.append((b.reward.clone(), b.terminated.clone(), b.hero.clone(), _frames(b)))
    keep = torch.from_numpy(la.steps.cpu().numpy() == H).to(a.device)
    assert keep.any()
    a.set_action_repeat(K)
    a.restore(leaf.snap)
    for t in range(M):
        a.step(acts[H + t].contiguous())
        r, te, h, o = ref[t]
        assert torch.equal(a.reward[keep], r[keep]) and torch.equal(a.terminated[keep], te[keep]), t
        assert torch.equal(a.hero[keep], h[keep]) and torch.equal(_frames(a)[keep], o[keep]), t
    a.close()
    b.close()


def test_isolation_and_repeat_1():
    """The live engine is untouched; repeat=1 through cbev_lookahead_repeat is byte-identical to cbev_lookahead_ex;
    the engine's own action repeat changes no lookahead result, and a lookahead does not change it."""
    import ctypes as C

    import torch

    from carlabev_env_b200 import engine as E

    n = 24
    eng = _engine(_scripted(16), n, autoreset=E.AUTORESET_NEXT_STEP)
    eng.reset(np.arange(n, dtype=np.int32) % 16)
    rng = np.random.default_rng(17)
    _warm(eng, rng, 8)
    roots = rng.integers(0, n, size=32)
    acts = _plan_actions(eng, rng, 10, 32)
    kw = dict(env_ids=roots, rewards=True, hero=True, obs=True, leaf=True)
    before = _live_state(eng)
    steps0 = eng.read_stats()[-1].item()
    ex = eng.lookahead(acts, **kw)
    ex_res, ex_leaf = _results(ex), ex.leaf.data.clone()
    r4 = eng.lookahead(acts, repeat=4, **kw)
    r4_res, r4_leaf = _results(r4), r4.leaf.data.clone()
    _same_state(before, _live_state(eng), "after the calls")
    assert eng.read_stats()[-1].item() == steps0 and eng.action_repeat == 1
    # repeat = 1 through the new entry point: same bytes, same launches
    out = {k: torch.full_like(v, 7) for k, v in ex_res.items() if k != "obs"}
    win = torch.full_like(ex.window, 7)
    leaf = torch.full_like(ex.leaf.data, 7)
    o = E.CbevLookaheadOut(*(out[k].data_ptr() for k in ("ret", "reward", "steps", "terminated", "truncated",
                                                          "cause", "hero")))
    info = E.CbevSnapshotInfo()
    ids = torch.from_numpy(roots.astype(np.int32)).to(eng.device)
    io = E.CbevLookaheadIo(None, None, ids.data_ptr(), win.data_ptr(), win.numel() * win.element_size(),
                           leaf.data_ptr(), leaf.numel(), C.pointer(info))
    l0 = eng.launches
    assert eng.lib.cbev_lookahead_repeat(eng.handle, C.byref(io), 32, 10, 1, acts.data_ptr(), 1.0, C.byref(o),
                                         eng._stream()) == 0
    l1 = eng.launches
    assert eng.lib.cbev_lookahead_ex(eng.handle, C.byref(io), 32, 10, acts.data_ptr(), 1.0, C.byref(o),
                                     eng._stream()) == 0
    assert l1 - l0 == eng.launches - l1 == 4
    for k, v in out.items():
        assert torch.equal(v, ex_res[k]), k
    assert torch.equal(win, ex.window) and torch.equal(leaf, ex_leaf)
    l0 = eng.launches
    eng.lookahead(acts, repeat=4, **kw)
    assert eng.launches - l0 == 4
    # the engine's own repeat does not apply to lookahead
    for k in (3, 1):
        eng.set_action_repeat(k)
        _same_results(ex_res, _results(eng.lookahead(acts, **kw)), f"repeat 1 at engine repeat {k}")
        got = eng.lookahead(acts, repeat=4, **kw)
        _same_results(r4_res, _results(got), f"repeat 4 at engine repeat {k}")
        assert torch.equal(got.leaf.data, r4_leaf) and eng.action_repeat == k
    eng.close()


@pytest.mark.parametrize("workload", ["c2", "c3"])
def test_scale(workload):
    """4096 branches on the c2 workload and 8192 on a c3-style pool (25 live vehicles: the 32-lane path) at K = 4;
    a 64-branch sample against the twin."""
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    def make(n, **kw):
        eng = E.Engine(n, ring_slots=7, autoreset=E.AUTORESET_DISABLED, seed=0, **kw)
        eng.upload_map(load_town01_map(128))
        return eng

    if workload == "c2":
        n, B, k = 256, 4096, 256
        a, b = (make(n, action_mode=E.ACTION_CONTINUOUS, max_actors=4) for _ in range(2))
        for eng in (a, b):
            eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    else:
        from carlabev_env_b200.pool import pack_pool

        n, B, k = 256, 8192, 8
        packed = pack_pool(_scenes("c3"))
        table = np.asarray([[0, 0, 0], [1, 0, 0], [0.5, -1, 0], [0.5, 1, 0], [0, 0, 1]], dtype=np.float32)
        a, b = (make(n, action_mode=E.ACTION_DISCRETE, discrete_table=table, max_actors=25, trajectory_steps=0,
                     mask_dtype="uint8") for _ in range(2))
        for eng in (a, b):
            eng.upload_pool(packed)
    ids = np.arange(n, dtype=np.int32) % k
    a.reset(ids)
    b.reset(ids)
    rng = np.random.default_rng(1)
    _warm(a, rng, 3)
    twin = Twin(a, b, 4)
    roots = rng.integers(0, n, size=B)
    acts = _plan_actions(a, rng, 8, B)
    la, snap, root_obs = _call(a, acts, 4, roots)
    sample = np.sort(rng.choice(B, size=64, replace=False))
    sel = torch.from_numpy(sample).to(a.device)
    sub = a.lookahead(acts[:, sel].contiguous(), env_ids=roots[sample], rewards=True, hero=True, obs=True, leaf=True,
                      repeat=4)
    for k2 in ("ret", "reward", "steps", "terminated", "truncated", "cause", "hero", "obs"):
        v = getattr(la, k2)
        v = v[:, sel] if k2 == "reward" else v[sel]
        assert torch.equal(v, getattr(sub, k2)), k2
    assert torch.equal(la.leaf.data[sel], sub.leaf.data)
    twin.check(sub, snap, roots[sample], acts[:, sel].contiguous(), 1.0, root_obs)
    a.close()
    b.close()
