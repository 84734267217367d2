"""Observation-free lookahead (Engine.lookahead / cbev_lookahead) on the GPU.

The reference for every branch is the engine itself: the roots' snapshot rows are restored as clones into the envs of
the same engine (auto-reset disabled) and stepped with the same actions.  Rewards of the steps taken, and flags, cause
and hero block of the last one, must be bit-identical; rewards after the last step are exactly 0.  Also: `ret`
reproduced in NumPy, the live engine left byte-identical (against a twin engine that never looked ahead), the oracle,
edge cases, and scale."""
import copy

import numpy as np
import pytest

from golden_util import load_map
from test_gpu_snapshot import _actions, _rdm, _scripted, _two_walkers

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]


def _engine(scenes, n, size=128, **kw):
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    args = dict(mask_mode="6-class", frame_stack=4, ring_slots=7, action_mode=E.ACTION_CONTINUOUS,
                autoreset=E.AUTORESET_DISABLED, max_actors=4, seed=3, size=size)
    args.update(kw)
    eng = E.Engine(n, **args)
    eng.upload_map(load_map(size))
    eng.upload_pool(pack_pool(scenes))
    return eng


def _plan_actions(eng, rng, H, B):
    import torch

    from carlabev_env_b200 import engine as E

    if eng.action_mode == E.ACTION_DISCRETE:
        return torch.from_numpy(rng.integers(0, eng.cfg.n_discrete, size=(H, B))).cuda()
    a = np.stack([rng.uniform(0, 1, (H, B)), rng.uniform(-1, 1, (H, B)), rng.uniform(0, 1, (H, B))], axis=2)
    return torch.from_numpy(a.astype(np.float32)).cuda()


def _warm(eng, rng, k):
    import torch

    from carlabev_env_b200 import engine as E

    for _ in range(k):
        if eng.action_mode == E.ACTION_DISCRETE:
            eng.step(torch.from_numpy(rng.integers(0, eng.cfg.n_discrete, size=eng.N)).cuda())
        else:
            eng.step(_actions(rng, eng.N))


def _stepping_reference(eng, snap, roots, acts):
    """Per-step reward / flags / cause / hero of each branch, from clones of the root rows stepped in the live engine
    (chunks of at most N branches).  Restores the whole snapshot afterwards."""
    import torch

    H, B = acts.shape[0], acts.shape[1]
    N = eng.N
    rew = np.zeros((H, B))
    term = np.zeros((H, B), bool)
    trunc = np.zeros((H, B), bool)
    cause = np.zeros((H, B), np.uint8)
    hero = np.zeros((H, B, eng.hero.shape[1]))
    for c0 in range(0, B, N):
        c1 = min(B, c0 + N)
        k = c1 - c0
        eng.restore(snap, env_ids=np.arange(k), rows=roots[c0:c1])
        for t in range(H):
            a = torch.zeros((N,) + tuple(acts.shape[2:]), dtype=acts.dtype, device=acts.device)
            a[:k] = acts[t, c0:c1]
            eng.step(a)
            rew[t, c0:c1] = eng.reward[:k].cpu().numpy()
            term[t, c0:c1] = eng.terminated[:k].cpu().numpy().astype(bool)
            trunc[t, c0:c1] = eng.truncated[:k].cpu().numpy().astype(bool)
            cause[t, c0:c1] = eng.cause[:k].cpu().numpy()
            hero[t, c0:c1] = eng.hero[:k].cpu().numpy()
    eng.restore(snap)
    return rew, term, trunc, cause, hero


def _check_against_stepping(eng, rng, roots, H, gamma=1.0):
    """Lookahead from `roots` with random actions against the stepping reference; returns (lookahead, rewards)."""
    B = len(roots)
    snap = eng.snapshot()
    done = snap.header().cpu().numpy()[:, 2].astype(bool)
    acts = _plan_actions(eng, rng, H, B)
    la = eng.lookahead(acts, env_ids=roots, gamma=gamma, rewards=True, hero=True)
    rew, term, trunc, cause, hero = _stepping_reference(eng, snap, roots, acts)
    steps = la.steps.cpu().numpy()
    L_rew = la.reward.cpu().numpy()
    L_term, L_trunc = la.terminated.cpu().numpy(), la.truncated.cpu().numpy()
    L_cause, L_hero = la.cause.cpu().numpy(), la.hero.cpu().numpy()
    for b in range(B):
        s = int(steps[b])
        if done[roots[b]]:
            assert s == 0 and not L_term[b] and not L_trunc[b] and L_cause[b] == 0, b
            assert not L_rew[:, b].any() and not L_hero[b].any() and la.ret[b].item() == 0.0, b
            continue
        ends = np.flatnonzero(term[:, b] | trunc[:, b])
        expect = int(ends[0]) + 1 if len(ends) else H
        assert s == expect, (b, s, expect)
        assert np.array_equal(L_rew[:s, b], rew[:s, b]), (b, "reward")
        assert np.all(L_rew[s:, b] == 0.0), (b, "reward after the last step")
        assert L_term[b] == term[s - 1, b] and L_trunc[b] == trunc[s - 1, b] and L_cause[b] == cause[s - 1, b], b
        assert np.array_equal(L_hero[b], hero[s - 1, b]), (b, "hero")
    return la, L_rew


def _ret_numpy(rew, steps, gamma):
    out = np.zeros(rew.shape[1])
    for b in range(rew.shape[1]):
        r, w = 0.0, 1.0
        for t in range(int(steps[b])):
            r = r + w * rew[t, b]
            w = w * gamma
        out[b] = r
    return out


CASES = ["carl_continuous", "carl_discrete", "shaping_truncation", "traj0", "traj8", "jaywalk_stop_return",
         "red_light_runner", "size64", "size256", "rdm25_wide"]


@pytest.mark.parametrize("case", CASES)
def test_branches_equal_stepping_bit_for_bit(case):
    from carlabev_env_b200 import engine as E

    n, size, kw, scenes, warm, H = 32, 128, {}, None, 12, 40
    if case == "carl_discrete" or case == "shaping_truncation":
        table = np.asarray([[0, 0, 0], [1, 0, 0], [0.5, -1, 0], [0.5, 1, 0], [0, 0, 1], [1, -0.5, 0], [1, 0.5, 0]],
                           dtype=np.float32)
        kw.update(action_mode=E.ACTION_DISCRETE, discrete_table=table)
    if case == "shaping_truncation":
        kw.update(reward_mode=E.REWARD_SHAPING, reward_params={"max_actions": 30})
        warm, H = 10, 32  # max_actions falls inside the horizon
    elif case == "traj0":
        kw["trajectory_steps"] = 0
    elif case == "traj8":
        kw["trajectory_steps"] = 8
        warm = 3  # the table -> live hand-over (episode step 8) happens inside the horizon
    elif case == "jaywalk_stop_return":
        scenes = _scripted(16, kinds=[("jaywalk", 3 + i % 2) for i in range(16)])
        kw["trajectory_steps"] = 0
        warm, H = 8, 64  # walkers yield, then start their retreat inside the horizon
    elif case == "red_light_runner":
        from carlabev_env_b200.scenes import build_pool

        scenes = build_pool([dict(scene="red_light_runner", scene_seed=i) for i in range(8)], pad=182)
        kw["max_actors"] = max(len(s["act_kind"]) for s in scenes)
    elif case in ("size64", "size256"):
        size = 64 if case == "size64" else 256
        scenes, kw["max_actors"] = _rdm(size), 16
    elif case == "rdm25_wide":
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options
        from carlabev_env_b200.scenes import build_pool

        scenes = build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                             for i in range(8)], pad=182)
        kw.update(max_actors=25, trajectory_steps=0)  # live actors, > 8 per scene: the 32-lane groups
    if scenes is None:
        scenes = _scripted(16)
    eng = _engine(scenes, n, size=size, **kw)
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(CASES.index(case))
    _warm(eng, rng, warm)
    # identity roots, then random repeated roots (more branches than envs)
    _check_against_stepping(eng, rng, np.arange(n), H)
    _check_against_stepping(eng, rng, rng.integers(0, n, size=3 * n // 2), H)
    eng.close()


@pytest.mark.parametrize("gamma", [1.0, 0.99])
def test_ret_is_reproduced_from_reward_in_numpy(gamma):
    eng = _engine(_scripted(16), 48)
    eng.reset(np.arange(48, dtype=np.int32) % 16)
    rng = np.random.default_rng(5)
    _warm(eng, rng, 10)
    la, rew = _check_against_stepping(eng, rng, rng.integers(0, 48, size=64), 48, gamma=gamma)
    steps = la.steps.cpu().numpy()
    assert (steps < 48).any() and (steps == 48).any(), "want branches that end early and branches that run out"
    assert np.array_equal(la.ret.cpu().numpy(), _ret_numpy(rew, steps, gamma))
    eng.close()


def _live_state(eng):
    import torch

    torch.cuda.synchronize()
    return {"rows": eng.snapshot().data.clone(), "ring": eng.ring.clone(), "stats": eng.read_stats().clone(),
            "reward": eng.reward.clone(), "terminated": eng.terminated.clone(), "hero": eng.hero.clone(),
            "head": eng.head}


def _same_state(a, b, what, twin=False):
    """Byte-identical, except the statistics vector of two different engines: its sums are accumulated with atomics
    in whatever order the envs finish, so twins agree only to rounding."""
    import torch

    for k in a:
        if k == "head":
            same = a[k] == b[k]
        elif k == "stats" and twin:
            same = torch.allclose(a[k], b[k], rtol=1e-12, atol=0.0)
        else:
            same = torch.equal(a[k], b[k])
        assert same, (what, k)


def test_live_engine_is_untouched():
    from carlabev_env_b200 import engine as E

    scenes = _scripted(16)
    n = 64
    engs = [_engine(scenes, n, autoreset=E.AUTORESET_NEXT_STEP) for _ in range(2)]
    rng = np.random.default_rng(17)
    for e in engs:
        e.reset(np.arange(n, dtype=np.int32) % len(scenes))
    for _ in range(25):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
    before = _live_state(engs[0])
    launches = engs[0].launches
    acts = _plan_actions(engs[0], rng, 64, 4 * n)  # long enough that many branches end an episode
    la = engs[0].lookahead(acts, env_ids=rng.integers(0, n, size=4 * n), rewards=True, hero=True)
    assert (la.terminated.cpu().numpy() & (la.steps.cpu().numpy() > 0)).any(), "no branch ended an episode"
    assert engs[0].launches == launches + 1
    _same_state(before, _live_state(engs[0]), "after lookahead")
    _same_state(_live_state(engs[1]), _live_state(engs[0]), "twin", twin=True)
    a = _actions(rng, n)
    for e in engs:
        e.step(a)
    _same_state(_live_state(engs[1]), _live_state(engs[0]), "one step later", twin=True)
    # the snapshot / step / restore recipe, by contrast, counts planning episodes in the statistics
    snap = engs[0].snapshot()
    stats0 = engs[0].read_stats().clone()
    for t in range(64):
        engs[0].step(acts[t, :n].contiguous())
    engs[0].restore(snap)
    assert not (engs[0].read_stats() == stats0).all(), "the clone/step/restore recipe left the statistics alone"
    for e in engs:
        e.close()


def test_branches_match_the_oracle():
    """Branches cloned from one source env, tracked by an OracleEnv, against deep copies of that oracle."""
    import torch

    from oracle.env import OracleEnv

    scenes = _scripted(16)
    n = 32
    eng = _engine(scenes, n)
    ids = np.arange(n) % len(scenes)
    eng.reset(ids.astype(np.int32))
    rng = np.random.default_rng(21)
    hist, alive = [], np.ones(n, bool)
    for _ in range(10):
        a = _actions(rng, n)
        eng.step(a)
        hist.append(a.cpu().numpy())
        alive &= ~(eng.terminated | eng.truncated).cpu().numpy().astype(bool)
    s = int(np.flatnonzero(alive)[0])
    oracle = OracleEnv(load_map(), action_mode="continuous")
    oracle.reset(scenes[ids[s]])
    for a in hist:
        oracle.step(a[s])
    B, H = 8, 30
    acts = _plan_actions(eng, rng, H, B)
    la = eng.lookahead(acts, env_ids=torch.full((B,), s, dtype=torch.int32, device=eng.device), rewards=True, hero=True)
    rew, steps, hero = la.reward.cpu().numpy(), la.steps.cpu().numpy(), la.hero.cpu().numpy()
    a_h = acts.cpu().numpy()
    for b in range(B):
        c = copy.deepcopy(oracle)
        for t in range(int(steps[b])):
            _, r, te, tr, _ = c.step(a_h[t, b])
            assert abs(r - rew[t, b]) < 1e-9, (b, t, r, rew[t, b])
            if te or tr:
                assert t + 1 == steps[b], (b, t)
                break
        ego = c.sim.ego
        assert np.allclose(hero[b, :4], [ego.x, ego.y, ego.yaw, ego.v], rtol=1e-9, atol=1e-9), b
    eng.close()


def test_edge_cases_and_argument_errors():
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    scenes = _scripted(12, kinds=[("jaywalk", 3)] * 12)
    n = 24
    eng = _engine(scenes, n, trajectory_steps=0)
    acts = _plan_actions(eng, np.random.default_rng(0), 4, n)
    with pytest.raises(E.CbevError, match="cbev error 3.*first reset"):
        eng.lookahead(acts)
    eng.reset(np.arange(n, dtype=np.int32) % len(scenes))
    rng = np.random.default_rng(9)
    # drive until some envs have ended their episode (autoreset disabled: they wait for a reset)
    for _ in range(200):
        eng.step(_actions(rng, n))
        done = eng.snapshot().header().cpu().numpy()[:, 2].astype(bool)
        if done.any() and not done.all():
            break
    assert done.any() and not done.all()
    la = eng.lookahead(_plan_actions(eng, rng, 6, n), rewards=True, hero=True)
    assert np.array_equal(la.steps.cpu().numpy() == 0, done)
    # B > N with repeated roots, and the branch state growing with B and with the retreat slots
    _check_against_stepping(eng, rng, rng.integers(0, n, size=5 * n), 24)
    grown = scenes + [_two_walkers(scenes[i], scenes[i + 1]) for i in range(0, 4, 2)]
    eng.upload_pool(pack_pool(grown))  # append-only: per-env retreat slots 1 -> 2
    eng.reset(np.arange(n, dtype=np.int32) % len(grown))
    _warm(eng, rng, 8)
    _check_against_stepping(eng, rng, rng.integers(0, n, size=6 * n), 40)
    # device roots out of range: steps = 0, nothing written out of bounds
    bad = torch.tensor([-1, n, 0, 10 ** 6], dtype=torch.int32, device=eng.device)
    la = eng.lookahead(_plan_actions(eng, rng, 3, 4), env_ids=bad)
    assert la.steps.cpu().tolist()[:2] == [0, 0] and la.steps[3].item() == 0
    # out= reuse
    acts = _plan_actions(eng, rng, 5, 16)
    r1 = eng.lookahead(acts, env_ids=np.arange(16), rewards=True)
    r2 = eng.lookahead(acts, env_ids=np.arange(16), rewards=True, out=r1)
    assert r2 is r1
    # host-side errors
    with pytest.raises(ValueError, match=r"\[0, 24\)"):
        eng.lookahead(acts, env_ids=np.arange(15, 31))
    with pytest.raises(ValueError, match="16 branches"):
        eng.lookahead(acts, env_ids=np.arange(8))
    with pytest.raises(ValueError, match="float32"):
        eng.lookahead(acts.double())
    with pytest.raises(ValueError, match="float32"):
        eng.lookahead(acts[:, :, :2].contiguous())
    with pytest.raises(ValueError, match="CUDA"):
        eng.lookahead(acts.cpu())
    with pytest.raises(ValueError, match="finite"):
        eng.lookahead(acts, gamma=float("nan"))
    with pytest.raises(ValueError, match="envs"):
        eng.lookahead(_plan_actions(eng, rng, 2, n + 1))
    with pytest.raises(ValueError, match="reward"):
        eng.lookahead(_plan_actions(eng, rng, 7, 16), rewards=True, out=r1)
    eng.close()


@pytest.mark.parametrize("workload", ["c2", "c3"])
def test_scale(workload):
    """4096 branches on the c2 workload (lead_brake pool, continuous) and 8192 on a c3-style pool (25-vehicle rt_hard_v1
    scenes, discrete), H = 32, against the stepping reference."""
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.vector_env import load_town01_map

    if workload == "c2":
        n = 4096
        eng = E.Engine(n, ring_slots=7, action_mode=E.ACTION_CONTINUOUS, autoreset=E.AUTORESET_DISABLED, max_actors=4,
                       seed=0, mask_dtype="uint8")
        eng.upload_map(load_town01_map(128))
        k = 1024
        eng.generate_scripted_pool(["lead_brake"] * k, [1 + i % 3 for i in range(k)], list(range(k)))
    else:
        from carlabev_env_b200.pool import pack_pool
        from carlabev_env_b200.reset import RandomNavigationReset, build_reset_options
        from carlabev_env_b200.scenes import build_pool

        n, k = 8192, 32
        scenes = build_pool([build_reset_options(RandomNavigationReset(difficulty_id="rt_hard_v1", scene_seed=i))
                             for i in range(k)], pad=182)
        table = np.asarray([[0, 0, 0], [1, 0, 0], [0.5, -1, 0], [0.5, 1, 0], [0, 0, 1]], dtype=np.float32)
        eng = E.Engine(n, ring_slots=7, action_mode=E.ACTION_DISCRETE, discrete_table=table,
                       autoreset=E.AUTORESET_DISABLED, max_actors=25, seed=0, mask_dtype="uint8")
        eng.upload_map(load_town01_map(128))
        eng.upload_pool(pack_pool(scenes))
    eng.reset(np.arange(n, dtype=np.int32) % k)
    rng = np.random.default_rng(1)
    _warm(eng, rng, 10)
    _check_against_stepping(eng, rng, np.arange(n), 32)
    eng.close()
