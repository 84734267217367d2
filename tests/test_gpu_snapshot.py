"""Snapshot / restore of whole environments (cbev_snapshot / cbev_restore) on the GPU.

The round trip: step K, snapshot, step M recording every output, restore, replay the same M actions -- observation
windows, rewards, flags, causes, hero blocks and the episode rows of terminal envs must be bit-identical.  K puts the
ring head in the mirror zone at the snapshot, M > L wraps the ring after the restore.  Also: restoring a subset
against a twin engine, cloning one row into every env (identical actions against the source, different actions
against deep copies of the oracle), the host state read-back, pool growth and the pool epoch, and the make_env
surface."""
import copy

import numpy as np
import pytest

from golden_util import load_map

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]


def _scripted(n, seed0=500, kinds=None):
    from carlabev_env_b200.scenes import build_scripted_scene

    cls = load_map()
    if kinds is None:
        kinds = [("lead_brake", 1 + i % 3) if i % 2 == 0 else ("jaywalk", 1 + i % 4) for i in range(n)]
    return [build_scripted_scene(k, seed0 + i, level=lv, cls_map=cls) for i, (k, lv) in enumerate(kinds)]


def _rdm(size, n=16):
    from carlabev_env_b200.scenes import build_pool

    pad = {64: 91, 128: 182, 256: 363}[size]
    return [s for s in build_pool([dict(scene="rdm", num_vehicles=12, route_dist_range=(30, 100), scene_seed=i)
                                   for i in range(n)], pad=pad, size=size, skip_invalid=True) if s is not None]


def _engine(scenes, n, size=128, **kw):
    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    args = dict(mask_mode="6-class", frame_stack=4, ring_slots=7, action_mode=E.ACTION_CONTINUOUS,
                autoreset=E.AUTORESET_NEXT_STEP, max_actors=4, seed=3, size=size)
    args.update(kw)
    if args.get("obs_mode") == E.OBS_RGB:
        args["ring_slots"] = None
    eng = E.Engine(n, **args)
    eng.upload_map(load_map(size))
    eng.upload_pool(pack_pool(scenes))
    return eng


def _actions(rng, n):
    import torch

    a = np.stack([rng.uniform(0, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 1, n)], axis=1).astype(np.float32)
    return torch.from_numpy(a).cuda()


def _outputs(eng, fusion=None):
    import torch

    done = (eng.terminated | eng.truncated).bool()
    ep = eng.episode.clone()
    ep[~done] = 0  # rows of terminal envs only
    obs = eng.obs() if fusion is None else eng.fuse(fusion)
    return {"obs": obs.clone(), "reward": eng.reward.clone(), "terminated": eng.terminated.clone(),
            "truncated": eng.truncated.clone(), "cause": eng.cause.clone(), "hero": eng.hero.clone(),
            "episode": ep, "done": done.to(torch.uint8)}


def _same(a, b, what, envs=None):
    import torch

    for k in a:
        x, y = a[k], b[k]
        if envs is not None:
            x, y = x[envs], y[envs]
        if k == "episode":
            assert np.array_equal(x.cpu().numpy(), y.cpu().numpy(), equal_nan=True), (what, k)
        else:
            assert torch.equal(x, y), (what, k, int((x != y).sum()))


def _step_to_mirror_zone(eng, rng, kmin):
    """Step at least kmin times and until the head is in the mirror zone (head >= L - F + 1)."""
    t = 0
    while t < kmin or (eng.F > 1 and eng.head < eng.L - eng.F + 1):
        eng.step(_actions(rng, eng.N))
        t += 1
    assert eng.F == 1 or eng.head >= eng.L - eng.F + 1
    return t


ROUND_TRIP = ["float32", "uint8", "gray", "rgb", "any64", "any256", "obs84", "vehicle_temporal", "vehicle_weighted",
              "traj0", "traj1024", "traj8", "jaywalk3", "disabled_masked_reset"]


@pytest.mark.parametrize("case", ROUND_TRIP)
def test_round_trip_is_bit_exact(case):
    import torch

    from carlabev_env_b200 import engine as E

    n, kw, fusion, kmin, size = 32, {}, None, 10, 128
    scenes = None
    if case == "uint8":
        kw["mask_dtype"] = "uint8"
    elif case == "gray":
        kw["obs_mode"] = E.OBS_GRAY
    elif case == "rgb":
        kw["obs_mode"] = E.OBS_RGB
    elif case in ("any64", "any256"):
        size = 64 if case == "any64" else 256
        scenes, kw["max_actors"] = _rdm(size), 16
    elif case == "obs84":
        kw["obs_size"] = (84, 84)
    elif case.startswith("vehicle_"):
        fusion = case
    elif case.startswith("traj"):
        kw["trajectory_steps"] = int(case[4:])
        kmin = 1 if case == "traj8" else kmin  # the table hand-over (step 8 of an episode) comes after the restore
    elif case == "jaywalk3":
        scenes = _scripted(16, kinds=[("jaywalk", 3 + i % 2) for i in range(16)])  # StopReturn walkers
    elif case == "disabled_masked_reset":
        kw["autoreset"] = E.AUTORESET_DISABLED
    if scenes is None:
        scenes = _scripted(16)
    eng = _engine(scenes, n, size=size, **kw)
    ids = torch.arange(n, dtype=torch.int32) % len(scenes)
    eng.reset(ids)
    rng = np.random.default_rng(7)
    _step_to_mirror_zone(eng, rng, kmin)
    at_snap = _outputs(eng, fusion)["obs"]
    snap = eng.snapshot()
    assert snap.data.shape == (n, eng.snapshot_row_bytes) and snap.row_bytes % 16 == 0
    M = max(eng.L, 7) + 25
    acts = [_actions(rng, n) for _ in range(M)]
    mask = torch.arange(n) % 3 == 0
    ids2 = (ids + 5) % len(scenes)

    def run():
        rec = []
        for t, a in enumerate(acts):
            eng.step(a)
            rec.append(_outputs(eng, fusion))
            if case == "disabled_masked_reset" and t == 5:
                eng.reset(ids2, mask)
                rec.append({"reset_obs": eng.obs().clone()})
        return rec

    first = run()
    obs = eng.restore(snap)
    if fusion is not None:
        obs = eng.fuse(fusion)
    assert torch.equal(obs, at_snap), "restore() does not return the snapshot's observation"
    second = run()
    assert len(first) == len(second)
    for t, (a, b) in enumerate(zip(first, second)):
        _same(a, b, (case, t))
    eng.close()


def test_restoring_a_subset_leaves_the_others_alone():
    """A third of the envs are restored; every other env stays bit-identical to a twin engine that never restored."""
    import torch

    scenes = _scripted(16)
    n = 48
    engs = [_engine(scenes, n) for _ in range(2)]
    ids = torch.arange(n, dtype=torch.int32) % len(scenes)
    for e in engs:
        e.reset(ids)
    rng = np.random.default_rng(3)
    for _ in range(12):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
    snap = engs[0].snapshot()
    at_snap = engs[0].obs().clone()
    for _ in range(9):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
    sub = np.arange(0, n, 3)
    others = torch.from_numpy(np.setdiff1d(np.arange(n), sub)).cuda()
    obs = engs[0].restore(snap, env_ids=sub, rows=sub)
    sub_t = torch.from_numpy(sub).cuda()
    assert torch.equal(obs[sub_t], at_snap[sub_t])
    _same({"obs": engs[0].obs()}, {"obs": engs[1].obs()}, "after restore", others)
    for t in range(20):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
        _same(_outputs(engs[0]), _outputs(engs[1]), t, others)
    for e in engs:
        e.close()


def test_clone_with_identical_actions_follows_the_source():
    """One row restored into every env (rows on the device); with the same action in every env, all of them equal the
    source's recorded continuation up to and including its first terminal step."""
    import torch

    scenes = _scripted(16)
    n = 64
    eng = _engine(scenes, n)
    eng.reset(torch.arange(n, dtype=torch.int32) % len(scenes))
    rng = np.random.default_rng(11)
    _step_to_mirror_zone(eng, rng, 6)
    snap = eng.snapshot()
    hdr = snap.header().cpu().numpy()
    s = int(np.flatnonzero(hdr[:, 2] == 0)[0])  # a source that is not about to auto-reset
    at_snap = eng.obs()[s].clone()
    acts = []
    for _ in range(40):
        a1 = _actions(rng, 1)
        acts.append(a1.expand(n, 3).contiguous())
    rec = []
    for a in acts:
        eng.step(a)
        rec.append({k: v[s].clone() for k, v in _outputs(eng).items()})
        if bool(rec[-1]["done"]):
            break
    rows = torch.full((n,), s, dtype=torch.int32, device=eng.device)
    obs = eng.restore(snap, rows=rows)
    assert torch.equal(obs, at_snap.expand_as(obs))
    for t, r in enumerate(rec):
        eng.step(acts[t])
        out = _outputs(eng)
        for k, v in r.items():
            assert torch.equal(out[k], v.unsqueeze(0).expand_as(out[k])), (t, k)
    eng.close()


def test_clones_with_different_actions_match_the_oracle():
    """A source env tracked by an OracleEnv up to the snapshot, then cloned into 32 envs that each take their own
    actions: 16 of them against deep copies of that oracle (observations and flags exact, poses and rewards to 1e-9)."""
    import torch

    from carlabev_env_b200 import engine as E
    from oracle.env import OracleEnv

    scenes = _scripted(16)
    n = 32
    eng = _engine(scenes, n, autoreset=E.AUTORESET_DISABLED)
    ids = np.arange(n) % len(scenes)
    eng.reset(torch.from_numpy(ids.astype(np.int32)))
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
    snap = eng.snapshot(env_ids=[s])
    obs = eng.restore(snap, rows=np.zeros(n, dtype=np.int64))
    sample = list(range(0, n, 2))
    clones = {j: copy.deepcopy(oracle) for j in sample}
    ref0 = oracle.sim  # the deep copies must not share simulator state with the original
    assert all(c.sim is not ref0 for c in clones.values())
    obs_h = obs.cpu().numpy()
    live = {j: True for j in sample}
    for t in range(30):
        a = _actions(rng, n)
        eng.step(a)
        a_h = a.cpu().numpy()
        obs_h, rew = eng.obs().cpu().numpy(), eng.reward.cpu().numpy()
        term = eng.terminated.cpu().numpy().astype(bool)
        hero = eng.hero.cpu().numpy()
        for j in sample:
            if not live[j]:
                continue
            o, r, te, _, _ = clones[j].step(a_h[j])
            ego = clones[j].sim.ego
            assert np.array_equal(obs_h[j], o), (t, j, "observation")
            assert te == term[j], (t, j, "terminated")
            assert abs(r - rew[j]) < 1e-9, (t, j, "reward", r, rew[j])
            assert np.allclose(hero[j, :4], [ego.x, ego.y, ego.yaw, ego.v], rtol=1e-9, atol=1e-9), (t, j, "pose")
            live[j] = not te
    eng.close()


def test_restored_host_state_equals_the_source():
    """get_state() after restoring a permutation of the rows equals the state each row was taken from."""
    import torch

    scenes = _scripted(16, kinds=[("jaywalk", 3 + i % 2) if i % 2 else ("lead_brake", 3) for i in range(16)])
    n = 24
    eng = _engine(scenes, n, trajectory_steps=0)
    eng.reset(torch.arange(n, dtype=torch.int32) % len(scenes))
    rng = np.random.default_rng(5)
    _step_to_mirror_zone(eng, rng, 15)
    ego0, act0 = eng.get_state()
    snap = eng.snapshot()
    for _ in range(11):
        eng.step(_actions(rng, n))
    perm = np.random.default_rng(0).permutation(n)
    eng.restore(snap, rows=perm)
    ego1, act1 = eng.get_state()
    assert np.array_equal(ego1, ego0[perm], equal_nan=True)
    assert np.array_equal(act1, act0[perm], equal_nan=True)
    eng.close()


def _two_walkers(a, b):
    """Scene a with the StopReturn pedestrian of scene b added: two retreat-route slots."""
    from carlabev_env_b200.pool import _PER_ACTOR

    s = dict(a)
    for k, _, _ in _PER_ACTOR:
        s[k] = np.concatenate([np.asarray(a[k]), np.asarray(b[k])])
    for off, keys in (("act_route_off", ("act_cx", "act_cy", "act_cyaw")), ("act_raw_off", ("act_raw_x", "act_raw_y"))):
        oa, ob = np.asarray(a[off]), np.asarray(b[off])
        s[off] = np.concatenate([oa, oa[-1] + ob[1:]]).astype(np.int32)
        for k in keys:
            s[k] = np.concatenate([np.asarray(a[k]), np.asarray(b[k])])
    return s


def test_pool_growth_keeps_rows_and_a_new_pool_voids_them():
    import torch

    from carlabev_env_b200 import engine as E
    from carlabev_env_b200.pool import pack_pool

    scenes = _scripted(12, kinds=[("jaywalk", 3)] * 12)
    n = 24
    eng = _engine(scenes, n, autoreset=E.AUTORESET_DISABLED, trajectory_steps=0)
    ids = torch.arange(n, dtype=torch.int32) % len(scenes)
    eng.reset(ids)
    rng = np.random.default_rng(9)
    _step_to_mirror_zone(eng, rng, 12)
    snap = eng.snapshot()
    acts = [_actions(rng, n) for _ in range(14)]
    first = []
    for a in acts:
        eng.step(a)
        first.append(_outputs(eng))
    # append scenes with two StopReturn walkers: the per-env retreat buffer widens from 1 to 2 slots
    grown = scenes + [_two_walkers(scenes[i], scenes[i + 1]) for i in range(0, 4, 2)]
    eng.upload_pool(pack_pool(grown))
    assert eng.snapshot_row_bytes > snap.row_bytes and snap.info.retreat_slots == 1
    eng.restore(snap)
    for t, a in enumerate(acts):
        eng.step(a)
        _same(first[t], _outputs(eng), ("grown pool", t))
    # rows taken at the wider R restore as well
    snap2 = eng.snapshot()
    assert snap2.info.retreat_slots == 2
    eng.restore(snap2)
    # an unrelated pool ends the epoch: before the next reset and after it, restore fails with the state code
    eng.invalidate()
    with pytest.raises(E.CbevError, match="cbev error 3"):
        eng.restore(snap2)
    eng.upload_pool(pack_pool(scenes))
    eng.reset(ids)
    with pytest.raises(E.CbevError, match="cbev error 3.*epoch"):
        eng.restore(snap2)
    eng.close()


def test_snapshot_argument_checks():
    import ctypes as C

    import torch

    from carlabev_env_b200 import engine as E

    scenes = _scripted(4)
    n = 8
    eng = _engine(scenes, n)
    lib = eng.lib
    rb = eng.snapshot_row_bytes
    buf = torch.zeros(n * rb + 16, dtype=torch.uint8, device=eng.device)
    info = E.CbevSnapshotInfo()
    s = eng._stream()
    # before the first reset
    assert lib.cbev_snapshot(eng.handle, None, n, buf.data_ptr(), n * rb, C.byref(info), s) == 3
    assert b"first reset" in lib.cbev_last_error()
    eng.reset(torch.arange(n, dtype=torch.int32) % len(scenes))
    for cnt, dst, nbytes, msg in ((0, 0, n * rb, b"1..8"), (n + 1, 0, (n + 1) * rb, b"1..8"),
                                  (n, 0, n * rb - 16, b"need"), (n, 8, n * rb, b"16-byte")):
        assert lib.cbev_snapshot(eng.handle, None, cnt, buf.data_ptr() + dst, nbytes, C.byref(info), s) == 1, msg
        assert msg in lib.cbev_last_error(), lib.cbev_last_error()
    assert lib.cbev_snapshot(eng.handle, None, n, buf.data_ptr(), n * rb, None, s) == 1
    snap = eng.snapshot()
    # identity rows need as many rows as targets
    part = eng.snapshot(env_ids=[1, 2])
    with pytest.raises(E.CbevError, match="identity rows"):
        eng.restore(part, env_ids=[0, 1, 2])
    with pytest.raises(ValueError, match="more than once"):
        eng.restore(snap, env_ids=[0, 0], rows=[1, 2])
    with pytest.raises(ValueError, match="rows"):
        eng.restore(part, rows=[0, 2])
    with pytest.raises(ValueError, match="same length"):
        eng.restore(snap, env_ids=[0, 1], rows=[1])
    with pytest.raises(ValueError, match="out="):
        eng.snapshot(out=part)
    # out= reuses the storage of an earlier snapshot
    again = eng.snapshot(env_ids=[3], out=part)
    assert again is part and part.n_rows == 1 and part.data.data_ptr() == part._buf.data_ptr()
    # a second engine does not take these rows
    other = _engine(scenes, n)
    other.reset(torch.arange(n, dtype=torch.int32) % len(scenes))
    with pytest.raises(E.CbevError, match="another engine"):
        other.restore(snap)
    other.close()
    eng.close()


def test_move_order_does_not_change_results():
    """The k_move order is not part of a snapshot: it is a permutation, and debug flag 128 (identity order) gives the
    same results, so a restore that leaves it as it is replays exactly."""
    import torch

    scenes = _scripted(16)
    n = 64
    engs = [_engine(scenes, n) for _ in range(2)]
    engs[1].set_debug_flags(128)
    ids = torch.arange(n, dtype=torch.int32) % len(scenes)
    for e in engs:
        e.reset(ids)
    rng = np.random.default_rng(13)
    done = 0
    for t in range(60):
        a = _actions(rng, n)
        for e in engs:
            e.step(a)
        _same(_outputs(engs[0]), _outputs(engs[1]), t)
        done += int(engs[0].terminated.sum())
    assert done > 0
    for e in engs:
        e.close()


def _env(n, autoreset, scenes):
    from carlabev_env_b200 import EnvConfig, RunConfig, make_env

    cfg = RunConfig(env=EnvConfig(action_mode="continuous"), num_envs=n)
    return make_env(cfg, scenes=scenes, autoreset=autoreset, ring_slots=8)


def test_make_env_round_trip_and_host_bookkeeping():
    scenes = _scripted(8)
    n = 8
    envs = _env(n, "next_step", scenes)
    envs.reset(options={"scene_ids": np.arange(n)})
    rng = np.random.default_rng(9)

    def act():
        return np.stack([rng.uniform(0.5, 1, n), rng.uniform(-1, 1, n), rng.uniform(0, 0.1, n)], axis=1).astype(np.float32)

    def step(a):  # observation, reward and flags are views of buffers the next step rewrites
        obs, rew, term, trunc, infos = envs.step(a)
        return obs.clone(), rew.clone(), term.clone(), trunc.clone(), infos

    for _ in range(5):
        envs.step(act())
    snap = envs.snapshot()
    at_snap = envs.engine.obs().clone()
    acts, first = [], []
    for t in range(400):
        acts.append(act())
        first.append(step(acts[-1]))
        if "episode_info" in first[-1][4] and len(acts) < 400:
            acts.append(act())
            first.append(step(acts[-1]))  # the step that consumes the device auto-reset
            break
    assert "episode_info" in first[-2][4], "no episode finished"
    import torch

    assert torch.equal(envs.restore(snap), at_snap)
    for t, a in enumerate(acts):
        res = envs.step(a)
        for k in range(4):
            assert torch.equal(res[k], first[t][k]), (t, k)
        assert ("episode_info" in res[4]) == ("episode_info" in first[t][4]), t
        if "episode_info" in res[4]:
            for key, col in first[t][4]["episode_info"].items():
                assert np.array_equal(res[4]["episode_info"][key], col), (t, key)
            assert np.array_equal(res[4]["episode"]["r"], first[t][4]["episode"]["r"])
    envs.recorder = object()  # capture_video on
    with pytest.raises(ValueError, match="capture_video"):
        envs.restore(snap)
    envs.recorder = None
    envs.close()
    # autoreset disabled: a restored terminal row needs a reset again
    envs = _env(n, "disabled", scenes)
    envs.reset(options={"scene_ids": np.arange(n)})
    for _ in range(400):
        envs.step(act())
        if envs._needs_reset.any():
            break
    done = envs._needs_reset.copy()
    assert done.any()
    snap = envs.snapshot()
    envs.reset(options={"scene_ids": (np.arange(n) + 3) % n, "reset_mask": done})
    assert not envs._needs_reset.any()
    envs.restore(snap, env_ids=np.flatnonzero(done), rows=np.flatnonzero(done))
    assert np.array_equal(envs._needs_reset, done)
    assert np.array_equal(envs._scene_of_env, np.arange(n))
    with pytest.raises(AssertionError, match="call reset"):
        envs.step(act())
    envs.close()
